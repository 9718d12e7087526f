// builtin_bfgs_batch.cu -- the batched BFGS launchers of the built-in scalar objectives that builtin_functors.cu lists: every
// instantiation of bfgs_batch_kernel for them (4 thread configurations each; the derivative modes are runtime flags). Functor code is
// compiled with -fmad=false.
#include "common.cuh"
#include "pnol/device/functor_kernels.cuh"

namespace pnol {

template <class F> pnol_bfgs_batch_launcher bfgs_batch_launcher() { return dev::ScalarTable<F>::bfgs_batch_; }

template pnol_bfgs_batch_launcher bfgs_batch_launcher<RosenbrockFunctor>();
template pnol_bfgs_batch_launcher bfgs_batch_launcher<PowerFunctor>();
template pnol_bfgs_batch_launcher bfgs_batch_launcher<BoothFunctor>();
template pnol_bfgs_batch_launcher bfgs_batch_launcher<GoldsteinFunctor>();
template pnol_bfgs_batch_launcher bfgs_batch_launcher<RastriginFunctor>();
template pnol_bfgs_batch_launcher bfgs_batch_launcher<ExpCurveSingleFunctor>();

} // namespace pnol
