// builtin_simplex_batch.cu -- the batched simplex launchers of the built-in scalar objectives that builtin_functors.cu lists: every
// instantiation of simplex_batch_kernel for them (4 group sizes each). Functor code is compiled with -fmad=false.
#include "common.cuh"
#include "pnol/device/functor_kernels.cuh"

namespace pnol {

template <class F> pnol_simplex_batch_launcher simplex_batch_launcher() { return dev::ScalarTable<F>::simplex_batch_; }

template pnol_simplex_batch_launcher simplex_batch_launcher<RosenbrockFunctor>();
template pnol_simplex_batch_launcher simplex_batch_launcher<PowerFunctor>();
template pnol_simplex_batch_launcher simplex_batch_launcher<BoothFunctor>();
template pnol_simplex_batch_launcher simplex_batch_launcher<GoldsteinFunctor>();
template pnol_simplex_batch_launcher simplex_batch_launcher<RastriginFunctor>();
template pnol_simplex_batch_launcher simplex_batch_launcher<ExpCurveSingleFunctor>();

} // namespace pnol
