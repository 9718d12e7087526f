// builtin_residual_functors.cu -- the records of the built-in residual models that builtin_functors.cu lists: every instantiation of the
// functor kernel templates for them. Functor code is compiled with -fmad=false.
#include "common.cuh"
#include "pnol/device/functor_kernels.cuh"

namespace pnol {

template <class R> KindTable residual_kind(int n_columns)
{
	static_assert(has_jacobian<R>::value, "a built-in residual model has an analytic Jacobian");
	KindTable k = {};
	k.vt = dev::ResidualTable<R>::make(n_columns);
	k.lm_batch = dev::ResidualTable<R>::lm_batch_;
	return k;
}

template KindTable residual_kind<ExpCurveFunctor>(int);
template KindTable residual_kind<CubicFunctor>(int);
template KindTable residual_kind<LorentzSumFunctor>(int);

} // namespace pnol
