// builtin_functors.cu -- the records of the nine built-in objectives (kind_table), filled from the launch tables a user kind registers
// as well (include/pnol/device/functor_kernels.cuh: ScalarTable / ResidualTable). The only place in csrc/ that lists the built-in kinds.
// This file holds every instantiation of the functor kernel templates for the built-in scalar objectives, builtin_residual_functors.cu
// those for the residual models. Functor code is compiled with -fmad=false.
#include "common.cuh"
#include "pnol/device/functor_kernels.cuh"

namespace pnol {

// builtin_bfgs_batch.cu: the batched BFGS launchers of the scalar objectives (bfgs_batch_kernel, 6 objectives x 4 configurations) take
// long to compile; in a file of their own they build in parallel with the other kernels
template <class F> pnol_bfgs_batch_launcher bfgs_batch_launcher();
// builtin_simplex_batch.cu: the batched simplex launchers (simplex_batch_kernel, 6 objectives x 4 group sizes), for the same reason
template <class F> pnol_simplex_batch_launcher simplex_batch_launcher();

namespace {

template <class F> KindTable scalar_kind(int n_columns)
{
	static_assert(has_partial<F>::value && has_partial2<F>::value, "a built-in scalar objective has an analytic gradient and Hessian");
	KindTable k = {};
	k.vt = dev::ScalarTable<F>::make(n_columns);
	k.gradient = dev::ScalarTable<F>::gradient_;
	k.hessian = dev::ScalarTable<F>::hessian_;
	k.slope = dev::ScalarTable<F>::alpha_slope_;
	k.bfgs_batch = bfgs_batch_launcher<F>();
	k.simplex_batch = simplex_batch_launcher<F>();
	return k;
}

struct BuiltinKind {
	int kind;
	KindTable table;
};

} // namespace

// builtin_residual_functors.cu: the residual models' kernels (lm_batch_kernel above all) take the longest to compile; in a file of their
// own they build in parallel with the scalar ones
template <class R> KindTable residual_kind(int n_columns);

const KindTable * builtin_kind_table(int kind)
{
	// built at the first lookup, which may come from another module's static initialiser; read-only after that, so no lock
	static const BuiltinKind kinds[] = {
		{PNOL_F_ROSENBROCK, scalar_kind<RosenbrockFunctor>(0)},
		{PNOL_F_POWER, scalar_kind<PowerFunctor>(0)},
		{PNOL_F_BOOTH, scalar_kind<BoothFunctor>(0)},
		{PNOL_F_GOLDSTEIN, scalar_kind<GoldsteinFunctor>(0)},
		{PNOL_F_RASTRIGIN, scalar_kind<RastriginFunctor>(0)},
		{PNOL_F_EXPCURVE_SINGLE, scalar_kind<ExpCurveSingleFunctor>(2)},
		{PNOL_F_EXPCURVE, residual_kind<ExpCurveFunctor>(2)},
		{PNOL_F_CUBIC, residual_kind<CubicFunctor>(3)},
		{PNOL_F_LORENTZ_SUM, residual_kind<LorentzSumFunctor>(2)},
	};
	for (const BuiltinKind & b : kinds)
		if (b.kind == kind) return &b.table;
	return nullptr;
}

} // namespace pnol
