// host_logic_hessian.cpp -- TEST INFRASTRUCTURE, never shipped. The CPU stand-in of the C-ABI extended by the analytic gradient
// (tests/host_logic_gradient.cpp, included here as it is) and by the analytic Hessian: pnol_hessian answered by the built-in scalar
// functors' host partial2() (include/pnol/functors.hpp, the definitions the kernels compile), upper triangle computed and mirrored as
// hessian_kernel does. tests/host_logic_hessian_lib.py builds it; with it the BFGS controllers run initHessFD with
// Runtime::setAnalyticHessian(true) on the CPU, and the GPU iterates are compared with theirs (tests/test_gpu_analytic_hessian.py).
#include "host_logic_gradient.cpp"

namespace {
template <class F> void host_hessian(const pnol_functor_params & P, const double * x, int n, double * H)
{
	const pnol::PtrAcc acc{x};
	for (int i = 0; i < n; i++)
		for (int j = i; j < n; j++) H[(size_t) i * n + j] = H[(size_t) j * n + i] = F::partial2(P, acc, n, i, j);
}
} // namespace

extern "C" int pnol_hessian(pnol_ctx * ctx, const pnol_functor * f, const double * x, int n, double * H_out)
{
	const pnol_functor_params P = host_params(f);
	switch (f->d.kind) {
		case PNOL_F_ROSENBROCK: host_hessian<pnol::RosenbrockFunctor>(P, x, n, H_out); return PNOL_OK;
		case PNOL_F_POWER: host_hessian<pnol::PowerFunctor>(P, x, n, H_out); return PNOL_OK;
		case PNOL_F_BOOTH: host_hessian<pnol::BoothFunctor>(P, x, n, H_out); return PNOL_OK;
		case PNOL_F_GOLDSTEIN: host_hessian<pnol::GoldsteinFunctor>(P, x, n, H_out); return PNOL_OK;
		case PNOL_F_RASTRIGIN: host_hessian<pnol::RastriginFunctor>(P, x, n, H_out); return PNOL_OK;
		case PNOL_F_EXPCURVE_SINGLE: host_hessian<pnol::ExpCurveSingleFunctor>(P, x, n, H_out); return PNOL_OK;
		default: return unavailable(ctx, "pnol_hessian for this functor kind");
	}
}
