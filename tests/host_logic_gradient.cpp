// host_logic_gradient.cpp -- TEST INFRASTRUCTURE, never shipped. The CPU stand-in of the C-ABI that the host-logic tests link the
// unmodified host sources against (oracle/host_logic_device.cpp, included here as it is) extended by the analytic gradient:
// pnol_gradient[_recur] answered by the built-in scalar functors' host partial() and eval() (include/pnol/functors.hpp, the definitions
// the kernels compile). tests/host_logic_gradient_lib.py builds it; with it the BFGS controllers run Runtime::setAnalyticGradient(true)
// on the CPU, and the GPU iterates are compared with theirs (tests/test_gpu_analytic_gradient.py). User kinds are not answered.
#include "../oracle/host_logic_device.cpp"
#include "../include/pnol/functors.hpp"

namespace {
pnol_functor_params host_params(const pnol_functor * f)
{
	pnol_functor_params P;
	std::memset(&P, 0, sizeof P);
	std::memcpy(P.scalars, f->d.scalars, sizeof P.scalars);
	std::memcpy(P.ints, f->d.ints, sizeof P.ints);
	for (int c = 0; c < f->d.n_columns && c < PNOL_MAX_COLUMNS; c++) P.col[c] = f->d.columns[c];
	P.m = f->d.m;
	return P;
}
// g[i] = df/dx_{pos[i]} (pos NULL: i; pos[i] < 0: 0), as gradient_kernel computes it; f0 = f(x)
template <class F> void host_gradient(const pnol_functor_params & P, const double * x, int n, const int * pos, int nvar, double * g, double * f0)
{
	const pnol::PtrAcc acc{x};
	for (int i = 0; i < nvar; i++) {
		const int j = pos ? pos[i] : i;
		g[i] = j >= 0 ? F::partial(P, acc, n, j) : 0.0;
	}
	if (f0) *f0 = F::eval(P, acc, n);
}
int gradient_at(pnol_ctx * ctx, const pnol_functor * f, const double * x, int n, const int * pos, int nvar, double * g, double * f0)
{
	const pnol_functor_params P = host_params(f);
	switch (f->d.kind) {
		case PNOL_F_ROSENBROCK: host_gradient<pnol::RosenbrockFunctor>(P, x, n, pos, nvar, g, f0); return PNOL_OK;
		case PNOL_F_POWER: host_gradient<pnol::PowerFunctor>(P, x, n, pos, nvar, g, f0); return PNOL_OK;
		case PNOL_F_BOOTH: host_gradient<pnol::BoothFunctor>(P, x, n, pos, nvar, g, f0); return PNOL_OK;
		case PNOL_F_GOLDSTEIN: host_gradient<pnol::GoldsteinFunctor>(P, x, n, pos, nvar, g, f0); return PNOL_OK;
		case PNOL_F_RASTRIGIN: host_gradient<pnol::RastriginFunctor>(P, x, n, pos, nvar, g, f0); return PNOL_OK;
		case PNOL_F_EXPCURVE_SINGLE: host_gradient<pnol::ExpCurveSingleFunctor>(P, x, n, pos, nvar, g, f0); return PNOL_OK;
		default: return unavailable(ctx, "pnol_gradient for this functor kind");
	}
}
} // namespace

extern "C" {

int pnol_gradient(pnol_ctx * ctx, const pnol_functor * f, const double * x, int n, double * g_out, double * f0_out)
{
	return gradient_at(ctx, f, x, n, nullptr, n, g_out, f0_out);
}

// the full point and the slot of every reduced entry, as the product assembles them (objEvalRecur's scatter,
// Source/PNOL_Objective.cpp:303-323; free variables beyond the reduced entries are 0); -1: no slot
int pnol_gradient_recur(pnol_ctx * ctx, const pnol_functor * f, const double * xr, int nr, const double * const_x, const unsigned char * const_ind,
                        int nfull, double * g_out, double * f0_out)
{
	std::vector<double> xf(nfull);
	std::vector<int> pos(nr, -1);
	int k = 0;
	for (int j = 0; j < nfull; j++) {
		if (const_ind[j]) { xf[j] = const_x[j]; continue; }
		xf[j] = k < nr ? xr[k] : 0.0;
		if (k < nr) pos[k] = j;
		k++;
	}
	return gradient_at(ctx, f, xf.data(), nfull, pos.data(), nr, g_out, f0_out);
}

} // extern "C"
