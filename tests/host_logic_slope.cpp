// host_logic_slope.cpp -- TEST INFRASTRUCTURE, never shipped. The CPU stand-in of the C-ABI extended by the analytic gradient and
// Hessian (tests/host_logic_hessian.cpp, included here as it is) and by the analytic line-search slope: pnol_alpha_pool_analytic answered
// by the built-in scalar functors' host eval() and partial() (include/pnol/functors.hpp, the definitions the kernels compile), with the
// point assembly, the sequential sum and the sentinel of alpha_slope_kernel / alpha_slope_finish_kernel. tests/host_logic_slope_lib.py
// builds it; with it the BFGS controllers run Runtime::setAnalyticSlope(true) on the CPU, and the GPU iterates are compared with theirs
// (tests/test_gpu_analytic_slope.py).
#include "host_logic_hessian.cpp"

namespace {
// phi = f(xa), dphi = sum_r p[r] * df/dx_{pos[r]}(xa) summed sequentially in r order (pos NULL: r; pos[r] < 0: 0 * p[r])
template <class F> void host_slope(const pnol_functor_params & P, const double * xa, int nfull, const int * pos, const double * p, int n,
                                   double * phi, double * dphi)
{
	const pnol::PtrAcc acc{xa};
	*phi = F::eval(P, acc, nfull);
	double s = 0.0;
	for (int r = 0; r < n; r++) {
		const int j = pos ? pos[r] : r;
		const double g = j >= 0 ? F::partial(P, acc, nfull, j) : 0.0;
		s = s + g * p[r];
	}
	*dphi = s;
}
} // namespace

extern "C" int pnol_alpha_pool_analytic(pnol_ctx * ctx, const pnol_functor * f, const double * x, const double * p, int n,
                                        const double * alpha, int npool, const unsigned char * eval_ind, const double * const_x,
                                        const unsigned char * const_ind, int nfull, double * phi, double * dphi, int * bad_out)
{
	if (!const_ind) nfull = n;
	// the full point and direction as the product assembles them (p = 0 on constants, free variables beyond the reduced entries 0)
	std::vector<double> xf(nfull), pf(nfull), xa(nfull);
	std::vector<int> pos(n, -1);
	int k = 0;
	for (int j = 0; j < nfull; j++) {
		if (const_ind && const_ind[j]) { xf[j] = const_x[j]; pf[j] = 0.0; continue; }
		xf[j] = k < n ? x[k] : 0.0;
		pf[j] = k < n ? p[k] : 0.0;
		if (k < n) pos[k] = j;
		k++;
	}
	const pnol_functor_params P = host_params(f);
	int bad = 0;
	for (int q = 0; q < npool; q++) {
		if (eval_ind && !eval_ind[q]) continue;
		for (int j = 0; j < nfull; j++) xa[j] = const_ind && const_ind[j] ? xf[j] : xf[j] + alpha[q] * pf[j];
		double ph, ds;
		switch (f->d.kind) {
			case PNOL_F_ROSENBROCK: host_slope<pnol::RosenbrockFunctor>(P, xa.data(), nfull, pos.data(), p, n, &ph, &ds); break;
			case PNOL_F_POWER: host_slope<pnol::PowerFunctor>(P, xa.data(), nfull, pos.data(), p, n, &ph, &ds); break;
			case PNOL_F_BOOTH: host_slope<pnol::BoothFunctor>(P, xa.data(), nfull, pos.data(), p, n, &ph, &ds); break;
			case PNOL_F_GOLDSTEIN: host_slope<pnol::GoldsteinFunctor>(P, xa.data(), nfull, pos.data(), p, n, &ph, &ds); break;
			case PNOL_F_RASTRIGIN: host_slope<pnol::RastriginFunctor>(P, xa.data(), nfull, pos.data(), p, n, &ph, &ds); break;
			case PNOL_F_EXPCURVE_SINGLE: host_slope<pnol::ExpCurveSingleFunctor>(P, xa.data(), nfull, pos.data(), p, n, &ph, &ds); break;
			default: return unavailable(ctx, "pnol_alpha_pool_analytic for this functor kind");
		}
		if (ph != ph || std::isinf(ph)) { ph = 1e10; bad++; }
		phi[q] = ph;
		dphi[q] = ds;
	}
	if (bad_out) *bad_out = bad;
	return PNOL_OK;
}
