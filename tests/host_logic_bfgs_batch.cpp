// host_logic_bfgs_batch.cpp -- TEST INFRASTRUCTURE, never shipped. The CPU stand-in of the C-ABI extended by the analytic derivatives
// (tests/host_logic_slope.cpp, included here as it is) and by pnol_bfgs_batch: every start is oracle_bfgs, a C++ restatement of
// BFGS::findMin (Source/BFGS_with_linesearch.cpp:12-385) over the built-in scalar functors' host eval(), partial() and partial2()
// (include/pnol/functors.hpp, the definitions the kernels compile) and the oracle's sequential dense helpers (oracle/pnol_oracle.cpp:
// oracle_matvec_neg, oracle_update_hinv, oracle_lu_solve). tests/host_logic_bfgs_batch_lib.py builds it; tests/test_bfgs_batch_cpu.py
// checks it bit for bit against the unmodified host BFGS controller on the same stand-in, and the GPU tests use it as the fast oracle.
#include "host_logic_slope.cpp"

#include <cmath>

namespace {

struct BfgsOut { double f0, fopt; int iters, stop; };

template <class F> struct Obj {
	const pnol_functor_params & P;
	int n;
	double f(const std::vector<double> & x) const { const pnol::PtrAcc a{x.data()}; return F::eval(P, a, n); }
};

double sgn(double x) { if (x > 0) return 1.0; if (x < 0) return -1.0; return 0.0; }

double cubic_interp_min(double alo, double ahi, double plo, double phh, double dlo, double dhh)
{
	double d1 = dlo + dhh - 3 * (plo - phh) / (alo - ahi);
	double d2 = sgn(ahi - alo) * std::sqrt(d1 * d1 - dlo * dhh);
	double a = ahi - (ahi - alo) * (dhh + d2 - d1) / (dhh - dlo + 2 * d2);
	if (alo < ahi) { if (a < alo) a = (ahi + alo) / 2; }
	else { if (a < ahi) a = (ahi + alo) / 2; }
	return a;
}

template <class F>
BfgsOut oracle_bfgs(const pnol_functor_params & P, double * Xb, int n, const pnol_bfgs_params & prm, int flags)
{
	const Obj<F> o{P, n};
	const bool agrad = flags & PNOL_BFGS_ANALYTIC_GRADIENT, aslope = flags & PNOL_BFGS_ANALYTIC_SLOPE;
	const bool ahess = flags & PNOL_BFGS_ANALYTIC_HESSIAN;
	std::vector<double> X(Xb, Xb + n), Xprev(n), dFdX(n), dFdXp(n), p(n), s(n), g(n), D((size_t) n * n), xt(n);
	auto gradient = [&]() {
		if (agrad) { const pnol::PtrAcc a{X.data()}; for (int i = 0; i < n; i++) dFdX[i] = F::partial(P, a, n, i); return; }
		const double f = o.f(X);                                             // oracle_fd_gradient
		for (int i = 0; i < n; i++) { xt = X; xt[i] = xt[i] + prm.dx_grad; dFdX[i] = (o.f(xt) - f) / prm.dx_grad; }
	};
	auto phi_and_slope = [&](double a, double & phi, double & dphi) {
		for (int i = 0; i < n; i++) xt[i] = X[i] + a * p[i];                 // lineSearchObj
		phi = o.f(xt);
		if (aslope) {                                                        // pnol_alpha_pool_analytic of the stand-in
			const pnol::PtrAcc acc{xt.data()};
			double sum = 0.0;
			for (int r = 0; r < n; r++) sum = sum + F::partial(P, acc, n, r) * p[r];
			dphi = sum;
			return;
		}
		for (int i = 0; i < n; i++) xt[i] = X[i] + (a + prm.dalpha) * p[i];    // lineSearchFDDerivative
		dphi = (o.f(xt) - phi) / prm.dalpha;
	};
	// D (:35-57): the inverse of the Hessian (oracle_fd_hessian or the analytic one), column by column with oracle_lu_solve, or I
	if (prm.init_hess_fd) {
		std::vector<double> B((size_t) n * n), e(n), col(n), xi(n), xj(n), xij(n);
		if (ahess) {
			const pnol::PtrAcc a{X.data()};
			for (int i = 0; i < n; i++) for (int j = i; j < n; j++) B[(size_t) i * n + j] = B[(size_t) j * n + i] = F::partial2(P, a, n, i, j);
		} else {
			const double f = o.f(X), h = prm.dx_hess;
			for (int i = 0; i < n; i++)
				for (int j = i; j < n; j++) {
					xi = X; xj = X; xij = X;
					xi[i] = xi[i] + h; xj[j] = xj[j] + h; xij[i] = xij[i] + h; xij[j] = xij[j] + h;
					B[(size_t) i * n + j] = (o.f(xij) - o.f(xi) - o.f(xj) + f) / (h * h);
				}
			for (int i = 0; i < n; i++) for (int j = 0; j < i; j++) B[(size_t) i * n + j] = B[(size_t) j * n + i];
		}
		for (int j = 0; j < n; j++) {
			for (int i = 0; i < n; i++) e[i] = i == j ? 1.0 : 0.0;
			oracle_lu_solve(B.data(), e.data(), n, col.data());
			for (int i = 0; i < n; i++) D[(size_t) i * n + j] = col[i];
		}
	} else {
		for (int i = 0; i < n; i++) for (int j = 0; j < n; j++) D[(size_t) i * n + j] = i == j ? 1.0 : 0.0;
	}
	gradient();                                                              // (:62-65)
	double Fx = o.f(X);
	const double f0 = Fx;
	int iter = 0;
	double xdiff = prm.x_min_diff * 2, g2 = 2 * prm.min_grad_2norm;
	while (iter < prm.max_iter && xdiff > prm.x_min_diff && g2 > prm.min_grad_2norm) {
		dFdXp = dFdX;
		oracle_matvec_neg(D.data(), dFdX.data(), n, p.data());
		// cubicInterpolationLineSearch (:177-291) and lineSearchZoom (:296-356)
		double alphaOpt = 0, Fopt = Fx;
		const double phi0 = Fx;
		double dphi0 = 0;
		for (int i = 0; i < n; i++) dphi0 = dphi0 + dFdX[i] * p[i];
		auto zoom = [&](double alo, double ahi, double plo, double phh, double dlo, double dhh) {
			for (int it = 0; it < prm.max_iter_ls; it++) {
				const double aj = cubic_interp_min(alo, ahi, plo, phh, dlo, dhh);
				double pj, dj;
				phi_and_slope(aj, pj, dj);
				if (pj > phi0 + prm.c1 * aj * dphi0 || pj >= plo) { ahi = aj; phh = pj; dhh = dj; }
				else {
					if (std::fabs(dj) <= std::fabs(prm.c2 * dphi0)) { alphaOpt = aj; Fopt = pj; break; }
					if (dj * (ahi - alo) >= 0) { ahi = alo; phh = plo; dhh = dlo; }
					alo = aj; plo = pj; dlo = dj;
				}
			}
		};
		double am1 = 0, phim1 = phi0, dm1 = dphi0, ai = prm.alpha_guess;
		for (int it = 0; it < prm.max_iter_ls; it++) {
			double phii, dphii;
			phi_and_slope(ai, phii, dphii);
			if ((phii > phi0 + prm.c1 * ai * dphi0) || (phii >= phim1 && it > 1)) { zoom(am1, ai, phim1, phii, dm1, dphii); break; }
			if (std::fabs(dphii) <= std::fabs(prm.c2 * dphi0)) { alphaOpt = ai; Fopt = phii; break; }
			if (dphii >= 0) { zoom(ai, am1, phii, phim1, dphii, dm1); break; }
			am1 = ai; phim1 = phii; dm1 = dphii; ai = 2 * ai;
		}
		for (int i = 0; i < n; i++) { Xprev[i] = X[i]; X[i] = X[i] + alphaOpt * p[i]; }
		Fx = Fopt;
		gradient();
		for (int i = 0; i < n; i++) { s[i] = alphaOpt * p[i]; g[i] = dFdX[i] - dFdXp[i]; }
		oracle_update_hinv(D.data(), g.data(), s.data(), n);
		xdiff = 0;
		for (int i = 0; i < n; i++) xdiff += std::fabs(X[i] - Xprev[i]);
		double s2 = 0;
		for (int i = 0; i < n; i++) s2 = s2 + dFdX[i] * dFdX[i];
		g2 = std::sqrt(s2);
		iter = iter + 1;
	}
	std::memcpy(Xb, X.data(), (size_t) n * sizeof(double));
	BfgsOut r;
	r.f0 = f0; r.fopt = Fx; r.iters = iter;
	r.stop = !(iter < prm.max_iter) ? 0 : (!(xdiff > prm.x_min_diff) ? 1 : 2);
	return r;
}

} // namespace

extern "C" int pnol_bfgs_batch(pnol_ctx * ctx, const pnol_functor * f, long long B, int n, double * X, const pnol_bfgs_params * prm,
                               int deriv_flags, double * f0_out, double * fopt_out, int * iters_out, int * stop_out)
{
	if (f->d.kind >= 100) { ctx->err = "bfgs_batch: not a scalar objective"; return PNOL_ERR_NO_FUNCTOR; }
	if (n < 1 || n > 64 || B < 0 || !prm) { ctx->err = "bfgs_batch: bad arguments"; return PNOL_ERR_INVALID; }
	if (B == 0) return PNOL_OK;
	const pnol_functor_params P = host_params(f);
	for (long long b = 0; b < B; b++) {
		BfgsOut r;
		double * Xb = X + b * n;
		switch (f->d.kind) {
			case PNOL_F_ROSENBROCK: r = oracle_bfgs<pnol::RosenbrockFunctor>(P, Xb, n, *prm, deriv_flags); break;
			case PNOL_F_POWER: r = oracle_bfgs<pnol::PowerFunctor>(P, Xb, n, *prm, deriv_flags); break;
			case PNOL_F_BOOTH: r = oracle_bfgs<pnol::BoothFunctor>(P, Xb, n, *prm, deriv_flags); break;
			case PNOL_F_GOLDSTEIN: r = oracle_bfgs<pnol::GoldsteinFunctor>(P, Xb, n, *prm, deriv_flags); break;
			case PNOL_F_RASTRIGIN: r = oracle_bfgs<pnol::RastriginFunctor>(P, Xb, n, *prm, deriv_flags); break;
			case PNOL_F_EXPCURVE_SINGLE: r = oracle_bfgs<pnol::ExpCurveSingleFunctor>(P, Xb, n, *prm, deriv_flags); break;
			default: return unavailable(ctx, "pnol_bfgs_batch for this functor kind");
		}
		f0_out[b] = r.f0; fopt_out[b] = r.fopt; iters_out[b] = r.iters; stop_out[b] = r.stop;
	}
	return PNOL_OK;
}
