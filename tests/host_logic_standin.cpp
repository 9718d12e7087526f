// host_logic_standin.cpp -- TEST INFRASTRUCTURE, never shipped. The CPU stand-in of the C-ABI that the host-logic tests link the
// unmodified host sources against (oracle/host_logic_device.cpp, included here as it is) extended by the entry points of the analytic
// derivatives and of the batched optimisers, answered by the functors' host definitions (include/pnol/functors.hpp, the definitions the
// kernels compile):
//   pnol_gradient[_recur]      partial() and eval(), as gradient_kernel computes them
//   pnol_hessian               partial2(), upper triangle computed and mirrored as hessian_kernel does
//   pnol_alpha_pool_analytic   eval() and partial() with the point assembly, the sequential sum and the sentinel of alpha_slope_kernel /
//                              alpha_slope_finish_kernel
//   pnol_bfgs_batch            every start is oracle_bfgs, a C++ restatement of BFGS::findMin (Source/BFGS_with_linesearch.cpp:12-385)
//                              over eval(), partial(), partial2() and the oracle's sequential dense helpers (oracle/pnol_oracle.cpp:
//                              oracle_matvec_neg, oracle_update_hinv, oracle_lu_solve)
//   pnol_lm_batch              every problem is oracle_lm (oracle/pnol_oracle.cpp) on its own rows -- the data columns sliced to
//                              [row_off[b], row_off[b+1]) -- and, with PNOL_JAC_ANALYTIC, the same loop with J from the models' jacobian()
//   pnol_simplex_batch         every start is oracle_simplex, a C++ restatement of SimplexSearch::findMin (Source/SimplexSearch.cpp:13-349)
//                              over eval(), which calls the library's own simplexSort and simplexDiff (host/SimplexSearch.cpp) rather than
//                              restating them; it also serves the test objectives of tests/user_functor/my_simplex_objectives.hpp and
//                              counts the sorts that left simplexSort's regime so that tests can show the quirk paths ran
// The built-in scalar objectives are answered; pnol_lm_batch answers the built-in residual models. tests/host_standin.py builds it. With
// it the host controllers run the analytic modes and the batch classes on the CPU, the batch restatements are checked bit for bit against
// the unmodified host controllers on the same stand-in (tests/test_{bfgs,lm,simplex}_batch_cpu.py), and the GPU tests use it as the oracle.
#include "../oracle/host_logic_device.cpp"

#include <cmath>

#include "../include/pnol/functors.hpp"
#include "../include/pnol/SimplexSearch.hpp"
#include "../include/pnol/device/simplex_sort.hpp"
#include "user_functor/my_simplex_objectives.hpp"

extern "C" {
int oracle_lm(int kind, const double * scalars, const long long * ints, const double * const * cols, long long m, double * X, int Nparam,
              double lambda0, double lambdaFactor, double dXGrad, int maxIter, double xMinDiff, double * F0, double * FOpt, double * chisq_out,
              double * lambda_out, double * trace);
}

namespace {

template <class F> struct functor_type { using type = F; };

// fn(functor_type<F>{}) with F the functor of a built-in scalar objective; any other kind is `what` not provided
template <class Fn> int with_scalar_functor(pnol_ctx * ctx, int kind, const char * what, Fn fn)
{
	switch (kind) {
		case PNOL_F_ROSENBROCK: return fn(functor_type<pnol::RosenbrockFunctor>{});
		case PNOL_F_POWER: return fn(functor_type<pnol::PowerFunctor>{});
		case PNOL_F_BOOTH: return fn(functor_type<pnol::BoothFunctor>{});
		case PNOL_F_GOLDSTEIN: return fn(functor_type<pnol::GoldsteinFunctor>{});
		case PNOL_F_RASTRIGIN: return fn(functor_type<pnol::RastriginFunctor>{});
		case PNOL_F_EXPCURVE_SINGLE: return fn(functor_type<pnol::ExpCurveSingleFunctor>{});
		default: return unavailable(ctx, what);
	}
}

// the same for the built-in residual models
template <class Fn> int with_residual_functor(pnol_ctx * ctx, int kind, const char * what, Fn fn)
{
	switch (kind) {
		case PNOL_F_EXPCURVE: return fn(functor_type<pnol::ExpCurveFunctor>{});
		case PNOL_F_CUBIC: return fn(functor_type<pnol::CubicFunctor>{});
		case PNOL_F_LORENTZ_SUM: return fn(functor_type<pnol::LorentzSumFunctor>{});
		default: return unavailable(ctx, what);
	}
}

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

// ---- pnol_gradient[_recur] ----

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
	return with_scalar_functor(ctx, f->d.kind, "pnol_gradient for this functor kind", [&](auto F) -> int {
		host_gradient<typename decltype(F)::type>(P, x, n, pos, nvar, g, f0);
		return PNOL_OK;
	});
}

// ---- pnol_hessian ----

template <class F> void host_hessian(const pnol_functor_params & P, const double * x, int n, double * H)
{
	const pnol::PtrAcc acc{x};
	for (int i = 0; i < n; i++)
		for (int j = i; j < n; j++) H[(size_t) i * n + j] = H[(size_t) j * n + i] = F::partial2(P, acc, n, i, j);
}

// ---- pnol_alpha_pool_analytic ----

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

// ---- pnol_bfgs_batch ----

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

// ---- pnol_lm_batch ----

double norm2(const double * v, long long n)
{
	double s = 0;
	for (long long i = 0; i < n; i++) s = s + v[i] * v[i];
	return std::sqrt(s);
}

template <class R> void host_jacobian_rows(const pnol_functor_params & P, const double * x, int n, long long m, double * J)
{
	const pnol::PtrAcc acc{x};
	for (long long i = 0; i < m; i++) R::jacobian(P, acc, n, i, J + i * n);
}

// oracle_lm's loop (LevMarqMPI::findMin, Source/LevenbergMarquardtMPI.cpp:12-173) with J = the model's analytic derivative
template <class R>
int lm_analytic(const pnol_functor * f, const pnol_functor_params & P, double * X, int n, double lambda, double factor, double xmin,
                int maxIter, double * chisq_out, double * lambda_out, int * stopped_out, double * Fopt)
{
	const long long m = P.m;
	std::vector<double> J((size_t) m * n), F(m), Ft(m), A((size_t) n * n), rhs(n), sigma(n), Xt(n);
	oracle_residual(f->d.kind, P.scalars, P.ints, P.col, m, X, n, F.data());
	double chi = std::pow(norm2(F.data(), m), 2);
	int iter = 0, stopped = 0;
	while (iter < maxIter) {
		host_jacobian_rows<R>(P, X, n, m, J.data());
		oracle_lm_normal_eq(J.data(), F.data(), m, n, lambda, nullptr, A.data(), rhs.data());
		oracle_lu_solve(A.data(), rhs.data(), n, sigma.data());
		for (int i = 0; i < n; i++) Xt[i] = X[i] + sigma[i];
		oracle_residual(f->d.kind, P.scalars, P.ints, P.col, m, Xt.data(), n, Ft.data());
		const double chit = std::pow(norm2(Ft.data(), m), 2);
		if (chit >= chi || chit != chit) {
			lambda = lambda * factor;
		} else {
			lambda = lambda / factor;
			chi = chit;
			for (int i = 0; i < n; i++) X[i] = Xt[i];
			F.swap(Ft);
			if (norm2(sigma.data(), n) < xmin) { stopped = 1; break; }
		}
		iter++;
	}
	if (Fopt) std::memcpy(Fopt, F.data(), (size_t) m * sizeof(double));
	*chisq_out = chi;
	*lambda_out = lambda;
	*stopped_out = stopped;
	return iter;
}

// ---- pnol_simplex_batch ----

long long gIrregularSorts = 0;

struct SimplexOut { double f0, fopt; int iters, stop; long long evals; };

// simplexSort outside its regime: a NaN entry, or a first maximum not in (0, inf) -- restated here, not taken from simplex_sort.hpp
bool sort_irregular(const double * f, int N)
{
	double M = f[0];
	bool nan = f[0] != f[0];
	for (int i = 1; i < N; i++) {
		if (f[i] != f[i]) nan = true;
		if (f[i] > M) M = f[i];
	}
	return nan || !(M > 0 && M < HUGE_VAL);
}

template <class F>
SimplexOut oracle_simplex(const pnol_functor_params & P, double * Xb, int n, const pnol_simplex_params & prm, const double * u)
{
	const int N = n + 1;
	std::vector<double> block((size_t) N * n), xbar(n), xr(n), xe(n), xc(n), fvec(N);
	std::vector<double *> rows(N);
	for (int k = 0; k < N; k++) rows[k] = block.data() + (size_t) k * n;
	double ** xvec = rows.data();
	auto f = [&](const double * x) { const pnol::PtrAcc a{x}; return F::eval(P, a, n); };
	auto sort = [&]() {
		if (sort_irregular(fvec.data(), N)) gIrregularSorts++;
		simplexSort(fvec.data(), xvec, n);
	};
	for (int j = 0; j < n; j++) xvec[0][j] = Xb[j];
	for (int i = 1; i < N; i++)
		for (int j = 0; j < n; j++) xvec[i][j] = xvec[0][j] + prm.init_rand_max * (u[(size_t) (i - 1) * n + j] - 0.5) * 2.0;
	for (int k = 0; k < N; k++) fvec[k] = f(xvec[k]);
	long long evals = N;
	const double f0 = fvec[0];
	sort();
	int iter = 0;
	double xdiff = prm.x_min_diff * 2;
	while (iter < prm.max_iter && xdiff > prm.x_min_diff) {
		for (int i = 0; i < n; i++) xbar[i] = 0.0;
		for (int i = 0; i < n; i++)
			for (int k = 0; k < n; k++) xbar[i] = xbar[i] + xvec[k][i] / ((double) n);
		double * worst = xvec[n];
		for (int i = 0; i < n; i++) xr[i] = xbar[i] + prm.alpha * (xbar[i] - worst[i]);
		const double fr = f(xr.data());
		evals++;
		if (fr >= fvec[0] && fr < fvec[n - 1]) {
			for (int i = 0; i < n; i++) worst[i] = xr[i];
			fvec[n] = fr;
		} else if (fr < fvec[0]) {
			for (int i = 0; i < n; i++) xe[i] = xbar[i] + prm.gamma * (xbar[i] - worst[i]);
			const double fe = f(xe.data());
			evals++;
			if (fe < fr) { for (int i = 0; i < n; i++) worst[i] = xe[i]; fvec[n] = fe; }
			else { for (int i = 0; i < n; i++) worst[i] = xr[i]; fvec[n] = fr; }
		} else {
			for (int i = 0; i < n; i++) xc[i] = xbar[i] + prm.rho * (worst[i] - xbar[i]);
			const double fc = f(xc.data());
			evals++;
			if (fc < fvec[n]) {
				for (int i = 0; i < n; i++) worst[i] = xc[i];
				fvec[n] = fc;
			} else {
				for (int k = 1; k < N; k++)
					for (int i = 0; i < n; i++) xvec[k][i] = xvec[0][i] + prm.sigma * (xvec[k][i] - xvec[0][i]);
				for (int k = 0; k < N; k++) fvec[k] = f(xvec[k]);
				evals += N;
			}
		}
		sort();
		xdiff = simplexDiff(xvec, n, N);
		iter = iter + 1;
	}
	std::memcpy(Xb, xvec[0], (size_t) n * sizeof(double));
	SimplexOut r;
	r.f0 = f0; r.fopt = fvec[0]; r.iters = iter; r.stop = !(iter < prm.max_iter) ? 0 : 1; r.evals = evals;
	return r;
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

int pnol_hessian(pnol_ctx * ctx, const pnol_functor * f, const double * x, int n, double * H_out)
{
	const pnol_functor_params P = host_params(f);
	return with_scalar_functor(ctx, f->d.kind, "pnol_hessian for this functor kind", [&](auto F) -> int {
		host_hessian<typename decltype(F)::type>(P, x, n, H_out);
		return PNOL_OK;
	});
}

int pnol_alpha_pool_analytic(pnol_ctx * ctx, const pnol_functor * f, const double * x, const double * p, int n, const double * alpha, int npool,
                             const unsigned char * eval_ind, const double * const_x, const unsigned char * const_ind, int nfull, double * phi,
                             double * dphi, int * bad_out)
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
		const int st = with_scalar_functor(ctx, f->d.kind, "pnol_alpha_pool_analytic for this functor kind", [&](auto F) -> int {
			host_slope<typename decltype(F)::type>(P, xa.data(), nfull, pos.data(), p, n, &ph, &ds);
			return PNOL_OK;
		});
		if (st != PNOL_OK) return st;
		if (ph != ph || std::isinf(ph)) { ph = 1e10; bad++; }
		phi[q] = ph;
		dphi[q] = ds;
	}
	if (bad_out) *bad_out = bad;
	return PNOL_OK;
}

int pnol_bfgs_batch(pnol_ctx * ctx, const pnol_functor * f, long long B, int n, double * X, const pnol_bfgs_params * prm, int deriv_flags,
                    double * f0_out, double * fopt_out, int * iters_out, int * stop_out)
{
	if (f->d.kind >= 100) { ctx->err = "bfgs_batch: not a scalar objective"; return PNOL_ERR_NO_FUNCTOR; }
	if (n < 1 || n > 64 || B < 0 || !prm) { ctx->err = "bfgs_batch: bad arguments"; return PNOL_ERR_INVALID; }
	if (B == 0) return PNOL_OK;
	const pnol_functor_params P = host_params(f);
	return with_scalar_functor(ctx, f->d.kind, "pnol_bfgs_batch for this functor kind", [&](auto F) -> int {
		for (long long b = 0; b < B; b++) {
			const BfgsOut r = oracle_bfgs<typename decltype(F)::type>(P, X + b * n, n, *prm, deriv_flags);
			f0_out[b] = r.f0; fopt_out[b] = r.fopt; iters_out[b] = r.iters; stop_out[b] = r.stop;
		}
		return PNOL_OK;
	});
}

int pnol_lm_batch(pnol_ctx * ctx, const pnol_functor * f, const long long * row_off, long long B, int n, double * X, const double * dx,
                  double lambda0, double lambda_factor, double x_min_diff, int max_iter, int jac_mode, double * chisq_out, double * lambda_out,
                  int * iters_out, int * stopped_out, double * F_out)
{
	if (f->d.kind < 100) { ctx->err = "lm_batch: not a residual model"; return PNOL_ERR_INVALID; }
	if (n < 1 || n > 64) { ctx->err = "lm_batch: n outside 1 .. 64"; return PNOL_ERR_INVALID; }
	return with_residual_functor(ctx, f->d.kind, "pnol_lm_batch for this functor kind", [&](auto R) -> int {
		const bool analytic = jac_mode == PNOL_JAC_ANALYTIC;
		if (!analytic && !dx) { ctx->err = "lm_batch: dx is required"; return PNOL_ERR_INVALID; }
		if (B == 0) return PNOL_OK;
		if (row_off[0] < 0 || row_off[B] > f->d.m) { ctx->err = "lm_batch: bad row_off"; return PNOL_ERR_INVALID; }
		for (long long b = 0; b < B; b++)
			if (row_off[b] > row_off[b + 1]) { ctx->err = "lm_batch: bad row_off"; return PNOL_ERR_INVALID; }
		for (int j = 1; j < n && !analytic; j++)
			if (dx[j] != dx[0]) return unavailable(ctx, "pnol_lm_batch with unequal dx entries (oracle_lm takes one dXGrad)");
		const pnol_functor_params P = host_params(f);
		for (long long b = 0; b < B; b++) {
			const long long base = row_off[b], mb = row_off[b + 1] - base;
			pnol_functor_params Pb = P;
			for (int c = 0; c < f->d.n_columns; c++) Pb.col[c] = P.col[c] + base;
			Pb.m = mb;
			double * Xb = X + b * n;
			double * Fb = F_out ? F_out + base : nullptr;
			if (analytic) {
				iters_out[b] = lm_analytic<typename decltype(R)::type>(f, Pb, Xb, n, lambda0, lambda_factor, x_min_diff, max_iter, chisq_out + b,
				                                                       lambda_out + b, stopped_out + b, Fb);
			} else {
				// the stopping rule fired when the loop left before max_iter passes
				iters_out[b] = oracle_lm(f->d.kind, Pb.scalars, Pb.ints, Pb.col, mb, Xb, n, lambda0, lambda_factor, dx[0], max_iter, x_min_diff,
				                         nullptr, Fb, chisq_out + b, lambda_out + b, nullptr);
				stopped_out[b] = iters_out[b] < max_iter;
			}
		}
		return PNOL_OK;
	});
}

int pnol_simplex_batch(pnol_ctx * ctx, const pnol_functor * f, long long B, int n, double * X, const pnol_simplex_params * prm,
                       const pnol_stream_desc * stream, uint64_t stream_offset, double * f0_out, double * fopt_out, int * iters_out,
                       int * stop_out, long long * evals_out)
{
	if (!ctx || !f) return PNOL_ERR_INVALID;
	const int kind = f->d.kind;
	if ((kind >= 100 && kind < PNOL_F_USER_SCALAR_BASE) || kind >= PNOL_F_USER_RESIDUAL_BASE) {
		ctx->err = "simplex_batch: not a scalar objective";
		return PNOL_ERR_NO_FUNCTOR;
	}
	if (n < 1 || n > 64 || B < 0 || B > 0x7fffffffLL || !prm || !stream) { ctx->err = "simplex_batch: bad arguments"; return PNOL_ERR_INVALID; }
	if (B == 0) return PNOL_OK;
	if (!X || !f0_out || !fopt_out || !iters_out || !stop_out) { ctx->err = "simplex_batch: an output is missing"; return PNOL_ERR_INVALID; }
	const uint64_t nn = (uint64_t) n * n, draws = (uint64_t) B * nn;
	if (stream->values && (stream_offset > stream->n_values || stream->n_values - stream_offset < draws)) {
		ctx->err = "simplex_batch: the explicit random stream is too short";
		return PNOL_ERR_STREAM;
	}
	const pnol_functor_params P = host_params(f);
	auto run = [&](auto F) -> int {
		std::vector<double> u(nn);
		for (long long b = 0; b < B; b++) {
			for (uint64_t t = 0; t < nn; t++) {
				const uint64_t pos = stream_offset + (uint64_t) b * nn + t;
				u[t] = stream->values ? stream->values[pos] : pnol_stream_uniform(stream->seed, pos, stream->scale);
			}
			const SimplexOut r = oracle_simplex<typename decltype(F)::type>(P, X + b * n, n, *prm, u.data());
			f0_out[b] = r.f0; fopt_out[b] = r.fopt; iters_out[b] = r.iters; stop_out[b] = r.stop;
			if (evals_out) evals_out[b] = r.evals;
		}
		return PNOL_OK;
	};
	switch (kind) {
		case MYS_F_NEGATIVE: return run(functor_type<SimplexNegativeFunctor>{});
		case MYS_F_QUANTIZED: return run(functor_type<SimplexQuantizedFunctor>{});
		case MYS_F_SIGNED_ZERO: return run(functor_type<SimplexSignedZeroFunctor>{});
		case MYS_F_NAN_REGION: return run(functor_type<SimplexNanRegionFunctor>{});
		default: return with_scalar_functor(ctx, kind, "pnol_simplex_batch for this functor kind", run);
	}
}

// the stand-in's pnol_simplex_batch on a functor of `kind` (scalars / ints as pnol_functor_desc holds them, no data columns)
int standin_simplex_batch(int kind, const double * scalars, const long long * ints, long long B, int n, double * X, const pnol_simplex_params * prm,
                          const pnol_stream_desc * stream, uint64_t stream_offset, double * f0_out, double * fopt_out, int * iters_out,
                          int * stop_out, long long * evals_out)
{
	pnol_ctx ctx;
	pnol_functor_desc d;
	std::memset(&d, 0, sizeof d);
	d.kind = kind;
	for (int k = 0; k < PNOL_MAX_SCALARS && scalars; k++) d.scalars[k] = scalars[k];
	for (int k = 0; k < PNOL_MAX_INTS && ints; k++) d.ints[k] = ints[k];
	pnol_functor * f = nullptr;
	int st = pnol_functor_create(&ctx, &d, &f);
	if (st != PNOL_OK) return st;
	st = pnol_simplex_batch(&ctx, f, B, n, X, prm, stream, stream_offset, f0_out, fopt_out, iters_out, stop_out, evals_out);
	pnol_functor_destroy(f);
	return st;
}

long long standin_simplex_irregular_sorts() { return gIrregularSorts; }

// simplexSort (the library's) on f (N entries): perm[k] is the entry place k received, f is left as simplexSort leaves it
void standin_simplex_sort_reference(double * f, int N, int * perm)
{
	const int nd = N - 1;
	std::vector<double> block((size_t) N * nd);
	std::vector<double *> rows(N);
	for (int k = 0; k < N; k++) {
		rows[k] = block.data() + (size_t) k * nd;
		for (int j = 0; j < nd; j++) rows[k][j] = k;
	}
	simplexSort(f, rows.data(), nd);
	for (int k = 0; k < N; k++) perm[k] = (int) rows[k][0];
}

// pnol::simplex_sort_perm (include/pnol/device/simplex_sort.hpp) with the stats of G lanes; returns 1 in the regime
int standin_simplex_sort_perm(double * f, int N, int G, int * perm) { return pnol::simplex_sort_perm(f, N, G, perm) ? 1 : 0; }

} // extern "C"
