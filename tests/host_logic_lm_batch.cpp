// host_logic_lm_batch.cpp -- TEST INFRASTRUCTURE, never shipped. The CPU stand-in of the C-ABI extended by the analytic derivatives
// (tests/host_logic_slope.cpp, included here as it is) and by pnol_lm_batch: every problem is oracle_lm (oracle/pnol_oracle.cpp) on its
// own rows -- the data columns sliced to [row_off[b], row_off[b+1]) -- and, with PNOL_JAC_ANALYTIC, the same loop with J from the
// built-in models' host jacobian() (include/pnol/functors.hpp, the definitions the kernels compile). tests/host_logic_lm_batch_lib.py
// builds it; with it LevMarqBatch runs on the CPU (tests/test_lm_batch_cpu.py).
#include "host_logic_slope.cpp"

#include <cmath>

extern "C" {
int oracle_lm(int kind, const double * scalars, const long long * ints, const double * const * cols, long long m, double * X, int Nparam,
              double lambda0, double lambdaFactor, double dXGrad, int maxIter, double xMinDiff, double * F0, double * FOpt, double * chisq_out,
              double * lambda_out, double * trace);
}

namespace {
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
int lm_analytic(const pnol_functor * f, const pnol_functor_params & P, double * X, int n, double lambda, double factor, double xmin,
                int maxIter, double * chisq_out, double * lambda_out, int * stopped_out, double * Fopt)
{
	const long long m = P.m;
	std::vector<double> J((size_t) m * n), F(m), Ft(m), A((size_t) n * n), rhs(n), sigma(n), Xt(n);
	oracle_residual(f->d.kind, P.scalars, P.ints, P.col, m, X, n, F.data());
	double chi = std::pow(norm2(F.data(), m), 2);
	int iter = 0, stopped = 0;
	while (iter < maxIter) {
		switch (f->d.kind) {
			case PNOL_F_EXPCURVE: host_jacobian_rows<pnol::ExpCurveFunctor>(P, X, n, m, J.data()); break;
			case PNOL_F_CUBIC: host_jacobian_rows<pnol::CubicFunctor>(P, X, n, m, J.data()); break;
			default: host_jacobian_rows<pnol::LorentzSumFunctor>(P, X, n, m, J.data()); break;
		}
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
} // namespace

extern "C" int pnol_lm_batch(pnol_ctx * ctx, const pnol_functor * f, const long long * row_off, long long B, int n, double * X,
                             const double * dx, double lambda0, double lambda_factor, double x_min_diff, int max_iter, int jac_mode,
                             double * chisq_out, double * lambda_out, int * iters_out, int * stopped_out, double * F_out)
{
	if (f->d.kind < 100) { ctx->err = "lm_batch: not a residual model"; return PNOL_ERR_INVALID; }
	if (n < 1 || n > 64) { ctx->err = "lm_batch: n outside 1 .. 64"; return PNOL_ERR_INVALID; }
	if (f->d.kind != PNOL_F_EXPCURVE && f->d.kind != PNOL_F_CUBIC && f->d.kind != PNOL_F_LORENTZ_SUM) return unavailable(ctx, "pnol_lm_batch for this functor kind");
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
			iters_out[b] = lm_analytic(f, Pb, Xb, n, lambda0, lambda_factor, x_min_diff, max_iter, chisq_out + b, lambda_out + b, stopped_out + b, Fb);
		} else {
			// the stopping rule fired when the loop left before max_iter passes
			iters_out[b] = oracle_lm(f->d.kind, Pb.scalars, Pb.ints, Pb.col, mb, Xb, n, lambda0, lambda_factor, dx[0], max_iter, x_min_diff,
			                         nullptr, Fb, chisq_out + b, lambda_out + b, nullptr);
			stopped_out[b] = iters_out[b] < max_iter;
		}
	}
	return PNOL_OK;
}
