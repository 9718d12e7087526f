// host_logic_simplex_batch.cpp -- TEST INFRASTRUCTURE, never shipped. The CPU stand-in of the C-ABI (oracle/host_logic_device.cpp, through
// tests/host_logic_gradient.cpp, included here as it is) extended by pnol_simplex_batch: every start is oracle_simplex, a C++ restatement
// of SimplexSearch::findMin (Source/SimplexSearch.cpp:13-349) over the functor's host eval() (include/pnol/functors.hpp, the definitions
// the kernels compile), which calls the library's own simplexSort and simplexDiff (host/SimplexSearch.cpp) rather than restating them.
// It serves the six built-in scalar objectives and the test objectives of tests/user_functor/my_simplex_objectives.hpp, and counts the
// sorts that left simplexSort's regime so that tests can show the quirk paths ran. tests/host_logic_simplex_batch_lib.py builds it;
// tests/test_simplex_batch_cpu.py checks it bit for bit against the unmodified host SimplexSearch controller on the same stand-in, and the
// GPU tests use it as the oracle.
#include "host_logic_gradient.cpp"

#include <cmath>

#include "../include/pnol/SimplexSearch.hpp"
#include "../include/pnol/device/simplex_sort.hpp"
#include "user_functor/my_simplex_objectives.hpp"

namespace {

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
	std::vector<double> u(nn);
	for (long long b = 0; b < B; b++) {
		for (uint64_t t = 0; t < nn; t++) {
			const uint64_t pos = stream_offset + (uint64_t) b * nn + t;
			u[t] = stream->values ? stream->values[pos] : pnol_stream_uniform(stream->seed, pos, stream->scale);
		}
		double * Xb = X + b * n;
		SimplexOut r;
		switch (kind) {
			case PNOL_F_ROSENBROCK: r = oracle_simplex<pnol::RosenbrockFunctor>(P, Xb, n, *prm, u.data()); break;
			case PNOL_F_POWER: r = oracle_simplex<pnol::PowerFunctor>(P, Xb, n, *prm, u.data()); break;
			case PNOL_F_BOOTH: r = oracle_simplex<pnol::BoothFunctor>(P, Xb, n, *prm, u.data()); break;
			case PNOL_F_GOLDSTEIN: r = oracle_simplex<pnol::GoldsteinFunctor>(P, Xb, n, *prm, u.data()); break;
			case PNOL_F_RASTRIGIN: r = oracle_simplex<pnol::RastriginFunctor>(P, Xb, n, *prm, u.data()); break;
			case PNOL_F_EXPCURVE_SINGLE: r = oracle_simplex<pnol::ExpCurveSingleFunctor>(P, Xb, n, *prm, u.data()); break;
			case MYS_F_NEGATIVE: r = oracle_simplex<SimplexNegativeFunctor>(P, Xb, n, *prm, u.data()); break;
			case MYS_F_QUANTIZED: r = oracle_simplex<SimplexQuantizedFunctor>(P, Xb, n, *prm, u.data()); break;
			case MYS_F_SIGNED_ZERO: r = oracle_simplex<SimplexSignedZeroFunctor>(P, Xb, n, *prm, u.data()); break;
			case MYS_F_NAN_REGION: r = oracle_simplex<SimplexNanRegionFunctor>(P, Xb, n, *prm, u.data()); break;
			default: return unavailable(ctx, "pnol_simplex_batch for this functor kind");
		}
		f0_out[b] = r.f0; fopt_out[b] = r.fopt; iters_out[b] = r.iters; stop_out[b] = r.stop;
		if (evals_out) evals_out[b] = r.evals;
	}
	return PNOL_OK;
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

}
