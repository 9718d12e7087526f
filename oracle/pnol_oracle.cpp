// TEST INFRASTRUCTURE -- CPU restatement ("port") of the reference's algorithm for the hot path.
//
// Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load this file's
// library (oracle/libpnol_oracle.so). The product (libpnol_b200.so, libpnol_b200_host.so) never links or calls it.
//
// Every function cites the reference file:line (under /root/reference/) it follows. Pinning: the arithmetic that
// lives in the reference tree (FD stencils, LM step control, updateHessianInv structure, GA operators, box
// helpers, example objectives) is checked bit-for-bit against the VERBATIM reference compiled from
// /root/reference/Source (oracle/_ref, see oracle/Makefile and tests/test_oracle_vs_ref.py) and against the
// fixtures under tests/golden/ generated from it. The dense helpers the reference takes from its un-vendored
// UtilityFunctionLibrary (matrixMultiply, luSolve, vector2Norm, dotProd, vectorMin/Max, linspace, timeRand) are
// NOT in the reference tree: here they follow oracle/shim (our stated conventions) -- "parity unpinned" at that
// boundary, see DESIGN.md.
//
// Plain sequential C++; no FMA contraction (-ffp-contract=off); built at -O2 like the reference (-O3) so that
// pow(x,2) folds to x*x exactly as in the reference build (SURVEY.md 7.1).

#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <vector>

using std::vector;

#include "oracle_objectives.h"

// ------------------------------------------------------------------------------------------------
// dense helpers: conventions of oracle/shim (un-vendored in the reference; "parity unpinned")
// ------------------------------------------------------------------------------------------------
static double o_norm2(const double * v, long long n)
{
	double s = 0;
	for (long long i = 0; i < n; i++) s = s + v[i] * v[i];
	return sqrt(s);
}
static double o_dot(const double * a, const double * b, int n)
{
	double s = 0;
	for (int i = 0; i < n; i++) s = s + a[i] * b[i];
	return s;
}
static void o_lu_solve(const double * A, const double * b, int n, double * x)
{
	vector<double> LU(A, A + (size_t) n * n);
	vector<int> piv(n);
	for (int i = 0; i < n; i++) piv[i] = i;
	for (int k = 0; k < n; k++) {
		int p = k; double best = fabs(LU[(size_t) k * n + k]);
		for (int i = k + 1; i < n; i++) if (fabs(LU[(size_t) i * n + k]) > best) { best = fabs(LU[(size_t) i * n + k]); p = i; }
		if (p != k) {
			for (int j = 0; j < n; j++) { double t = LU[(size_t) p * n + j]; LU[(size_t) p * n + j] = LU[(size_t) k * n + j]; LU[(size_t) k * n + j] = t; }
			int t = piv[p]; piv[p] = piv[k]; piv[k] = t;
		}
		for (int i = k + 1; i < n; i++) {
			LU[(size_t) i * n + k] = LU[(size_t) i * n + k] / LU[(size_t) k * n + k];
			for (int j = k + 1; j < n; j++) LU[(size_t) i * n + j] = LU[(size_t) i * n + j] - LU[(size_t) i * n + k] * LU[(size_t) k * n + j];
		}
	}
	vector<double> y(n);
	for (int i = 0; i < n; i++) {
		double s = b[piv[i]];
		for (int k = 0; k < i; k++) s = s - LU[(size_t) i * n + k] * y[k];
		y[i] = s;
	}
	for (int i = n - 1; i >= 0; i--) {
		double s = y[i];
		for (int k = i + 1; k < n; k++) s = s - LU[(size_t) i * n + k] * x[k];
		x[i] = s / LU[(size_t) i * n + i];
	}
}

static double o_stream_u(uint64_t seed, uint64_t k, double scale)
{
	uint64_t z = seed + (k + 1ULL) * 0x9E3779B97F4A7C15ULL;
	z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
	z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
	z = z ^ (z >> 31);
	return ((double) (z >> 11) * (1.0 / 9007199254740992.0)) * scale;
}

struct OStream {
	const double * values; uint64_t n_values; uint64_t seed; double scale; uint64_t pos; int exhausted;
	double next()
	{
		if (values) {
			if (pos >= n_values) { exhausted = 1; pos++; return 0.0; }
			return values[pos++];
		}
		return o_stream_u(seed, pos++, scale);
	}
};

extern "C" {

// ------------------------------------------------------------------------------------------------
// objective evaluation
// ------------------------------------------------------------------------------------------------
double oracle_obj_eval(int kind, const double * scalars, const long long * ints, const double * const * cols, long long m,
                       const double * X, int n)
{
	OFunctor f = {kind, scalars, ints, cols, m};
	return o_scalar(f, X, n);
}

// GeneticAlgorithm::evaluatePopulation, Source/GeneticAlgorithm.cpp:301-311 (== the P=1 result of
// GeneticAlgorithmMPI::evaluatePopulationParallel, Source/GeneticAlgorithmMPI.cpp:283-414)
void oracle_eval_batch(int kind, const double * scalars, const long long * ints, const double * const * cols, long long m,
                       const double * pts, long long B, int n, long long ld, const unsigned char * indicator, double * f_out)
{
	OFunctor f = {kind, scalars, ints, cols, m};
	for (long long b = 0; b < B; b++)
		if (!indicator || indicator[b]) f_out[b] = o_scalar(f, pts + b * ld, n);
}

void oracle_residual(int kind, const double * scalars, const long long * ints, const double * const * cols, long long m,
                     const double * X, int n, double * F)
{
	OFunctor f = {kind, scalars, ints, cols, m};
	o_residual(f, X, n, F);
}

// ------------------------------------------------------------------------------------------------
// FD stencils
// ------------------------------------------------------------------------------------------------
// Objective::gradientApproximation, Source/PNOL_Objective.cpp:12-34 (MPI twin :88-159 gives identical bits)
void oracle_fd_gradient(int kind, const double * scalars, const long long * ints, const double * const * cols, long long m,
                        const double * X, const double * dX, int N, double * dFdX, double * f0)
{
	OFunctor f = {kind, scalars, ints, cols, m};
	vector<double> XdX(N, 0);
	double F = o_scalar(f, X, N);
	for (int i = 0; i < N; i++) {
		for (int j = 0; j < N; j++) XdX[j] = X[j];
		XdX[i] = XdX[i] + dX[i];
		double FdX = o_scalar(f, XdX.data(), N);
		dFdX[i] = (FdX - F) / dX[i];
	}
	if (f0) *f0 = F;
}

// Objective::objEvalRecur, Source/PNOL_Objective.cpp:303-333
static double o_eval_recur(const OFunctor & f, const double * Xrecur, const double * constantX, const unsigned char * ind, int Nparam)
{
	vector<double> X(Nparam, 0);
	int iRecur = 0;
	for (int i = 0; i < Nparam; i++) {
		if (ind[i]) X[i] = constantX[i];
		else { X[i] = Xrecur[iRecur]; iRecur++; }
	}
	return o_scalar(f, X.data(), Nparam);
}

double oracle_eval_recur(int kind, const double * scalars, const long long * ints, const double * const * cols, long long m,
                         const double * Xr, int Nr, const double * constantX, const unsigned char * ind, int Nparam)
{
	(void) Nr;
	OFunctor f = {kind, scalars, ints, cols, m};
	return o_eval_recur(f, Xr, constantX, ind, Nparam);
}

// Objective::gradientApproximationRecur, Source/PNOL_Objective.cpp:337-360 (MPI twin :366-459)
void oracle_fd_gradient_recur(int kind, const double * scalars, const long long * ints, const double * const * cols, long long m,
                              const double * X, const double * dX, int N, const double * constantX, const unsigned char * ind,
                              int Nparam, double * dFdX, double * f0)
{
	OFunctor f = {kind, scalars, ints, cols, m};
	vector<double> XdX(N, 0);
	double F = o_eval_recur(f, X, constantX, ind, Nparam);
	for (int i = 0; i < N; i++) {
		for (int j = 0; j < N; j++) XdX[j] = X[j];
		XdX[i] = XdX[i] + dX[i];
		double FdX = o_eval_recur(f, XdX.data(), constantX, ind, Nparam);
		dFdX[i] = (FdX - F) / dX[i];
	}
	if (f0) *f0 = F;
}

// Objective::hessianApproximation, Source/PNOL_Objective.cpp:38-85
void oracle_fd_hessian(int kind, const double * scalars, const long long * ints, const double * const * cols, long long m,
                       const double * X, const double * dX, int N, double * B)
{
	OFunctor f = {kind, scalars, ints, cols, m};
	vector<double> XdXi(N), XdXj(N), XdXij(N);
	double F = o_scalar(f, X, N);
	for (int i = 0; i < N; i++)
		for (int j = i; j < N; j++) {
			for (int k = 0; k < N; k++) { XdXi[k] = X[k]; XdXj[k] = X[k]; XdXij[k] = X[k]; }
			XdXi[i] = XdXi[i] + dX[i];
			XdXj[j] = XdXj[j] + dX[j];
			XdXij[i] = XdXij[i] + dX[i];
			XdXij[j] = XdXij[j] + dX[j];
			double FdXi = o_scalar(f, XdXi.data(), N);
			double FdXj = o_scalar(f, XdXj.data(), N);
			double FdXij = o_scalar(f, XdXij.data(), N);
			B[(size_t) i * N + j] = (FdXij - FdXi - FdXj + F) / (dX[i] * dX[j]);
		}
	for (int i = 0; i < N; i++)
		for (int j = 0; j < i; j++) B[(size_t) i * N + j] = B[(size_t) j * N + i];
}

// MultiObjective::gradientApproximation, Source/PNOL_Objective.cpp:165-197 (MPI twin :202-299). J is m x n row-major.
void oracle_fd_jacobian(int kind, const double * scalars, const long long * ints, const double * const * cols, long long m,
                        const double * X, const double * dX, int N, double * J, double * Fout)
{
	OFunctor f = {kind, scalars, ints, cols, m};
	vector<double> XdX(N, 0), F(m, 0), FdX(m, 0);
	o_residual(f, X, N, F.data());
	for (int j = 0; j < N; j++) {
		for (int k = 0; k < N; k++) XdX[k] = X[k];
		XdX[j] = XdX[j] + dX[j];
		o_residual(f, XdX.data(), N, FdX.data());
		for (long long i = 0; i < m; i++) J[(size_t) i * N + j] = (FdX[i] - F[i]) / dX[j];
	}
	if (Fout) memcpy(Fout, F.data(), (size_t) m * sizeof(double));
}

// ------------------------------------------------------------------------------------------------
// Levenberg-Marquardt
// ------------------------------------------------------------------------------------------------
// normal equations, Source/LevenbergMarquardtMPI.cpp:64-85 with the shim's i-j-k sequential products.
// (JTJ[i][j] = sum_k JT[i][k] J[k][j], k ascending; rhs = -(JT F), k ascending)
void oracle_lm_normal_eq(const double * J, const double * F, long long m, int n, double lambda, double * JTJ, double * A, double * rhs)
{
	for (int i = 0; i < n; i++)
		for (int j = 0; j < n; j++) {
			double s = 0;
			for (long long k = 0; k < m; k++) s = s + J[(size_t) k * n + i] * J[(size_t) k * n + j];
			if (JTJ) JTJ[(size_t) i * n + j] = s;
			if (A) A[(size_t) i * n + j] = (i == j) ? (1 + lambda) * s : s;
		}
	if (rhs)
		for (int i = 0; i < n; i++) {
			double s = 0;
			for (long long k = 0; k < m; k++) s = s + J[(size_t) k * n + i] * F[k];
			rhs[i] = -s;
		}
}

void oracle_lu_solve(const double * A, const double * b, int n, double * x) { o_lu_solve(A, b, n, x); }

// LevMarqMPI::findMin, Source/LevenbergMarquardtMPI.cpp:12-173 (serial twin LevenbergMarquardt.cpp:11-177).
// trace (optional, (maxIter+1) x (n+2)): per loop pass k the values [X after the pass | chiSq | lambda].
// Returns the iteration counter at exit.
int oracle_lm(int kind, const double * scalars, const long long * ints, const double * const * cols, long long m,
              double * X, int Nparam, double lambda0, double lambdaFactor, double dXGrad, int maxIter, double xMinDiff,
              double * F0, double * FOpt, double * chisq_out, double * lambda_out, double * trace)
{
	OFunctor f = {kind, scalars, ints, cols, m};
	long long Ndata = m;
	double chiSq;
	double lambda = lambda0;
	vector<double> A((size_t) Nparam * Nparam), J((size_t) Ndata * Nparam), rhs(Nparam, 0.0), dX(Nparam, dXGrad);
	vector<double> F(Ndata, 0), Fprev(Ndata, 0), sigma(Nparam, 0), Xprev(Nparam, 0), F0v(Ndata, 0);

	o_residual(f, X, Nparam, F0v.data());                       // :42
	for (long long k = 0; k < Ndata; k++) { F[k] = F0v[k]; Fprev[k] = F[k]; }
	for (int k = 0; k < Nparam; k++) Xprev[k] = X[k];
	chiSq = pow(o_norm2(F.data(), Ndata), 2);                   // :51

	int iter = 0;
	double xdiff2Norm = xMinDiff * 2;
	while (iter < maxIter) {                                    // :55
		oracle_fd_jacobian(kind, scalars, ints, cols, m, X, dX.data(), Nparam, J.data(), nullptr);   // :60
		oracle_lm_normal_eq(J.data(), F.data(), Ndata, Nparam, lambda, nullptr, A.data(), rhs.data()); // :64-85
		o_lu_solve(A.data(), rhs.data(), Nparam, sigma.data());  // :88
		for (int k = 0; k < Nparam; k++) Xprev[k] = X[k];        // :91-94
		for (long long k = 0; k < Ndata; k++) Fprev[k] = F[k];
		for (int i = 0; i < Nparam; i++) X[i] = X[i] + sigma[i]; // :97-100
		o_residual(f, X, Nparam, F.data());                      // :103
		double chiSqPrev = chiSq;                                // :107
		chiSq = pow(o_norm2(F.data(), Ndata), 2);                // :108
		bool stop = false;
		if (chiSq >= chiSqPrev || chiSq != chiSq) {              // :110
			chiSq = chiSqPrev;
			for (int i = 0; i < Nparam; i++) X[i] = Xprev[i];
			for (long long k = 0; k < Ndata; k++) F[k] = Fprev[k];
			lambda = lambda * lambdaFactor;                      // :129
		} else {
			lambda = lambda / lambdaFactor;                      // :135
			xdiff2Norm = o_norm2(sigma.data(), Nparam);          // :138
			if (xdiff2Norm < xMinDiff) stop = true;              // :139-140
		}
		if (trace) {
			double * row = trace + (size_t) iter * (Nparam + 2);
			for (int i = 0; i < Nparam; i++) row[i] = X[i];
			row[Nparam] = chiSq; row[Nparam + 1] = lambda;
		}
		if (stop) break;
		iter++;
	}
	if (F0) memcpy(F0, F0v.data(), (size_t) Ndata * sizeof(double));
	if (FOpt) for (long long k = 0; k < Ndata; k++) FOpt[k] = F[k];   // :159-162
	if (chisq_out) *chisq_out = chiSq;
	if (lambda_out) *lambda_out = lambda;
	return iter;
}

// ------------------------------------------------------------------------------------------------
// BFGS dense pieces
// ------------------------------------------------------------------------------------------------
// updateHessianInv, Source/BFGS_with_linesearch.cpp:389-432 (shim matrixMultiply: i-j-k, sequential k)
void oracle_update_hinv(double * D, const double * g, const double * s, int n)
{
	size_t nn = (size_t) n * n;
	vector<double> M1(nn), M2(nn), M3(nn), A(nn);
	double rho = 1 / o_dot(g, s, n);                            // :397
	for (int i = 0; i < n; i++)
		for (int j = 0; j < n; j++) {
			double m1 = 0, m2 = 0;
			if (i == j) { m1 = 1; m2 = 1; }
			M1[(size_t) i * n + j] = m1 - rho * s[i] * g[j];     // :412
			M2[(size_t) i * n + j] = m2 - rho * g[i] * s[j];     // :413
			M3[(size_t) i * n + j] = rho * s[i] * s[j];          // :414
		}
	for (int i = 0; i < n; i++)                                  // matrixMultiply(M1, D, A)  :421
		for (int j = 0; j < n; j++) {
			double acc = 0;
			for (int k = 0; k < n; k++) acc = acc + M1[(size_t) i * n + k] * D[(size_t) k * n + j];
			A[(size_t) i * n + j] = acc;
		}
	for (int i = 0; i < n; i++)                                  // matrixMultiply(A, M2, D)  :422
		for (int j = 0; j < n; j++) {
			double acc = 0;
			for (int k = 0; k < n; k++) acc = acc + A[(size_t) i * n + k] * M2[(size_t) k * n + j];
			D[(size_t) i * n + j] = acc;
		}
	for (size_t e = 0; e < nn; e++) D[e] = D[e] + M3[e];         // :424-430
}

// p = -D g, Source/BFGS_bnd_linesearch_MPI_SW.cpp:143-144
void oracle_matvec_neg(const double * D, const double * g, int n, double * p)
{
	for (int i = 0; i < n; i++) {
		double s = 0;
		for (int k = 0; k < n; k++) s = s + D[(size_t) i * n + k] * g[k];
		p[i] = -s;
	}
}

void oracle_dgemm_nn(const double * A, const double * B, double * C, int M, int N, int K)
{
	for (int i = 0; i < M; i++)
		for (int j = 0; j < N; j++) {
			double acc = 0;
			for (int k = 0; k < K; k++) acc = acc + A[(size_t) i * K + k] * B[(size_t) k * N + j];
			C[(size_t) i * N + j] = acc;
		}
}

// lineSearchObj / lineSearchFDDerivative + sentinel, Source/BFGS_bnd_linesearch_MPI_SW.cpp:599-734
// (also BFGS_with_linesearch.cpp:140-172). const_ind == NULL: no active set.
void oracle_alpha_pool(int kind, const double * scalars, const long long * ints, const double * const * cols, long long m,
                       const double * X, const double * p, int n, const double * alpha, int npool, double dalpha,
                       const unsigned char * eval_ind, const double * constantX, const unsigned char * const_ind, int nfull,
                       double * phi, double * dphi, int * bad)
{
	OFunctor f = {kind, scalars, ints, cols, m};
	vector<double> Xt(n);
	int nbad = 0;
	for (int k = 0; k < npool; k++) {
		if (eval_ind && !eval_ind[k]) continue;
		for (int i = 0; i < n; i++) Xt[i] = X[i] + alpha[k] * p[i];
		double ph = const_ind ? o_eval_recur(f, Xt.data(), constantX, const_ind, nfull) : o_scalar(f, Xt.data(), n);
		if (dphi) {
			for (int i = 0; i < n; i++) Xt[i] = X[i] + (alpha[k] + dalpha) * p[i];
			double ph2 = const_ind ? o_eval_recur(f, Xt.data(), constantX, const_ind, nfull) : o_scalar(f, Xt.data(), n);
			dphi[k] = (ph2 - ph) / dalpha;     // (:719-734) no sentinel on the slope
		}
		if (ph != ph || isinf(ph)) { ph = 1e10; nbad++; }
		phi[k] = ph;
	}
	if (bad) *bad = nbad;
}

// checkBoxBounds, Source/Box_boundary_functions.cpp:11-40
int oracle_check_box_bounds(double * X, const double * Xlb, const double * Xub, int n)
{
	int cnt = 0;
	for (int i = 0; i < n; i++)
		if (X[i] - Xlb[i] < -fabs(Xlb[i]) / 1000 || X[i] - Xub[i] > fabs(Xub[i]) / 1000) { X[i] = (Xlb[i] + Xub[i]) / 2.0; cnt++; }
	return cnt;
}

// computeAlphaBnd, Source/BFGS_with_bnd_linsearch_MPI.cpp:665-708
double oracle_compute_alpha_bnd(const double * X, const double * Xlb, const double * Xub, const double * p, int Nprm)
{
	double alphaBnd = 0;
	for (int i = 0; i < Nprm; i++) {
		double alpha1i = (Xub[i] - X[i]) / p[i];
		double alpha2i = (Xlb[i] - X[i]) / p[i];
		double alphaBndi;
		if (alpha1i > 0) alphaBndi = alpha1i;
		else if (alpha2i > 0) alphaBndi = alpha2i;
		else alphaBndi = 0;
		if (i == 0) alphaBnd = alphaBndi;
		if (alphaBnd > alphaBndi) alphaBnd = alphaBndi;
	}
	return alphaBnd;
}

double oracle_stream_uniform(uint64_t seed, uint64_t k, double scale) { return o_stream_u(seed, k, scale); }

// ------------------------------------------------------------------------------------------------
// genetic algorithm
// ------------------------------------------------------------------------------------------------
// checkPopulationBoundsAndReplace, Source/GeneticAlgorithm.cpp:347-365
static void o_check_bounds(double * Xpop, long long Npop, int n, const double * Xlb, const double * Xub, unsigned char * ind, OStream & st)
{
	for (long long i = 0; i < Npop; i++)
		for (int j = 0; j < n; j++)
			if (Xpop[i * n + j] > Xub[j] || Xpop[i * n + j] < Xlb[j]) {
				Xpop[i * n + j] = Xlb[j] + (Xub[j] - Xlb[j]) * st.next();
				if (ind) ind[i] = 1;
			}
}

// checkIndenticalChildAndReplace, Source/GeneticAlgorithm.cpp:313-344 (O(Npop^2) as written)
static void o_check_identical(double * Xpop, long long Npop, int n, const double * Xlb, const double * Xub, unsigned char * ind, OStream & st)
{
	for (long long i = 0; i < Npop; i++)
		for (long long k = i + 1; k < Npop; k++) {
			int Nsame = 0;
			for (int j = 0; j < n; j++) if (Xpop[i * n + j] == Xpop[k * n + j]) Nsame++;
			if (Nsame == n) {
				for (int j = 0; j < n; j++) Xpop[i * n + j] = Xlb[j] + (Xub[j] - Xlb[j]) * st.next();
				if (ind) ind[i] = 1;
			}
		}
}

// popSort, Source/GeneticAlgorithm.cpp:370-412: repeated first-minimum extraction with a 2*FMax sentinel
static void o_pop_sort(double * Xpop, double * F, long long Npop, int n)
{
	vector<double> Xt((size_t) Npop * n), Ft(Npop);
	double FMax = F[0];
	for (long long i = 1; i < Npop; i++) if (F[i] > FMax) FMax = F[i];
	for (long long k = 0; k < Npop; k++) {
		double Fmin = F[0]; long long idxMin = 0;
		for (long long i = 1; i < Npop; i++) if (F[i] < Fmin) { Fmin = F[i]; idxMin = i; }
		for (int j = 0; j < n; j++) Xt[k * n + j] = Xpop[idxMin * n + j];
		Ft[k] = F[idxMin];
		F[idxMin] = 2 * FMax;
	}
	for (long long k = 0; k < Npop; k++) {
		F[k] = Ft[k];
		for (int j = 0; j < n; j++) Xpop[k * n + j] = Xt[k * n + j];
	}
}

void oracle_ga_pop_sort(double * Xpop, double * F, long long Npop, int n) { o_pop_sort(Xpop, F, Npop, n); }

uint64_t oracle_ga_check_bounds(double * Xpop, long long Npop, int n, const double * Xlb, const double * Xub, unsigned char * ind,
                                const double * values, uint64_t n_values, uint64_t seed, double scale, uint64_t pos)
{
	OStream st = {values, n_values, seed, scale, pos, 0};
	o_check_bounds(Xpop, Npop, n, Xlb, Xub, ind, st);
	return st.pos;
}

uint64_t oracle_ga_check_identical(double * Xpop, long long Npop, int n, const double * Xlb, const double * Xub, unsigned char * ind,
                                   const double * values, uint64_t n_values, uint64_t seed, double scale, uint64_t pos)
{
	OStream st = {values, n_values, seed, scale, pos, 0};
	o_check_identical(Xpop, Npop, n, Xlb, Xub, ind, st);
	return st.pos;
}

// GeneticAlgorithmMPI::findMinBnd, Source/GeneticAlgorithmMPI.cpp:12-276, at P = 1 (evaluatePopulationParallel
// reduces to "evaluate rows whose indicator is set"). timeRand() -> the host-supplied stream.
// A trial whose index rounds to Npop (undefined behaviour in the reference, :138-140) counts as rejected.
// Outputs (all optional): Xpop_out (Npop x n sorted), F_out, per-generation parent indices of the LAST generation
// run: cross_idx (Ncross x n), mut_idx (Nrand), elite_idx (NeliteMut x n); stream_pos_out.
// Returns the number of generations completed (iter at exit), or -1 if the fractions are invalid (the reference
// calls exit(0), :40-44). stopAfter >= 0 ends the loop early with maxGenerations (hence the mutation schedule) unchanged.
// fn != NULL: the objective is fn(x, n) (a user objective compiled into the caller) instead of the built-in kind.
int oracle_ga_fn(int kind, const double * scalars, const long long * ints, const double * const * cols, long long m,
                 double (*fn)(const double *, int), double * X, const double * Xlb, const double * Xub, int Nparam, int Npop,
                 int maxGenerations, double eliteFrac, double crossFrac, double eliteMutationFrac, double mutationSize,
                 double eliteMutationSize, double NstaticGenerations, int stopAfter, const double * values, uint64_t n_values,
                 uint64_t seed, double scale, double * f0_out, double * fOpt_out, double * Xpop_out, double * F_out, int * cross_idx,
                 int * mut_idx, int * elite_idx, uint64_t * stream_pos_out)
{
	OFunctor fobj = {kind, scalars, ints, cols, m};
	auto objective = [&](const double * x) { return fn ? fn(x, Nparam) : o_scalar(fobj, x, Nparam); };
	OStream st = {values, n_values, seed, scale, 0, 0};
	size_t NN = (size_t) Npop * Nparam;
	vector<double> Xpop(NN, 0.0), XpopNew(NN, 0.0), F(Npop, 0), Fnew(Npop, 0), fitness(Npop, 0);
	vector<unsigned char> ind(Npop, 1);

	int Nelite = (int) ceil(eliteFrac * Npop);                  // :33-36
	int NeliteMut = (int) ceil(eliteMutationFrac * Npop);
	int Ncross = (int) ceil(crossFrac * Npop);
	int Nrand = Npop - Nelite - NeliteMut - Ncross;
	if (Nrand <= 0) return -1;                                  // :37-44

	for (int i = 0; i < Nparam; i++) Xpop[i] = X[i];            // :58-61
	for (int i = 1; i < Npop; i++)
		for (int j = 0; j < Nparam; j++)
			Xpop[(size_t) i * Nparam + j] = Xpop[j] + ((Xub[j] - Xlb[j]) * st.next() + Xlb[j]);   // :66
	o_check_identical(XpopNew.data(), Npop, Nparam, Xlb, Xub, ind.data(), st);                    // :71 (sic: XpopNew)
	o_check_bounds(Xpop.data(), Npop, Nparam, Xlb, Xub, ind.data(), st);                           // :74
	for (int i = 0; i < Npop; i++) if (ind[i]) F[i] = objective(&Xpop[(size_t) i * Nparam]);   // :77
	double f0 = F[0];                                           // :78
	o_pop_sort(Xpop.data(), F.data(), Npop, Nparam);            // :81

	double FbestPrev = F[0];
	int Nstatic = 0;
	int iter = 0;
	// stopAfter (test hook, not in the reference): leave the loop after that many completed generations (< 0: never)
	while (iter < maxGenerations && (stopAfter < 0 || iter < stopAfter)) {   // :87
		for (int k = 0; k < Npop; k++) fitness[k] = pow(F[Npop - 1] - F[k], 2);   // :101-104
		double maxFitness = fitness[0];
		for (int k = 0; k < Npop; k++) ind[k] = 1;
		int popIdx = 0;
		for (int k = 0; k < Nelite; k++) {                      // :109-124
			for (int i = 0; i < Nparam; i++) XpopNew[(size_t) popIdx * Nparam + i] = Xpop[(size_t) popIdx * Nparam + i];
			Fnew[popIdx] = F[popIdx];
			ind[popIdx] = 0;
			popIdx++;
		}
		for (int k = 0; k < Ncross; k++) {                      // :128-153
			vector<int> indices(Nparam, 0);
			for (int i = 0; i < Nparam; i++) {
				while (indices[i] == 0) {
					int randomIndex = (int) round(st.next() * Npop);
					double selectValue = st.next();
					if (st.exhausted) return -2;
					if (randomIndex < Npop && selectValue <= fitness[randomIndex] / maxFitness) indices[i] = randomIndex;
				}
			}
			for (int i = 0; i < Nparam; i++) {
				XpopNew[(size_t) popIdx * Nparam + i] = Xpop[(size_t) indices[i] * Nparam + i];
				if (cross_idx) cross_idx[(size_t) k * Nparam + i] = indices[i];
			}
			popIdx++;
		}
		double spreadRatio = mutationSize * (maxGenerations - iter) / maxGenerations;   // :159
		for (int k = 0; k < Nrand; k++) {                       // :164-190
			int index = 0;
			for (int j = 0; j < Nparam; j++) {
				while (index == 0) {
					int randomIndex = (int) round(st.next() * Npop);
					double selectValue = st.next();
					if (st.exhausted) return -2;
					if (randomIndex < Npop && selectValue <= fitness[randomIndex] / maxFitness) index = randomIndex;
				}
			}
			if (mut_idx) mut_idx[k] = index;
			for (int j = 0; j < Nparam; j++) {
				double mutation = spreadRatio * (Xub[j] - Xlb[j]) * st.next();
				XpopNew[(size_t) popIdx * Nparam + j] = Xpop[(size_t) index * Nparam + j] + mutation;
			}
			popIdx++;
		}
		for (int k = 0; k < NeliteMut; k++) {                   // :195-207
			for (int j = 0; j < Nparam; j++) {
				int randomEliteIdx = (int) round(st.next() * Nelite);
				double mutation = eliteMutationSize * (Xub[j] - Xlb[j]) * st.next();
				XpopNew[(size_t) popIdx * Nparam + j] = Xpop[(size_t) randomEliteIdx * Nparam + j] + mutation;
				if (elite_idx) elite_idx[(size_t) k * Nparam + j] = randomEliteIdx;
			}
			popIdx++;
		}
		o_check_identical(XpopNew.data(), Npop, Nparam, Xlb, Xub, ind.data(), st);   // :211
		o_check_bounds(XpopNew.data(), Npop, Nparam, Xlb, Xub, ind.data(), st);      // :214
		for (int i = 0; i < Npop; i++) if (ind[i]) Fnew[i] = objective(&XpopNew[(size_t) i * Nparam]);   // :217
		o_pop_sort(XpopNew.data(), Fnew.data(), Npop, Nparam);                        // :220
		for (int i = 0; i < Npop; i++) {                        // :223-230
			F[i] = Fnew[i];
			for (int j = 0; j < Nparam; j++) Xpop[(size_t) i * Nparam + j] = XpopNew[(size_t) i * Nparam + j];
		}
		double Fbest = F[0];                                    // :234-249
		if (Fbest == FbestPrev) Nstatic++; else Nstatic = 0;
		if (Nstatic > NstaticGenerations) break;
		FbestPrev = Fbest;
		iter++;
	}
	if (st.exhausted) return -2;
	if (fOpt_out) *fOpt_out = F[0];                             // :255-259
	for (int i = 0; i < Nparam; i++) X[i] = Xpop[i];
	if (f0_out) *f0_out = f0;
	if (Xpop_out) memcpy(Xpop_out, Xpop.data(), NN * sizeof(double));
	if (F_out) memcpy(F_out, F.data(), (size_t) Npop * sizeof(double));
	if (stream_pos_out) *stream_pos_out = st.pos;
	return iter;
}

int oracle_ga(int kind, const double * scalars, const long long * ints, const double * const * cols, long long m,
              double * X, const double * Xlb, const double * Xub, int Nparam, int Npop, int maxGenerations, double eliteFrac,
              double crossFrac, double eliteMutationFrac, double mutationSize, double eliteMutationSize,
              double NstaticGenerations, int stopAfter, const double * values, uint64_t n_values, uint64_t seed, double scale,
              double * f0_out, double * fOpt_out, double * Xpop_out, double * F_out, int * cross_idx, int * mut_idx,
              int * elite_idx, uint64_t * stream_pos_out)
{
	return oracle_ga_fn(kind, scalars, ints, cols, m, nullptr, X, Xlb, Xub, Nparam, Npop, maxGenerations, eliteFrac, crossFrac,
	                    eliteMutationFrac, mutationSize, eliteMutationSize, NstaticGenerations, stopAfter, values, n_values, seed, scale,
	                    f0_out, fOpt_out, Xpop_out, F_out, cross_idx, mut_idx, elite_idx, stream_pos_out);
}

} // extern "C"
