/* This Source Code Form is subject to the terms of the Mozilla Public License, v. 2.0 (LICENSE at the repository root).
 * It mirrors the interface / host control flow of briandaniel/ParallelNonlinearOptimizationLibrary (MPL-2.0); see NOTICE. */
/*
 * functors.hpp -- device functors: ONE __host__ __device__ definition per objective.
 *
 * A functor is the device twin of a PNOL Objective / MultiObjective (Source/PNOL_Objective.hpp:25-62 of
 * the reference). The same source is used by
 *   - the CUDA kernels (one perturbed point per thread; the point is seen through an accessor so the base
 *     point can sit in shared memory while a single coordinate is perturbed in a register), and
 *   - the host objEval of the matching C++ plugin class (include/pnol/ExampleObjectives.hpp),
 * so that host and device agree bit for bit (compiled with -fmad=false / -ffp-contract=off).
 *
 * Scalar functor concept:
 *     struct F { static constexpr int kKind;  template<class Acc> static double eval(const FunctorParams&, const Acc& X, int n); };
 * Residual functor concept (row i of the residual vector, data columns in FunctorParams::col):
 *     struct R { static constexpr int kKind;  template<class Acc> static double residual(const FunctorParams&, const Acc& X, int n, long long i); };
 * Acc needs only `double operator[](int) const`.
 * Batch contract (pnol_lm_batch, which fits many problems whose rows lie back to back in one functor): residual row i reads only row i
 * of each data column and does not use P.m. All three built-in models below keep it.
 * A residual functor MAY also define its analytic Jacobian row (PNOL_JAC_ANALYTIC; detected by has_jacobian below):
 *     template<class Acc> static void jacobian(const FunctorParams&, const Acc& X, int n, long long i, double * Ji);
 * which writes all n entries Ji[j] = d r_i / d x_j. That one definition is the specification: the kernels (the generic template of
 * device/functor_kernels.cuh and any specialised kernel of a built-in model) return its bits, host and device alike.
 * A scalar functor MAY likewise define one partial derivative per coordinate (pnol_gradient; detected by has_partial below):
 *     template<class Acc> static double partial(const FunctorParams&, const Acc& X, int n, int j);      // d f / d x_j
 * gradient_kernel (device/functor_kernels.cuh) runs one coordinate per thread and returns its bits. Every built-in scalar objective
 * defines one; each states its operation order, which the tests restate.
 * And one second derivative per pair (pnol_hessian; detected by has_partial2 below):
 *     template<class Acc> static double partial2(const FunctorParams&, const Acc& X, int n, int i, int j);   // d2 f / dx_i dx_j
 * It is only ever called with i <= j: hessian_kernel (device/functor_kernels.cuh) evaluates each unordered pair once and mirrors it,
 * so H[j][i] has the bits of H[i][j] by construction. Every built-in scalar objective defines one; each states its operation order.
 */
#ifndef PNOL_FUNCTORS_HPP_
#define PNOL_FUNCTORS_HPP_

#include "pnol_math.h"
#include "../pnol_b200.h"

namespace pnol {

/* parameters of a functor as the kernels see them (POD, passed by value as a kernel argument): scalars[PNOL_MAX_SCALARS],
 * ints[PNOL_MAX_INTS], col[PNOL_MAX_COLUMNS] (data columns; device pointers on the device side), m -- the C struct of pnol_b200.h */
typedef pnol_functor_params FunctorParams;

/* ---- accessors ---- */
struct PtrAcc {                      /* plain array */
	const double * p;
	PNOL_HD double operator[](int j) const { return p[j]; }
};
struct PerturbAcc {                  /* base point with ONE coordinate replaced (forward-difference stencil) */
	const double * base; int i; double xi;
	PNOL_HD double operator[](int j) const { return j == i ? xi : base[j]; }
};
struct Perturb2Acc {                 /* base point with TWO coordinates replaced (FD Hessian) */
	const double * base; int i; double xi; int j2; double xj;
	PNOL_HD double operator[](int j) const { return j == i ? xi : (j == j2 ? xj : base[j]); }
};

/* ---- scalar objectives ---- */

/* Source/ExampleObjectives.hpp:87-103: sum_k 100 (x_{k+1} - x_k^2)^2 + (1 - x_k)^2, sequential sum.
 * pow(.,2) is written as a product: GCC folds the literal pow(x,2) to x*x at -O2 (SURVEY.md 7.1). */
struct RosenbrockFunctor {
	static constexpr int kKind = PNOL_F_ROSENBROCK;
	template <class Acc> PNOL_HD static double eval(const FunctorParams &, const Acc & X, int n)
	{
		double value = 0;
		double xk = X[0];
		for (int k = 0; k < n - 1; k++) {
			double xk1 = X[k + 1];
			double a = xk1 - xk * xk;
			double b = 1 - xk;
			value = value + (100.0 * (a * a) + b * b);
			xk = xk1;
		}
		return value;
	}
	/* [j >= 1] 200 (x_j - x_{j-1}^2)  +  [j <= n-2] (-400 x_j (x_{j+1} - x_j^2) - 2 (1 - x_j)), in this order; a term whose condition
	 * fails is left out (not added as 0), so n = 1 gives 0 */
	template <class Acc> PNOL_HD static double partial(const FunctorParams &, const Acc & X, int n, int j)
	{
		const double xj = X[j];
		double a = 0.0, b = 0.0;
		if (j >= 1) {
			const double xp = X[j - 1];
			a = 200.0 * (xj - xp * xp);
		}
		if (j <= n - 2) {
			const double xn = X[j + 1];
			b = -400.0 * xj * (xn - xj * xj) - 2.0 * (1 - xj);
		}
		if (j >= 1 && j <= n - 2) return a + b;
		return j >= 1 ? a : b;
	}
	/* H_jj = [j >= 1] 200  +  [j <= n-2] (1200 (x_j x_j) - 400 x_{j+1} + 2), in this order, a term whose condition fails left out (n = 1
	 * gives 0); H_{j,j+1} = -400 x_j; every other entry 0 */
	template <class Acc> PNOL_HD static double partial2(const FunctorParams &, const Acc & X, int n, int i, int j)
	{
		if (j == i + 1) return -400.0 * X[i];
		if (j != i) return 0.0;
		double b = 0.0;
		if (j <= n - 2) {
			const double xj = X[j], xn = X[j + 1];
			b = 1200.0 * (xj * xj) - 400.0 * xn + 2.0;
		}
		if (j >= 1 && j <= n - 2) return 200.0 + b;
		return j >= 1 ? 200.0 : b;
	}
};

/* Source/ExampleObjectives.hpp:214-224 with the runtime pow(X[k], power) replaced by repeated
 * multiplication ((x*x)*x...): libm pow is not reproducible on the device (SURVEY.md 7.1). */
struct PowerFunctor {
	static constexpr int kKind = PNOL_F_POWER;
	/* separable: f = init + term(x_0) + term(x_1) + ... summed in index order (see the note above RastriginFunctor) */
	static constexpr bool kSeparable = true;
	PNOL_HD static double sep_init(const FunctorParams &, int) { return 0.0; }
	PNOL_HD static double sep_term(const FunctorParams & P, double x)
	{
		int power = (int) P.ints[0];
		double v = 1.0;
		for (int q = 0; q < power; q++) v = v * x;
		return v;
	}
	template <class Acc> PNOL_HD static double eval(const FunctorParams & P, const Acc & X, int n)
	{
		double value = sep_init(P, n);
		for (int k = 0; k < n; k++) value = value + sep_term(P, X[k]);
		return value;
	}
	/* p x^(p-1): v = x^(p-1) by the same repeated multiplication ((x*x)*x...), then p * v; 0 for p <= 0 (f is then the constant n) */
	template <class Acc> PNOL_HD static double partial(const FunctorParams & P, const Acc & X, int, int j)
	{
		const int power = (int) P.ints[0];
		if (power <= 0) return 0.0;
		const double x = X[j];
		double v = 1.0;
		for (int q = 0; q < power - 1; q++) v = v * x;
		return (double) power * v;
	}
	/* diagonal p (p-1) x^(p-2): v = x^(p-2) by the same repeated multiplication, then (double) (p (p-1)) * v; 0 for p <= 1 and off the
	 * diagonal */
	template <class Acc> PNOL_HD static double partial2(const FunctorParams & P, const Acc & X, int, int i, int j)
	{
		const int power = (int) P.ints[0];
		if (i != j || power <= 1) return 0.0;
		const double x = X[j];
		double v = 1.0;
		for (int q = 0; q < power - 2; q++) v = v * x;
		return (double) (power * (power - 1)) * v;
	}
};

/* Source/ExampleObjectives.hpp:58-69 */
struct BoothFunctor {
	static constexpr int kKind = PNOL_F_BOOTH;
	template <class Acc> PNOL_HD static double eval(const FunctorParams &, const Acc & X, int)
	{
		double x = X[0], y = X[1];
		double a = x + 2 * y - 7;
		double b = 2 * x + y - 5;
		return a * a + b * b;
	}
	/* a, b as in eval: d/dx = 2 a + 4 b, d/dy = 4 a + 2 b; 0 for j >= 2 */
	template <class Acc> PNOL_HD static double partial(const FunctorParams &, const Acc & X, int, int j)
	{
		if (j >= 2) return 0.0;
		double x = X[0], y = X[1];
		double a = x + 2 * y - 7;
		double b = 2 * x + y - 5;
		return j == 0 ? 2 * a + 4 * b : 4 * a + 2 * b;
	}
	/* the constant [[10, 8], [8, 10]]; 0 when i or j >= 2 */
	template <class Acc> PNOL_HD static double partial2(const FunctorParams &, const Acc &, int, int i, int j)
	{
		if (i >= 2 || j >= 2) return 0.0;
		return i == j ? 10.0 : 8.0;
	}
};

/* Source/ExampleObjectives.hpp:27-39 */
struct GoldsteinFunctor {
	static constexpr int kKind = PNOL_F_GOLDSTEIN;
	template <class Acc> PNOL_HD static double eval(const FunctorParams &, const Acc & X, int)
	{
		double x = X[0], y = X[1];
		double s = x + y + 1;
		double d = 2 * x - 3 * y;
		return (1 + (s * s) * (19 - 14 * x + 3 * (x * x) - 14 * y + 6 * x * y + 3 * (y * y))) *
		       (30 + (d * d) * (18 - 32 * x + 12 * (x * x) + 48 * y - 36 * x * y + 27 * (y * y)));
	}
	/* product rule on f = A B, A = 1 + s^2 U, B = 30 + d^2 V (U, V the two polynomials of eval, in eval's order):
	 *   dA = (2 s) U + s^2 (-14 + 6 x + 6 y)                 (the same for x and y)
	 *   dB = (4 d) V + d^2 (-32 + 24 x - 36 y)     for x,    (-6 d) V + d^2 (48 - 36 x + 54 y)   for y
	 *   df = dA B + A dB;  0 for j >= 2 */
	template <class Acc> PNOL_HD static double partial(const FunctorParams &, const Acc & X, int, int j)
	{
		if (j >= 2) return 0.0;
		double x = X[0], y = X[1];
		double s = x + y + 1;
		double d = 2 * x - 3 * y;
		double U = 19 - 14 * x + 3 * (x * x) - 14 * y + 6 * x * y + 3 * (y * y);
		double V = 18 - 32 * x + 12 * (x * x) + 48 * y - 36 * x * y + 27 * (y * y);
		double s2 = s * s, d2 = d * d;
		double A = 1 + s2 * U, B = 30 + d2 * V;
		double dA = (2 * s) * U + s2 * (-14 + 6 * x + 6 * y);
		double dB = j == 0 ? (4 * d) * V + d2 * (-32 + 24 * x - 36 * y) : (-6 * d) * V + d2 * (48 - 36 * x + 54 * y);
		return dA * B + A * dB;
	}
	/* product rule on f = A B:  f_ij = A_ij B + A_i B_j + A_j B_i + A B_ij, in this order, with partial()'s names and order for s, d, U, V,
	 * A, B, dA (= A_x = A_y) and dB (B_x, B_y), and Ux = -14 + 6 x + 6 y, Vx = -32 + 24 x - 36 y, Vy = 48 - 36 x + 54 y:
	 *   A_ij = 2 U + (4 s) Ux + 6 s2                                   (the same for every pair: U_xx = U_xy = U_yy = 6)
	 *   B_xx = 8 V + (8 d) Vx + 24 d2,   B_xy = -12 V + (4 d) Vy - (6 d) Vx - 36 d2,   B_yy = 18 V - (12 d) Vy + 54 d2
	 * 0 when i or j >= 2 */
	template <class Acc> PNOL_HD static double partial2(const FunctorParams &, const Acc & X, int, int i, int j)
	{
		if (i >= 2 || j >= 2) return 0.0;
		double x = X[0], y = X[1];
		double s = x + y + 1;
		double d = 2 * x - 3 * y;
		double U = 19 - 14 * x + 3 * (x * x) - 14 * y + 6 * x * y + 3 * (y * y);
		double V = 18 - 32 * x + 12 * (x * x) + 48 * y - 36 * x * y + 27 * (y * y);
		double s2 = s * s, d2 = d * d;
		double A = 1 + s2 * U, B = 30 + d2 * V;
		double Ux = -14 + 6 * x + 6 * y;
		double Vx = -32 + 24 * x - 36 * y, Vy = 48 - 36 * x + 54 * y;
		double dA = (2 * s) * U + s2 * Ux;
		double Bx = (4 * d) * V + d2 * Vx, By = (-6 * d) * V + d2 * Vy;
		double A2 = 2 * U + (4 * s) * Ux + 6 * s2;
		double Bi = i == 0 ? Bx : By, Bj = j == 0 ? Bx : By;
		double B2 = i != j ? -12 * V + (4 * d) * Vy - (6 * d) * Vx - 36 * d2 : (i == 0 ? 8 * V + (8 * d) * Vx + 24 * d2 : 18 * V - (12 * d) * Vy + 54 * d2);
		return A2 * B + dA * Bj + dA * Bi + A * B2;
	}
};

/* ours (BASELINE.json config 4): f = 10 n + sum_k (x_k^2 - 10 cos(2 pi x_k)), sequential sum.
 * A functor may declare itself SEPARABLE (kSeparable, sep_init, sep_term): f = init + term(x_0) + term(x_1) + ... with the sum
 * taken in index order. The population sweep then computes the terms one gene per LANE straight from coalesced loads and
 * only the (cheap, order-preserving) summation one individual per lane -- same bits as eval(), which is defined through the
 * same two functions. */
struct RastriginFunctor {
	static constexpr int kKind = PNOL_F_RASTRIGIN;
	static constexpr bool kSeparable = true;
	PNOL_HD static double sep_init(const FunctorParams &, int n) { return 10.0 * n; }
	PNOL_HD static double sep_term(const FunctorParams &, double x) { return x * x - 10.0 * cos2pi(x); }
	template <class Acc> PNOL_HD static double eval(const FunctorParams & P, const Acc & X, int n)
	{
		double value = sep_init(P, n);
		PNOL_UNROLL(4)
		for (int k = 0; k < n; k++) value = value + sep_term(P, X[k]);
		return value;
	}
	/* 2 x + 20 pi sin(2 pi x), as 2 * x + RN(20 pi) * sin2pi(x) (pnol_math.h) */
	template <class Acc> PNOL_HD static double partial(const FunctorParams &, const Acc & X, int, int j)
	{
		const double x = X[j];
		return 2 * x + 62.83185307179586 * sin2pi(x);
	}
	/* diagonal 2 + 40 pi^2 cos(2 pi x), as 2 + RN(40 pi^2) * cos2pi(x) (pnol_math.h); 0 off the diagonal */
	template <class Acc> PNOL_HD static double partial2(const FunctorParams &, const Acc & X, int, int i, int j)
	{
		if (i != j) return 0.0;
		return 2 + 394.78417604357435 * cos2pi(X[j]);
	}
};

/* Source/ExampleObjectives.hpp:287-298 with exp -> exp_hd; columns {x, y} */
struct ExpCurveSingleFunctor {
	static constexpr int kKind = PNOL_F_EXPCURVE_SINGLE;
	template <class Acc> PNOL_HD static double eval(const FunctorParams & P, const Acc & X, int)
	{
		double Fnorm = 0;
		double x0 = X[0], x1 = X[1], x2 = X[2];
		for (long long k = 0; k < P.m; k++) {
			double func = x0 * exp_hd(x1 * P.col[0][k]) + x2;
			double d = P.col[1][k] - func;
			Fnorm = Fnorm + d * d;
		}
		return Fnorm;
	}
	/* with e, func, d as in eval and c = -(d + d): the terms c e (x0), c ((x0 e) t) (x1), c (x2), summed sequentially in row order
	 * from 0; 0 for j >= 3 */
	template <class Acc> PNOL_HD static double partial(const FunctorParams & P, const Acc & X, int, int j)
	{
		if (j >= 3) return 0.0;
		double g = 0;
		double x0 = X[0], x1 = X[1], x2 = X[2];
		for (long long k = 0; k < P.m; k++) {
			double t = P.col[0][k];
			double e = exp_hd(x1 * t);
			double func = x0 * e + x2;
			double d = P.col[1][k] - func;
			double c = -(d + d);
			double term = j == 0 ? c * e : (j == 1 ? c * ((x0 * e) * t) : c);
			g = g + term;
		}
		return g;
	}
	/* with e, func, d as in eval: the terms 2 (g_i g_j) - (2 d) h_ij, summed sequentially in row order from 0, where g = (e, (x0 e) t, 1)
	 * is the derivative of func and h its second derivative: h_01 = e t, h_11 = ((x0 e) t) t, every other h_ij = 0 (still multiplied
	 * and subtracted); 0 when i or j >= 3 */
	template <class Acc> PNOL_HD static double partial2(const FunctorParams & P, const Acc & X, int, int i, int j)
	{
		if (i >= 3 || j >= 3) return 0.0;
		double H = 0;
		double x0 = X[0], x1 = X[1], x2 = X[2];
		for (long long k = 0; k < P.m; k++) {
			double t = P.col[0][k];
			double e = exp_hd(x1 * t);
			double func = x0 * e + x2;
			double d = P.col[1][k] - func;
			double g1 = (x0 * e) * t;
			double gi = i == 0 ? e : (i == 1 ? g1 : 1.0);
			double gj = j == 0 ? e : (j == 1 ? g1 : 1.0);
			double h = i == 0 && j == 1 ? e * t : (i == 1 && j == 1 ? g1 * t : 0.0);
			double term = 2.0 * (gi * gj) - (2.0 * d) * h;
			H = H + term;
		}
		return H;
	}
};

/* ---- residual models ---- */

/* Source/ExampleObjectives.hpp:123-132 with exp -> exp_hd; columns {x, y} */
struct ExpCurveFunctor {
	static constexpr int kKind = PNOL_F_EXPCURVE;
	template <class Acc> PNOL_HD static double residual(const FunctorParams & P, const Acc & X, int, long long i)
	{
		double func = X[0] * exp_hd(X[1] * P.col[0][i]) + X[2];
		return P.col[1][i] - func;
	}
	/* r = y - (x0 e + x2), e = exp(x1 t):  dr/dx0 = -e, dr/dx1 = -((x0 e) t), dr/dx2 = -1 */
	template <class Acc> PNOL_HD static void jacobian(const FunctorParams & P, const Acc & X, int, long long i, double * Ji)
	{
		const double t = P.col[0][i];
		const double e = exp_hd(X[1] * t);
		Ji[0] = -e;
		Ji[1] = -((X[0] * e) * t);
		Ji[2] = -1.0;
	}
};

/* Source/ExampleObjectives.hpp:170-179; columns {x^3 computed by the host's pow(x,3), x, y}; pow(x,2) -> x*x */
struct CubicFunctor {
	static constexpr int kKind = PNOL_F_CUBIC;
	template <class Acc> PNOL_HD static double residual(const FunctorParams & P, const Acc & X, int, long long i)
	{
		double x3 = P.col[0][i], x = P.col[1][i];
		double func = X[0] * x3 + X[1] * (x * x) + X[2] * x + X[3];
		return P.col[2][i] - func;
	}
	/* dr/dx = -(x^3, x*x, x, 1) */
	template <class Acc> PNOL_HD static void jacobian(const FunctorParams & P, const Acc &, int, long long i, double * Ji)
	{
		const double x3 = P.col[0][i], x = P.col[1][i];
		Ji[0] = -x3;
		Ji[1] = -(x * x);
		Ji[2] = -x;
		Ji[3] = -1.0;
	}
};

/* ours (BASELINE.json configs 2 and 5): r_i = y_i - S_i,  S_i = balanced-tree sum over k < K of
 *   term_k = a_k / (1 + w (t_i - c_k)^2),   x = (a_0, c_0, a_1, c_1, ...), n = 2K, K a power of two.
 * The tree is the adjacent-pairs tree: level l sums nodes 2j and 2j+1 of level l-1. A single-parameter
 * perturbation changes one leaf, hence only log2 K nodes: the structured Jacobian kernel exploits that and
 * returns the same bits as n+1 black-box evaluations of this function. */
PNOL_HD double lorentz_term(double a, double c, double w, double t)
{
	double d = t - c;
	double q = d * d;
	double e = w * q;
	double den = 1.0 + e;
	return a / den;
}

/* Derivatives of one term of the residual r = y - S: ja = dr/da = -1/den, jc = dr/dc = -2 a w (t - c) / den^2, in this operation
 * order (the first four operations are lorentz_term's). Every kernel and test of the analytic Jacobian follows it. */
PNOL_HD void lorentz_term_grad(double a, double c, double w, double t, double & ja, double & jc)
{
	double d = t - c;
	double q = d * d;
	double e = w * q;
	double den = 1.0 + e;
	double u = 1.0 / den;
	ja = -u;
	jc = -((a * u) * u * ((w + w) * d));
}

struct LorentzSumFunctor {
	static constexpr int kKind = PNOL_F_LORENTZ_SUM;
	static constexpr int kMaxLog2K = 12;
	template <class Acc> PNOL_HD static double residual(const FunctorParams & P, const Acc & X, int n, long long i)
	{
		double w = P.scalars[0];
		double t = P.col[0][i];
		int K = n / 2;
		/* adjacent-pairs tree evaluated as a binary counter: stack[l] holds a finished subtree of 2^l leaves */
		double stack[kMaxLog2K + 1];
		for (int k = 0; k < K; k++) {
			double v = lorentz_term(X[2 * k], X[2 * k + 1], w, t);
			int l = 0;
			int kk = k;
			while (kk & 1) { v = stack[l] + v; kk >>= 1; l++; }
			stack[l] = v;
		}
		int top = 0;
		while ((1 << top) < K) top++;
		return P.col[1][i] - stack[top];
	}
	/* the terms are independent: Ji = (ja_0, jc_0, ja_1, jc_1, ...), no tree */
	template <class Acc> PNOL_HD static void jacobian(const FunctorParams & P, const Acc & X, int n, long long i, double * Ji)
	{
		const double w = P.scalars[0];
		const double t = P.col[0][i];
		for (int k = 0; k < n / 2; k++) lorentz_term_grad(X[2 * k], X[2 * k + 1], w, t, Ji[2 * k], Ji[2 * k + 1]);
	}
};

/* has_jacobian<R>::value: R defines the analytic Jacobian row of the concept above */
template <class R> struct has_jacobian {
	template <class T>
	static constexpr bool test(decltype(&T::template jacobian<PtrAcc>)) { return true; }
	template <class T> static constexpr bool test(...) { return false; }
	static constexpr bool value = test<R>(nullptr);
};

/* has_partial<F>::value: F defines the per-coordinate analytic gradient of the concept above */
template <class F> struct has_partial {
	template <class T>
	static constexpr bool test(decltype(&T::template partial<PtrAcc>)) { return true; }
	template <class T> static constexpr bool test(...) { return false; }
	static constexpr bool value = test<F>(nullptr);
};

/* has_partial2<F>::value: F defines the per-pair analytic Hessian of the concept above */
template <class F> struct has_partial2 {
	template <class T>
	static constexpr bool test(decltype(&T::template partial2<PtrAcc>)) { return true; }
	template <class T> static constexpr bool test(...) { return false; }
	static constexpr bool value = test<F>(nullptr);
};

} // namespace pnol

#endif /* PNOL_FUNCTORS_HPP_ */
