/* Scalar objectives with hand-written analytic Hessians (pnol_hessian), defined OUTSIDE the library (tests/test_user_hessian_cpu.py,
 * tests/test_gpu_analytic_hessian.py; INTEGRATION.md section A). Their kinds are new: registering a kind of my_objectives or
 * my_gradients again would replace that kind's table. */
#ifndef MY_HESSIANS_HPP_
#define MY_HESSIANS_HPP_

#include "pnol/functors.hpp"
#include "my_objectives.hpp"

enum {
	MYH_F_QUADFORM = PNOL_F_USER_SCALAR_BASE + 301,      /* dense quadratic form, A one data column of length n * n, with partial2 */
	MYH_F_STYBLINSKI = PNOL_F_USER_SCALAR_BASE + 302     /* Styblinski-Tang with a user scale (separable), with partial2 */
};

/* f = 1/2 sum_i sum_j A_ij x_i x_j, A row-major in col[0] (m = n * n, not necessarily symmetric): the sum ((A_ij x_i) x_j) taken row by
 * row, then halved. d2f / dx_i dx_j = 0.5 * (A[i n + j] + A[j n + i]), in this order: a dense Hessian that reads A at (i, j) and at
 * (j, i) */
struct MyQuadFormFunctor {
	static constexpr int kKind = MYH_F_QUADFORM;
	template <class Acc> PNOL_HD static double eval(const pnol::FunctorParams & P, const Acc & X, int n)
	{
		const double * A = P.col[0];
		double v = 0;
		for (int i = 0; i < n; i++) {
			const double xi = X[i];
			for (int j = 0; j < n; j++) v = v + (A[(long long) i * n + j] * xi) * X[j];
		}
		return 0.5 * v;
	}
	template <class Acc> PNOL_HD static double partial2(const pnol::FunctorParams & P, const Acc &, int n, int i, int j)
	{
		const double * A = P.col[0];
		return 0.5 * (A[(long long) i * n + j] + A[(long long) j * n + i]);
	}
};

/* f = s sum_i (x_i^4 - 16 x_i^2 + 5 x_i), scalars[0] = s:  d2f / dx_j^2 = s (12 (x x) - 32) with x = x_j, in this order; 0 off the
 * diagonal */
struct MyHessStyblinskiFunctor {
	static constexpr int kKind = MYH_F_STYBLINSKI;
	static constexpr bool kSeparable = true;
	PNOL_HD static double sep_init(const pnol::FunctorParams & P, int n) { return StyblinskiFunctor::sep_init(P, n); }
	PNOL_HD static double sep_term(const pnol::FunctorParams & P, double x) { return StyblinskiFunctor::sep_term(P, x); }
	template <class Acc> PNOL_HD static double eval(const pnol::FunctorParams & P, const Acc & X, int n)
	{
		return StyblinskiFunctor::eval(P, X, n);
	}
	template <class Acc> PNOL_HD static double partial2(const pnol::FunctorParams & P, const Acc & X, int, int i, int j)
	{
		if (i != j) return 0.0;
		const double x = X[j];
		return P.scalars[0] * (12.0 * (x * x) - 32.0);
	}
};

#endif
