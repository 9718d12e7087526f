/* Scalar objectives with hand-written analytic gradients (pnol_gradient), defined OUTSIDE the library
 * (tests/test_user_gradient_cpu.py, tests/test_gpu_analytic_gradient.py; INTEGRATION.md section A). Their kinds are new: registering
 * MY_F_TRID or MY_F_STYBLINSKI again would replace my_objectives' tables. */
#ifndef MY_GRADIENTS_HPP_
#define MY_GRADIENTS_HPP_

#include "pnol/functors.hpp"
#include "my_objectives.hpp"

enum {
	MYG_F_TRID = PNOL_F_USER_SCALAR_BASE + 201,          /* Trid (neighbours coupled), with partial */
	MYG_F_STYBLINSKI = PNOL_F_USER_SCALAR_BASE + 202     /* Styblinski-Tang with a user scale (separable), with partial */
};

/* f = sum_i (x_i - 1)^2 - sum_{i >= 1} x_i x_{i-1}:  df/dx_j = 2 (x_j - 1) - [j >= 1] x_{j-1} - [j <= n-2] x_{j+1}, in this order */
struct MyTridFunctor {
	static constexpr int kKind = MYG_F_TRID;
	template <class Acc> PNOL_HD static double eval(const pnol::FunctorParams & P, const Acc & X, int n) { return TridFunctor::eval(P, X, n); }
	template <class Acc> PNOL_HD static double partial(const pnol::FunctorParams &, const Acc & X, int n, int j)
	{
		double g = 2.0 * (X[j] - 1.0);
		if (j >= 1) g = g - X[j - 1];
		if (j <= n - 2) g = g - X[j + 1];
		return g;
	}
};

/* f = s sum_i (x_i^4 - 16 x_i^2 + 5 x_i), scalars[0] = s:  df/dx_j = s (4 (x2 x) - 32 x + 5) with x = x_j, x2 = x * x */
struct MyStyblinskiFunctor {
	static constexpr int kKind = MYG_F_STYBLINSKI;
	static constexpr bool kSeparable = true;
	PNOL_HD static double sep_init(const pnol::FunctorParams & P, int n) { return StyblinskiFunctor::sep_init(P, n); }
	PNOL_HD static double sep_term(const pnol::FunctorParams & P, double x) { return StyblinskiFunctor::sep_term(P, x); }
	template <class Acc> PNOL_HD static double eval(const pnol::FunctorParams & P, const Acc & X, int n)
	{
		return StyblinskiFunctor::eval(P, X, n);
	}
	template <class Acc> PNOL_HD static double partial(const pnol::FunctorParams & P, const Acc & X, int, int j)
	{
		const double x = X[j];
		const double x2 = x * x;
		return P.scalars[0] * (4.0 * (x2 * x) - 32.0 * x + 5.0);
	}
};

#endif
