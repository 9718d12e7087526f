/* Residual models with hand-written analytic Jacobians (PNOL_JAC_ANALYTIC), defined OUTSIDE the library
 * (tests/test_user_jacobian_cpu.py, tests/test_gpu_analytic_jacobian.py; INTEGRATION.md section A). */
#ifndef MY_JACOBIANS_HPP_
#define MY_JACOBIANS_HPP_

#include "pnol/functors.hpp"

enum {
	MYJ_F_LORENTZ = PNOL_F_USER_RESIDUAL_BASE + 101,      /* user copy of the sum of Lorentzians, with jacobian */
	MYJ_F_GAUSS = PNOL_F_USER_RESIDUAL_BASE + 102,        /* Gaussian peak, with jacobian */
	MYJ_F_GAUSS_V1 = PNOL_F_USER_RESIDUAL_BASE + 103,     /* the Gaussian peak registered through a version-1 table */
	MYJ_F_GAUSS_NOJAC = PNOL_F_USER_RESIDUAL_BASE + 104   /* the Gaussian peak without jacobian (version-2 table) */
};

/* r_i = y_i - tree-sum_k a_k / (1 + w (t_i - c_k)^2): the library's model, its residual taken as is, its derivative written here on
 * the public per-term helper lorentz_term_grad. scalars[0] = w, columns {t, y}. */
struct MyLorentzFunctor {
	static constexpr int kKind = MYJ_F_LORENTZ;
	template <class Acc> PNOL_HD static double residual(const pnol::FunctorParams & P, const Acc & X, int n, long long i)
	{
		return pnol::LorentzSumFunctor::residual(P, X, n, i);
	}
	template <class Acc> PNOL_HD static void jacobian(const pnol::FunctorParams & P, const Acc & X, int n, long long i, double * Ji)
	{
		const double w = P.scalars[0], t = P.col[0][i];
		for (int k = 0; k < n / 2; k++) pnol::lorentz_term_grad(X[2 * k], X[2 * k + 1], w, t, Ji[2 * k], Ji[2 * k + 1]);
	}
};

/* Gaussian peak r_i = y_i - (A e + c0), e = exp(-(d*d) s), d = t_i - mu, x = (A, mu, s), scalars[0] = c0, columns {t, y}:
 *   dr/dA = -e,   dr/dmu = -((A e) ((s + s) d)),   dr/ds = (A e) (d*d) */
struct MyGaussFunctor {
	static constexpr int kKind = MYJ_F_GAUSS;
	template <class Acc> PNOL_HD static double residual(const pnol::FunctorParams & P, const Acc & X, int, long long i)
	{
		const double d = P.col[0][i] - X[1];
		const double model = X[0] * pnol::exp_hd(-(d * d) * X[2]) + P.scalars[0];
		return P.col[1][i] - model;
	}
	template <class Acc> PNOL_HD static void jacobian(const pnol::FunctorParams & P, const Acc & X, int, long long i, double * Ji)
	{
		const double d = P.col[0][i] - X[1];
		const double e = pnol::exp_hd(-(d * d) * X[2]);
		const double ae = X[0] * e;
		Ji[0] = -e;
		Ji[1] = -(ae * ((X[2] + X[2]) * d));
		Ji[2] = ae * (d * d);
	}
};

/* the same model without a derivative: PNOL_JAC_ANALYTIC is refused for it */
struct MyGaussNoJacFunctor {
	static constexpr int kKind = MYJ_F_GAUSS_NOJAC;
	template <class Acc> PNOL_HD static double residual(const pnol::FunctorParams & P, const Acc & X, int n, long long i)
	{
		return MyGaussFunctor::residual(P, X, n, i);
	}
};

#endif
