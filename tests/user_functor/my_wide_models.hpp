/* A residual model of any width n with O(1) work per row, defined OUTSIDE the library (tests/test_gpu_functor_kernels_exact.py):
 * it lets the forward-difference and analytic Jacobian kernels of include/pnol/device/functor_kernels.cuh run at every n up to their
 * shared-memory limits while the m x n stencils stay cheap on the host. */
#ifndef MY_WIDE_MODELS_HPP_
#define MY_WIDE_MODELS_HPP_

#include "pnol/functors.hpp"

enum {
	MYW_F_WIDE = PNOL_F_USER_RESIDUAL_BASE + 201      /* two columns per row, with jacobian */
};

/* Row i touches columns a = i mod n and b = (7 i + 3) mod n (a == b happens):
 *   r_i = y_i - (x_a t_i + (x_b x_b) s_i),   columns {t, s, y}
 *   dr/dx_a = -t_i,  dr/dx_b = -((x_b + x_b) s_i),  their sum when a == b,  every other entry 0 */
struct MyWideFunctor {
	static constexpr int kKind = MYW_F_WIDE;
	PNOL_HD static int col_a(long long i, int n) { return (int) (i % n); }
	PNOL_HD static int col_b(long long i, int n) { return (int) ((7 * i + 3) % n); }
	template <class Acc> PNOL_HD static double residual(const pnol::FunctorParams & P, const Acc & X, int n, long long i)
	{
		const double xa = X[col_a(i, n)], xb = X[col_b(i, n)];
		return P.col[2][i] - (xa * P.col[0][i] + (xb * xb) * P.col[1][i]);
	}
	template <class Acc> PNOL_HD static void jacobian(const pnol::FunctorParams & P, const Acc & X, int n, long long i, double * Ji)
	{
		const int a = col_a(i, n), b = col_b(i, n);
		const double xb = X[b];
		const double ja = -P.col[0][i], jb = -((xb + xb) * P.col[1][i]);
		for (int j = 0; j < n; j++) Ji[j] = 0.0;
		if (a == b) {
			Ji[a] = ja + jb;
		} else {
			Ji[a] = ja;
			Ji[b] = jb;
		}
	}
};

#endif
