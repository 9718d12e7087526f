/* Four objectives for the batched simplex tests (tests/test_gpu_simplex_batch.py), written to the functor concept of
 * include/pnol/functors.hpp, each steering simplexSort into one of its quirks. my_simplex_objectives.cu registers them with the library
 * (compiled out of tree, as my_objectives.cu is) and the CPU stand-in (tests/host_logic_standin.cpp) includes this header for
 * its oracle, so the host and device definitions are the same source. */
#ifndef MY_SIMPLEX_OBJECTIVES_HPP_
#define MY_SIMPLEX_OBJECTIVES_HPP_

#include <math.h>

#include "pnol/functors.hpp"

enum {
	MYS_F_NEGATIVE = PNOL_F_USER_SCALAR_BASE + 401,
	MYS_F_QUANTIZED = PNOL_F_USER_SCALAR_BASE + 402,
	MYS_F_SIGNED_ZERO = PNOL_F_USER_SCALAR_BASE + 403,
	MYS_F_NAN_REGION = PNOL_F_USER_SCALAR_BASE + 404
};

/* f = -1 / (1 + |x|^2): negative everywhere, so the largest f is never positive and every sort is outside simplexSort's regime (its
 * sentinel 2 max f lies BELOW the entries: vertices get taken twice) */
struct SimplexNegativeFunctor {
	template <class Acc> PNOL_HD static double eval(const pnol::FunctorParams &, const Acc & X, int n)
	{
		double s = 0;
		for (int k = 0; k < n; k++) s = s + X[k] * X[k];
		return -1.0 / (1.0 + s);
	}
};

/* f = 1 + floor(4 |x|^2): positive steps; many vertices tie, at the minimum too (index 1 goes first there) */
struct SimplexQuantizedFunctor {
	template <class Acc> PNOL_HD static double eval(const pnol::FunctorParams &, const Acc & X, int n)
	{
		double s = 0;
		for (int k = 0; k < n; k++) s = s + X[k] * X[k];
		return 1.0 + floor(4.0 * s);
	}
};

/* -0 where |x|^2 < 1/2, +0 where 1/2 <= |x|^2 < 1, |x|^2 elsewhere: near the minimum every f is a zero of either sign (largest f 0:
 * outside the regime, the sentinel is a zero too) */
struct SimplexSignedZeroFunctor {
	template <class Acc> PNOL_HD static double eval(const pnol::FunctorParams &, const Acc & X, int n)
	{
		double s = 0;
		for (int k = 0; k < n; k++) s = s + X[k] * X[k];
		if (s >= 1.0) return s;
		return s < 0.5 ? -0.0 : 0.0;
	}
};

/* sum_k (x_k - 1)^2, NaN where x_0 > 2: vertices in that region carry NaN into the sort */
struct SimplexNanRegionFunctor {
	template <class Acc> PNOL_HD static double eval(const pnol::FunctorParams &, const Acc & X, int n)
	{
		double s = 0;
		for (int k = 0; k < n; k++) s = s + (X[k] - 1.0) * (X[k] - 1.0);
		return X[0] > 2.0 ? NAN : s;
	}
};

#endif
