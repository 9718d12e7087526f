/* Two objectives for the GA tests (tests/test_ga_fast_reference.py, tests/test_gpu_ga_large.py), written to the functor concept of
 * include/pnol/functors.hpp. my_ga_objectives.cu registers them with the library (compiled out of tree, as my_objectives.cu is) and
 * tests/ga_fast_reference.cpp includes this header for the CPU reference, so the host and device definitions are the same source. */
#ifndef MY_GA_OBJECTIVES_HPP_
#define MY_GA_OBJECTIVES_HPP_

#include <math.h>

#include "pnol/functors.hpp"

enum { MY_F_QUANTIZED = PNOL_F_USER_SCALAR_BASE + 11, MY_F_SIGNED_ZERO = PNOL_F_USER_SCALAR_BASE + 12 };

/* Step function of 33 levels: f = min(32, floor(|x|^2 / 2)). Many rows tie. While the best row is at level 0 and the worst at level 32,
 * the selection ratio (F_worst - F)^2 / (F_worst - F_best)^2 = (32 - f)^2 / 1024 lies exactly on a bucket edge of the GA's acceptance
 * table (csrc/ga_pipeline.cu, pipe_accept) */
struct QuantizedFunctor {
	static constexpr int kKind = MY_F_QUANTIZED;
	template <class Acc> PNOL_HD static double eval(const pnol::FunctorParams &, const Acc & X, int n)
	{
		double s = 0;
		for (int k = 0; k < n; k++) s = s + X[k] * X[k];
		const double level = floor(s * 0.5);
		return level < 32.0 ? level : 32.0;
	}
};

/* -0.0 where |x|^2 < 1/2, +0.0 where 1/2 <= |x|^2 < 1, |x|^2 elsewhere (so max F > 0). The two zeros compare equal under the
 * reference's <, so its popSort keeps them in row order */
struct SignedZeroFunctor {
	static constexpr int kKind = MY_F_SIGNED_ZERO;
	template <class Acc> PNOL_HD static double eval(const pnol::FunctorParams &, const Acc & X, int n)
	{
		double s = 0;
		for (int k = 0; k < n; k++) s = s + X[k] * X[k];
		if (s >= 1.0) return s;
		return s < 0.5 ? -0.0 : 0.0;
	}
};

#endif
