/* This Source Code Form is subject to the terms of the Mozilla Public License, v. 2.0 (LICENSE at the repository root). */
// random_stream.cuh -- the random stream on the device: the "host-supplied" uniform stream u_0, u_1, ... (include/pnol_b200.h,
// pnol_stream_desc), an explicit device array or the counter generator of pnol_stream_uniform. Header-only, so that the launchers of
// out-of-tree functors (device/functor_kernels.cuh) draw the same values as the library's kernels.
#pragma once

#include <cuda_runtime.h>

namespace pnol {

struct StreamDev {
	const double * values;      // explicit stream (device copy) or nullptr
	unsigned long long n_values;
	unsigned long long seed;
	double scale;
	// A read past the end of an explicit stream gives 0.0: kernels read speculatively (trial windows), and the host decides
	// exhaustion from the draws the sequential algorithm consumed
	__device__ __forceinline__ double u(unsigned long long k) const
	{
		if (values) return k < n_values ? values[k] : 0.0;
		return from_state(state(k));
	}
	// counter mode in two steps, for loops over equally spaced positions: state(k + d) = state(k) + d * kGamma saves the 64-bit
	// multiply of the first step (a quarter of the generator's integer work, which is what the selection kernels are bound by)
	static constexpr unsigned long long kGamma = 0x9E3779B97F4A7C15ULL;
	__device__ __forceinline__ unsigned long long state(unsigned long long k) const { return seed + (k + 1ULL) * kGamma; }
	__device__ __forceinline__ double from_state(unsigned long long z) const
	{
		z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
		z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
		z = z ^ (z >> 31);
		return ((double) (z >> 11) * (1.0 / 9007199254740992.0)) * scale;
	}
};

} // namespace pnol
