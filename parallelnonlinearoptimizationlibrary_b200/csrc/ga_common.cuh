// ga_common.cuh -- pieces shared by the genetic-algorithm translation units (ga.cu: state object, initial population and
// stand-alone stages; ga_pipeline.cu: the fused, sync-free generation).
#pragma once

#include "common.cuh"

namespace pnol {

// ---------------------------------------------------------------------------------------------------
// random stream on the device: the "host-supplied" uniform stream u_0, u_1, ... (include/pnol_b200.h, pnol_stream_desc)
// ---------------------------------------------------------------------------------------------------
struct StreamDev {
	const double * values;      // explicit stream (device copy) or nullptr
	unsigned long long n_values;
	unsigned long long seed;
	double scale;
	int * exhausted;            // set to 1 when an explicit stream is read past its end
	__device__ __forceinline__ double u(unsigned long long k) const
	{
		if (values) {
			if (k >= n_values) { if (exhausted) *exhausted = 1; return 0.0; }    // exhausted == nullptr: speculative reads (ga_pipeline.cu)
			return values[k];
		}
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

// order-preserving map of a double onto an unsigned 64-bit key (and back)
__host__ __device__ __forceinline__ unsigned long long double_to_key(double d)
{
#if defined(__CUDA_ARCH__)
	unsigned long long b = (unsigned long long) __double_as_longlong(d);
#else
	unsigned long long b; memcpy(&b, &d, 8);
#endif
	return (b >> 63) ? ~b : (b | 0x8000000000000000ULL);
}
__device__ __forceinline__ double key_to_double(unsigned long long k)
{
	unsigned long long b = (k >> 63) ? (k & 0x7FFFFFFFFFFFFFFFULL) : ~k;
	return __longlong_as_double((long long) b);
}

// contribution of gene j (value v) to the order-independent 64-bit row hash of the duplicate check; +0 and -0 compare equal in
// the reference's == (Source/GeneticAlgorithm.cpp:325), so they hash alike
__device__ __forceinline__ unsigned long long gene_hash(double v, int j)
{
	if (v == 0.0) v = 0.0;
	unsigned long long b = (unsigned long long) __double_as_longlong(v);
	b ^= (unsigned long long) (j + 1) * 0x9E3779B97F4A7C15ULL;
	b = (b ^ (b >> 30)) * 0xBF58476D1CE4E5B9ULL;
	b = (b ^ (b >> 27)) * 0x94D049BB133111EBULL;
	return b ^ (b >> 31);
}

// Where the rows of a population live. One GPU: base[0], per = Npop. Several GPUs: rank o owns rows [o per, (o+1) per) in ITS
// memory, base[o] is that block as seen from this GPU (CUDA IPC mapping over NVLink, or a local replica)
constexpr int kGaMaxRanks = 16;
struct RowTable {
	const double * base[kGaMaxRanks];
	long long per;
	int n;
	int nranks;
	// (row numbers fit 32 bits: a 64-bit division here cost more than the gene fetch it addresses)
	__device__ __forceinline__ const double * row(unsigned r) const
	{
		if (nranks <= 1) return base[0] + (size_t) r * n;
		const unsigned o = r / (unsigned) per;
		return base[o] + (size_t) (r - o * (unsigned) per) * n;
	}
};

constexpr int kScanTile = 2048;      // elements per block of the three-kernel prefix sum (256 threads x 8)
constexpr int kSortTile = 2048;      // keys per block of the radix sort of ga.cu's stages: 8 warps x 8 rounds x 32 lanes
constexpr int kSortWarps = 8;

struct SortScratch {
	unsigned long long * keys_alt;
	unsigned * vals_alt;
	unsigned * counts;              // [8][256][nblocks]
	unsigned long long * offsets;   // [256][nblocks]
	unsigned long long * scan_tmp;
	int * skip;                     // [8]
	static size_t bytes(long long n)
	{
		long long nb = (n + kSortTile - 1) / kSortTile;
		if (nb < 1) nb = 1;
		size_t s = 0;
		s += (size_t) n * 8 + 256;                 // keys_alt
		s += (size_t) n * 4 + 256;                 // vals_alt
		s += (size_t) 8 * 256 * nb * 4 + 256;      // counts
		s += (size_t) 256 * nb * 8 + 256;          // offsets
		s += (size_t) ((256 * nb + kScanTile - 1) / kScanTile + 1) * 8 + 256;
		s += 256;
		return s;
	}
	void carve(void * base, long long n)
	{
		long long nb = (n + kSortTile - 1) / kSortTile;
		if (nb < 1) nb = 1;
		unsigned char * p = (unsigned char *) base;
		auto take = [&](size_t b) { void * r = p; p += (b + 255) & ~(size_t) 255; return r; };
		keys_alt = (unsigned long long *) take((size_t) n * 8);
		vals_alt = (unsigned *) take((size_t) n * 4);
		counts = (unsigned *) take((size_t) 8 * 256 * nb * 4);
		offsets = (unsigned long long *) take((size_t) 256 * nb * 8);
		scan_tmp = (unsigned long long *) take((size_t) ((256 * nb + kScanTile - 1) / kScanTile + 1) * 8);
		skip = (int *) take(64);
	}
};


} // namespace pnol

// state object of the C-ABI (pnol_ga_create ... pnol_ga_destroy)
struct pnol_ga {
	pnol_ctx * ctx;
	const pnol_functor * f;
	pnol_ga_params prm;
	int n;
	int nelite, nelmut, ncross, nrand;
	// device state
	double * Xpop, * Xnew, * F, * Fnew, * fitness, * lb, * ub, * x0;
	unsigned char * indicator;
	int * cross_idx, * mut_idx, * elite_idx;
	long long * mut_pos;
	double * stream_values;
	int * exhausted;
	// scratch
	void * sort_mem; pnol::SortScratch sort;
	unsigned long long * keys; unsigned * perm;
	unsigned * u32a; unsigned long long * u64a; unsigned long long * scan_tmp; unsigned long long * total_dev;
	double * gather = nullptr;           // all-gather buffer of the sharded fitness sweep (multi-GPU)
	// host state
	pnol_stream_desc stream;
	uint64_t pos;
	int generation, n_static, stopped;
	double f_best_prev, f_best;
	std::vector<void *> owned;
	// the fused generation pipeline (ga_pipeline.cu); created by pnol_ga_create, nullptr only while it is being built or torn down
	struct GaPipe * pipe = nullptr;
};


namespace pnol {
// ga_pipeline.cu
int ga_pipe_create(pnol_ga * ga);                 // allocates the pipeline state (after the buffers of pnol_ga_init exist)
void ga_pipe_destroy(pnol_ga * ga);
int ga_pipe_reset(pnol_ga * ga);                  // after pnol_ga_init: sorted population -> pipeline representation
int ga_pipe_generation(pnol_ga * ga);
int ga_pipe_get_population(pnol_ga * ga, double * xpop, double * F);
int ga_pipe_get_indices(pnol_ga * ga, int * cross_idx, int * mut_idx, int * elite_idx);
int ga_pipe_peer_mode(pnol_ga * ga);
// comm.cu
int comm_allgather_bytes_dev(pnol_ctx * ctx, const void * send, void * recv, size_t bytes_per_rank);
}
