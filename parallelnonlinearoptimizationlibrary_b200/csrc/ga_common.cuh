// ga_common.cuh -- pieces shared by the genetic-algorithm translation units (ga.cu: the C-ABI layer and the start population;
// ga_pipeline.cu: the generation's kernels and stages, which pnol_ga_init and the stand-alone stages run too).
#pragma once

#include "common.cuh"
#include "pnol/device/random_stream.cuh"      // StreamDev: the random stream on the device

namespace pnol {

// order-preserving map of a double onto an unsigned 64-bit key (and back). -0 and +0 get the same key: the reference's popSort compares
// with < (Source/GeneticAlgorithm.cpp:370-412), so the two zeros tie and keep their row order. The key of zero does not tell which zero
// it was: the sort kernels read that value from F[row] (sorted_value)
__host__ __device__ __forceinline__ unsigned long long double_to_key(double d)
{
#if defined(__CUDA_ARCH__)
	unsigned long long b = (unsigned long long) __double_as_longlong(d);
#else
	unsigned long long b; memcpy(&b, &d, 8);
#endif
	if (b == 0x8000000000000000ULL) b = 0;
	return (b >> 63) ? ~b : (b | 0x8000000000000000ULL);
}
constexpr unsigned long long kZeroKey = 0x8000000000000000ULL;     // double_to_key(+0.0) == double_to_key(-0.0)
__device__ __forceinline__ double key_to_double(unsigned long long k)
{
	unsigned long long b = (k >> 63) ? (k & 0x7FFFFFFFFFFFFFFFULL) : ~k;
	return __longlong_as_double((long long) b);
}
// the objective value of sorted key k, row r: rebuilt from the key, except a zero, whose sign only F[r] holds
__device__ __forceinline__ double sorted_value(unsigned long long k, unsigned r, const double * F)
{
	return k == kZeroKey ? F[r] : key_to_double(k);
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

} // namespace pnol

// state object of the C-ABI (pnol_ga_create ... pnol_ga_destroy)
struct pnol_ga {
	pnol_ctx * ctx;
	const pnol_functor * f;
	pnol_ga_params prm;
	int n;
	int nelite, nelmut, ncross, nrand;
	// device state
	double * Xnew;                       // Npop x n, replicated: pnol_ga_init's start population, pnol_ga_get_population's staging
	double * fitness, * lb, * ub, * x0;
	int * cross_idx, * mut_idx, * elite_idx;
	long long * mut_pos;
	double * stream_values;
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
// the GA's random stream as the kernels read it
inline StreamDev ga_stream(const pnol_ga * ga)
{
	StreamDev st;
	st.values = ga->stream_values; st.n_values = ga->stream.n_values; st.seed = ga->stream.seed; st.scale = ga->stream.scale;
	return st;
}
// ga_pipeline.cu
int ga_pipe_create(pnol_ga * ga);
void ga_pipe_destroy(pnol_ga * ga);
int ga_pipe_init(pnol_ga * ga, double * f0_out);  // pnol_ga_init after the start population is in ga->Xnew (see there)
int ga_pipe_generation(pnol_ga * ga);
int ga_pipe_get_population(pnol_ga * ga, double * xpop, double * F);
int ga_pipe_get_indices(pnol_ga * ga, int * cross_idx, int * mut_idx, int * elite_idx);
int ga_pipe_peer_mode(pnol_ga * ga);
// stand-alone stages on device arrays (pnol_ga_pop_sort, pnol_ga_check_identical, pnol_ga_check_bounds)
int ga_stage_pop_sort(pnol_ctx * ctx, double * X, double * F, long long npop, int n);
int ga_stage_repair(pnol_ctx * ctx, bool identical, double * X, long long npop, int n, const double * lb, const double * ub,
                    unsigned char * indicator, const StreamDev & st, unsigned long long pos, unsigned long long * pos_end);
// comm.cu
int comm_allgather_bytes_dev(pnol_ctx * ctx, const void * send, void * recv, size_t bytes_per_rank);
}
