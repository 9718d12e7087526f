// ga.cu -- genetic algorithm on the device (a15 / a16): the state object of GeneticAlgorithmMPI::findMinBnd
// (Source/GeneticAlgorithmMPI.cpp:12-276), its initial population (:55-81), and the free functions popSort /
// checkIndenticalChildAndReplace / checkPopulationBoundsAndReplace (Source/GeneticAlgorithm.cpp:313-412) as stand-alone
// stages. One generation runs in the fused pipeline of ga_pipeline.cu.
//
// The reference draws every random number from ONE sequential stream (timeRand()); which draw feeds which decision
// depends on the data. The stages below reproduce exactly that consumption order in parallel:
//   * duplicates : rows are hashed, (hash,row) sorted, equal-hash runs compared exactly; replaced rows take n draws
//                  each in row order (prefix sum);
//   * bounds     : out-of-box genes take one draw each in row-major order (prefix sum over per-row counts);
//   * popSort    : stable LSD radix sort of the objective values (== repeated first-minimum extraction).
// Integer / index work is bit-exact against the oracle by construction; see tests/test_gpu_ga.py.
#include "ga_common.cuh"

#include <math.h>
#include <utility>

namespace pnol {

// ---------------------------------------------------------------------------------------------------
// exclusive prefix sum of unsigned ints (three kernels, deterministic)
// ---------------------------------------------------------------------------------------------------

__global__ void __launch_bounds__(256)
scan_reduce_kernel(const unsigned * __restrict__ in, long long n, unsigned long long * __restrict__ block_sums)
{
	__shared__ unsigned long long red[256];
	long long base = (long long) blockIdx.x * kScanTile;
	unsigned long long s = 0;
	for (int e = 0; e < 8; e++) {
		long long i = base + threadIdx.x * 8 + e;
		if (i < n) s += in[i];
	}
	red[threadIdx.x] = s;
	__syncthreads();
	for (int o = 128; o > 0; o >>= 1) {
		if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
		__syncthreads();
	}
	if (threadIdx.x == 0) block_sums[blockIdx.x] = red[0];
}

// single block: exclusive scan of block sums in place; total -> *total
__global__ void __launch_bounds__(1024)
scan_sums_kernel(unsigned long long * __restrict__ sums, int nb, unsigned long long * __restrict__ total)
{
	__shared__ unsigned long long part[1024];
	const int per = (nb + 1023) / 1024;
	const int b0 = threadIdx.x * per;
	unsigned long long s = 0;
	for (int e = 0; e < per; e++) if (b0 + e < nb) s += sums[b0 + e];
	part[threadIdx.x] = s;
	__syncthreads();
	// Hillis-Steele inclusive scan over 1024 partials
	for (int o = 1; o < 1024; o <<= 1) {
		unsigned long long v = threadIdx.x >= o ? part[threadIdx.x - o] : 0;
		__syncthreads();
		part[threadIdx.x] += v;
		__syncthreads();
	}
	unsigned long long run = threadIdx.x ? part[threadIdx.x - 1] : 0;
	for (int e = 0; e < per; e++)
		if (b0 + e < nb) { unsigned long long v = sums[b0 + e]; sums[b0 + e] = run; run += v; }
	if (threadIdx.x == 1023 && total) *total = part[1023];
}

__global__ void __launch_bounds__(256)
scan_apply_kernel(const unsigned * __restrict__ in, long long n, const unsigned long long * __restrict__ block_offs,
                  unsigned long long * __restrict__ out)
{
	__shared__ unsigned long long tsum[256];
	long long base = (long long) blockIdx.x * kScanTile;
	unsigned v[8];
	unsigned long long s = 0;
	for (int e = 0; e < 8; e++) {
		long long i = base + threadIdx.x * 8 + e;
		v[e] = i < n ? in[i] : 0;
		s += v[e];
	}
	tsum[threadIdx.x] = s;
	__syncthreads();
	for (int o = 1; o < 256; o <<= 1) {
		unsigned long long t = threadIdx.x >= o ? tsum[threadIdx.x - o] : 0;
		__syncthreads();
		tsum[threadIdx.x] += t;
		__syncthreads();
	}
	unsigned long long run = block_offs[blockIdx.x] + (threadIdx.x ? tsum[threadIdx.x - 1] : 0);
	for (int e = 0; e < 8; e++) {
		long long i = base + threadIdx.x * 8 + e;
		if (i < n) out[i] = run;
		run += v[e];
	}
}

// out[i] = sum_{j<i} in[j]; *total_dev = sum of all. scratch: ceil(n/2048) u64
static int exclusive_scan_u32(pnol_ctx * ctx, const unsigned * in, long long n, unsigned long long * out,
                              unsigned long long * scratch, unsigned long long * total_dev)
{
	int nb = (int) ((n + kScanTile - 1) / kScanTile);
	if (nb < 1) nb = 1;
	PNOL_LAUNCH(ctx, scan_reduce_kernel, nb, 256, 0, in, n, scratch);
	PNOL_LAUNCH(ctx, scan_sums_kernel, 1, 1024, 0, scratch, nb, total_dev);
	PNOL_LAUNCH(ctx, scan_apply_kernel, nb, 256, 0, in, n, scratch, out);
	return PNOL_OK;
}

// ---------------------------------------------------------------------------------------------------
// stable LSD radix sort of (u64 key, u32 value) pairs, 8-bit digits; passes whose digit is constant are skipped
// ---------------------------------------------------------------------------------------------------

// counts[pass][digit][block] for every pass in ONE read of the keys
__global__ void __launch_bounds__(256)
sort_hist_kernel(const unsigned long long * __restrict__ keys, long long n, int nblocks, unsigned * __restrict__ counts)
{
	__shared__ unsigned h[8][256];
	for (int e = threadIdx.x; e < 8 * 256; e += 256) (&h[0][0])[e] = 0;
	__syncthreads();
	long long base = (long long) blockIdx.x * kSortTile;
	for (int e = threadIdx.x; e < kSortTile; e += 256) {
		long long i = base + e;
		if (i < n) {
			unsigned long long k = keys[i];
#pragma unroll
			for (int p = 0; p < 8; p++) atomicAdd(&h[p][(k >> (8 * p)) & 255], 1u);
		}
	}
	__syncthreads();
	for (int e = threadIdx.x; e < 8 * 256; e += 256) {
		int p = e >> 8, d = e & 255;
		counts[((size_t) p * 256 + d) * nblocks + blockIdx.x] = h[p][d];
	}
}

// per pass: is one digit value holding every key? (skip[p] = 1; skip[] zeroed by the caller). One warp per (pass, digit) counter
// row: the first version summed the 2048 x nblocks counters in ONE block, 8 rows per thread -- 0.30 ms per sort at 1M keys, a
// fifth of a GA generation.
__global__ void __launch_bounds__(256)
sort_skip_kernel(const unsigned * __restrict__ counts, int nblocks, long long n, int * __restrict__ skip)
{
	const int e = (int) ((blockIdx.x * blockDim.x + threadIdx.x) >> 5);      // (pass, digit) = (e >> 8, e & 255)
	const int lane = threadIdx.x & 31;
	if (e >= 8 * 256) return;
	const unsigned * c = counts + (size_t) e * nblocks;
	unsigned long long s = 0;
	for (int b = lane; b < nblocks; b += 32) s += c[b];
	for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
	if (lane == 0 && s == (unsigned long long) n) skip[e >> 8] = 1;
}

__global__ void __launch_bounds__(kSortWarps * 32)
sort_scatter_kernel(const unsigned long long * __restrict__ keys_in, const unsigned * __restrict__ vals_in, long long n,
                    int pass, int nblocks, const unsigned long long * __restrict__ offsets /* [256][nblocks] exclusive */,
                    unsigned long long * __restrict__ keys_out, unsigned * __restrict__ vals_out)
{
	__shared__ unsigned wcount[kSortWarps][256];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	for (int e = threadIdx.x; e < kSortWarps * 256; e += blockDim.x) (&wcount[0][0])[e] = 0;
	__syncthreads();
	const long long base = (long long) blockIdx.x * kSortTile + warp * 256;
	unsigned long long k[8];
	unsigned v[8];
	unsigned short rank[8];
	// warp w owns 256 consecutive keys; round r covers keys base + r*32 + lane, so (warp, round, lane) is key order
#pragma unroll
	for (int r = 0; r < 8; r++) {
		long long i = base + r * 32 + lane;
		bool valid = i < n;
		k[r] = valid ? keys_in[i] : 0xFFFFFFFFFFFFFFFFULL;
		v[r] = valid ? vals_in[i] : 0;
		unsigned d = valid ? (unsigned) ((k[r] >> (8 * pass)) & 255) : 256u;
		unsigned mask = __match_any_sync(0xffffffffu, d);
		unsigned before = __popc(mask & ((1u << lane) - 1));
		unsigned prev = 0;
		if (valid) prev = wcount[warp][d];
		__syncwarp();
		if (valid && before == 0) wcount[warp][d] = prev + __popc(mask);
		__syncwarp();
		rank[r] = (unsigned short) (prev + before);
	}
	__syncthreads();
	// exclusive scan over warps, per digit (thread d handles digit d)
	{
		int d = threadIdx.x;
		if (d < 256) {
			unsigned run = 0;
			for (int w = 0; w < kSortWarps; w++) { unsigned c = wcount[w][d]; wcount[w][d] = run; run += c; }
		}
	}
	__syncthreads();
#pragma unroll
	for (int r = 0; r < 8; r++) {
		long long i = base + r * 32 + lane;
		if (i < n) {
			unsigned d = (unsigned) ((k[r] >> (8 * pass)) & 255);
			unsigned long long pos = offsets[(size_t) d * nblocks + blockIdx.x] + wcount[warp][d] + rank[r];
			keys_out[pos] = k[r];
			vals_out[pos] = v[r];
		}
	}
}

// sorts (keys, vals) in place (result ends in the given arrays); stable
static int radix_sort_pairs(pnol_ctx * ctx, unsigned long long * keys, unsigned * vals, long long n, SortScratch & sc)
{
	if (n <= 1) return PNOL_OK;
	int nblocks = (int) ((n + kSortTile - 1) / kSortTile);
	PNOL_LAUNCH(ctx, sort_hist_kernel, nblocks, 256, 0, keys, n, nblocks, sc.counts);
	PNOL_CUDA(ctx, cudaMemsetAsync(sc.skip, 0, 8 * sizeof(int), ctx->stream));
	PNOL_LAUNCH(ctx, sort_skip_kernel, 8 * 256 * 32 / 256, 256, 0, sc.counts, nblocks, n, sc.skip);
	int skip[8];
	PNOL_CUDA(ctx, cudaMemcpyAsync(skip, sc.skip, sizeof skip, cudaMemcpyDeviceToHost, ctx->stream));
	PNOL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	unsigned long long * kin = keys, * kout = sc.keys_alt;
	unsigned * vin = vals, * vout = sc.vals_alt;
	for (int pass = 0; pass < 8; pass++) {
		if (skip[pass]) continue;
		// the per-pass digit histogram of a tile does not depend on the order of the keys inside the whole array?
		// It does (tiles change as keys move), so the histogram is recomputed from the current key order.
		if (kin != keys || pass > 0) PNOL_LAUNCH(ctx, sort_hist_kernel, nblocks, 256, 0, kin, n, nblocks, sc.counts);
		PNOL_CHECK(exclusive_scan_u32(ctx, sc.counts + (size_t) pass * 256 * nblocks, (long long) 256 * nblocks, sc.offsets,
		                              sc.scan_tmp, nullptr));
		PNOL_LAUNCH(ctx, sort_scatter_kernel, nblocks, kSortWarps * 32, 0, kin, vin, n, pass, nblocks, sc.offsets, kout, vout);
		unsigned long long * tk = kin; kin = kout; kout = tk;
		unsigned * tv = vin; vin = vout; vout = tv;
	}
	if (kin != keys) {
		PNOL_CUDA(ctx, cudaMemcpyAsync(keys, kin, (size_t) n * 8, cudaMemcpyDeviceToDevice, ctx->stream));
		PNOL_CUDA(ctx, cudaMemcpyAsync(vals, vin, (size_t) n * 4, cudaMemcpyDeviceToDevice, ctx->stream));
	}
	return PNOL_OK;
}

// ---------------------------------------------------------------------------------------------------
// popSort  (Source/GeneticAlgorithm.cpp:370-412)
// ---------------------------------------------------------------------------------------------------
__global__ void make_sort_keys_kernel(const double * __restrict__ F, long long n, unsigned long long * __restrict__ keys,
                                      unsigned * __restrict__ vals)
{
	long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n) { keys[i] = double_to_key(F[i]); vals[i] = (unsigned) i; }
}

// dst[k] = src[perm[k]] for rows of n doubles; one warp per row, coalesced
__global__ void __launch_bounds__(256)
gather_rows_kernel(const double * __restrict__ src, const unsigned * __restrict__ perm, long long npop, int n,
                   double * __restrict__ dst, const double * __restrict__ Fsrc, double * __restrict__ Fdst)
{
	long long row = ((long long) blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	int lane = threadIdx.x & 31;
	if (row >= npop) return;
	unsigned from = perm[row];
	const double * s = src + (long long) from * n;
	double * d = dst + row * n;
	for (int j = lane; j < n; j += 32) d[j] = s[j];
	if (lane == 0 && Fsrc) Fdst[row] = Fsrc[from];
}

// ---------------------------------------------------------------------------------------------------
// checkPopulationBoundsAndReplace  (Source/GeneticAlgorithm.cpp:347-365)
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
bounds_count_kernel(const double * __restrict__ X, long long npop, int n, const double * __restrict__ lb,
                    const double * __restrict__ ub, unsigned * __restrict__ rowcount)
{
	long long row = ((long long) blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	int lane = threadIdx.x & 31;
	if (row >= npop) return;
	const double * x = X + row * n;
	unsigned c = 0;
	for (int j = lane; j < n; j += 32) { double v = x[j]; if (v > ub[j] || v < lb[j]) c++; }
	for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
	if (lane == 0) rowcount[row] = c;
}

__global__ void __launch_bounds__(256)
bounds_fix_kernel(double * __restrict__ X, long long npop, int n, const double * __restrict__ lb, const double * __restrict__ ub,
                  const unsigned * __restrict__ rowcount, const unsigned long long * __restrict__ rowoff, StreamDev st,
                  unsigned long long pos, unsigned char * __restrict__ indicator)
{
	long long row = (long long) blockIdx.x * blockDim.x + threadIdx.x;
	if (row >= npop || rowcount[row] == 0) return;
	double * x = X + row * n;
	unsigned long long k = pos + rowoff[row];
	for (int j = 0; j < n; j++) {
		double v = x[j];
		if (v > ub[j] || v < lb[j]) { x[j] = lb[j] + (ub[j] - lb[j]) * st.u(k); k++; }
	}
	if (indicator) indicator[row] = 1;
}

// ---------------------------------------------------------------------------------------------------
// checkIndenticalChildAndReplace  (Source/GeneticAlgorithm.cpp:313-344)
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
row_hash_kernel(const double * __restrict__ X, long long npop, int n, unsigned long long * __restrict__ keys, unsigned * __restrict__ vals,
                unsigned long long * __restrict__ fullhash)
{
	long long row = ((long long) blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	int lane = threadIdx.x & 31;
	if (row >= npop) return;
	const double * x = X + row * n;
	unsigned long long h = 0;
	for (int j = lane; j < n; j += 32) {
		double v = x[j];
		if (v == 0.0) v = 0.0;                              // +0 and -0 compare equal in the reference's ==
		unsigned long long b = (unsigned long long) __double_as_longlong(v);
		b ^= (unsigned long long) (j + 1) * 0x9E3779B97F4A7C15ULL;
		b = (b ^ (b >> 30)) * 0xBF58476D1CE4E5B9ULL;
		b = (b ^ (b >> 27)) * 0x94D049BB133111EBULL;
		h += b ^ (b >> 31);                                 // order independent across lanes
	}
	for (int o = 16; o > 0; o >>= 1) h += __shfl_xor_sync(0xffffffffu, h, o);
	// only the top 32 bits are SORTED on (the radix sort skips the four all-zero low digits: half the passes); the full hash is
	// compared inside the few runs of equal top halves
	if (lane == 0) { keys[row] = h & 0xFFFFFFFF00000000ULL; fullhash[row] = h; vals[row] = (unsigned) row; }
}

// sorted by (top half of the hash, row): element s is a duplicate iff some later element of its run has the same full hash and an
// equal row
__global__ void __launch_bounds__(256)
dup_flag_kernel(const double * __restrict__ X, long long npop, int n, const unsigned long long * __restrict__ keys,
                const unsigned * __restrict__ vals, const unsigned long long * __restrict__ fullhash, unsigned * __restrict__ dupflag)
{
	long long s = (long long) blockIdx.x * blockDim.x + threadIdx.x;
	if (s >= npop) return;
	unsigned long long h = keys[s];
	unsigned row = vals[s];
	const unsigned long long hf = fullhash[row];
	unsigned flag = 0;
	for (long long t = s + 1; t < npop && keys[t] == h; t++) {
		if (fullhash[vals[t]] != hf) continue;
		const double * a = X + (long long) row * n;
		const double * b = X + (long long) vals[t] * n;
		int same = 0;
		for (int j = 0; j < n; j++) if (a[j] == b[j]) same++;
		if (same == n) { flag = 1; break; }
	}
	dupflag[row] = flag;
}

__global__ void __launch_bounds__(256)
dup_fix_kernel(double * __restrict__ X, long long npop, int n, const double * __restrict__ lb, const double * __restrict__ ub,
               const unsigned * __restrict__ dupflag, const unsigned long long * __restrict__ dupoff, StreamDev st,
               unsigned long long pos, unsigned char * __restrict__ indicator)
{
	long long row = ((long long) blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	int lane = threadIdx.x & 31;
	if (row >= npop || !dupflag[row]) return;
	double * x = X + row * n;
	unsigned long long k = pos + dupoff[row] * (unsigned long long) n;
	for (int j = lane; j < n; j += 32) x[j] = lb[j] + (ub[j] - lb[j]) * st.u(k + j);
	if (lane == 0 && indicator) indicator[row] = 1;
}

// ---------------------------------------------------------------------------------------------------
// initial population (Source/GeneticAlgorithmMPI.cpp:58-68)
// ---------------------------------------------------------------------------------------------------
__global__ void ga_init_pop_kernel(double * __restrict__ X, long long npop, int n, const double * __restrict__ x0,
                                   const double * __restrict__ lb, const double * __restrict__ ub, StreamDev st, unsigned long long pos)
{
	long long e = (long long) blockIdx.x * blockDim.x + threadIdx.x;
	if (e >= npop * n) return;
	long long i = e / n;
	int j = (int) (e - i * n);
	if (i == 0) X[e] = x0[j];
	else X[e] = x0[j] + ((ub[j] - lb[j]) * st.u(pos + (unsigned long long) (e - n)) + lb[j]);
}

} // namespace pnol

using namespace pnol;

// ---------------------------------------------------------------------------------------------------
// state object
// ---------------------------------------------------------------------------------------------------
static StreamDev ga_stream_dev(pnol_ga * ga)
{
	StreamDev st;
	st.values = ga->stream_values;
	st.n_values = ga->stream.n_values;
	st.seed = ga->stream.seed;
	st.scale = ga->stream.scale;
	st.exhausted = ga->exhausted;
	return st;
}

template <class T> static int ga_alloc(pnol_ga * ga, T ** p, size_t count);

// The fitness sweep of one population (GeneticAlgorithmMPI::evaluatePopulationParallel, Source/GeneticAlgorithmMPI.cpp:283-414).
// With a communicator the individuals are SHARDED: rank r evaluates rows [r per, (r+1) per) and the objective values are
// all-gathered (the reference round-robins the individuals and sums zero-padded copies, :344-401). Every other stage of a
// generation is replicated: all ranks hold the same population and consume the same random stream, so they stay bit-identical.
static int ga_evaluate(pnol_ga * ga, const double * X, const unsigned char * indicator, double * Fout)
{
	pnol_ctx * ctx = ga->ctx;
	const int Npop = ga->prm.npop, n = ga->n;
	if (ctx->nranks <= 1) return launch_eval_batch(ctx, ga->f, X, Npop, n, n, indicator, Fout);
	const int R = ctx->nranks;
	const long long per = ((long long) Npop + R - 1) / R;
	if (!ga->gather) PNOL_CHECK(ga_alloc(ga, &ga->gather, (size_t) per * R));
	const long long lo = per * ctx->rank < Npop ? per * ctx->rank : Npop;
	const long long hi = lo + per < Npop ? lo + per : Npop;
	if (hi > lo) PNOL_CHECK(launch_eval_batch(ctx, ga->f, X + lo * n, hi - lo, n, n, indicator ? indicator + lo : nullptr, Fout + lo));
	// rows that were not evaluated (elites) already hold the same value on every rank, so gathering whole shards is exact
	double * slot = ga->gather + per * ctx->rank;
	PNOL_CUDA(ctx, cudaMemsetAsync(slot, 0, (size_t) per * sizeof(double), ctx->stream));
	if (hi > lo) PNOL_CUDA(ctx, cudaMemcpyAsync(slot, Fout + lo, (size_t) (hi - lo) * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
	PNOL_CHECK(comm_allgather_dev(ctx, slot, ga->gather, (size_t) per));
	PNOL_CUDA(ctx, cudaMemcpyAsync(Fout, ga->gather, (size_t) Npop * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
	return PNOL_OK;
}

template <class T> static int ga_alloc(pnol_ga * ga, T ** p, size_t count)
{
	void * d = nullptr;
	PNOL_CUDA(ga->ctx, cudaMalloc(&d, (count ? count : 1) * sizeof(T)));
	ga->owned.push_back(d);
	*p = (T *) d;
	return PNOL_OK;
}

extern "C" void pnol_ga_destroy(pnol_ga * ga)
{
	if (!ga) return;
	cudaStreamSynchronize(ga->ctx->stream);
	ga_pipe_destroy(ga);
	for (void * p : ga->owned) cudaFree(p);
	delete ga;
}

extern "C" int pnol_ga_create(pnol_ctx * ctx, const pnol_functor * f, const pnol_ga_params * prm, int n, const double * xlb,
                              const double * xub, const pnol_stream_desc * stream, pnol_ga ** out)
{
	if (!ctx || !f || !prm || !xlb || !xub || !stream || !out) return PNOL_ERR_INVALID;
	*out = nullptr;
	PNOL_REQUIRE(ctx, prm->npop >= 2 && n >= 1, "ga: need npop >= 2 and n >= 1");
	const int Npop = prm->npop;
	// population sizes (Source/GeneticAlgorithmMPI.cpp:33-36); the reference prints and calls exit(0) when Nrand <= 0
	int nelite = (int) ceil(prm->elite_frac * Npop);
	int nelmut = (int) ceil(prm->elite_mutation_frac * Npop);
	int ncross = (int) ceil(prm->cross_frac * Npop);
	int nrand = Npop - nelite - nelmut - ncross;
	PNOL_REQUIRE(ctx, nrand > 0, "GA fractions set incorrectly: their sum must be below 1 (Nrand = %d)", nrand);
	PNOL_REQUIRE(ctx, nelite >= 0 && nelmut >= 0 && ncross >= 0 && nelite < Npop, "ga: negative fraction");
	pnol_ga * ga = new pnol_ga();
	ga->ctx = ctx; ga->f = f; ga->prm = *prm; ga->n = n;
	ga->nelite = nelite; ga->nelmut = nelmut; ga->ncross = ncross; ga->nrand = nrand;
	ga->stream = *stream; ga->pos = 0; ga->generation = 0; ga->n_static = 0; ga->stopped = 0;
	ga->f_best = ga->f_best_prev = 0; ga->stream_values = nullptr;
	size_t NN = (size_t) Npop * n;
	int st = PNOL_OK;
#define GA_TRY(x) do { st = (x); if (st != PNOL_OK) { pnol_ga_destroy(ga); return st; } } while (0)
	GA_TRY(ga_alloc(ga, &ga->Xpop, NN));
	GA_TRY(ga_alloc(ga, &ga->Xnew, NN));
	GA_TRY(ga_alloc(ga, &ga->F, Npop));
	GA_TRY(ga_alloc(ga, &ga->Fnew, Npop));
	GA_TRY(ga_alloc(ga, &ga->fitness, Npop));
	GA_TRY(ga_alloc(ga, &ga->lb, n));
	GA_TRY(ga_alloc(ga, &ga->ub, n));
	GA_TRY(ga_alloc(ga, &ga->x0, n));
	GA_TRY(ga_alloc(ga, &ga->indicator, Npop));
	GA_TRY(ga_alloc(ga, &ga->cross_idx, (size_t) ncross * n));
	GA_TRY(ga_alloc(ga, &ga->mut_idx, nrand));
	GA_TRY(ga_alloc(ga, &ga->mut_pos, nrand));
	GA_TRY(ga_alloc(ga, &ga->elite_idx, (size_t) nelmut * n));
	GA_TRY(ga_alloc(ga, &ga->exhausted, 4));
	GA_TRY(ga_alloc(ga, &ga->keys, Npop));
	GA_TRY(ga_alloc(ga, &ga->perm, Npop));
	GA_TRY(ga_alloc(ga, &ga->u32a, (size_t) Npop + 16));
	GA_TRY(ga_alloc(ga, &ga->u64a, (size_t) Npop + 16));
	GA_TRY(ga_alloc(ga, &ga->scan_tmp, (size_t) Npop / kScanTile + 16));
	GA_TRY(ga_alloc(ga, &ga->total_dev, 4));
	{
		void * sm = nullptr;
		cudaError_t e = cudaMalloc(&sm, SortScratch::bytes(Npop));
		if (e != cudaSuccess) { PNOL_SET_ERR(ctx, "ga: sort scratch: %s", cudaGetErrorString(e)); pnol_ga_destroy(ga); return PNOL_ERR_CUDA; }
		ga->owned.push_back(sm);
		ga->sort_mem = sm;
		ga->sort.carve(sm, Npop);
	}
	if (stream->values && stream->n_values) {
		GA_TRY(ga_alloc(ga, &ga->stream_values, stream->n_values));
		cudaError_t e = cudaMemcpyAsync(ga->stream_values, stream->values, stream->n_values * sizeof(double), cudaMemcpyDefault, ctx->stream);
		if (e != cudaSuccess) { PNOL_SET_ERR(ctx, "ga: stream upload: %s", cudaGetErrorString(e)); pnol_ga_destroy(ga); return PNOL_ERR_CUDA; }
	}
	cudaMemcpyAsync(ga->lb, xlb, n * sizeof(double), cudaMemcpyDefault, ctx->stream);
	cudaMemcpyAsync(ga->ub, xub, n * sizeof(double), cudaMemcpyDefault, ctx->stream);
	cudaMemsetAsync(ga->exhausted, 0, 16, ctx->stream);
	GA_TRY(finish(ctx));
	GA_TRY(ga_pipe_create(ga));
#undef GA_TRY
	*out = ga;
	return PNOL_OK;
}

// ---- stage helpers on raw device buffers (shared by the state machine and the stand-alone entry points) ----
struct GaScratch {
	unsigned long long * keys; unsigned * perm; SortScratch * sort;
	unsigned * u32a; unsigned long long * u64a; unsigned long long * scan_tmp; unsigned long long * total_dev;
};

static int ga_pop_sort_dev(pnol_ctx * ctx, const double * Xsrc, const double * Fsrc, long long npop, int n, double * Xdst,
                           double * Fdst, GaScratch & sc)
{
	TimerScope ts(ctx, "ga_pop_sort");
	PNOL_LAUNCH(ctx, make_sort_keys_kernel, (unsigned) ((npop + 255) / 256), 256, 0, Fsrc, npop, sc.keys, sc.perm);
	PNOL_CHECK(radix_sort_pairs(ctx, sc.keys, sc.perm, npop, *sc.sort));
	PNOL_LAUNCH(ctx, gather_rows_kernel, (unsigned) ((npop * 32 + 255) / 256), 256, 0, Xsrc, sc.perm, npop, n, Xdst, Fsrc, Fdst);
	return PNOL_OK;
}

static int ga_check_bounds_dev(pnol_ctx * ctx, double * X, long long npop, int n, const double * lb, const double * ub,
                               unsigned char * indicator, StreamDev st, uint64_t * pos, GaScratch & sc)
{
	TimerScope ts(ctx, "ga_check_bounds");
	PNOL_LAUNCH(ctx, bounds_count_kernel, (unsigned) ((npop * 32 + 255) / 256), 256, 0, X, npop, n, lb, ub, sc.u32a);
	PNOL_CHECK(exclusive_scan_u32(ctx, sc.u32a, npop, sc.u64a, sc.scan_tmp, sc.total_dev));
	PNOL_LAUNCH(ctx, bounds_fix_kernel, (unsigned) ((npop + 255) / 256), 256, 0, X, npop, n, lb, ub, sc.u32a, sc.u64a, st,
	            (unsigned long long) *pos, indicator);
	unsigned long long total = 0;
	PNOL_CUDA(ctx, cudaMemcpyAsync(&total, sc.total_dev, sizeof total, cudaMemcpyDeviceToHost, ctx->stream));
	PNOL_CHECK(finish(ctx));
	*pos += total;
	return PNOL_OK;
}

static int ga_check_identical_dev(pnol_ctx * ctx, double * X, long long npop, int n, const double * lb, const double * ub,
                                  unsigned char * indicator, StreamDev st, uint64_t * pos, GaScratch & sc)
{
	TimerScope ts(ctx, "ga_check_identical");
	// sc.u64a carries the full hashes until the flags are known; the scan below then reuses it for the offsets
	PNOL_LAUNCH(ctx, row_hash_kernel, (unsigned) ((npop * 32 + 255) / 256), 256, 0, X, npop, n, sc.keys, sc.perm, sc.u64a);
	PNOL_CHECK(radix_sort_pairs(ctx, sc.keys, sc.perm, npop, *sc.sort));
	PNOL_LAUNCH(ctx, dup_flag_kernel, (unsigned) ((npop + 255) / 256), 256, 0, X, npop, n, sc.keys, sc.perm, sc.u64a, sc.u32a);
	PNOL_CHECK(exclusive_scan_u32(ctx, sc.u32a, npop, sc.u64a, sc.scan_tmp, sc.total_dev));
	unsigned long long total = 0;
	PNOL_CUDA(ctx, cudaMemcpyAsync(&total, sc.total_dev, sizeof total, cudaMemcpyDeviceToHost, ctx->stream));
	PNOL_CHECK(finish(ctx));
	if (total) {
		PNOL_LAUNCH(ctx, dup_fix_kernel, (unsigned) ((npop * 32 + 255) / 256), 256, 0, X, npop, n, lb, ub, sc.u32a, sc.u64a, st,
		            (unsigned long long) *pos, indicator);
		*pos += total * (unsigned long long) n;
	}
	return PNOL_OK;
}

static GaScratch ga_scratch(pnol_ga * ga)
{
	GaScratch sc;
	sc.keys = ga->keys; sc.perm = ga->perm; sc.sort = &ga->sort; sc.u32a = ga->u32a; sc.u64a = ga->u64a;
	sc.scan_tmp = ga->scan_tmp; sc.total_dev = ga->total_dev;
	return sc;
}

static int ga_check_stream(pnol_ga * ga)
{
	if (!ga->stream_values) return PNOL_OK;
	int ex = 0;
	PNOL_CUDA(ga->ctx, cudaMemcpyAsync(&ex, ga->exhausted, sizeof ex, cudaMemcpyDeviceToHost, ga->ctx->stream));
	PNOL_CHECK(finish(ga->ctx));
	if (ex) { PNOL_SET_ERR(ga->ctx, "ga: the explicit random stream (%llu values) is exhausted", (unsigned long long) ga->stream.n_values); return PNOL_ERR_STREAM; }
	return PNOL_OK;
}

// Source/GeneticAlgorithmMPI.cpp:55-81
extern "C" int pnol_ga_init(pnol_ga * ga, const double * x0, double * f0_out)
{
	if (!ga || !x0) return PNOL_ERR_INVALID;
	pnol_ctx * ctx = ga->ctx;
	const long long Npop = ga->prm.npop;
	const int n = ga->n;
	StreamDev st = ga_stream_dev(ga);
	GaScratch sc = ga_scratch(ga);
	ga->pos = 0; ga->generation = 0; ga->n_static = 0; ga->stopped = 0;
	PNOL_CUDA(ctx, cudaMemcpyAsync(ga->x0, x0, n * sizeof(double), cudaMemcpyDefault, ctx->stream));
	PNOL_LAUNCH(ctx, ga_init_pop_kernel, (unsigned) ((Npop * n + 255) / 256), 256, 0, ga->Xpop, Npop, n, ga->x0, ga->lb, ga->ub, st,
	            (unsigned long long) ga->pos);
	ga->pos += (uint64_t) (Npop - 1) * n;
	// the reference checks the all-zero XpopNew for identical children here (:71, sic): every row but the last is
	// "identical to a later one" and is re-randomised, which only burns (Npop-1)*n draws. Run the real kernel on zeros.
	PNOL_CUDA(ctx, cudaMemsetAsync(ga->Xnew, 0, (size_t) Npop * n * sizeof(double), ctx->stream));
	PNOL_CUDA(ctx, cudaMemsetAsync(ga->indicator, 1, (size_t) Npop, ctx->stream));
	PNOL_CHECK(ga_check_identical_dev(ctx, ga->Xnew, Npop, n, ga->lb, ga->ub, ga->indicator, st, &ga->pos, sc));
	PNOL_CHECK(ga_check_bounds_dev(ctx, ga->Xpop, Npop, n, ga->lb, ga->ub, ga->indicator, st, &ga->pos, sc));   // (:74)
	PNOL_CHECK(ga_evaluate(ga, ga->Xpop, nullptr, ga->F));                                                      // (:77)
	double f0 = 0;
	PNOL_CUDA(ctx, cudaMemcpyAsync(&f0, ga->F, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));         // (:78)
	// popSort (:81): sort into Xnew / Fnew, then swap the buffers
	PNOL_CHECK(ga_pop_sort_dev(ctx, ga->Xpop, ga->F, Npop, n, ga->Xnew, ga->Fnew, sc));
	std::swap(ga->Xpop, ga->Xnew);
	std::swap(ga->F, ga->Fnew);
	double fb = 0;
	PNOL_CUDA(ctx, cudaMemcpyAsync(&fb, ga->F, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
	PNOL_CHECK(finish(ctx));
	PNOL_CHECK(ga_check_stream(ga));
	ga->f_best_prev = fb; ga->f_best = fb;
	if (f0_out) *f0_out = f0;
	return ga_pipe_reset(ga);
}

// Source/GeneticAlgorithmMPI.cpp:87-249 (one pass of the while loop)
extern "C" int pnol_ga_generation(pnol_ga * ga)
{
	if (!ga) return PNOL_ERR_INVALID;
	if (ga->stopped || ga->generation >= ga->prm.max_generations) return PNOL_OK;
	return ga_pipe_generation(ga);
}

extern "C" int pnol_ga_status_get(pnol_ga * ga, pnol_ga_status * s)
{
	if (!ga || !s) return PNOL_ERR_INVALID;
	s->generation = ga->generation; s->n_static = ga->n_static; s->stopped = ga->stopped; s->f_best = ga->f_best;
	s->stream_pos = ga->pos; s->n_elite = ga->nelite; s->n_elite_mut = ga->nelmut; s->n_cross = ga->ncross; s->n_rand = ga->nrand;
	return PNOL_OK;
}

extern "C" int pnol_ga_set_sharding(pnol_ctx * ctx, int mode)
{
	if (!ctx) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, mode >= 0 && mode <= 3, "ga_set_sharding: mode %d (0 auto, 1 rows, 2 sweep, 3 none)", mode);
	ctx->ga_sharding = mode;
	return PNOL_OK;
}

extern "C" int pnol_ga_peer_mode(pnol_ga * ga)
{
	return ga ? ga_pipe_peer_mode(ga) : 0;
}

extern "C" int pnol_ga_get_population(pnol_ga * ga, double * xpop, double * F)
{
	if (!ga) return PNOL_ERR_INVALID;
	return ga_pipe_get_population(ga, xpop, F);
}

extern "C" int pnol_ga_get_indices(pnol_ga * ga, int * cross_idx, int * mut_idx, int * elite_idx)
{
	if (!ga) return PNOL_ERR_INVALID;
	return ga_pipe_get_indices(ga, cross_idx, mut_idx, elite_idx);
}

// ---------------------------------------------------------------------------------------------------
// stand-alone stages on caller data
// ---------------------------------------------------------------------------------------------------
struct StageScratch {
	pnol_ctx * ctx;
	std::vector<void *> owned;
	GaScratch sc;
	SortScratch sort;
	double * stream_values = nullptr;
	int * exhausted = nullptr;
	~StageScratch() { cudaStreamSynchronize(ctx->stream); for (void * p : owned) cudaFree(p); }
	int init(pnol_ctx * c, long long npop, const pnol_stream_desc * stream)
	{
		ctx = c;
		auto alloc = [&](void ** p, size_t bytes) -> int {
			PNOL_CUDA(ctx, cudaMalloc(p, bytes ? bytes : 1));
			owned.push_back(*p);
			return PNOL_OK;
		};
		void * p;
		PNOL_CHECK(alloc(&p, (size_t) npop * 8)); sc.keys = (unsigned long long *) p;
		PNOL_CHECK(alloc(&p, (size_t) npop * 4)); sc.perm = (unsigned *) p;
		PNOL_CHECK(alloc(&p, (size_t) (npop + 16) * 4)); sc.u32a = (unsigned *) p;
		PNOL_CHECK(alloc(&p, (size_t) (npop + 16) * 8)); sc.u64a = (unsigned long long *) p;
		PNOL_CHECK(alloc(&p, (size_t) (npop / kScanTile + 16) * 8)); sc.scan_tmp = (unsigned long long *) p;
		PNOL_CHECK(alloc(&p, 64)); sc.total_dev = (unsigned long long *) p;
		PNOL_CHECK(alloc(&p, SortScratch::bytes(npop))); sort.carve(p, npop); sc.sort = &sort;
		PNOL_CHECK(alloc(&p, 64)); exhausted = (int *) p;
		PNOL_CUDA(ctx, cudaMemsetAsync(exhausted, 0, 16, ctx->stream));
		if (stream && stream->values && stream->n_values) {
			PNOL_CHECK(alloc(&p, stream->n_values * sizeof(double))); stream_values = (double *) p;
			PNOL_CUDA(ctx, cudaMemcpyAsync(stream_values, stream->values, stream->n_values * sizeof(double), cudaMemcpyDefault, ctx->stream));
		}
		return PNOL_OK;
	}
	StreamDev dev(const pnol_stream_desc * stream)
	{
		StreamDev st;
		st.values = stream_values; st.n_values = stream ? stream->n_values : 0; st.seed = stream ? stream->seed : 0;
		st.scale = stream ? stream->scale : 1.0; st.exhausted = exhausted;
		return st;
	}
	int check_stream()
	{
		int ex = 0;
		PNOL_CUDA(ctx, cudaMemcpyAsync(&ex, exhausted, sizeof ex, cudaMemcpyDeviceToHost, ctx->stream));
		PNOL_CHECK(finish(ctx));
		if (ex) { PNOL_SET_ERR(ctx, "ga: the explicit random stream is exhausted"); return PNOL_ERR_STREAM; }
		return PNOL_OK;
	}
};

extern "C" int pnol_ga_pop_sort(pnol_ctx * ctx, double * xpop, double * F, long long npop, int n)
{
	if (!ctx) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, xpop && F && npop >= 1 && n >= 1, "ga_pop_sort: bad arguments");
	StageScratch ss;
	PNOL_CHECK(ss.init(ctx, npop, nullptr));
	DevOut<double> dX, dF;
	PNOL_CHECK(dX.init(ctx, xpop, (size_t) npop * n, true));
	PNOL_CHECK(dF.init(ctx, F, (size_t) npop, true));
	double * Xs = nullptr; double * Fs = nullptr;
	PNOL_CUDA(ctx, cudaMalloc((void **) &Xs, (size_t) npop * n * sizeof(double))); ss.owned.push_back(Xs);
	PNOL_CUDA(ctx, cudaMalloc((void **) &Fs, (size_t) npop * sizeof(double))); ss.owned.push_back(Fs);
	PNOL_CHECK(ga_pop_sort_dev(ctx, dX.get(), dF.get(), npop, n, Xs, Fs, ss.sc));
	PNOL_CUDA(ctx, cudaMemcpyAsync(dX.get(), Xs, (size_t) npop * n * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
	PNOL_CUDA(ctx, cudaMemcpyAsync(dF.get(), Fs, (size_t) npop * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
	PNOL_CHECK(dX.commit());
	PNOL_CHECK(dF.commit());
	return finish(ctx);
}

static int ga_stage_common(pnol_ctx * ctx, bool identical, double * xpop, long long npop, int n, const double * xlb, const double * xub,
                           unsigned char * indicator, const pnol_stream_desc * stream, uint64_t * stream_pos)
{
	PNOL_REQUIRE(ctx, xpop && xlb && xub && stream && stream_pos && npop >= 1 && n >= 1, "ga stage: bad arguments");
	StageScratch ss;
	PNOL_CHECK(ss.init(ctx, npop, stream));
	DevOut<double> dX; DevIn<double> dlb, dub; DevOut<unsigned char> dind;
	PNOL_CHECK(dX.init(ctx, xpop, (size_t) npop * n, true));
	PNOL_CHECK(dlb.init(ctx, xlb, n));
	PNOL_CHECK(dub.init(ctx, xub, n));
	PNOL_CHECK(dind.init(ctx, indicator, (size_t) npop, true));
	StreamDev st = ss.dev(stream);
	if (identical) PNOL_CHECK(ga_check_identical_dev(ctx, dX.get(), npop, n, dlb.get(), dub.get(), dind.get(), st, stream_pos, ss.sc));
	else PNOL_CHECK(ga_check_bounds_dev(ctx, dX.get(), npop, n, dlb.get(), dub.get(), dind.get(), st, stream_pos, ss.sc));
	PNOL_CHECK(dX.commit());
	PNOL_CHECK(dind.commit());
	PNOL_CHECK(finish(ctx));
	return ss.check_stream();
}

extern "C" int pnol_ga_check_bounds(pnol_ctx * ctx, double * xpop, long long npop, int n, const double * xlb, const double * xub,
                                    unsigned char * indicator, const pnol_stream_desc * stream, uint64_t * stream_pos)
{
	if (!ctx) return PNOL_ERR_INVALID;
	return ga_stage_common(ctx, false, xpop, npop, n, xlb, xub, indicator, stream, stream_pos);
}

extern "C" int pnol_ga_check_identical(pnol_ctx * ctx, double * xpop, long long npop, int n, const double * xlb, const double * xub,
                                       unsigned char * indicator, const pnol_stream_desc * stream, uint64_t * stream_pos)
{
	if (!ctx) return PNOL_ERR_INVALID;
	return ga_stage_common(ctx, true, xpop, npop, n, xlb, xub, indicator, stream, stream_pos);
}
