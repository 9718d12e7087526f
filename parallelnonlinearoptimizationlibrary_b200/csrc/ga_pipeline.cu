// ga_pipeline.cu -- one generation of GeneticAlgorithmMPI::findMinBnd (Source/GeneticAlgorithmMPI.cpp:87-249) as a fused,
// sync-free kernel pipeline: every stage reads the stream position it starts from out of a status block in device memory, so the
// host enqueues the whole generation and synchronises ONCE at its end to read that block (stream position, best objective, error
// bits). Bit-exact with the oracle (tests/test_gpu_ga.py).
//
// What changed against the stage-by-stage generation of round 1 (2.25 ms at 1M x 32, ~105 launches, 8 host round trips):
//   * the population is never physically sorted. Rows stay where the generation that made them wrote them ("child order");
//     `perm` maps sorted position -> row. Parents are fetched through perm (they are random accesses anyway), so popSort's
//     gather of 256 MB in and 256 MB out per generation is gone; only pnol_ga_get_population materialises the sorted rows;
//   * crossover (:128-153): ONE kernel. Trials are evaluated once, accepted trials are ranked by a chained ("decoupled
//     look-back") prefix sum over ticketed tiles, and the tile that knows its ranks gathers the parent genes and writes the
//     children (three kernels + a host-driven batch loop before);
//   * mutation (:159-190): the sequential parser state at a block boundary is the offset of the next trial start; every CTA
//     tabulates offset -> (exit offset, children) for its sub-blocks, one small kernel composes the CTA tables, a third emits the
//     children of every sub-block. The window is sized from the measured acceptance rate; a window that turns out short sets an
//     error bit and the generation is redone with a longer one (the old population is untouched until the generation commits);
//   * child writers compute the row hash and the out-of-box gene count of the duplicate / bounds checks while they hold the row;
//   * duplicates (GeneticAlgorithm.cpp:313-344): "row i equals a LATER row" through an open-addressing table keyed by the row hash
//     that keeps the largest row index per hash; candidates are compared exactly, a hash collision without equality goes to an
//     exhaustive scan (never seen, but exact);
//   * bounds repair (:347-365) and duplicate replacement take their draws at positions from ONE packed prefix sum;
//   * popSort (:370-412): stable LSD radix sort of (key(F), row) in ONE cooperative kernel (grid-wide barriers between the
//     histogram and scatter phases of the passes, constant digits skipped on the device);
//   * several GPUs: rank r creates, repairs and evaluates child rows [r per, (r+1) per) only; parents are read from the owner's
//     memory over NVLink (CUDA IPC mappings), or from a local replica refreshed by an all-gather when peer mappings are
//     unavailable. Row hashes / box counts and objective values are all-gathered (two small collectives per generation).
#include "ga_common.cuh"

#include <cooperative_groups.h>
#include <math.h>
#include <algorithm>

namespace cg = cooperative_groups;

namespace pnol {

// error bits of GaDevStatus::error
enum { kGaErrDegenerate = 1, kGaErrCrossWindow = 2, kGaErrMutWindow = 4, kGaErrStream = 8 };

// device-resident bookkeeping of one generation
struct GaDevStatus {
	unsigned long long pos0;            // stream position at the start of the generation
	long long cross_last_trial;         // trial whose acceptance completed the crossover children (-1: no crossover)
	long long mut_last_q;               // stream offset (from the start of the mutation stage) of the last child's accepted trial
	long long mut_children;             // children the mutation window reaches
	unsigned long long pos_elite;       // start of the elite-mutation stage (set by the mutation emit kernel)
	unsigned long long ndup;            // duplicate rows replaced
	unsigned long long noob;            // out-of-box genes repaired
	unsigned long long pos_end;         // stream position after the generation
	double fbest;
	double max_fitness;
	int error;
	unsigned int pad0;
	int pad1;
	unsigned int nsuspect;              // rows whose hash matched a later row that is NOT equal (exhaustive check)
	int sort_result_in_alt;             // which buffer the radix sort ended in
	int sort_fallback;                  // bucket sort: a bucket outgrew one CTA, the radix kernel sorts instead
};

// Acceptance test of a selection trial, selectValue <= fitness[randomIndex] / maxFitness (Source/GeneticAlgorithmMPI.cpp:141), without
// the look-up for all but one trial in a thousand. The population is sorted by objective value, so ratio[k] = fitness[k] / maxFitness
// falls with k, and "ratio[k] >= s" holds exactly for k below a threshold. ga_prep_kernel tabulates K[b] = #{k : ratio[k] >= b / B},
// b = 0 .. B (B = kAccBuckets, stored behind the ratio array); for s in [b / B, (b + 1) / B):
//     k <  K[b + 1]  =>  ratio[k] >= (b + 1) / B > s   accepted,
//     k >= K[b]      =>  ratio[k] <  b / B <= s        rejected,
// and only K[b + 1] <= k < K[b] -- a fraction 1 / B of the trials -- reads ratio[k] itself. The table is 4 KB and stays in L1; the
// ratio array is 8 MB, and its 44 M random 8-byte reads per generation (one 32-byte L2 sector each) were what bounded the trial scans.
constexpr int kAccBuckets = 1024;

// K: the threshold table (global: behind the ratio array, read through L1; or a shared-memory copy). Branch-free up to the rare
// look-up: both thresholds are loaded unconditionally and only the ambiguous band touches ratio[].
__device__ __forceinline__ bool pipe_accept(double selectValue, int randomIndex, const double * __restrict__ ratio, const unsigned * K)
{
	const bool in01 = selectValue >= 0.0 && selectValue < 1.0;                                      // a draw of a [0, 1) stream
	const int b = in01 ? (int) (selectValue * kAccBuckets) : 0;
	const unsigned k_hi = K[b], k_lo = K[b + 1];
	bool acc = (unsigned) randomIndex < k_lo;
	if (!in01 || ((unsigned) randomIndex >= k_lo && (unsigned) randomIndex < k_hi)) acc = selectValue <= ratio[randomIndex];
	return acc;
}
__device__ __forceinline__ const unsigned * pipe_thresholds(const double * __restrict__ ratio, int Npop) { return reinterpret_cast<const unsigned *>(ratio + Npop); }

// index of the selection trial at stream position q (Source/GeneticAlgorithmMPI.cpp:134-144): round(u(q) Npop); 0 = rejected.
// ratio[k] = fitness[k] / maxFitness is tabulated once per generation (the same IEEE division, 1M instead of ~40M times)
__device__ __forceinline__ int pipe_trial(const StreamDev & st, unsigned long long q, const double * __restrict__ ratio, int Npop, const unsigned * K)
{
	const int randomIndex = (int) round(st.u(q) * Npop);
	const double selectValue = st.u(q + 1);
	if (randomIndex <= 0 || randomIndex >= Npop) return 0;
	return pipe_accept(selectValue, randomIndex, ratio, K) ? randomIndex : 0;
}

// the same for a counter stream whose state at position q is at hand (the second draw's state is one increment on)
__device__ __forceinline__ int pipe_trial_state(const StreamDev & st, unsigned long long z, const double * __restrict__ ratio, int Npop, const unsigned * K)
{
	int randomIndex = (int) round(st.from_state(z) * Npop);
	const double selectValue = st.from_state(z + StreamDev::kGamma);
	const bool in_range = randomIndex > 0 && randomIndex < Npop;
	if (!in_range) randomIndex = 0;                       // a valid index for the (discarded) test
	return (pipe_accept(selectValue, randomIndex, ratio, K) && in_range) ? randomIndex : 0;
}

// ---------------------------------------------------------------------------------------------------
// 0. fitness, acceptance ratios, elite objective values, status reset   (:101-124)
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
ga_prep_kernel(const double * __restrict__ Fs, int Npop, int Nelite, double * __restrict__ fitness, double * __restrict__ ratio,
               double * __restrict__ Fchild, GaDevStatus * __restrict__ S, unsigned long long pos0)
{
	const int k = blockIdx.x * blockDim.x + threadIdx.x;
	const double fw = Fs[Npop - 1];
	const double d0 = fw - Fs[0];
	const double maxFitness = d0 * d0;                                     // fitness[0]
	if (k < Npop) {
		const double d = fw - Fs[k];
		const double fit = d * d;                                          // pow(F[Npop-1] - F[k], 2)
		fitness[k] = fit;
		const double r = fit / maxFitness;
		ratio[k] = r;
		if (k < Nelite) Fchild[k] = Fs[k];
		// K[b] = k + 1 for the b with ratio[k] >= b / B > ratio[k + 1] (pipe_accept; B a power of two: ratio * B is exact). A
		// degenerate generation (NaN / inf ratios) is stopped by S->error before any trial reads the table.
		unsigned * K = reinterpret_cast<unsigned *>(ratio + Npop);
		if (r >= 0.0 && r <= 1.0) {
			const int hi_b = (int) (r * kAccBuckets);
			int lo_b = -1;
			if (k + 1 < Npop) {
				const double dn = fw - Fs[k + 1];
				const double rn = (dn * dn) / maxFitness;
				lo_b = (rn >= 0.0 && rn <= 1.0) ? (int) (rn * kAccBuckets) : hi_b;
			}
			for (int b = lo_b + 1; b <= hi_b; b++) K[b] = (unsigned) (k + 1);
		}
	}
	if (k == 0) {
		S->pos0 = pos0; S->cross_last_trial = -1; S->mut_last_q = -1; S->mut_children = 0; S->pos_elite = 0;
		S->ndup = 0; S->noob = 0; S->pos_end = 0; S->fbest = 0; S->max_fitness = maxFitness;
		// every trial would compare against NaN / inf: the reference spins forever in its while loops (SURVEY App. B)
		S->error = (!(maxFitness > 0) || isinf(maxFitness)) ? kGaErrDegenerate : 0;
		S->nsuspect = 0; S->sort_result_in_alt = 0; S->sort_fallback = 1;      // cleared by the bucket sort when it takes the sort
	}
}

// Row kernels: a warp holds FOUR rows, eight lanes each (lane g of a group takes genes g, g + 8, ...). With one row per warp a
// warp had a single 256-byte request in flight behind three dependent look-ups (child -> parent index -> perm -> row): these
// kernels ran at the latency of that chain, 0.07-0.2 ms each at 1M x 32. Four independent chains per warp instead.
constexpr int kRowLanes = 8;
constexpr int kRowsPerBlock = 256 / kRowLanes;
__device__ __forceinline__ unsigned long long group_sum(unsigned long long v)
{
	v += __shfl_xor_sync(0xffffffffu, v, 4); v += __shfl_xor_sync(0xffffffffu, v, 2); v += __shfl_xor_sync(0xffffffffu, v, 1);
	return v;
}
__device__ __forceinline__ unsigned group_sum(unsigned v)
{
	v += __shfl_xor_sync(0xffffffffu, v, 4); v += __shfl_xor_sync(0xffffffffu, v, 2); v += __shfl_xor_sync(0xffffffffu, v, 1);
	return v;
}

// elite rows (:108-118): child row k = sorted row k, for the rows this rank owns. The row hash is computed from the genes copied: the
// previous generation's hash of a row predates the duplicate replacement and bounds repair of ga_fix_kernel, which rewrite genes
__global__ void __launch_bounds__(256)
ga_elite_copy_kernel(RowTable cur, const unsigned * __restrict__ perm, long long lo, long long hi, int n, double * __restrict__ Xloc,
                     unsigned long long * __restrict__ hash_new, unsigned * __restrict__ bcount)
{
	const long long row = lo + (((long long) blockIdx.x * blockDim.x + threadIdx.x) / kRowLanes);
	const int g = threadIdx.x % kRowLanes;
	const bool live = row < hi;
	unsigned long long h = 0;
	if (live) {
		const double * s = cur.row(perm[row]);
		double * d = Xloc + (row - lo) * n;
		for (int j = g; j < n; j += kRowLanes) { const double v = __ldcg(s + j); d[j] = v; h += gene_hash(v, j); }
	}
	h = group_sum(h);
	if (live && g == 0) { hash_new[row] = h; bcount[row] = 0; }
}

// ---------------------------------------------------------------------------------------------------
// 1. crossover (:128-153) in one cooperative kernel. Trial t uses the draws (pos + 2t, pos + 2t + 1) whatever its outcome, and the
// g-th gene (child g / n, gene g % n) takes the g-th ACCEPTED trial. Per round every CTA owns a contiguous range of trials:
//   phase 1  evaluate the range, keep the acceptance bits in shared memory, publish the range's count;
//   -------  grid barrier: every CTA adds up the counts of the ranges before it (a few hundred values) = its first rank;
//   phase 2  walk the bits in chunks: accepted trials are compacted in rank order into shared memory, then all threads fetch the
//            parent genes (random reads) and write children and indices with consecutive threads on consecutive ranks.
// Rounds repeat until `need` genes are filled (the range length comes from the measured acceptance rate, so normally once).
// A first version ranked tiles with a chained look-back prefix instead: with ~900 tiles in flight every tile summed up to 28
// batches of predecessors before it could write, 0.41 ms; the barrier costs 3 us.
// ---------------------------------------------------------------------------------------------------
constexpr int kCrossThreads = 512;
constexpr int kCrossChunkWords = 256;                          // words (32 trials each) compacted at a time
constexpr int kCrossMaxWords = 6144;                           // per CTA and round (dynamic shared memory: 8 bytes per word)

__global__ void __launch_bounds__(kCrossThreads)
ga_cross_kernel(StreamDev st, GaDevStatus * __restrict__ S, const double * __restrict__ ratio, int Npop, long long need, int W,
                int max_rounds, unsigned long long * __restrict__ cta_counts, int * __restrict__ sel, RowTable cur,
                const unsigned * __restrict__ perm, int n, double * __restrict__ Xloc, long long own_lo, long long own_hi,
                long long row0)
{
	// own_lo / own_hi: child rows of the whole new population this rank owns; crossover child c is row row0 + c
	cg::grid_group grid = cg::this_grid();
	extern __shared__ unsigned cross_sm[];
	unsigned * s_bits = cross_sm;                                // W acceptance words
	unsigned * s_woff = cross_sm + W;                            // W: exclusive prefix of the words' popcounts inside the CTA
	unsigned short * s_list = (unsigned short *) (cross_sm + 2 * W);   // accepted trials of a chunk (offset inside the chunk), rank order
	__shared__ unsigned s_K[kAccBuckets + 1];                    // acceptance thresholds (pipe_accept)
	__shared__ unsigned long long s_red[kCrossThreads / 32];
	__shared__ unsigned long long s_before, s_total;
	if (S->error) return;                                        // set before the launch: uniform over the grid
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const int G = gridDim.x, cta = blockIdx.x;
	const unsigned long long pos = S->pos0;
	for (int b = tid; b <= kAccBuckets; b += kCrossThreads) s_K[b] = pipe_thresholds(ratio, Npop)[b];
	__syncthreads();
	unsigned long long done = 0;                                 // ranks filled by earlier rounds
	for (int pass = 0; pass < max_rounds; pass++) {
		const long long tb = ((long long) pass * G + cta) * (long long) W * 32;      // first trial of this CTA's range
		// ---- phase 1: acceptance bits and count of the range ----
		unsigned cnt = 0;
		if (st.values == nullptr) {
			// counter stream: the generator state of the lane's trial advances by a constant from word to word
			unsigned long long z = st.state(pos + 2ULL * (unsigned long long) (tb + (long long) warp * 32 + lane));
			const unsigned long long dz = (unsigned long long) (2 * 32 * (kCrossThreads / 32)) * StreamDev::kGamma;
			int w = warp;
			constexpr int kWS = kCrossThreads / 32;                  // word stride of a warp
			for (; w + 3 * kWS < W; w += 4 * kWS, z += 4 * dz) {
				// four independent trials per lane in flight
				const bool acc0 = pipe_trial_state(st, z, ratio, Npop, s_K) != 0;
				const bool acc1 = pipe_trial_state(st, z + dz, ratio, Npop, s_K) != 0;
				const bool acc2 = pipe_trial_state(st, z + 2 * dz, ratio, Npop, s_K) != 0;
				const bool acc3 = pipe_trial_state(st, z + 3 * dz, ratio, Npop, s_K) != 0;
				const unsigned m0 = __ballot_sync(0xffffffffu, acc0), m1 = __ballot_sync(0xffffffffu, acc1);
				const unsigned m2 = __ballot_sync(0xffffffffu, acc2), m3 = __ballot_sync(0xffffffffu, acc3);
				if (lane == 0) { s_bits[w] = m0; s_bits[w + kWS] = m1; s_bits[w + 2 * kWS] = m2; s_bits[w + 3 * kWS] = m3; }
				cnt += __popc(m0) + __popc(m1) + __popc(m2) + __popc(m3);      // the same in every lane
			}
			for (; w < W; w += kWS, z += dz) {
				const bool acc = pipe_trial_state(st, z, ratio, Npop, s_K) != 0;
				const unsigned m = __ballot_sync(0xffffffffu, acc);
				if (lane == 0) s_bits[w] = m;
				cnt += __popc(m);
			}
		} else {
			for (int w = warp; w < W; w += kCrossThreads / 32) {
				const long long t = tb + (long long) w * 32 + lane;
				const bool acc = pipe_trial(st, pos + 2ULL * (unsigned long long) t, ratio, Npop, s_K) != 0;
				const unsigned m = __ballot_sync(0xffffffffu, acc);
				if (lane == 0) s_bits[w] = m;
				cnt += __popc(m);
			}
		}
		if (lane == 0) s_red[warp] = cnt;
		__syncthreads();
		if (tid == 0) {
			unsigned long long c = 0;
			for (int w = 0; w < kCrossThreads / 32; w++) c += s_red[w];
			cta_counts[cta] = c;
		}
		grid.sync();
		// ---- first rank of this range = ranks of earlier rounds + counts of the ranges before it ----
		{
			unsigned long long before = 0, total = 0;
			for (int c = tid; c < G; c += kCrossThreads) { const unsigned long long v = cta_counts[c]; total += v; if (c < cta) before += v; }
			for (int o = 16; o > 0; o >>= 1) { before += __shfl_xor_sync(0xffffffffu, before, o); total += __shfl_xor_sync(0xffffffffu, total, o); }
			__syncthreads();                                     // s_red of phase 1 has been read
			if (lane == 0) { s_red[warp] = before; }
			__syncthreads();
			if (tid == 0) { unsigned long long b = 0; for (int w = 0; w < kCrossThreads / 32; w++) b += s_red[w]; s_before = b; }
			__syncthreads();
			if (lane == 0) { s_red[warp] = total; }
			__syncthreads();
			if (tid == 0) { unsigned long long b = 0; for (int w = 0; w < kCrossThreads / 32; w++) b += s_red[w]; s_total = b; }
			__syncthreads();
		}
		const unsigned long long first = done + s_before;
		const unsigned long long total = s_total;
		if (first < (unsigned long long) need) {
			// ---- exclusive prefix of the word popcounts (thread t owns words [t per, t per + per)) ----
			const int per = (W + kCrossThreads - 1) / kCrossThreads;
			unsigned loc = 0;
			for (int e = 0; e < per; e++) { const int w = tid * per + e; if (w < W) loc += __popc(s_bits[w]); }
			unsigned incl = loc;
#pragma unroll
			for (int o = 1; o < 32; o <<= 1) { const unsigned v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
			__syncthreads();
			if (lane == 31) s_red[warp] = incl;
			__syncthreads();
			if (tid == 0) { unsigned long long run = 0; for (int w = 0; w < kCrossThreads / 32; w++) { const unsigned long long v = s_red[w]; s_red[w] = run; run += v; } }
			__syncthreads();
			unsigned run = (unsigned) s_red[warp] + incl - loc;
			for (int e = 0; e < per; e++) { const int w = tid * per + e; if (w < W) { s_woff[w] = run; run += __popc(s_bits[w]); } }
			__syncthreads();
			// ---- phase 2: chunks of 256 words ----
			for (int c0 = 0; c0 < W; c0 += kCrossChunkWords) {
				const int c1 = c0 + kCrossChunkWords < W ? c0 + kCrossChunkWords : W;
				const unsigned coff = s_woff[c0];
				if (first + coff >= (unsigned long long) need) break;                        // uniform
				const unsigned cend = c1 < W ? s_woff[c1] : s_woff[W - 1] + __popc(s_bits[W - 1]);
				for (int w = c0 + warp; w < c1; w += kCrossThreads / 32) {
					const unsigned m = s_bits[w];
					if ((m >> lane) & 1u) s_list[s_woff[w] - coff + __popc(m & ((1u << lane) - 1))] = (unsigned short) ((w - c0) * 32 + lane);
				}
				__syncthreads();
				const unsigned long long left = (unsigned long long) need - (first + coff);
				const unsigned used = (unsigned long long) (cend - coff) < left ? (cend - coff) : (unsigned) left;
				// XpopNew[popIdx][i] = Xpop[indices[i]][i]  (:147-150): rank r is gene r % n of child r / n. One 64-bit division per
				// chunk, 32-bit arithmetic per element
				const long long r0 = (long long) (first + coff);
				const long long child0 = r0 / n;
				const unsigned gene0 = (unsigned) (r0 - child0 * n);
				for (unsigned e0 = tid; e0 < used; e0 += 4 * kCrossThreads) {
					// four independent chains (draw -> perm -> gene) per thread
					int parent[4];
					unsigned slot[4];
#pragma unroll
					for (int u = 0; u < 4; u++) {
						const unsigned e = e0 + u * kCrossThreads;
						parent[u] = 0;
						if (e < used) {
							const long long t = tb + (long long) c0 * 32 + s_list[e];
							parent[u] = (int) round(st.u(pos + 2ULL * (unsigned long long) t) * Npop);
							if (r0 + e == need - 1) S->cross_last_trial = t;
						}
					}
#pragma unroll
					for (int u = 0; u < 4; u++) slot[u] = perm[parent[u]];
#pragma unroll
					for (int u = 0; u < 4; u++) {
						const unsigned e = e0 + u * kCrossThreads;
						if (e < used) {
							sel[r0 + e] = parent[u];
							const unsigned ge = gene0 + e, dc = ge / (unsigned) n;
							const unsigned gene = ge - dc * (unsigned) n;
							const long long row = row0 + child0 + dc;
							if (row >= own_lo && row < own_hi) Xloc[(row - own_lo) * n + gene] = __ldcg(cur.row(slot[u]) + gene);
						}
					}
				}
				__syncthreads();
			}
		}
		done += total;
		if (done >= (unsigned long long) need) return;           // the same `total` in every CTA: uniform
		grid.sync();                                             // cta_counts is rewritten by the next round
	}
	if (cta == 0 && tid == 0) atomicOr(&S->error, kGaErrCrossWindow);
}

// row hash (and a zero box count: every gene of a crossover child is a parent's gene, which is inside the box) of rows [lo, hi)
__global__ void __launch_bounds__(256)
ga_rows_hash_kernel(const double * __restrict__ Xloc, long long own_lo, long long lo, long long hi, int n,
                    unsigned long long * __restrict__ hash_new, unsigned * __restrict__ bcount)
{
	const long long row = lo + (((long long) blockIdx.x * blockDim.x + threadIdx.x) / kRowLanes);
	const int g = threadIdx.x % kRowLanes;
	const bool live = row < hi;
	unsigned long long h = 0;
	if (live) {
		const double * x = Xloc + (row - own_lo) * n;
		for (int j = g; j < n; j += kRowLanes) h += gene_hash(x[j], j);
	}
	h = group_sum(h);
	if (live && g == 0) { hash_new[row] = h; if (bcount) bcount[row] = 0; }
}

// ---------------------------------------------------------------------------------------------------
// 2. mutation (:159-190). Stream layout from the stage start P1: [rejected trial (2 draws)]* [accepted trial (2)] [n mutation
// draws] per child. Trial starts are multiples of g = gcd(2, n + 2); "candidate" j is stream offset g j. A trial at candidate j
// moves the parser to j + stepA when accepted (stepA = (n + 2) / g) and to j + stepR otherwise (stepR = 2 / g).
// ---------------------------------------------------------------------------------------------------
constexpr int kMutSub = 1024;            // candidates per sub-block
constexpr int kMutThreads = 256;

struct MutGeom {
	int g, stepA, stepR, SD;             // SD = stepA: entry offsets 0 .. stepA-1 (in candidates) a block can be entered at
	int nsub;                            // sub-blocks per CTA
	int nctas;
};

__device__ __forceinline__ unsigned long long mut_stage_pos(const GaDevStatus * S)
{
	return S->pos0 + 2ULL * (unsigned long long) (S->cross_last_trial + 1);
}

// acceptance bits of the CTA's candidates, sub-block tables entry offset -> (exit offset, children), CTA table
__global__ void __launch_bounds__(kMutThreads)
ga_mut_tables_kernel(StreamDev st, const GaDevStatus * __restrict__ S, const double * __restrict__ ratio, int Npop, MutGeom G,
                     unsigned * __restrict__ accbits, int * __restrict__ sub_exit, int * __restrict__ sub_cnt,
                     int * __restrict__ cta_exit, int * __restrict__ cta_cnt)
{
	extern __shared__ unsigned mut_sm[];
	if (S->error) return;
	const int tid = threadIdx.x, lane = tid & 31;
	const int words = G.nsub * (kMutSub / 32);
	unsigned * bits = mut_sm;                                        // words
	int * t_exit = (int *) (bits + words);                           // nsub x SD
	int * t_cnt = t_exit + G.nsub * G.SD;                            // nsub x SD
	const unsigned long long P1 = mut_stage_pos(S);
	const long long cand0 = (long long) blockIdx.x * G.nsub * kMutSub;
	if (st.values == nullptr) {
		unsigned long long z = st.state(P1 + (unsigned long long) G.g * (unsigned long long) (cand0 + (long long) (tid >> 5) * 32 + lane));
		const unsigned long long dz = (unsigned long long) (G.g * 32 * (kMutThreads / 32)) * StreamDev::kGamma;
		for (int w = tid >> 5; w < words; w += kMutThreads / 32, z += dz) {
			const bool acc = pipe_trial_state(st, z, ratio, Npop, pipe_thresholds(ratio, Npop)) != 0;
			const unsigned m = __ballot_sync(0xffffffffu, acc);
			if (lane == 0) { bits[w] = m; accbits[(size_t) blockIdx.x * words + w] = m; }
		}
	} else {
		for (int w = tid >> 5; w < words; w += kMutThreads / 32) {
			const long long j = cand0 + (long long) w * 32 + lane;
			const bool acc = pipe_trial(st, P1 + (unsigned long long) G.g * (unsigned long long) j, ratio, Npop, pipe_thresholds(ratio, Npop)) != 0;
			const unsigned m = __ballot_sync(0xffffffffu, acc);
			if (lane == 0) { bits[w] = m; accbits[(size_t) blockIdx.x * words + w] = m; }
		}
	}
	__syncthreads();
	for (int e = tid; e < G.nsub * G.SD; e += kMutThreads) {
		const int sub = e / G.SD, d = e - sub * G.SD;
		const unsigned * b = bits + sub * (kMutSub / 32);
		int j = d, cnt = 0;
		while (j < kMutSub) {
			if ((b[j >> 5] >> (j & 31)) & 1u) { cnt++; j += G.stepA; } else j += G.stepR;
		}
		t_exit[e] = j - kMutSub; t_cnt[e] = cnt;
		sub_exit[(size_t) blockIdx.x * G.nsub * G.SD + e] = j - kMutSub;
		sub_cnt[(size_t) blockIdx.x * G.nsub * G.SD + e] = cnt;
	}
	__syncthreads();
	for (int d0 = tid; d0 < G.SD; d0 += kMutThreads) {
		int d = d0;
		int cnt = 0;
		for (int sub = 0; sub < G.nsub; sub++) {
			if (d >= kMutSub) { d -= kMutSub; continue; }            // a jump longer than a sub-block (n + 2 > 1024 g)
			cnt += t_cnt[sub * G.SD + d];
			d = t_exit[sub * G.SD + d];
		}
		cta_exit[(size_t) blockIdx.x * G.SD + d0] = d;
		cta_cnt[(size_t) blockIdx.x * G.SD + d0] = cnt;
	}
}

// entry offset and first child of every CTA; children the window reaches. Composition of the CTA tables in two levels out of
// shared memory: segments of 32 CTAs are composed for every entry offset in parallel, one thread walks the segments, then one
// thread per segment walks its CTAs. (One thread walking all CTA tables in global memory paid an L2 round trip per CTA: 0.2 ms.)
constexpr int kMutSeg = 32;
__global__ void __launch_bounds__(1024)
ga_mut_compose_kernel(GaDevStatus * __restrict__ S, MutGeom G, const int * __restrict__ cta_exit, const int * __restrict__ cta_cnt,
                      int * __restrict__ cta_entry, long long * __restrict__ cta_base, long long Nrand, int in_smem)
{
	extern __shared__ int compose_sm[];
	if (S->error) return;
	const size_t total = (size_t) G.nctas * G.SD;
	const int nseg = (G.nctas + kMutSeg - 1) / kMutSeg;
	int * s_cnt = compose_sm;                                        // nctas x SD   (only with in_smem)
	int * s_exit = compose_sm + (in_smem ? total : 0);               // nctas x SD
	int * g_exit = s_exit + (in_smem ? total : 0);                   // nseg x SD: segment tables
	long long * g_cnt = (long long *) (g_exit + (((size_t) nseg * G.SD + 1) & ~(size_t) 1));      // nseg x SD
	int * seg_entry = (int *) (g_cnt + (size_t) nseg * G.SD);        // nseg
	long long * seg_base = (long long *) (seg_entry + ((nseg + 1) & ~1));                          // nseg
	if (in_smem) {
		for (size_t e = threadIdx.x; e < total; e += blockDim.x) { s_cnt[e] = cta_cnt[e]; s_exit[e] = cta_exit[e]; }
		__syncthreads();
	}
	const int * cnt_t = in_smem ? s_cnt : cta_cnt;
	const int * exit_t = in_smem ? s_exit : cta_exit;
	const long long span = (long long) G.nsub * kMutSub;
	// a jump longer than a CTA's span cannot happen: SD <= span by construction (ga_pipe_enqueue)
	for (int e = threadIdx.x; e < nseg * G.SD; e += blockDim.x) {
		const int seg = e / G.SD;
		int d = e - seg * G.SD;
		long long cnt = 0;
		const int c1 = min(G.nctas, (seg + 1) * kMutSeg);
		for (int c = seg * kMutSeg; c < c1; c++) { cnt += cnt_t[(size_t) c * G.SD + d]; d = exit_t[(size_t) c * G.SD + d]; }
		g_exit[e] = d; g_cnt[e] = cnt;
	}
	__syncthreads();
	if (threadIdx.x == 0) {
		int d = 0;
		long long cnt = 0;
		for (int seg = 0; seg < nseg; seg++) {
			seg_entry[seg] = d; seg_base[seg] = cnt;
			cnt += g_cnt[seg * G.SD + d];
			d = g_exit[seg * G.SD + d];
		}
		S->mut_children = cnt;
		if (cnt < Nrand) atomicOr(&S->error, kGaErrMutWindow);
	}
	__syncthreads();
	for (int seg = threadIdx.x; seg < nseg; seg += blockDim.x) {
		int d = seg_entry[seg];
		long long cnt = seg_base[seg];
		const int c1 = min(G.nctas, (seg + 1) * kMutSeg);
		for (int c = seg * kMutSeg; c < c1; c++) {
			cta_entry[c] = d; cta_base[c] = cnt;
			cnt += cnt_t[(size_t) c * G.SD + d];
			d = exit_t[(size_t) c * G.SD + d];
		}
	}
	(void) span;
}

// every sub-block walks from its entry offset and records (stream offset of the accepted trial, parent index) of its children
__global__ void __launch_bounds__(kMutThreads)
ga_mut_emit_kernel(StreamDev st, GaDevStatus * __restrict__ S, int Npop, int n, MutGeom G, const unsigned * __restrict__ accbits,
                   const int * __restrict__ sub_exit, const int * __restrict__ sub_cnt, const int * __restrict__ cta_entry,
                   const long long * __restrict__ cta_base, long long Nrand, long long NeliteMutGenes,
                   long long * __restrict__ child_q, int * __restrict__ child_idx)
{
	extern __shared__ int emit_sm[];
	if (S->error) return;
	const int words = G.nsub * (kMutSub / 32);
	int * s_entry = emit_sm;                                         // nsub
	long long * s_base = (long long *) (emit_sm + ((G.nsub + 1) & ~1));      // nsub
	unsigned * s_bits = (unsigned *) (s_base + G.nsub);              // words
	const long long base0 = cta_base[blockIdx.x];
	if (base0 >= Nrand) return;
	int * s_texit = (int *) (s_bits + words);                        // nsub x SD
	int * s_tcnt = s_texit + G.nsub * G.SD;                          // nsub x SD
	for (int w = threadIdx.x; w < words; w += kMutThreads) s_bits[w] = accbits[(size_t) blockIdx.x * words + w];
	for (int e = threadIdx.x; e < G.nsub * G.SD; e += kMutThreads) {
		s_texit[e] = sub_exit[(size_t) blockIdx.x * G.nsub * G.SD + e];
		s_tcnt[e] = sub_cnt[(size_t) blockIdx.x * G.nsub * G.SD + e];
	}
	__syncthreads();
	if (threadIdx.x == 0) {
		// entry offsets of the sub-blocks: a serial walk, so out of shared memory (from global memory every step was an L2 round trip)
		int d = cta_entry[blockIdx.x];
		long long cnt = base0;
		for (int sub = 0; sub < G.nsub; sub++) {
			s_entry[sub] = d; s_base[sub] = cnt;
			if (d >= kMutSub) { d -= kMutSub; continue; }
			cnt += s_tcnt[sub * G.SD + d];
			d = s_texit[sub * G.SD + d];
		}
	}
	__syncthreads();
	const unsigned long long P1 = mut_stage_pos(S);
	for (int sub = threadIdx.x; sub < G.nsub; sub += kMutThreads) {
		long long k = s_base[sub];
		if (k >= Nrand) continue;
		const unsigned * b = s_bits + sub * (kMutSub / 32);
		const long long cand0 = ((long long) blockIdx.x * G.nsub + sub) * kMutSub;
		int j = s_entry[sub];
		while (j < kMutSub && k < Nrand) {
			if ((b[j >> 5] >> (j & 31)) & 1u) {
				const long long q = (long long) G.g * (cand0 + j);
				child_q[k] = q;
				child_idx[k] = (int) round(st.u(P1 + (unsigned long long) q) * Npop);
				if (k == Nrand - 1) {
					S->mut_last_q = q;
					S->pos_elite = P1 + (unsigned long long) q + 2ULL + (unsigned long long) n;
				}
				k++;
				j += G.stepA;
			} else j += G.stepR;
		}
	}
}

// XpopNew[popIdx][j] = Xpop[index][j] + spreadRatio (Xub[j] - Xlb[j]) timeRand()   (:182-186), one warp per child of this rank;
// row hash and out-of-box gene count on the way
__global__ void __launch_bounds__(256)
ga_mut_apply_kernel(StreamDev st, const GaDevStatus * __restrict__ S, RowTable cur, const unsigned * __restrict__ perm,
                    const long long * __restrict__ child_q, const int * __restrict__ child_idx, long long k_lo, long long k_hi,
                    long long row0, long long own_lo, int n, const double * __restrict__ lb, const double * __restrict__ ub,
                    double spreadRatio, double * __restrict__ Xloc, unsigned long long * __restrict__ hash_new,
                    unsigned * __restrict__ bcount)
{
	if (S->error) return;
	const long long k = k_lo + (((long long) blockIdx.x * blockDim.x + threadIdx.x) / kRowLanes);
	const int g = threadIdx.x % kRowLanes;
	const bool live = k < k_hi;
	unsigned long long h = 0;
	unsigned oob = 0;
	const long long row = row0 + k;
	if (live) {
		const unsigned long long q = mut_stage_pos(S) + (unsigned long long) child_q[k] + 2ULL;
		const double * src = cur.row(perm[child_idx[k]]);
		double * dst = Xloc + (row - own_lo) * n;
		// four genes of the lane at a time, all parent loads issued before the first store (the compiler keeps a load behind an
		// earlier store it cannot tell apart: one HBM round trip per gene otherwise)
		for (int j0 = g; j0 < n; j0 += 4 * kRowLanes) {
			double pv[4];
#pragma unroll
			for (int u = 0; u < 4; u++) { const int j = j0 + u * kRowLanes; pv[u] = j < n ? __ldcg(src + j) : 0.0; }
#pragma unroll
			for (int u = 0; u < 4; u++) {
				const int j = j0 + u * kRowLanes;
				if (j < n) {
					const double mutation = spreadRatio * (ub[j] - lb[j]) * st.u(q + (unsigned long long) j);
					const double v = pv[u] + mutation;
					dst[j] = v;
					h += gene_hash(v, j);
					oob += (v > ub[j] || v < lb[j]) ? 1u : 0u;
				}
			}
		}
	}
	h = group_sum(h); oob = group_sum(oob);
	if (live && g == 0) { hash_new[row] = h; bcount[row] = oob; }
}

// ---------------------------------------------------------------------------------------------------
// 3. mutations of the elite children (:195-207): two draws per gene at fixed positions
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
ga_elite_mut_kernel(StreamDev st, const GaDevStatus * __restrict__ S, RowTable cur, const unsigned * __restrict__ perm,
                    long long c_lo, long long c_hi, long long row0, long long own_lo, int n, int Nelite,
                    const double * __restrict__ lb, const double * __restrict__ ub, double eliteMutationSize,
                    double * __restrict__ Xloc, unsigned long long * __restrict__ hash_new, unsigned * __restrict__ bcount,
                    int * __restrict__ elite_idx)
{
	if (S->error) return;
	const long long c = c_lo + (((long long) blockIdx.x * blockDim.x + threadIdx.x) / kRowLanes);
	const int g = threadIdx.x % kRowLanes;
	const bool live = c < c_hi;
	const long long row = row0 + c;
	unsigned long long h = 0;
	unsigned oob = 0;
	if (live) {
		const unsigned long long P2 = S->pos_elite;
		double * dst = Xloc + (row - own_lo) * n;
		// four genes of the lane at a time: the four chains draw -> perm -> gene run side by side, stores last (see ga_mut_apply_kernel)
		for (int j0 = g; j0 < n; j0 += 4 * kRowLanes) {
			int idx[4];
			unsigned slot[4];
			double pv[4];
#pragma unroll
			for (int u = 0; u < 4; u++) {
				const int j = j0 + u * kRowLanes;
				const unsigned long long e = (unsigned long long) c * (unsigned long long) n + (unsigned long long) j;
				idx[u] = j < n ? (int) round(st.u(P2 + 2ULL * e) * Nelite) : 0;
			}
#pragma unroll
			for (int u = 0; u < 4; u++) slot[u] = perm[idx[u]];
#pragma unroll
			for (int u = 0; u < 4; u++) { const int j = j0 + u * kRowLanes; pv[u] = j < n ? __ldcg(cur.row(slot[u]) + j) : 0.0; }
#pragma unroll
			for (int u = 0; u < 4; u++) {
				const int j = j0 + u * kRowLanes;
				if (j < n) {
					const unsigned long long e = (unsigned long long) c * (unsigned long long) n + (unsigned long long) j;
					const double mutation = eliteMutationSize * (ub[j] - lb[j]) * st.u(P2 + 2ULL * e + 1ULL);
					const double v = pv[u] + mutation;
					dst[j] = v;
					elite_idx[e] = idx[u];
					h += gene_hash(v, j);
					oob += (v > ub[j] || v < lb[j]) ? 1u : 0u;
				}
			}
		}
	}
	h = group_sum(h); oob = group_sum(oob);
	if (live && g == 0) { hash_new[row] = h; bcount[row] = oob; }
}

// parent indices of ALL elite-mutation genes (pnol_ga_get_indices on a rank that only made its own children)
__global__ void ga_elite_idx_kernel(StreamDev st, unsigned long long P2, long long count, int Nelite, int * __restrict__ elite_idx)
{
	const long long e = (long long) blockIdx.x * blockDim.x + threadIdx.x;
	if (e < count) elite_idx[e] = (int) round(st.u(P2 + 2ULL * (unsigned long long) e) * Nelite);
}

// ---------------------------------------------------------------------------------------------------
// 4. identical children (GeneticAlgorithm.cpp:313-344): row i is replaced iff a LATER row equals it
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
ga_dup_insert_kernel(const unsigned long long * __restrict__ hash, long long Npop, unsigned long long * __restrict__ tkeys,
                     unsigned * __restrict__ tmax, unsigned mask)
{
	const long long row = (long long) blockIdx.x * blockDim.x + threadIdx.x;
	if (row >= Npop) return;
	unsigned long long h = hash[row];
	if (h == 0) h = 1;                                               // 0 marks an empty slot
	unsigned slot = (unsigned) (h >> 17) & mask;
	for (;;) {
		const unsigned long long prev = atomicCAS(&tkeys[slot], 0ULL, h);
		if (prev == 0ULL || prev == h) { atomicMax(&tmax[slot], (unsigned) row); return; }
		slot = (slot + 1) & mask;
	}
}

__device__ __forceinline__ bool rows_equal(const double * a, const double * b, int n)
{
	int same = 0;
	for (int j = 0; j < n; j++) same += (__ldcg(a + j) == __ldcg(b + j)) ? 1 : 0;      // the reference counts Nsame, NaN != NaN
	return same == n;
}

__global__ void __launch_bounds__(256)
ga_dup_query_kernel(const unsigned long long * __restrict__ hash, long long Npop, const unsigned long long * __restrict__ tkeys,
                    const unsigned * __restrict__ tmax, unsigned mask, RowTable xnew, int n, unsigned char * __restrict__ dupflag,
                    GaDevStatus * __restrict__ S, unsigned * __restrict__ suspects)
{
	const long long row = (long long) blockIdx.x * blockDim.x + threadIdx.x;
	if (row >= Npop) return;
	unsigned long long h = hash[row];
	if (h == 0) h = 1;
	unsigned slot = (unsigned) (h >> 17) & mask;
	while (tkeys[slot] != h) slot = (slot + 1) & mask;
	const unsigned last = tmax[slot];                                // largest row with this hash
	unsigned char flag = 0;
	if (last > (unsigned) row) {
		if (rows_equal(xnew.row((unsigned) row), xnew.row(last), n)) flag = 1;
		else suspects[atomicAdd(&S->nsuspect, 1u)] = (unsigned) row;   // a later row shares the hash but differs: look at all of them
	}
	dupflag[row] = flag;
}

// exhaustive check for the suspects (hash collisions, rows holding NaN): any later row with the same hash and equal genes?
__global__ void __launch_bounds__(256)
ga_dup_resolve_kernel(const unsigned long long * __restrict__ hash, long long Npop, RowTable xnew, int n,
                      unsigned char * __restrict__ dupflag, const GaDevStatus * __restrict__ S, const unsigned * __restrict__ suspects)
{
	__shared__ int found;
	const unsigned ns = S->nsuspect;
	for (unsigned s = blockIdx.x; s < ns; s += gridDim.x) {
		const unsigned row = suspects[s];
		const unsigned long long h = hash[row];
		if (threadIdx.x == 0) found = 0;
		__syncthreads();
		for (long long k = (long long) row + 1 + threadIdx.x; k < Npop; k += blockDim.x)
			if (hash[k] == h && rows_equal(xnew.row(row), xnew.row((unsigned) k), n)) found = 1;
		__syncthreads();
		if (threadIdx.x == 0 && found) dupflag[row] = 1;
		__syncthreads();
	}
}

// ---------------------------------------------------------------------------------------------------
// 5. stream offsets of the replaced rows and of the repaired genes: exclusive prefix sum of the packed value
//    (duplicate ? 1 : 0) << 40 | (duplicate ? 0 : out-of-box genes)     -- a replaced row is inside the box afterwards
// ---------------------------------------------------------------------------------------------------
constexpr int kPackTile = 2048;
__device__ __forceinline__ unsigned long long pack_row(const unsigned char * dupflag, const unsigned * bcount, long long row)
{
	return dupflag[row] ? (1ULL << 40) : (unsigned long long) bcount[row];
}

__global__ void __launch_bounds__(256)
ga_pack_sums_kernel(const unsigned char * __restrict__ dupflag, const unsigned * __restrict__ bcount, long long Npop,
                    unsigned long long * __restrict__ block_sums)
{
	__shared__ unsigned long long red[256];
	const long long base = (long long) blockIdx.x * kPackTile;
	unsigned long long s = 0;
	for (int e = 0; e < 8; e++) {
		const long long i = base + threadIdx.x * 8 + e;
		if (i < Npop) s += pack_row(dupflag, bcount, i);
	}
	red[threadIdx.x] = s;
	__syncthreads();
	for (int o = 128; o > 0; o >>= 1) {
		if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
		__syncthreads();
	}
	if (threadIdx.x == 0) block_sums[blockIdx.x] = red[0];
}

// every block adds up the sums of the blocks before it (a few hundred values), then scans its own tile
__global__ void __launch_bounds__(256)
ga_pack_scan_kernel(const unsigned char * __restrict__ dupflag, const unsigned * __restrict__ bcount, long long Npop,
                    const unsigned long long * __restrict__ block_sums, int nblocks, unsigned long long * __restrict__ offs,
                    GaDevStatus * __restrict__ S, long long NeliteMutGenes, int n)
{
	__shared__ unsigned long long red[256];
	unsigned long long before = 0;
	for (int b = threadIdx.x; b < (int) blockIdx.x; b += 256) before += block_sums[b];
	red[threadIdx.x] = before;
	__syncthreads();
	for (int o = 128; o > 0; o >>= 1) {
		if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
		__syncthreads();
	}
	before = red[0];
	__syncthreads();
	const long long base = (long long) blockIdx.x * kPackTile;
	unsigned long long v[8], s = 0;
	for (int e = 0; e < 8; e++) {
		const long long i = base + threadIdx.x * 8 + e;
		v[e] = i < Npop ? pack_row(dupflag, bcount, i) : 0;
		s += v[e];
	}
	red[threadIdx.x] = s;
	__syncthreads();
	for (int o = 1; o < 256; o <<= 1) {
		const unsigned long long t = threadIdx.x >= o ? red[threadIdx.x - o] : 0;
		__syncthreads();
		red[threadIdx.x] += t;
		__syncthreads();
	}
	unsigned long long run = before + (threadIdx.x ? red[threadIdx.x - 1] : 0);
	for (int e = 0; e < 8; e++) {
		const long long i = base + threadIdx.x * 8 + e;
		if (i < Npop) offs[i] = run;
		run += v[e];
	}
	if ((int) blockIdx.x == nblocks - 1 && threadIdx.x == 255) {
		S->ndup = run >> 40;
		S->noob = run & ((1ULL << 40) - 1);
	}
}

// replacement of duplicate rows and repair of out-of-box genes for the rows of this rank (eight lanes per row); evaluation flags
__global__ void __launch_bounds__(256)
ga_fix_kernel(StreamDev st, const GaDevStatus * __restrict__ S, long long own_lo, long long own_hi, int n, int Nelite,
              long long NeliteMutGenes, const double * __restrict__ lb, const double * __restrict__ ub,
              const unsigned char * __restrict__ dupflag, const unsigned * __restrict__ bcount,
              const unsigned long long * __restrict__ offs, double * __restrict__ Xloc, unsigned char * __restrict__ indicator)
{
	if (S->error) return;
	const long long row = own_lo + (((long long) blockIdx.x * blockDim.x + threadIdx.x) / kRowLanes);
	const int lane = threadIdx.x & 31, g = lane % kRowLanes, gshift = lane - g;
	const bool live = row < own_hi;
	const bool dup = live && dupflag[row] != 0;
	const unsigned cnt = live ? bcount[row] : 0;
	if (live && g == 0) indicator[row - own_lo] = (row >= Nelite || dup) ? 1 : 0;      // elites keep their value unless replaced (:116, :220)
	const bool work = dup || cnt != 0;
	if (!__any_sync(0xffffffffu, work)) return;
	const unsigned long long P3 = S->pos_elite + 2ULL * (unsigned long long) NeliteMutGenes;       // after the elite mutations
	const unsigned long long o = work ? offs[row] : 0;
	double * x = Xloc + (live ? (row - own_lo) * n : 0);
	// one draw per out-of-box gene in row-major order (GeneticAlgorithm.cpp:352-361), after all the replacement draws;
	// a replaced row takes n draws, Xpop[i][j] = Xlb[j] + (Xub[j] - Xlb[j]) timeRand(), rows in order (:335-338)
	unsigned long long k = dup ? P3 + (o >> 40) * (unsigned long long) n : P3 + S->ndup * (unsigned long long) n + (o & ((1ULL << 40) - 1));
	for (int j0 = 0; j0 < n; j0 += kRowLanes) {              // n is the same for every group: the ballots below are warp-uniform
		const int j = j0 + g;
		const bool in = work && j < n;
		const double v = in && !dup ? x[j] : 0.0;
		const bool out = in && (dup || v > ub[j] || v < lb[j]);
		const unsigned m = (__ballot_sync(0xffffffffu, out) >> gshift) & ((1u << kRowLanes) - 1);     // this group's genes
		if (out) x[j] = lb[j] + (ub[j] - lb[j]) * st.u(k + (unsigned long long) __popc(m & ((1u << g) - 1)));
		k += (unsigned long long) __popc(m);
	}
}

// ---------------------------------------------------------------------------------------------------
// 6. popSort (GeneticAlgorithm.cpp:370-412) == stable sort by objective value: LSD radix sort of (key(F), row), 8-bit digits,
// in ONE cooperative kernel. Each CTA owns a contiguous range of the array; per pass: digit counts of the range -> grid barrier
// -> every CTA derives its scatter offsets from all counts (and finds out whether one digit holds every key: pass skipped by all)
// -> stable ranking inside the range and scatter -> grid barrier.
// ---------------------------------------------------------------------------------------------------
constexpr int kSortThreads = 1024;
constexpr int kSortPerThread = 8;
constexpr int kSortChunk = kSortThreads * kSortPerThread;          // keys ranked at a time

__global__ void __launch_bounds__(kSortThreads, 1)
ga_sort_kernel(const double * __restrict__ F, long long N, long long range, unsigned long long * __restrict__ keys0,
               unsigned * __restrict__ vals0, unsigned long long * __restrict__ keys1, unsigned * __restrict__ vals1,
               unsigned * __restrict__ counts /* [256][gridDim] */, GaDevStatus * __restrict__ S, double * __restrict__ Fsorted,
               unsigned * __restrict__ perm_out)
{
	cg::grid_group grid = cg::this_grid();
	if (!S->sort_fallback) return;                                   // the bucket sort has produced Fsorted / perm_out (uniform over the grid)
	__shared__ unsigned wcount[kSortThreads / 32][256];              // 32 KB
	__shared__ unsigned long long dbase[256];
	__shared__ unsigned long long dtot[256];
	__shared__ int s_skip;
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const int G = gridDim.x, cta = blockIdx.x;
	const long long lo = (long long) cta * range < N ? (long long) cta * range : N, hi = lo + range < N ? lo + range : N;
	// keys from the objective values, values = row numbers
	for (long long i = lo + tid; i < hi; i += kSortThreads) { keys0[i] = double_to_key(F[i]); vals0[i] = (unsigned) i; }
	unsigned long long * kin = keys0, * kout = keys1;
	unsigned * vin = vals0, * vout = vals1;
	for (int pass = 0; pass < 8; pass++) {
		const int shift = 8 * pass;
		// ---- digit counts of this CTA's range ----
		for (int e = tid; e < (kSortThreads / 32) * 256; e += kSortThreads) (&wcount[0][0])[e] = 0;
		__syncthreads();
		// (warp-private counters, equal digits of a warp's 32 keys added once: the high bytes of the keys hold a handful of values,
		// and 7000 shared-memory atomics on one address per CTA and pass were the longest phase of the sort)
		for (long long c0 = lo; c0 < hi; c0 += kSortChunk) {
			// (all loads of the chunk first: the warp-synchronous counting below would otherwise pay one L2 round trip per round)
			unsigned dg[kSortPerThread];
#pragma unroll
			for (int r = 0; r < kSortPerThread; r++) {
				const long long i = c0 + (long long) r * kSortThreads + tid;
				dg[r] = i < hi ? (unsigned) ((kin[i] >> shift) & 255) : 256u;
			}
#pragma unroll
			for (int r = 0; r < kSortPerThread; r++) {
				const unsigned m = __match_any_sync(0xffffffffu, dg[r]);
				if (dg[r] < 256u && (m & ((1u << lane) - 1)) == 0) wcount[warp][dg[r]] += __popc(m);
				__syncwarp();
			}
		}
		__syncthreads();
		if (tid < 256) {
			unsigned c = 0;
			for (int w = 0; w < kSortThreads / 32; w++) c += wcount[w][tid];
			counts[(size_t) tid * G + cta] = c;
		}
		grid.sync();
		// ---- offsets of this range: total of the smaller digits + the same digit in the ranges before ----
		// (four threads per digit, loads issued in batches: one thread per digit adding G counts one after the other waited for
		// an L2 round trip per count, 40 us per pass)
		{
			const int d = tid & 255, part = tid >> 8;                // kSortThreads / 256 = 4 parts
			unsigned tot = 0, before = 0;
			const unsigned * c = counts + (size_t) d * G;
#pragma unroll 8
			for (int b = part; b < G; b += kSortThreads / 256) { const unsigned v = c[b]; tot += v; before += b < cta ? v : 0u; }
			wcount[part][d] = tot;
			wcount[4 + part][d] = before;
		}
		if (tid == 0) s_skip = 0;
		__syncthreads();
		if (tid < 256) {
			dtot[tid] = (unsigned long long) wcount[0][tid] + wcount[1][tid] + wcount[2][tid] + wcount[3][tid];
			dbase[tid] = (unsigned long long) wcount[4][tid] + wcount[5][tid] + wcount[6][tid] + wcount[7][tid];
		}
		__syncthreads();
		if (tid < 256 && dtot[tid] == (unsigned long long) N) s_skip = 1;      // one digit value holds every key: nothing moves
		__syncthreads();
		if (s_skip) { grid.sync(); continue; }                                 // uniform over the grid: all CTAs see the same totals
		if (warp == 0) {
			// dbase[d] += total of the smaller digits: lane l owns digits 8 l .. 8 l + 7 (a one-thread loop over 256 dependent
			// shared-memory updates took 8 us per pass)
			unsigned long long t[8], sum = 0;
#pragma unroll
			for (int e = 0; e < 8; e++) { t[e] = dtot[lane * 8 + e]; sum += t[e]; }
			unsigned long long incl = sum;
#pragma unroll
			for (int o = 1; o < 32; o <<= 1) { const unsigned long long v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
			unsigned long long run = incl - sum;
#pragma unroll
			for (int e = 0; e < 8; e++) { dbase[lane * 8 + e] += run; run += t[e]; }
		}
		__syncthreads();
		// ---- stable ranking and scatter, kSortChunk keys at a time ----
		for (long long c0 = lo; c0 < hi; c0 += kSortChunk) {
			for (int e = tid; e < (kSortThreads / 32) * 256; e += kSortThreads) (&wcount[0][0])[e] = 0;
			__syncthreads();
			// warp w owns 256 consecutive keys of the chunk; round r covers keys base + 32 r + lane: (warp, round, lane) is key order
			const long long base = c0 + (long long) warp * (32 * kSortPerThread);
			unsigned long long k[kSortPerThread];
			unsigned v[kSortPerThread];
			unsigned short rank[kSortPerThread];
#pragma unroll
			for (int r = 0; r < kSortPerThread; r++) {
				const long long i = base + r * 32 + lane;
				const bool valid = i < hi;
				k[r] = valid ? kin[i] : 0xFFFFFFFFFFFFFFFFULL;
				v[r] = valid ? vin[i] : 0;
			}
#pragma unroll
			for (int r = 0; r < kSortPerThread; r++) {
				const long long i = base + r * 32 + lane;
				const bool valid = i < hi;
				const unsigned d = valid ? (unsigned) ((k[r] >> shift) & 255) : 256u;
				const unsigned m = __match_any_sync(0xffffffffu, d);
				const unsigned ahead = __popc(m & ((1u << lane) - 1));
				unsigned prev = 0;
				if (valid) prev = wcount[warp][d];
				__syncwarp();
				if (valid && ahead == 0) wcount[warp][d] = prev + __popc(m);
				__syncwarp();
				rank[r] = (unsigned short) (prev + ahead);
			}
			__syncthreads();
			if (tid < 256) {                                        // exclusive scan over the warps, per digit
				unsigned run = 0;
				for (int w = 0; w < kSortThreads / 32; w++) { const unsigned c = wcount[w][tid]; wcount[w][tid] = run; run += c; }
				dtot[tid] = run;                                    // keys of this digit in the chunk
			}
			__syncthreads();
#pragma unroll
			for (int r = 0; r < kSortPerThread; r++) {
				const long long i = base + r * 32 + lane;
				if (i < hi) {
					const unsigned d = (unsigned) ((k[r] >> shift) & 255);
					const unsigned long long p = dbase[d] + wcount[warp][d] + rank[r];
					kout[p] = k[r];
					vout[p] = v[r];
				}
			}
			__syncthreads();
			if (tid < 256) dbase[tid] += dtot[tid];
			__syncthreads();
		}
		{ unsigned long long * t = kin; kin = kout; kout = t; unsigned * u = vin; vin = vout; vout = u; }
		grid.sync();
	}
	// sorted objective values and the permutation sorted position -> row
	for (long long i = lo + tid; i < hi; i += kSortThreads) { const unsigned r = vin[i]; Fsorted[i] = sorted_value(kin[i], r, F); perm_out[i] = r; }
	if (cta == 0 && tid == 0) S->sort_result_in_alt = (kin != keys0);
}

// ---------------------------------------------------------------------------------------------------
// 6'. popSort at large Npop: splitter buckets + one shared-memory sort per bucket, four short launches instead of the seven
// passes (fourteen grid barriers) of the radix kernel above (0.27 ms at 1M keys). The PREVIOUS generation's sorted objective values
// are the splitters (every Npop / 4096-th one): the distribution moves slowly from one generation to the next, so the buckets come
// out balanced (about 250 keys each; a CTA of four warps sorts up to kBsCap = 1024, a second launch the few buckets up to 8192). Keys are (key(F), row), unique, so the order inside a bucket
// before its sort does not matter and the result is the stable sort of the radix kernel, bit for bit. A bucket that outgrows
// kBsCapLarge (a population collapsing onto few values, a distribution that jumped) sets GaDevStatus::sort_fallback and the radix
// kernel, which is always enqueued behind and otherwise returns at once, redoes the sort.
// ---------------------------------------------------------------------------------------------------
constexpr int kBsBuckets = 4096;
constexpr int kBsLog2 = 12;
constexpr int kBsCap = 1024;       // keys of a bucket the small-bucket instantiation sorts
constexpr int kBsCapLarge = 8192;  // ... and the large-bucket one
constexpr int kBsCountThreads = 1024;

// bucket of a key = number of splitters <= key; tag[i] = bucket | rank inside (CTA, bucket) << kBsLog2; totals[bucket] += CTA counts
__global__ void __launch_bounds__(kBsCountThreads)
ga_bsort_count_kernel(const double * __restrict__ F, long long N, const double * __restrict__ Fs_old, unsigned * __restrict__ tag,
                      unsigned * __restrict__ totals)
{
	extern __shared__ unsigned long long bs_smem[];
	unsigned long long * spl = bs_smem;                            // spl[b], b >= 1: lower end of bucket b
	unsigned * hist = reinterpret_cast<unsigned *>(bs_smem + kBsBuckets);
	for (int b = threadIdx.x; b < kBsBuckets; b += kBsCountThreads) {
		spl[b] = b ? double_to_key(Fs_old[(long long) b * N / kBsBuckets]) : 0ULL;
		hist[b] = 0;
	}
	__syncthreads();
	const long long per = (N + gridDim.x - 1) / gridDim.x;
	const long long lo = min(N, (long long) blockIdx.x * per), hi = min(N, lo + per);
	const int lane = threadIdx.x & 31;
	for (long long i = lo + threadIdx.x; i < hi; i += kBsCountThreads) {
		const unsigned long long k = double_to_key(F[i]);
		int b = 0;                                                 // largest b with spl[b] <= k (spl[0] = 0)
#pragma unroll
		for (int step = kBsBuckets / 2; step > 0; step >>= 1)
			if (spl[b + step] <= k) b += step;
		// one atomic per distinct bucket of the warp: the elite rows arrive sorted, 32 neighbours share a bucket, and 6000 atomics of
		// one CTA on a few dozen addresses were the longest part of this kernel
		const unsigned act = __activemask();
		const unsigned m = __match_any_sync(act, b);
		const int leader = __ffs(m) - 1;
		unsigned base = 0;
		if (lane == leader) base = atomicAdd(&hist[b], (unsigned) __popc(m));
		base = __shfl_sync(act, base, leader);
		tag[i] = (unsigned) b | ((base + (unsigned) __popc(m & ((1u << lane) - 1))) << kBsLog2);
	}
	__syncthreads();
	for (int b = threadIdx.x; b < kBsBuckets; b += kBsCountThreads)
		if (hist[b]) atomicAdd(&totals[b], hist[b]);
}

// bucket starts (exclusive scan of the totals), scatter cursors = starts, totals cleared for the next sort
__global__ void __launch_bounds__(1024)
ga_bsort_scan_kernel(unsigned * __restrict__ totals, unsigned * __restrict__ bstart /* kBsBuckets + 1 */, unsigned * __restrict__ cursor,
                     GaDevStatus * __restrict__ S, unsigned * __restrict__ large /* [0]: count, then the buckets of more than kBsCap keys */)
{
	__shared__ unsigned wsum[32];
	__shared__ unsigned s_nlarge;
	if (threadIdx.x == 0) s_nlarge = 0;
	__syncthreads();
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	unsigned c[4];
#pragma unroll
	for (int q = 0; q < 4; q++) c[q] = totals[4 * tid + q];
	const unsigned mine = c[0] + c[1] + c[2] + c[3];
	unsigned incl = mine;
	for (int o = 1; o < 32; o <<= 1) { const unsigned v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
	if (lane == 31) wsum[warp] = incl;
	__syncthreads();
	if (warp == 0) {
		unsigned w = wsum[lane], wi = w;
		for (int o = 1; o < 32; o <<= 1) { const unsigned v = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= o) wi += v; }
		wsum[lane] = wi - w;
	}
	__syncthreads();
	unsigned run = wsum[warp] + incl - mine;
#pragma unroll
	for (int q = 0; q < 4; q++) {
		bstart[4 * tid + q] = run; cursor[4 * tid + q] = run; run += c[q]; totals[4 * tid + q] = 0;
		if (c[q] > (unsigned) kBsCap) large[1 + atomicAdd(&s_nlarge, 1u)] = (unsigned) (4 * tid + q);      // order is irrelevant
	}
	if (tid == 1023) bstart[kBsBuckets] = run;
	const int overflow = __syncthreads_or(c[0] > (unsigned) kBsCapLarge || c[1] > (unsigned) kBsCapLarge || c[2] > (unsigned) kBsCapLarge || c[3] > (unsigned) kBsCapLarge);
	if (tid == 0) { S->sort_fallback = overflow; large[0] = s_nlarge; }
}
static_assert(kBsBuckets == 4096 && (1 << kBsLog2) == kBsBuckets, "ga_bsort_scan_kernel scans four buckets per thread of one 1024-thread CTA");

// (key, row) of every entry to its bucket's region; a CTA reserves its share of a bucket with one atomic on the bucket's cursor
__global__ void __launch_bounds__(kBsCountThreads)
ga_bsort_scatter_kernel(const double * __restrict__ F, long long N, const unsigned * __restrict__ tag, unsigned * __restrict__ cursor,
                        unsigned long long * __restrict__ keys, unsigned * __restrict__ vals)
{
	__shared__ unsigned base[kBsBuckets];
	for (int b = threadIdx.x; b < kBsBuckets; b += kBsCountThreads) base[b] = 0;
	__syncthreads();
	const long long per = (N + gridDim.x - 1) / gridDim.x;          // the same ranges as ga_bsort_count_kernel (same grid)
	const long long lo = min(N, (long long) blockIdx.x * per), hi = min(N, lo + per);
	for (long long i = lo + threadIdx.x; i < hi; i += kBsCountThreads) atomicAdd(&base[tag[i] & (kBsBuckets - 1)], 1u);
	__syncthreads();
	for (int b = threadIdx.x; b < kBsBuckets; b += kBsCountThreads) {
		const unsigned c = base[b];
		base[b] = c ? atomicAdd(&cursor[b], c) : 0u;
	}
	__syncthreads();
	for (long long i = lo + threadIdx.x; i < hi; i += kBsCountThreads) {
		const unsigned t = tag[i];
		const unsigned p = base[t & (kBsBuckets - 1)] + (t >> kBsLog2);
		keys[p] = double_to_key(F[i]);
		vals[p] = (unsigned) i;
	}
}

// one CTA per bucket. The keys of a bucket lie between two neighbouring splitters, spread about evenly: a second, interpolating
// bucket pass inside the CTA (sub-bucket = floor((key - min) * nsub / (max - min + 1)), monotone in the key, about one key per
// sub-bucket) leaves almost nothing to compare -- every key counts the smaller (key, row) pairs of its own sub-bucket and that is
// its place. (A bitonic network over the bucket in shared memory: 2700 instructions per key, 78 us for the 4096 buckets.)
// Two instantiations: <128, 8> takes the buckets of up to 1024 keys (nearly all of them: 16 KB of shared memory, 13 CTAs per SM), <512, 16>
// the ones between 1025 and kBsCapLarge = 8192 keys (the first generations after a start, when the distribution still moves: the
// good children of a generation pile up below the old 10 % mark). Every CTA looks at its bucket's size and leaves if it is not its.
template <int kThreads, int kPer>
__global__ void __launch_bounds__(kThreads)
ga_bsort_bucket_kernel(const double * __restrict__ F, const unsigned long long * __restrict__ keys, const unsigned * __restrict__ vals,
                       const unsigned * __restrict__ bstart, const GaDevStatus * __restrict__ S, double * __restrict__ Fsorted, unsigned * __restrict__ perm_out, unsigned min_cnt,
                       const unsigned * __restrict__ list /* nullptr: bucket = blockIdx.x; else [0] = count, buckets follow */)
{
	constexpr int kCap = kThreads * kPer;
	extern __shared__ unsigned long long bs_smem[];
	unsigned long long * sk = bs_smem;                                   // kCap
	unsigned * sv = reinterpret_cast<unsigned *>(bs_smem + kCap);      // kCap
	unsigned * sstart = sv + kCap;                                       // kCap + 1: sub-bucket counts, then starts
	__shared__ unsigned long long red[2][kThreads / 32];
	__shared__ unsigned wtot[kThreads / 32];
	if (S->sort_fallback) return;
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const unsigned n_list = list ? list[0] : 1u;
	for (unsigned li = list ? blockIdx.x : 0u; li < n_list; li += gridDim.x) {
	const unsigned bucket = list ? list[1 + li] : blockIdx.x;
	const unsigned b0 = bstart[bucket], cnt = bstart[bucket + 1] - b0;
	if (cnt <= min_cnt || cnt > (unsigned) kCap) { if (list) continue; else return; }
	unsigned nsub = 32;
	while (nsub < cnt) nsub <<= 1;                      // <= kCap
	unsigned long long k[kPer];
	unsigned v[kPer], sub[kPer], slot[kPer];
	unsigned long long kmin = ~0ULL, kmax = 0ULL;
#pragma unroll
	for (int q = 0; q < kPer; q++) {
		const unsigned e = tid + q * kThreads;
		k[q] = e < cnt ? keys[b0 + e] : 0ULL;
		v[q] = e < cnt ? vals[b0 + e] : 0u;
		if (e < cnt) { kmin = min(kmin, k[q]); kmax = max(kmax, k[q]); }
	}
	for (unsigned e = tid; e <= nsub; e += kThreads) sstart[e] = 0;
	for (int o = 16; o > 0; o >>= 1) { kmin = min(kmin, __shfl_xor_sync(0xffffffffu, kmin, o)); kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, o)); }
	if (lane == 0) { red[0][warp] = kmin; red[1][warp] = kmax; }
	__syncthreads();
#pragma unroll
	for (int w = 0; w < kThreads / 32; w++) { kmin = min(kmin, red[0][w]); kmax = max(kmax, red[1][w]); }
	const double scale = (double) nsub / ((double) (kmax - kmin) + 1.0);
#pragma unroll
	for (int q = 0; q < kPer; q++) {
		const unsigned e = tid + q * kThreads;
		if (e < cnt) {
			const unsigned sb = (unsigned) min((double) (nsub - 1), (double) (k[q] - kmin) * scale);      // monotone in the key
			sub[q] = sb;
			slot[q] = atomicAdd(&sstart[sb], 1u);
		}
	}
	__syncthreads();
	// exclusive scan of the nsub counts: thread t owns entries [t per, (t + 1) per)
	{
		const unsigned per = nsub / kThreads > 0 ? nsub / kThreads : 1;      // nsub >= 32; with fewer entries than threads the tail threads idle
		unsigned c[kPer], mine = 0;
#pragma unroll
		for (int q = 0; q < kPer; q++) {
			const unsigned e = tid * per + q;
			c[q] = (q < (int) per && e < nsub) ? sstart[e] : 0u;
			mine += c[q];
		}
		unsigned incl = mine;
		for (int o = 1; o < 32; o <<= 1) { const unsigned t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
		if (lane == 31) wtot[warp] = incl;
		__syncthreads();
		unsigned run = incl - mine;
#pragma unroll
		for (int w = 0; w < kThreads / 32; w++) run += w < warp ? wtot[w] : 0u;
#pragma unroll
		for (int q = 0; q < kPer; q++) {
			const unsigned e = tid * per + q;
			if (q < (int) per && e < nsub) { sstart[e] = run; run += c[q]; }
		}
		if (tid == 0) sstart[nsub] = cnt;
	}
	__syncthreads();
#pragma unroll
	for (int q = 0; q < kPer; q++) {
		const unsigned e = tid + q * kThreads;
		if (e < cnt) { const unsigned p = sstart[sub[q]] + slot[q]; sk[p] = k[q]; sv[p] = v[q]; }
	}
	__syncthreads();
#pragma unroll
	for (int q = 0; q < kPer; q++) {
		const unsigned e = tid + q * kThreads;
		if (e < cnt) {
			const unsigned s0 = sstart[sub[q]], s1 = sstart[sub[q] + 1];
			unsigned smaller = 0;
			for (unsigned j = s0; j < s1; j++) {
				const unsigned long long kj = sk[j];
				smaller += (kj < k[q] || (kj == k[q] && sv[j] < v[q])) ? 1u : 0u;
			}
			Fsorted[b0 + s0 + smaller] = sorted_value(k[q], v[q], F);
			perm_out[b0 + s0 + smaller] = v[q];
		}
	}
	__syncthreads();          // shared memory is reused by the next bucket of the list
	}
}

constexpr size_t bsort_bucket_smem(int cap) { return (size_t) cap * 12 + ((size_t) cap + 1) * 4 + 8; }


// end of the generation: stream position, best objective. The kernels above read the stream speculatively (trial windows), so
// exhaustion of an explicit stream is decided here: the sequential algorithm consumed exactly the draws [0, pos_end)
__global__ void ga_finish_kernel(GaDevStatus * __restrict__ S, const double * __restrict__ Fsorted, long long NeliteMutGenes, int n,
                                 unsigned long long n_values)
{
	if (threadIdx.x != 0 || blockIdx.x != 0) return;
	if (S->error) return;
	S->pos_end = S->pos_elite + 2ULL * (unsigned long long) NeliteMutGenes + S->ndup * (unsigned long long) n + S->noob;
	S->fbest = Fsorted[0];
	if (S->pos_end > n_values) S->error |= kGaErrStream;
}

// dst[k] = src row perm[k] (materialising the sorted population for pnol_ga_get_population)
__global__ void __launch_bounds__(256)
ga_gather_sorted_kernel(RowTable cur, const unsigned * __restrict__ perm, long long k0, long long k1, int n, double * __restrict__ dst)
{
	const long long k = k0 + (((long long) blockIdx.x * blockDim.x + threadIdx.x) / kRowLanes);
	const int g = threadIdx.x % kRowLanes;
	if (k >= k1) return;
	const double * s = cur.row(perm[k]);
	double * d = dst + (k - k0) * n;
	for (int j = g; j < n; j += kRowLanes) d[j] = __ldcg(s + j);
}

__global__ void ga_iota_kernel(unsigned * __restrict__ perm, long long n)
{
	const long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n) perm[i] = (unsigned) i;
}

} // namespace pnol

using namespace pnol;

// ---------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------
struct GaPipe {
	// population rows of THIS rank, double-buffered: XL[cur] holds rows [lo, hi) of the current population in child order
	double * XL[2] = {nullptr, nullptr};
	int cur = 0;
	long long per = 0, lo = 0, hi = 0;               // rows per rank, own range
	RowTable table[2];                               // where all ranks' rows of XL[0] / XL[1] are, as seen from this GPU
	void * peer_maps[2][kGaMaxRanks] = {};           // IPC mappings to close
	double * replica[2] = {nullptr, nullptr};        // fallback without peer mappings: full copies refreshed by all-gather
	bool use_ipc = false;
	int R = 1;                                        // row partitions: the communicator's ranks (rows sharded) or 1 (rows replicated, sweep sharded)
	long long eper = 0;                               // rows replicated: rows of the fitness sweep per rank
	bool shard_sweep = true;                          // rows replicated: split the sweep and all-gather F (false: every rank sweeps everything)
	// replicated per-row arrays (sorted order: Fs, ratio, perm; child order: hash, bcount, dupflag, Fchild, offs)
	unsigned * perm[2] = {nullptr, nullptr};
	double * Fs[2] = {nullptr, nullptr};
	unsigned long long * hash[2] = {nullptr, nullptr};
	double * ratio = nullptr, * Fchild = nullptr;
	unsigned * bcount = nullptr;
	unsigned char * dupflag = nullptr, * indicator = nullptr;
	unsigned long long * offs = nullptr, * block_sums = nullptr;
	unsigned * suspects = nullptr;
	// gather staging (several ranks): [hash (8) | bcount (4)] per row, per rank slots
	unsigned char * hb_send = nullptr, * hb_recv = nullptr;
	double * f_recv = nullptr;
	// crossover
	unsigned long long * cross_counts = nullptr; int cross_grid = 0;
	// mutation
	void * mut_mem = nullptr; size_t mut_bytes = 0;
	// duplicate table
	unsigned long long * tkeys = nullptr; unsigned * tmax = nullptr; unsigned tmask = 0;
	// sort
	unsigned long long * skeys[2] = {nullptr, nullptr}; unsigned * svals[2] = {nullptr, nullptr}; unsigned * scounts = nullptr;
	int sort_grid = 0; long long sort_range = 0;
	unsigned * bs_tag = nullptr, * bs_totals = nullptr, * bs_start = nullptr, * bs_cursor = nullptr, * bs_large = nullptr; bool bs_on = false; int bs_grid = 0;
	// status
	GaDevStatus * status = nullptr; GaDevStatus * status_host = nullptr;
	unsigned long long pos_elite_last = 0;           // start of the last generation's elite-mutation stage (for get_indices)
	bool elite_idx_complete = true;
	double accept_rate = 0.25;
	std::vector<void *> owned;
};

namespace {

template <class T> int pipe_alloc(pnol_ga * ga, T ** p, size_t count)
{
	void * d = nullptr;
	PNOL_CUDA(ga->ctx, cudaMalloc(&d, (count ? count : 1) * sizeof(T)));
	ga->pipe->owned.push_back(d);
	*p = (T *) d;
	return PNOL_OK;
}

StreamDev pipe_stream(pnol_ga * ga)
{
	StreamDev st;
	st.values = ga->stream_values; st.n_values = ga->stream.n_values; st.seed = ga->stream.seed; st.scale = ga->stream.scale;
	st.exhausted = nullptr;            // speculative reads past the end are fine; ga_finish_kernel decides exhaustion
	return st;
}

unsigned blocks_for(long long threads, int per_block) { return (unsigned) std::max<long long>(1, (threads + per_block - 1) / per_block); }

// peer mappings of the ranks' row blocks (CUDA IPC over NVLink); false when any step fails (the caller falls back to replicas)
bool pipe_open_peers(pnol_ga * ga)
{
	pnol_ctx * ctx = ga->ctx;
	GaPipe * P = ga->pipe;
	const int R = ctx->nranks;
	static const bool disabled = [] { const char * e = getenv("PNOL_GA_NO_IPC"); return e && atoi(e) != 0; }();
	int ok = disabled ? 0 : 1;
	cudaIpcMemHandle_t mine[2];
	for (int b = 0; b < 2 && ok; b++) if (cudaIpcGetMemHandle(&mine[b], P->XL[b]) != cudaSuccess) { cudaGetLastError(); ok = 0; }
	// everybody must take the same path: exchange [ok | handles] through the communicator
	const size_t slot = 8 + 2 * sizeof(cudaIpcMemHandle_t);
	std::vector<unsigned char> send(slot, 0), recv(slot * R, 0);
	send[0] = (unsigned char) ok;
	memcpy(send.data() + 8, mine, sizeof mine);
	unsigned char * dsend = nullptr, * drecv = nullptr;
	if (cudaMalloc((void **) &dsend, slot) != cudaSuccess || cudaMalloc((void **) &drecv, slot * R) != cudaSuccess) return false;
	cudaMemcpyAsync(dsend, send.data(), slot, cudaMemcpyHostToDevice, ctx->stream);
	bool good = comm_allgather_bytes_dev(ctx, dsend, drecv, slot) == PNOL_OK;
	cudaMemcpyAsync(recv.data(), drecv, slot * R, cudaMemcpyDeviceToHost, ctx->stream);
	cudaStreamSynchronize(ctx->stream);
	cudaFree(dsend); cudaFree(drecv);
	if (!good) return false;
	for (int r = 0; r < R; r++) if (!recv[(size_t) r * slot]) return false;
	bool opened = true;
	for (int b = 0; b < 2; b++)
		for (int r = 0; r < R; r++) {
			if (r == ctx->rank) { P->table[b].base[r] = P->XL[b]; continue; }
			cudaIpcMemHandle_t h;
			memcpy(&h, recv.data() + (size_t) r * slot + 8 + b * sizeof h, sizeof h);
			void * p = nullptr;
			if (cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); opened = false; p = nullptr; }
			P->peer_maps[b][r] = p;
			P->table[b].base[r] = (const double *) p;
		}
	// again a common decision: one failed mapping anywhere sends every rank to the replica path
	double flag = opened ? 0.0 : 1.0;
	double * dflag = nullptr;
	if (cudaMalloc((void **) &dflag, sizeof(double)) != cudaSuccess) return false;
	cudaMemcpyAsync(dflag, &flag, sizeof flag, cudaMemcpyHostToDevice, ctx->stream);
	comm_allreduce_dev(ctx, dflag, 1);
	cudaMemcpyAsync(&flag, dflag, sizeof flag, cudaMemcpyDeviceToHost, ctx->stream);
	cudaStreamSynchronize(ctx->stream);
	cudaFree(dflag);
	if (flag != 0.0) {
		for (int b = 0; b < 2; b++)
			for (int r = 0; r < R; r++) if (P->peer_maps[b][r]) { cudaIpcCloseMemHandle(P->peer_maps[b][r]); P->peer_maps[b][r] = nullptr; }
		return false;
	}
	return true;
}

} // namespace

namespace pnol {

int ga_pipe_create(pnol_ga * ga)
{
	pnol_ctx * ctx = ga->ctx;
	const long long Npop = ga->prm.npop;
	const int n = ga->n;
	PNOL_REQUIRE(ctx, ctx->nranks <= kGaMaxRanks, "ga: at most %d ranks", kGaMaxRanks);
	GaPipe * P = new GaPipe();
	ga->pipe = P;
	// Several GPUs, two ways to split a generation (pnol_ga_set_sharding):
	//   rows  : rank r owns child rows [r per, (r+1) per): it creates, repairs and evaluates them, parents are read from their
	//           owners over NVLink. Memory per GPU falls with the GPU count; at 1M x 32 the gene-wise parent reads (8 bytes each,
	//           millions of them per rank) are latency-bound on the link and the generation is SLOWER than on one GPU
	//           (1.41 against 1.09 ms at 2 GPUs, profiles/).
	//   sweep : every rank keeps the whole population and makes all children (no row ever crosses a link); the fitness sweep
	//           is split and the objective values are all-gathered, as in the reference's evaluatePopulationParallel.
	//   none  : every rank keeps the population, makes all children AND sweeps all of them: replicas, no collective at all. For a
	//           cheap objective the split sweep does not pay for its all-gather: at 1M x 32 Rastrigin the whole sweep is 0.057 ms,
	//           an eighth of it 0.015 ms, the all-gather of the 8 MB of objective values 0.06 / 0.11 / 0.17 ms at 2 / 4 / 8 GPUs
	//           (a generation: 1.12 ms with the split sweep against 0.88 ms on one GPU).
	// auto = rows when two copies of the population exceed a quarter of the GPU's memory; otherwise sweep when the part of the sweep
	// that the other ranks take over costs more than the all-gather (built-in objectives: streaming time of the population at 4.6 TB/s
	// against 0.02 ms + 18 ns per KB gathered, the measured figures above; user functors: always, their cost is unknown), else none.
	int mode = ctx->ga_sharding;
	if (mode == 0) {
		size_t free_b = 0, total_b = 0;
		cudaMemGetInfo(&free_b, &total_b);
		if ((size_t) Npop * n * 16 > total_b / 4) mode = 1;
		else {
			const double Rr = (double) (ctx->nranks > 1 ? ctx->nranks : 1);
			const double sweep_ms = (double) Npop * (n + 1) * 8.0 / 4.6e9;
			const double gather_ms = 0.02 + (double) Npop * 8.0 / 1024.0 * 18e-6 * (1.0 - 1.0 / Rr) / 0.875;
			mode = (is_user_kind(ga->f->kind) || sweep_ms * (1.0 - 1.0 / Rr) > gather_ms) ? 2 : 3;
		}
	}
	P->shard_sweep = mode != 3;
	const int R = (ctx->nranks > 1 && mode == 1) ? ctx->nranks : 1;
	P->R = R;
	P->per = (Npop + R - 1) / R;
	P->lo = R > 1 ? std::min<long long>(P->per * ctx->rank, Npop) : 0;
	P->hi = R > 1 ? std::min<long long>(P->lo + P->per, Npop) : Npop;
	P->eper = (Npop + ctx->nranks - 1) / ctx->nranks;
	for (int b = 0; b < 2; b++) {
		PNOL_CHECK(pipe_alloc(ga, &P->XL[b], (size_t) P->per * n));
		PNOL_CHECK(pipe_alloc(ga, &P->perm[b], (size_t) Npop));
		PNOL_CHECK(pipe_alloc(ga, &P->Fs[b], (size_t) Npop));
		PNOL_CHECK(pipe_alloc(ga, &P->hash[b], (size_t) P->per * R));
		PNOL_CHECK(pipe_alloc(ga, &P->skeys[b], (size_t) Npop));
		PNOL_CHECK(pipe_alloc(ga, &P->svals[b], (size_t) Npop));
		P->table[b].per = P->per; P->table[b].n = n; P->table[b].nranks = R;
		for (int r = 0; r < kGaMaxRanks; r++) P->table[b].base[r] = nullptr;
		P->table[b].base[0] = P->XL[b];
	}
	PNOL_CHECK(pipe_alloc(ga, &P->ratio, (size_t) Npop + kAccBuckets / 2 + 2));      // + the acceptance thresholds K[0 .. kAccBuckets] (pipe_accept)
	PNOL_CHECK(pipe_alloc(ga, &P->Fchild, std::max((size_t) P->per * R, (size_t) P->eper * ctx->nranks)));
	PNOL_CHECK(pipe_alloc(ga, &P->bcount, (size_t) P->per * R));
	PNOL_CHECK(pipe_alloc(ga, &P->dupflag, (size_t) Npop));
	PNOL_CHECK(pipe_alloc(ga, &P->indicator, (size_t) P->per));
	PNOL_CHECK(pipe_alloc(ga, &P->offs, (size_t) Npop));
	PNOL_CHECK(pipe_alloc(ga, &P->block_sums, (size_t) (Npop + kPackTile - 1) / kPackTile + 1));
	PNOL_CHECK(pipe_alloc(ga, &P->suspects, (size_t) Npop));
	PNOL_CHECK(pipe_alloc(ga, &P->status, 1));
	PNOL_CUDA(ctx, cudaMallocHost((void **) &P->status_host, sizeof(GaDevStatus)));
	// crossover: cooperative grid (all CTAs resident), one count per CTA
	{
		int per_sm = 0;
		const size_t smem_max = (size_t) kCrossMaxWords * 8 + (size_t) kCrossChunkWords * 32 * 2;
		PNOL_CUDA(ctx, cudaFuncSetAttribute(ga_cross_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem_max));
		PNOL_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ga_cross_kernel, kCrossThreads, smem_max));
		PNOL_REQUIRE(ctx, per_sm >= 1, "ga: the crossover kernel does not fit an SM");
		P->cross_grid = ctx->sm_count * std::min(per_sm, 4);
		PNOL_CHECK(pipe_alloc(ga, &P->cross_counts, (size_t) P->cross_grid));
	}
	// duplicate table: at least 2 slots per row, power of two
	{
		unsigned slots = 1024;
		while ((long long) slots < 2 * Npop) slots <<= 1;
		P->tmask = slots - 1;
		PNOL_CHECK(pipe_alloc(ga, &P->tkeys, (size_t) slots));
		PNOL_CHECK(pipe_alloc(ga, &P->tmax, (size_t) slots));
	}
	// sort: one CTA per SM at most (cooperative launch), contiguous ranges that are multiples of the ranking chunk
	{
		int per_sm = 0;
		PNOL_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ga_sort_kernel, kSortThreads, 0));
		PNOL_REQUIRE(ctx, per_sm >= 1, "ga: the sort kernel does not fit an SM");
		const int maxg = ctx->sm_count * per_sm;
		long long range = (Npop + maxg - 1) / maxg;
		range = (range + kSortChunk - 1) / kSortChunk * kSortChunk;
		P->sort_range = range;
		P->sort_grid = (int) ((Npop + range - 1) / range);
		PNOL_CHECK(pipe_alloc(ga, &P->scounts, (size_t) 256 * P->sort_grid));
		// bucket sort in front of it at large Npop (PNOL_GA_SORT=radix: radix kernel only -- A/B runs and the equivalence test)
		const char * sort_env = getenv("PNOL_GA_SORT");              // read per pnol_ga_create
		const bool radix_only = sort_env && strcmp(sort_env, "radix") == 0;
		P->bs_on = !radix_only && Npop >= 65536;
		if (P->bs_on) {
			P->bs_grid = 2 * ctx->sm_count;                          // two 1024-thread CTAs per SM (count: 48 KB, scatter: 16 KB of shared memory)
			PNOL_CHECK(pipe_alloc(ga, &P->bs_tag, (size_t) Npop));
			PNOL_CHECK(pipe_alloc(ga, &P->bs_totals, (size_t) kBsBuckets));
			PNOL_CHECK(pipe_alloc(ga, &P->bs_start, (size_t) kBsBuckets + 1));
			PNOL_CHECK(pipe_alloc(ga, &P->bs_cursor, (size_t) kBsBuckets));
			PNOL_CHECK(pipe_alloc(ga, &P->bs_large, (size_t) kBsBuckets + 1));
			PNOL_CUDA(ctx, cudaMemsetAsync(P->bs_totals, 0, kBsBuckets * sizeof(unsigned), ctx->stream));
			PNOL_CUDA(ctx, cudaFuncSetAttribute(ga_bsort_count_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kBsBuckets * 12));
			PNOL_CUDA(ctx, cudaFuncSetAttribute(ga_bsort_bucket_kernel<512, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bsort_bucket_smem(kBsCapLarge)));
		}
	}
	if (ctx->nranks > 1) PNOL_CHECK(pipe_alloc(ga, &P->f_recv, std::max((size_t) P->per * R, (size_t) P->eper * ctx->nranks)));
	if (R > 1) {
		PNOL_CHECK(pipe_alloc(ga, &P->hb_send, (size_t) P->per * 12));
		PNOL_CHECK(pipe_alloc(ga, &P->hb_recv, (size_t) P->per * 12 * R));
		P->use_ipc = pipe_open_peers(ga);
		if (!P->use_ipc) {
			for (int b = 0; b < 2; b++) {
				PNOL_CHECK(pipe_alloc(ga, &P->replica[b], (size_t) P->per * R * n));
				for (int r = 0; r < R; r++) P->table[b].base[r] = P->replica[b] + (size_t) r * P->per * n;
			}
		}
	}
	return PNOL_OK;
}

void ga_pipe_destroy(pnol_ga * ga)
{
	GaPipe * P = ga->pipe;
	if (!P) return;
	cudaStreamSynchronize(ga->ctx->stream);
	for (int b = 0; b < 2; b++)
		for (int r = 0; r < kGaMaxRanks; r++) if (P->peer_maps[b][r]) cudaIpcCloseMemHandle(P->peer_maps[b][r]);
	for (void * p : P->owned) cudaFree(p);
	if (P->mut_mem) cudaFree(P->mut_mem);
	if (P->status_host) cudaFreeHost(P->status_host);
	delete P;
	ga->pipe = nullptr;
}

// refresh the local replica of buffer b from every rank's block (path without peer mappings)
static int pipe_refresh_replica(pnol_ga * ga, int b)
{
	GaPipe * P = ga->pipe;
	if (P->R <= 1 || P->use_ipc) return PNOL_OK;
	return comm_allgather_dev(ga->ctx, P->XL[b], P->replica[b], (size_t) P->per * ga->n);
}

// after pnol_ga_init: ga->Xpop / ga->F hold the sorted start population (replicated). Rows -> this rank's block, perm = identity.
int ga_pipe_reset(pnol_ga * ga)
{
	pnol_ctx * ctx = ga->ctx;
	GaPipe * P = ga->pipe;
	const long long Npop = ga->prm.npop;
	const int n = ga->n;
	P->cur = 0;
	if (P->hi > P->lo)
		PNOL_CUDA(ctx, cudaMemcpyAsync(P->XL[0], ga->Xpop + P->lo * n, (size_t) (P->hi - P->lo) * n * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
	PNOL_CUDA(ctx, cudaMemcpyAsync(P->Fs[0], ga->F, (size_t) Npop * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
	PNOL_LAUNCH(ctx, ga_iota_kernel, blocks_for(Npop, 256), 256, 0, P->perm[0], Npop);
	PNOL_CHECK(pipe_refresh_replica(ga, 0));
	P->elite_idx_complete = true;
	return PNOL_OK;
}

static int pipe_mut_reserve(pnol_ga * ga, size_t bytes)
{
	GaPipe * P = ga->pipe;
	if (bytes <= P->mut_bytes) return PNOL_OK;
	if (P->mut_mem) { PNOL_CUDA(ga->ctx, cudaStreamSynchronize(ga->ctx->stream)); cudaFree(P->mut_mem); P->mut_mem = nullptr; P->mut_bytes = 0; }
	PNOL_CUDA(ga->ctx, cudaMalloc(&P->mut_mem, bytes + bytes / 4));
	P->mut_bytes = bytes + bytes / 4;
	return PNOL_OK;
}

// enqueue one generation; window_scale > 1 after a short mutation window
static int pipe_enqueue(pnol_ga * ga, double window_scale)
{
	pnol_ctx * ctx = ga->ctx;
	GaPipe * P = ga->pipe;
	const int Npop = ga->prm.npop, n = ga->n, R = P->R;
	const long long Nelite = ga->nelite, Ncross = ga->ncross, Nrand = ga->nrand, NeliteMut = ga->nelmut;
	const int cur = P->cur, nxt = cur ^ 1;
	const RowTable & T = P->table[cur];
	const RowTable & Tn = P->table[nxt];
	StreamDev st = pipe_stream(ga);
	GaDevStatus * S = P->status;
	double * Xloc = P->XL[nxt];
	const long long lo = P->lo, hi = P->hi;
	auto clampr = [&](long long a, long long b, long long & x0, long long & x1) {   // [a, b) cut to the own rows
		x0 = std::max(a, lo); x1 = std::min(b, hi); if (x1 < x0) x1 = x0;
	};

	// 0. fitness / ratios / status
	{
		TimerScope ts(ctx, "ga_prep");
		PNOL_LAUNCH(ctx, ga_prep_kernel, blocks_for(Npop, 256), 256, 0, P->Fs[cur], Npop, (int) Nelite, ga->fitness, P->ratio, P->Fchild, S,
		            (unsigned long long) ga->pos);
		long long a, b;
		clampr(0, Nelite, a, b);
		if (b > a) PNOL_LAUNCH(ctx, ga_elite_copy_kernel, blocks_for((b - a) * kRowLanes, 256), 256, 0, T, P->perm[cur], a, b, n,
		                       Xloc + (a - lo) * n, P->hash[nxt], P->bcount);
	}
	// 1. crossover
	if (Ncross > 0) {
		TimerScope ts(ctx, "ga_crossover");
		long long need = Ncross * n;
		// range length per CTA from the measured acceptance rate (+ 8 %); a short range costs another round, not an error
		const double rate = std::max(P->accept_rate, 1.0 / 512);
		int W = (int) std::min<double>(kCrossMaxWords, std::max(8.0, (double) need / rate * 1.08 / (32.0 * P->cross_grid) + 1.0));
		int max_rounds = 1 << 16, npop_i = Npop, n_i = n;
		long long own_lo = lo, own_hi = hi, row0 = Nelite;
		const double * ratio = P->ratio;
		unsigned long long * counts = P->cross_counts;
		int * sel = ga->cross_idx;
		const unsigned * perm_c = P->perm[cur];
		RowTable Tc = T;
		void * args[] = {(void *) &st, (void *) &S, (void *) &ratio, (void *) &npop_i, (void *) &need, (void *) &W, (void *) &max_rounds, (void *) &counts,
		                 (void *) &sel, (void *) &Tc, (void *) &perm_c, (void *) &n_i, (void *) &Xloc, (void *) &own_lo, (void *) &own_hi, (void *) &row0};
		const size_t smem = (size_t) W * 8 + (size_t) kCrossChunkWords * 32 * 2;
		PNOL_CUDA(ctx, cudaLaunchCooperativeKernel((const void *) ga_cross_kernel, dim3(P->cross_grid), dim3(kCrossThreads), args, smem, ctx->stream));
		ctx->launches++;
		long long a, b;
		clampr(Nelite, Nelite + Ncross, a, b);
		if (b > a) PNOL_LAUNCH(ctx, ga_rows_hash_kernel, blocks_for((b - a) * kRowLanes, 256), 256, 0, Xloc, lo, a, b, n, P->hash[nxt], P->bcount);
	}
	// 2. mutation
	{
		TimerScope ts(ctx, "ga_mutation");
		const double spreadRatio = ga->prm.mutation_size * (ga->prm.max_generations - ga->generation) / ga->prm.max_generations;   // (:159)
		MutGeom G;
		G.g = (n % 2 == 0) ? 2 : 1;
		G.stepA = (n + 2) / G.g; G.stepR = 2 / G.g; G.SD = G.stepA;
		const double rate = std::max(P->accept_rate, 1e-3);
		// candidates per child: one accepted trial (stepA) and 1/rate - 1 rejected ones (stepR each)
		double cand = (double) Nrand * (G.stepA + G.stepR * (1.0 / rate - 1.0)) * 1.12 * window_scale + 8.0 * kMutSub;
		const size_t smem_cap = 96 * 1024;
		int nsub_max = (int) (smem_cap / ((size_t) (kMutSub / 32) * 4 + (size_t) G.SD * 8));
		PNOL_REQUIRE(ctx, nsub_max >= 1, "ga: n = %d is too large for the mutation tables", n);
		long long subs = (long long) (cand / kMutSub) + 1;
		const long long min_subs = ((long long) G.SD + kMutSub - 1) / kMutSub;            // a CTA spans at least the longest jump
		int nsub = (int) std::max<long long>(min_subs, std::min<long long>(nsub_max, (subs + 6LL * ctx->sm_count - 1) / (6LL * ctx->sm_count)));
		PNOL_REQUIRE(ctx, nsub <= nsub_max, "ga: n = %d is too large for the mutation tables", n);
		G.nsub = nsub;
		G.nctas = (int) ((subs + nsub - 1) / nsub);
		const size_t words = (size_t) G.nctas * nsub * (kMutSub / 32);
		const size_t tabs = (size_t) G.nctas * nsub * G.SD;
		const size_t ctab = (size_t) G.nctas * G.SD;
		size_t bytes = words * 4 + tabs * 8 + ctab * 12 + (size_t) G.nctas * 12 + 4096;
		PNOL_CHECK(pipe_mut_reserve(ga, bytes));
		unsigned char * p = (unsigned char *) P->mut_mem;
		auto take = [&](size_t b) { void * r = p; p += (b + 255) & ~(size_t) 255; return r; };
		int * cta_cnt = (int *) take(ctab * 4);
		long long * cta_base = (long long *) take((size_t) G.nctas * 8);
		unsigned * accbits = (unsigned *) take(words * 4);
		int * sub_exit = (int *) take(tabs * 4);
		int * sub_cnt = (int *) take(tabs * 4);
		int * cta_exit = (int *) take(ctab * 4);
		int * cta_entry = (int *) take((size_t) G.nctas * 4);
		const size_t smem1 = (size_t) nsub * (kMutSub / 32) * 4 + (size_t) nsub * G.SD * 8;
		PNOL_CUDA(ctx, cudaFuncSetAttribute(ga_mut_tables_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem1));
		PNOL_LAUNCH(ctx, ga_mut_tables_kernel, G.nctas, kMutThreads, smem1, st, S, P->ratio, Npop, G, accbits, sub_exit, sub_cnt, cta_exit, cta_cnt);
		{
			const int nseg = (G.nctas + kMutSeg - 1) / kMutSeg;
			const size_t seg_bytes = (size_t) nseg * G.SD * 12 + (size_t) nseg * 12 + 64;
			const int in_smem = ctab * 8 + seg_bytes <= 200 * 1024 ? 1 : 0;
			const size_t smem2 = (in_smem ? ctab * 8 : 0) + seg_bytes;
			PNOL_REQUIRE(ctx, smem2 <= 200 * 1024, "ga: n = %d is too large for the mutation tables", n);
			PNOL_CUDA(ctx, cudaFuncSetAttribute(ga_mut_compose_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem2));
			PNOL_LAUNCH(ctx, ga_mut_compose_kernel, 1, 1024, smem2, S, G, cta_exit, cta_cnt, cta_entry, cta_base, Nrand, in_smem);
		}
		const size_t smem3 = (size_t) ((nsub + 1) & ~1) * 4 + (size_t) nsub * 8 + (size_t) nsub * (kMutSub / 32) * 4 + (size_t) nsub * G.SD * 8;
		PNOL_CUDA(ctx, cudaFuncSetAttribute(ga_mut_emit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem3));
		PNOL_LAUNCH(ctx, ga_mut_emit_kernel, G.nctas, kMutThreads, smem3, st, S, Npop, n, G, accbits, sub_exit, sub_cnt, cta_entry, cta_base, Nrand,
		            NeliteMut * n, ga->mut_pos, ga->mut_idx);
		long long a, b;
		clampr(Nelite + Ncross, Nelite + Ncross + Nrand, a, b);
		if (b > a)
			PNOL_LAUNCH(ctx, ga_mut_apply_kernel, blocks_for((b - a) * kRowLanes, 256), 256, 0, st, S, T, P->perm[cur], ga->mut_pos, ga->mut_idx,
			            a - (Nelite + Ncross), b - (Nelite + Ncross), Nelite + Ncross, lo, n, ga->lb, ga->ub, spreadRatio, Xloc, P->hash[nxt], P->bcount);
	}
	// 3. elite mutations
	if (NeliteMut > 0) {
		TimerScope ts(ctx, "ga_elite_mutation");
		const long long row0 = Nelite + Ncross + Nrand;
		long long a, b;
		clampr(row0, row0 + NeliteMut, a, b);
		if (b > a)
			PNOL_LAUNCH(ctx, ga_elite_mut_kernel, blocks_for((b - a) * kRowLanes, 256), 256, 0, st, S, T, P->perm[cur], a - row0, b - row0, row0, lo, n,
			            (int) Nelite, ga->lb, ga->ub, ga->prm.elite_mutation_size, Xloc, P->hash[nxt], P->bcount, ga->elite_idx);
	}
	// hashes and box counts of all rows on every rank; the new rows where the duplicate check of another rank may look at them
	if (R > 1) {
		TimerScope ts(ctx, "ga_gather_hash");
		const size_t own = (size_t) (hi - lo);
		PNOL_CUDA(ctx, cudaMemsetAsync(P->hb_send, 0, (size_t) P->per * 12, ctx->stream));
		if (own) {
			PNOL_CUDA(ctx, cudaMemcpyAsync(P->hb_send, P->hash[nxt] + lo, own * 8, cudaMemcpyDeviceToDevice, ctx->stream));
			PNOL_CUDA(ctx, cudaMemcpyAsync(P->hb_send + (size_t) P->per * 8, P->bcount + lo, own * 4, cudaMemcpyDeviceToDevice, ctx->stream));
		}
		PNOL_CHECK(comm_allgather_bytes_dev(ctx, P->hb_send, P->hb_recv, (size_t) P->per * 12));
		for (int r = 0; r < R; r++) {
			const unsigned char * slot = P->hb_recv + (size_t) r * P->per * 12;
			PNOL_CUDA(ctx, cudaMemcpyAsync(P->hash[nxt] + (size_t) r * P->per, slot, (size_t) P->per * 8, cudaMemcpyDeviceToDevice, ctx->stream));
			PNOL_CUDA(ctx, cudaMemcpyAsync(P->bcount + (size_t) r * P->per, slot + (size_t) P->per * 8, (size_t) P->per * 4, cudaMemcpyDeviceToDevice, ctx->stream));
		}
		PNOL_CHECK(pipe_refresh_replica(ga, nxt));
	}
	// 4. identical children
	{
		TimerScope ts(ctx, "ga_check_identical");
		PNOL_CUDA(ctx, cudaMemsetAsync(P->tkeys, 0, ((size_t) P->tmask + 1) * 8, ctx->stream));
		PNOL_CUDA(ctx, cudaMemsetAsync(P->tmax, 0, ((size_t) P->tmask + 1) * 4, ctx->stream));
		PNOL_LAUNCH(ctx, ga_dup_insert_kernel, blocks_for(Npop, 256), 256, 0, P->hash[nxt], (long long) Npop, P->tkeys, P->tmax, P->tmask);
		PNOL_LAUNCH(ctx, ga_dup_query_kernel, blocks_for(Npop, 256), 256, 0, P->hash[nxt], (long long) Npop, P->tkeys, P->tmax, P->tmask, Tn, n,
		            P->dupflag, S, P->suspects);
		PNOL_LAUNCH(ctx, ga_dup_resolve_kernel, 64, 256, 0, P->hash[nxt], (long long) Npop, Tn, n, P->dupflag, S, P->suspects);
	}
	// 5. stream offsets, replacement and repair, evaluation flags
	{
		TimerScope ts(ctx, "ga_check_bounds");
		const int nb = (int) blocks_for(Npop, kPackTile);
		PNOL_LAUNCH(ctx, ga_pack_sums_kernel, nb, 256, 0, P->dupflag, P->bcount, (long long) Npop, P->block_sums);
		PNOL_LAUNCH(ctx, ga_pack_scan_kernel, nb, 256, 0, P->dupflag, P->bcount, (long long) Npop, P->block_sums, nb, P->offs, S, NeliteMut * n, n);
		if (hi > lo)
			PNOL_LAUNCH(ctx, ga_fix_kernel, blocks_for((hi - lo) * kRowLanes, 256), 256, 0, st, S, lo, hi, n, (int) Nelite, NeliteMut * n, ga->lb, ga->ub,
			            P->dupflag, P->bcount, P->offs, Xloc, P->indicator);
	}
	// 6. the fitness sweep over this rank's rows (:217)
	if (R == 1 && ctx->nranks > 1 && P->shard_sweep) {
		// rows replicated: this rank sweeps individuals [r eper, (r+1) eper) and the objective values are all-gathered
		// (GeneticAlgorithmMPI::evaluatePopulationParallel, Source/GeneticAlgorithmMPI.cpp:283-414)
		const long long elo = std::min<long long>(P->eper * ctx->rank, Npop), ehi = std::min<long long>(elo + P->eper, Npop);
		if (ehi > elo) PNOL_CHECK(launch_eval_batch(ctx, ga->f, Xloc + elo * n, ehi - elo, n, n, P->indicator + elo, P->Fchild + elo));
		TimerScope ts(ctx, "ga_gather_f");
		PNOL_CHECK(comm_allgather_dev(ctx, P->Fchild + elo, P->f_recv, (size_t) P->eper));
		PNOL_CUDA(ctx, cudaMemcpyAsync(P->Fchild, P->f_recv, (size_t) Npop * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
	} else if (hi > lo) PNOL_CHECK(launch_eval_batch(ctx, ga->f, Xloc, hi - lo, n, n, P->indicator, P->Fchild + lo));
	if (R > 1) {
		TimerScope ts(ctx, "ga_gather_f");
		// rows that were not evaluated (elites) already hold the same value on every rank, so gathering whole blocks is exact
		PNOL_CHECK(comm_allgather_dev(ctx, P->Fchild + lo, P->f_recv, (size_t) P->per));
		PNOL_CUDA(ctx, cudaMemcpyAsync(P->Fchild, P->f_recv, (size_t) P->per * R * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
		PNOL_CHECK(pipe_refresh_replica(ga, nxt));      // repaired / replaced genes
	}
	// 7. popSort (:220): sorted objective values and the permutation, rows stay where they are
	{
		TimerScope ts(ctx, "ga_pop_sort");
		const double * Fc = P->Fchild;
		long long N = Npop, range = P->sort_range;
		unsigned long long * k0 = P->skeys[0], * k1 = P->skeys[1];
		unsigned * v0 = P->svals[0], * v1 = P->svals[1], * sc = P->scounts, * po = P->perm[nxt];
		double * Fo = P->Fs[nxt];
		if (P->bs_on) {
			PNOL_LAUNCH(ctx, ga_bsort_count_kernel, P->bs_grid, kBsCountThreads, kBsBuckets * 12, Fc, N, (const double *) P->Fs[cur], P->bs_tag, P->bs_totals);
			PNOL_LAUNCH(ctx, ga_bsort_scan_kernel, 1, 1024, 0, P->bs_totals, P->bs_start, P->bs_cursor, S, P->bs_large);
			PNOL_LAUNCH(ctx, ga_bsort_scatter_kernel, P->bs_grid, kBsCountThreads, 0, Fc, N, (const unsigned *) P->bs_tag, P->bs_cursor, k0, v0);
			PNOL_LAUNCH(ctx, (ga_bsort_bucket_kernel<128, 8>), kBsBuckets, 128, bsort_bucket_smem(kBsCap), Fc, (const unsigned long long *) k0, (const unsigned *) v0,
			            (const unsigned *) P->bs_start, (const GaDevStatus *) S, Fo, po, 0u, (const unsigned *) nullptr);
			// the large buckets from the list the scan kernel made (4096 CTAs of 131 KB that only look and leave took 20 us)
			PNOL_LAUNCH(ctx, (ga_bsort_bucket_kernel<512, 16>), ctx->sm_count, 512, bsort_bucket_smem(kBsCapLarge), Fc, (const unsigned long long *) k0, (const unsigned *) v0,
			            (const unsigned *) P->bs_start, (const GaDevStatus *) S, Fo, po, (unsigned) kBsCap, (const unsigned *) P->bs_large);
		}
		void * args[] = {(void *) &Fc, (void *) &N, (void *) &range, (void *) &k0, (void *) &v0, (void *) &k1, (void *) &v1, (void *) &sc, (void *) &S,
		                 (void *) &Fo, (void *) &po};
		PNOL_CUDA(ctx, cudaLaunchCooperativeKernel((const void *) ga_sort_kernel, dim3(P->sort_grid), dim3(kSortThreads), args, 0, ctx->stream));
		ctx->launches++;
	}
	PNOL_LAUNCH(ctx, ga_finish_kernel, 1, 32, 0, S, P->Fs[nxt], NeliteMut * n, n,
	            ga->stream_values ? (unsigned long long) ga->stream.n_values : ~0ULL);
	PNOL_CUDA(ctx, cudaMemcpyAsync(P->status_host, S, sizeof(GaDevStatus), cudaMemcpyDeviceToHost, ctx->stream));
	return PNOL_OK;
}

// Source/GeneticAlgorithmMPI.cpp:87-249 (one pass of the while loop)
int ga_pipe_generation(pnol_ga * ga)
{
	pnol_ctx * ctx = ga->ctx;
	GaPipe * P = ga->pipe;
	const int n = ga->n;
	double scale = 1.0;
	for (int attempt = 0;; attempt++) {
		PNOL_CHECK(pipe_enqueue(ga, scale));
		PNOL_CHECK(finish(ctx));
		const GaDevStatus & H = *P->status_host;
		if (H.error & kGaErrStream) {
			PNOL_SET_ERR(ctx, "ga: the explicit random stream (%llu values) is exhausted", (unsigned long long) ga->stream.n_values);
			return PNOL_ERR_STREAM;
		}
		if (H.error & kGaErrDegenerate) {
			PNOL_SET_ERR(ctx, "ga: degenerate population (best and worst objective coincide or are not finite): selection cannot proceed");
			return PNOL_ERR_NONFINITE;
		}
		if (H.error & kGaErrCrossWindow) { PNOL_SET_ERR(ctx, "ga: selection accepts (almost) no trial"); return PNOL_ERR_NONFINITE; }
		if (H.error & kGaErrMutWindow) {
			// the mutation window was too short for Nrand children: nothing has been committed, redo the generation with a longer one
			if (attempt >= 6) { PNOL_SET_ERR(ctx, "ga: mutation selection accepts (almost) no trial"); return PNOL_ERR_NONFINITE; }
			const double got = (double) std::max<long long>(H.mut_children, 1);
			scale *= std::max(2.0, 1.3 * (double) ga->nrand / got);
			continue;
		}
		// commit
		if (ga->ncross > 0) P->accept_rate = (double) ga->ncross * n / (double) (H.cross_last_trial + 1);
		else if (H.mut_last_q >= 0) {
			const double g = (n % 2 == 0) ? 2.0 : 1.0;
			const double per_child = (double) (H.mut_last_q + 2 + n) / (double) ga->nrand;       // n + 2 / rate
			P->accept_rate = std::min(1.0, std::max(1e-3, 2.0 / std::max(per_child - n, 2.0)));
			(void) g;
		}
		P->pos_elite_last = H.pos_elite;
		P->elite_idx_complete = P->R <= 1;
		P->cur ^= 1;
		ga->pos = H.pos_end;
		const double Fbest = H.fbest;
		ga->f_best = Fbest;
		if (Fbest == ga->f_best_prev) ga->n_static++; else ga->n_static = 0;                    // (:234-249)
		if (ga->n_static > ga->prm.n_static_generations) { ga->stopped = 1; return PNOL_OK; }
		ga->f_best_prev = Fbest;
		ga->generation++;
		return PNOL_OK;
	}
}

int ga_pipe_peer_mode(pnol_ga * ga)
{
	if (ga->ctx->nranks <= 1) return 0;
	if (ga->pipe->R <= 1) return ga->pipe->shard_sweep ? 3 : 4;
	return ga->pipe->use_ipc ? 1 : 2;
}

int ga_pipe_get_population(pnol_ga * ga, double * xpop, double * F)
{
	pnol_ctx * ctx = ga->ctx;
	GaPipe * P = ga->pipe;
	const long long Npop = ga->prm.npop;
	const int n = ga->n;
	if (xpop) {
		// sorted rows into the full-size buffer that pnol_ga_init sorts through (idle between generations)
		PNOL_LAUNCH(ctx, ga_gather_sorted_kernel, blocks_for(Npop * kRowLanes, 256), 256, 0, P->table[P->cur], P->perm[P->cur], 0LL, Npop, n, ga->Xnew);
		PNOL_CUDA(ctx, cudaMemcpyAsync(xpop, ga->Xnew, (size_t) Npop * n * sizeof(double), cudaMemcpyDefault, ctx->stream));
	}
	if (F) PNOL_CUDA(ctx, cudaMemcpyAsync(F, P->Fs[P->cur], (size_t) Npop * sizeof(double), cudaMemcpyDefault, ctx->stream));
	PNOL_CHECK(finish(ctx));
	return PNOL_OK;
}

int ga_pipe_get_indices(pnol_ga * ga, int * cross_idx, int * mut_idx, int * elite_idx)
{
	pnol_ctx * ctx = ga->ctx;
	GaPipe * P = ga->pipe;
	if (elite_idx && !P->elite_idx_complete && ga->nelmut > 0) {
		const long long count = (long long) ga->nelmut * ga->n;
		PNOL_LAUNCH(ctx, ga_elite_idx_kernel, blocks_for(count, 256), 256, 0, pipe_stream(ga), P->pos_elite_last, count, ga->nelite, ga->elite_idx);
		P->elite_idx_complete = true;
	}
	if (cross_idx) PNOL_CUDA(ctx, cudaMemcpyAsync(cross_idx, ga->cross_idx, (size_t) ga->ncross * ga->n * sizeof(int), cudaMemcpyDefault, ctx->stream));
	if (mut_idx) PNOL_CUDA(ctx, cudaMemcpyAsync(mut_idx, ga->mut_idx, (size_t) ga->nrand * sizeof(int), cudaMemcpyDefault, ctx->stream));
	if (elite_idx) PNOL_CUDA(ctx, cudaMemcpyAsync(elite_idx, ga->elite_idx, (size_t) ga->nelmut * ga->n * sizeof(int), cudaMemcpyDefault, ctx->stream));
	return finish(ctx);
}

} // namespace pnol
