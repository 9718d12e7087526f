/* This Source Code Form is subject to the terms of the Mozilla Public License, v. 2.0 (LICENSE at the repository root). */
/*
 * functor_kernels.cuh -- the library's generic kernels and launchers as templates over a device functor, so that an objective
 * that is NOT one of the built-ins gets the same device path WITHOUT rebuilding libpnol_b200.so.
 *
 * The reference lets a user plug any objective into every stencil and algorithm by subclassing Objective / MultiObjective and
 * implementing objEval (Source/PNOL_Objective.hpp:29, :57). Here the device side of that plug-in point is:
 *
 *   1. write the functor once, __host__ __device__, to the concept of include/pnol/functors.hpp (scalar: eval(P, X, n), optionally
 *      partial(P, X, n, j) for pnol_gradient[_recur] and pnol_alpha_pool_analytic, and partial2(P, X, n, i, j) for pnol_hessian; residual
 *      model: residual(P, X, n, i), optionally jacobian(P, X, n, i, Ji) for
 *      PNOL_JAC_ANALYTIC; optionally kSeparable / sep_init / sep_term for the fast population sweep);
 *   2. in ONE .cu file of your own, compiled with
 *        nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -Xcompiler -ffp-contract=off -I<repo>/include ...
 *      write   PNOL_REGISTER_SCALAR_FUNCTOR(kind, MyFunctor, n_columns)   or   PNOL_REGISTER_RESIDUAL_FUNCTOR(kind, MyModel, n_columns)
 *      with a kind in [PNOL_F_USER_SCALAR_BASE, +1000) resp. [PNOL_F_USER_RESIDUAL_BASE, +1000);
 *   3. link that object into your program / shared library next to libpnol_b200.so. The macro registers a launch table
 *      (pnol_functor_vtable, include/pnol_b200.h) at load time, and for a scalar functor with partial() also its gradient and slope
 *      launchers (pnol_register_functor_gradient / _slope), with partial2() its Hessian launcher (pnol_register_functor_hessian), for
 *      a residual model its batched LM launcher (pnol_register_functor_lm_batch), for every scalar functor its batched BFGS and simplex
 *      launchers (pnol_register_functor_bfgs_batch / _simplex_batch);
 *      pnol_functor_create(kind) and every entry point that takes a functor -- pnol_eval_batch, pnol_fd_gradient[_recur],
 *      pnol_gradient[_recur], pnol_fd_hessian, pnol_hessian, pnol_alpha_pool, pnol_alpha_pool_analytic, the GA, pnol_residual_eval,
 *      pnol_fd_jacobian, pnol_lm_step / pnol_lm_iterate, pnol_lm_batch, pnol_bfgs_batch, pnol_simplex_batch -- then launch YOUR instantiations of the kernels below on the
 *      context's stream. The built-in objectives run through exactly these templates and tables (csrc/builtin_functors.cu).
 *
 * Everything here is header-only device / launch code; it needs nothing from the library but pnol_register_functor.
 */
#ifndef PNOL_DEVICE_FUNCTOR_KERNELS_CUH_
#define PNOL_DEVICE_FUNCTOR_KERNELS_CUH_

#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>

#include "../../pnol_b200.h"
#include "../functors.hpp"
#include "exact_div.cuh"
#include "random_stream.cuh"
#include "simplex_sort.hpp"

namespace pnol {
namespace dev {

/* ---- launch plumbing over the C launch environment (include/pnol_b200.h: pnol_launch_env) ---- */
#define PNOL_DEV_ERR(env, ...)                                                   \
	do {                                                                         \
		if ((env)->err && (env)->err_len) snprintf((env)->err, (env)->err_len, __VA_ARGS__); \
	} while (0)
#define PNOL_DEV_CUDA(env, call)                                                                      \
	do {                                                                                              \
		cudaError_t _e = (call);                                                                      \
		if (_e != cudaSuccess) {                                                                      \
			PNOL_DEV_ERR(env, "%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e));  \
			return PNOL_ERR_CUDA;                                                                     \
		}                                                                                             \
	} while (0)
#define PNOL_DEV_REQUIRE(env, cond, ...)        \
	do {                                        \
		if (!(cond)) {                          \
			PNOL_DEV_ERR(env, __VA_ARGS__);     \
			return PNOL_ERR_INVALID;            \
		}                                       \
	} while (0)
/* every launch is counted: pnol_ctx_launches() stays exact for user functors too */
#define PNOL_DEV_LAUNCH(env, kernel, grid, block, smem, ...)                                          \
	do {                                                                                              \
		kernel<<<(grid), (block), (smem), (cudaStream_t) (env)->stream>>>(__VA_ARGS__);               \
		if ((env)->launches) ++*(env)->launches;                                                      \
		cudaError_t _e = cudaGetLastError();                                                          \
		if (_e != cudaSuccess) {                                                                      \
			PNOL_DEV_ERR(env, "%s:%d: launch %s -> %s", __FILE__, __LINE__, #kernel, cudaGetErrorString(_e)); \
			return PNOL_ERR_CUDA;                                                                     \
		}                                                                                             \
	} while (0)

// ---------------------------------------------------------------------------------------------------
// a1 / a15: batch sweep. Replaces GeneticAlgorithmMPI::evaluatePopulationParallel
// (Source/GeneticAlgorithmMPI.cpp:283-414): F[i] = objEval(Xpop[i]) for rows with evaluateIndicator[i].
// ---------------------------------------------------------------------------------------------------
constexpr int kSweepThreads = 128;

template <class F>
__global__ void __launch_bounds__(kSweepThreads)
eval_batch_tile_kernel(FunctorParams P, const double * __restrict__ pts, long long B, int n, long long ld,
                       const unsigned char * __restrict__ indicator, double * __restrict__ f_out, int pitch)
{
	extern __shared__ double tile[];   // kSweepThreads rows x pitch
	const int tid = threadIdx.x;
	for (long long row0 = (long long) blockIdx.x * kSweepThreads; row0 < B; row0 += (long long) gridDim.x * kSweepThreads) {
		const int rows = (int) min((long long) kSweepThreads, B - row0);
		const bool mine = tid < rows && (indicator == nullptr || indicator[row0 + tid] != 0);
		// skip tiles with nothing to evaluate (the elite block of a GA generation)
		if (!__syncthreads_or(mine)) continue;

		if (ld == n && (n & 1) == 0 && ((((size_t) (pts + row0 * ld)) & 15) == 0)) {
			// contiguous tile: 16-byte coalesced loads
			const double2 * src = reinterpret_cast<const double2 *>(pts + row0 * ld);
			const int n2 = n >> 1;
			const int total2 = rows * n2;
			for (int e = tid; e < total2; e += kSweepThreads) {
				double2 v = __ldg(src + e);
				int r = e / n2, c = (e - r * n2) * 2;
				tile[r * pitch + c] = v.x;
				tile[r * pitch + c + 1] = v.y;
			}
		} else {
			const int total = rows * n;
			for (int e = tid; e < total; e += kSweepThreads) {
				int r = e / n, c = e - r * n;
				tile[r * pitch + c] = pts[(row0 + r) * ld + c];
			}
		}
		__syncthreads();
		if (mine) {
			PtrAcc acc{tile + tid * pitch};
			f_out[row0 + tid] = F::eval(P, acc, n);
		}
		__syncthreads();
	}
}

// Separable objectives (functors.hpp: kSeparable): f = init + sum_k term(x_k) in index order. One WARP takes 32 individuals:
// the terms are computed one gene per lane directly from coalesced row loads (no staging of the inputs, no block-wide
// barrier, so the warps of an SM drift apart and loads overlap arithmetic), parked in the warp's private shared-memory tile
// (odd pitch), and lane r then adds up the terms of individual r in index order -- the same operations in the same order as
// F::eval, hence the same bits. The tile kernel below spends its time in lock-step load / compute phases instead.
template <class F> struct is_separable {
	template <class T> static constexpr bool test(decltype(T::kSeparable) *) { return T::kSeparable; }
	template <class T> static constexpr bool test(...) { return false; }
	static constexpr bool value = test<F>(nullptr);
};

constexpr int kSepThreads = 128;

template <class F, int G>
__global__ void __launch_bounds__(kSepThreads)
eval_batch_separable_kernel(FunctorParams P, const double * __restrict__ pts, long long B, int n, long long ld,
                            const unsigned char * __restrict__ indicator, double * __restrict__ f_out, int pitch)
{
	extern __shared__ double sm[];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	double * tile = sm + (size_t) warp * 32 * pitch;
	const long long nbatch = (B + 31) / 32;
	const long long gwarp = (long long) blockIdx.x * (kSepThreads / 32) + warp, gwarps = (long long) gridDim.x * (kSepThreads / 32);
	for (long long b = gwarp; b < nbatch; b += gwarps) {
		const long long row0 = b * 32;
		const int rows = (int) min((long long) 32, B - row0);
		const bool mine = lane < rows && (indicator == nullptr || indicator[row0 + lane] != 0);
		if (!__any_sync(0xffffffffu, mine)) continue;       // e.g. the elite block of a GA generation
		const double * src = pts + row0 * ld;
		if (n == 32 && rows == 32) {
			// software pipeline: the loads of the next 8 rows are in flight while the terms of these 8 are computed
			double cur[G], nxt[G];
#pragma unroll
			for (int q = 0; q < G; q++) cur[q] = __ldg(src + q * ld + lane);
#pragma unroll
			for (int r0 = 0; r0 < 32; r0 += G) {
				if (r0 + G < 32) {
#pragma unroll
					for (int q = 0; q < G; q++) nxt[q] = __ldg(src + (r0 + G + q) * ld + lane);
				}
#pragma unroll
				for (int q = 0; q < G; q++) tile[(r0 + q) * pitch + lane] = F::sep_term(P, cur[q]);
#pragma unroll
				for (int q = 0; q < G; q++) cur[q] = nxt[q];
			}
		} else if (n == 32) {
			for (int r = 0; r < rows; r++) tile[r * pitch + lane] = F::sep_term(P, __ldg(src + r * ld + lane));
		} else {
			for (int r = 0; r < rows; r++)
				for (int k = lane; k < n; k += 32) tile[r * pitch + k] = F::sep_term(P, __ldg(src + r * ld + k));
		}
		__syncwarp();
		if (mine) {
			double v = F::sep_init(P, n);
			const double * mt = tile + lane * pitch;
#pragma unroll 8
			for (int k = 0; k < n; k++) v = v + mt[k];
			f_out[row0 + lane] = v;
		}
		__syncwarp();
	}
}

// Variant without shared memory: one individual per THREAD, its genes read with 256-bit loads (one full 32-byte sector per
// load, so the uncoalesced row walk still moves only the bytes it needs), four independent term chains in flight per thread.
__device__ __forceinline__ void ldg_f64x4(const double * p, double (&v)[4])
{
	asm volatile("ld.global.nc.L1::no_allocate.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(v[0]), "=d"(v[1]), "=d"(v[2]), "=d"(v[3]) : "l"(p));
}

__device__ __forceinline__ void ldg_f64x4p(const double * p, double * v)
{
	asm volatile("ld.global.nc.L1::no_allocate.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(v[0]), "=d"(v[1]), "=d"(v[2]), "=d"(v[3]) : "l"(p));
}

template <class F>
__global__ void __launch_bounds__(128)
eval_batch_rowwise_kernel(FunctorParams P, const double * __restrict__ pts, long long B, int n, long long ld,
                          const unsigned char * __restrict__ indicator, double * __restrict__ f_out)
{
	const long long b = (long long) blockIdx.x * blockDim.x + threadIdx.x;
	if (b >= B) return;
	if (indicator && !indicator[b]) return;
	const double * row = pts + b * ld;
	double v = F::sep_init(P, n);
	double cur[4], nxt[4];
	ldg_f64x4(row, cur);
	for (int k = 0; k < n; k += 4) {
		if (k + 4 < n) ldg_f64x4(row + k + 4, nxt);
		const double t0 = F::sep_term(P, cur[0]), t1 = F::sep_term(P, cur[1]), t2 = F::sep_term(P, cur[2]), t3 = F::sep_term(P, cur[3]);
		v = v + t0; v = v + t1; v = v + t2; v = v + t3;
#pragma unroll
		for (int q = 0; q < 4; q++) cur[q] = nxt[q];
	}
	f_out[b] = v;
}

// same, n a multiple of 16: four 256-bit loads (16 genes) in flight per thread ahead of the arithmetic, so that the memory system
// keeps working through the FP64-heavy terms (the kernel's FP64 issue time and its HBM time are about equal; with one load ahead
// they overlapped badly). Same order of additions, hence the same bits.
template <class F>
__global__ void __launch_bounds__(128)
eval_batch_rowwise16_kernel(FunctorParams P, const double * __restrict__ pts, long long B, int n, long long ld,
                            const unsigned char * __restrict__ indicator, double * __restrict__ f_out)
{
	const long long b = (long long) blockIdx.x * blockDim.x + threadIdx.x;
	if (b >= B) return;
	if (indicator && !indicator[b]) return;
	const double * row = pts + b * ld;
	double v = F::sep_init(P, n);
	double cur[16], nxt[16];
#pragma unroll
	for (int q = 0; q < 4; q++) ldg_f64x4p(row + 4 * q, cur + 4 * q);
	for (int k = 0; k < n; k += 16) {
		if (k + 16 < n) {
#pragma unroll
			for (int q = 0; q < 4; q++) ldg_f64x4p(row + k + 16 + 4 * q, nxt + 4 * q);
		}
#pragma unroll
		for (int q = 0; q < 16; q++) v = v + F::sep_term(P, cur[q]);
#pragma unroll
		for (int q = 0; q < 16; q++) cur[q] = nxt[q];
	}
	f_out[b] = v;
}

// large-n fallback: one thread per row straight from global memory
template <class F>
__global__ void eval_batch_direct_kernel(FunctorParams P, const double * __restrict__ pts, long long B, int n, long long ld,
                                         const unsigned char * __restrict__ indicator, double * __restrict__ f_out)
{
	long long b = (long long) blockIdx.x * blockDim.x + threadIdx.x;
	if (b >= B) return;
	if (indicator && !indicator[b]) return;
	PtrAcc acc{pts + b * ld};
	f_out[b] = F::eval(P, acc, n);
}


template <class F, bool kSep = is_separable<F>::value> struct SeparableLaunch {
	static int run(const pnol_launch_env *, const FunctorParams &, const double *, long long, int, long long, const unsigned char *, double *, bool * done)
	{
		*done = false;
		return PNOL_OK;
	}
};
template <class F> struct SeparableLaunch<F, true> {
	static int run(const pnol_launch_env * env, const FunctorParams & P, const double * pts, long long B, int n, long long ld,
	               const unsigned char * indicator, double * f_out, bool * done)
	{
		*done = false;
		const int pitch = n | 1;
		const size_t smem = (size_t) (kSepThreads / 32) * 32 * pitch * sizeof(double);
		const bool rowwise_ok = n % 4 == 0 && ld % 4 == 0 && (((size_t) pts) & 31) == 0;
		if (!rowwise_ok && (smem > env->smem_optin / 2 || B < 64 || n < 24)) return PNOL_OK;   // long / very short genomes, tiny batches: the generic kernels
		// aligned rows: the row-wise kernel (0.059 ms at 1M x 32, 68 % of the HBM roofline; the warp-tile kernel below it 0.078 ms)
		if (rowwise_ok) {
			if (n % 16 == 0)
				PNOL_DEV_LAUNCH(env, eval_batch_rowwise16_kernel<F>, (unsigned) ((B + 127) / 128), 128, 0, P, pts, B, n, ld, indicator, f_out);
			else
				PNOL_DEV_LAUNCH(env, eval_batch_rowwise_kernel<F>, (unsigned) ((B + 127) / 128), 128, 0, P, pts, B, n, ld, indicator, f_out);
			*done = true;
			return PNOL_OK;
		}
		// unaligned rows: the warp-tile kernel with eight rows loaded ahead, at most one wave of CTAs
		auto kern = eval_batch_separable_kernel<F, 8>;
		PNOL_DEV_CUDA(env, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
		int per_sm = 1;
		PNOL_DEV_CUDA(env, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kSepThreads, smem));
		if (per_sm < 1) per_sm = 1;
		const long long blocks = ((B + 31) / 32 + kSepThreads / 32 - 1) / (kSepThreads / 32);
		const long long grid = blocks < (long long) env->sm_count * per_sm ? blocks : (long long) env->sm_count * per_sm;
		PNOL_DEV_LAUNCH(env, kern, (unsigned) grid, kSepThreads, smem, P, pts, B, n, ld, indicator, f_out, pitch);
		*done = true;
		return PNOL_OK;
	}
};

/* a1 / a15: f_out[b] = F(pts[b * ld ..]) for rows with indicator[b] != 0 */
template <class F>
int eval_batch(const pnol_launch_env * env, const FunctorParams & P, const double * pts, long long B, int n, long long ld,
               const unsigned char * indicator, double * f_out)
{
	if (B <= 0) return PNOL_OK;
	bool done = false;
	int st = SeparableLaunch<F>::run(env, P, pts, B, n, ld, indicator, f_out, &done);
	if (st != PNOL_OK || done) return st;
	int pitch = n | 1;
	size_t smem = (size_t) kSweepThreads * pitch * sizeof(double);
	if (smem <= env->smem_optin) {
		auto kern = eval_batch_tile_kernel<F>;
		PNOL_DEV_CUDA(env, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
		long long tiles = (B + kSweepThreads - 1) / kSweepThreads;
		size_t q = env->smem_optin / (smem > 0 ? smem : 1);
		int per_sm = (int) (q < 1 ? 1 : (q > 8 ? 8 : q));
		long long grid = tiles < (long long) env->sm_count * per_sm ? tiles : (long long) env->sm_count * per_sm;
		PNOL_DEV_LAUNCH(env, kern, (unsigned) grid, kSweepThreads, smem, P, pts, B, n, ld, indicator, f_out, pitch);
	} else {
		auto kern = eval_batch_direct_kernel<F>;
		PNOL_DEV_LAUNCH(env, kern, (unsigned) ((B + 127) / 128), 128, 0, P, pts, B, n, ld, indicator, f_out);
	}
	return PNOL_OK;
}

// ---------------------------------------------------------------------------------------------------
// a3 / a4 / a5: forward-difference stencil points. Point i in [i0, i1) is the base point with coordinate
// pos[i] (pos == nullptr: i itself) incremented by dx[i]; the base value f0 is produced by one extra thread
// when f0_out != nullptr. Replaces the evaluation loops of Objective::gradientApproximation[MPI]
// (Source/PNOL_Objective.cpp:19-32, 125-145) and the Recur variants (:345-358, :399-420).
// ---------------------------------------------------------------------------------------------------
constexpr int kFdThreads = 32;

template <class F>
__global__ void __launch_bounds__(kFdThreads)
fd_points_kernel(FunctorParams P, const double * __restrict__ xfull, int nfull, const int * __restrict__ pos,
                 const double * __restrict__ dx, int i0, int i1, double * __restrict__ fdx_out, double * __restrict__ f0_out)
{
	extern __shared__ double xs[];
	for (int j = threadIdx.x; j < nfull; j += blockDim.x) xs[j] = xfull[j];
	__syncthreads();
	int i = i0 + blockIdx.x * blockDim.x + threadIdx.x;
	if (i < i1) {
		// pos[i] < 0: reduced variable i has no slot in the full point (more reduced entries than free variables: the reference's
		// objEvalRecur never reads it, Source/PNOL_Objective.cpp:311-323), so its stencil point is the base point itself
		int pi = pos ? pos[i] : i;
		PerturbAcc acc{xs, pi, pi >= 0 ? xs[pi] + dx[i] : 0.0};   // XdX[i] = XdX[i] + dX[i]  (Source/PNOL_Objective.cpp:27)
		fdx_out[i] = F::eval(P, acc, nfull);
	} else if (i == i1 && f0_out) {
		PtrAcc acc{xs};
		*f0_out = F::eval(P, acc, nfull);
	}
}


template <class F>
int fd_points(const pnol_launch_env * env, const FunctorParams & P, const double * xfull, int nfull, const int * pos,
              const double * dx, int i0, int i1, double * fdx_out, double * f0_out)
{
	int npts = (i1 - i0) + (f0_out ? 1 : 0);
	if (npts <= 0) return PNOL_OK;
	size_t smem = (size_t) nfull * sizeof(double);
	PNOL_DEV_REQUIRE(env, smem <= env->smem_optin, "fd stencil: n = %d does not fit in shared memory", nfull);
	auto kern = fd_points_kernel<F>;
	PNOL_DEV_CUDA(env, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
	PNOL_DEV_LAUNCH(env, kern, (unsigned) ((npts + kFdThreads - 1) / kFdThreads), kFdThreads, smem, P, xfull, nfull, pos, dx, i0, i1,
	                fdx_out, f0_out);
	return PNOL_OK;
}

// ---------------------------------------------------------------------------------------------------
// a3 / a5, analytic: g[i] = F::partial(x, pos[i]) for i in [i0, i1) (pos == nullptr: i itself) of a scalar functor that defines partial
// (functors.hpp: has_partial). One coordinate per thread, so the depth of a gradient is that of ONE partial (O(1) for a locally coupled
// objective) where the forward difference runs a whole evaluation per thread. The base point is staged in shared memory with coalesced
// loads; each thread writes its entry straight to g, coalesced. pos[i] < 0 (a reduced entry without a slot, see fd_points_kernel) gives
// 0.0, what the forward difference gives there. f0 (f(x)) only when f0_out != nullptr: one extra thread runs F::eval, the one long
// dependent chain of the kernel, so it is not run when nobody asks for it.
// ---------------------------------------------------------------------------------------------------
constexpr int kGradThreads = 128;

template <class F>
__global__ void __launch_bounds__(kGradThreads)
gradient_kernel(FunctorParams P, const double * __restrict__ xfull, int nfull, const int * __restrict__ pos, int i0, int i1,
                double * __restrict__ g_out, double * __restrict__ f0_out)
{
	extern __shared__ double xs[];
#pragma unroll 4
	for (int j = threadIdx.x; j < nfull; j += blockDim.x) xs[j] = xfull[j];
	__syncthreads();
	const PtrAcc acc{xs};
	const int i = i0 + blockIdx.x * blockDim.x + threadIdx.x;
	if (i < i1) {
		const int pi = pos ? pos[i] : i;
		g_out[i] = pi >= 0 ? F::partial(P, acc, nfull, pi) : 0.0;
	} else if (i == i1 && f0_out) {
		*f0_out = F::eval(P, acc, nfull);
	}
}

template <class F>
int gradient(const pnol_launch_env * env, const FunctorParams & P, const double * xfull, int nfull, const int * pos, int i0, int i1,
             double * g_out, double * f0_out)
{
	const int nthreads = (i1 - i0) + (f0_out ? 1 : 0);
	if (nthreads <= 0) return PNOL_OK;
	size_t smem = (size_t) nfull * sizeof(double);
	PNOL_DEV_REQUIRE(env, smem <= env->smem_optin, "gradient: n = %d does not fit in shared memory", nfull);
	auto kern = gradient_kernel<F>;
	PNOL_DEV_CUDA(env, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
	PNOL_DEV_LAUNCH(env, kern, (unsigned) ((nthreads + kGradThreads - 1) / kGradThreads), kGradThreads, smem, P, xfull, nfull, pos, i0, i1,
	                g_out, f0_out);
	return PNOL_OK;
}

// pair -> (i, j), i <= j, row-major over the upper triangle of an n x n matrix: row i starts at s(i) = i*n - i*(i-1)/2; solved by a
// floating estimate, then fixed up
__device__ __forceinline__ void unrank_upper(long long pair, int n, int & i, int & j)
{
	double nn = (double) n;
	double est = (2.0 * nn + 1.0 - sqrt((2.0 * nn + 1.0) * (2.0 * nn + 1.0) - 8.0 * (double) pair)) * 0.5;
	i = (int) est;
	if (i < 0) i = 0;
	if (i > n - 1) i = n - 1;
	while (i > 0 && (long long) i * n - (long long) i * (i - 1) / 2 > pair) i--;
	while ((long long) (i + 1) * n - (long long) (i + 1) * i / 2 <= pair) i++;
	j = i + (int) (pair - ((long long) i * n - (long long) i * (i - 1) / 2));
}

// ---------------------------------------------------------------------------------------------------
// a6: forward-difference Hessian (Objective::hessianApproximation, Source/PNOL_Objective.cpp:38-85).
// One thread per pair (i <= j): B_ij = (f_ij - f_i - f_j + f) / (dx_i dx_j), mirrored. f_i are the n stencil
// values already produced by fd_points_kernel (the reference recomputes the same value for every pair).
// ---------------------------------------------------------------------------------------------------
template <class F>
__global__ void __launch_bounds__(kFdThreads)
fd_hessian_kernel(FunctorParams P, const double * __restrict__ x, const double * __restrict__ dx, int n,
                  const double * __restrict__ fdx, const double * __restrict__ f0, double * __restrict__ Bout)
{
	extern __shared__ double xs[];
	for (int j = threadIdx.x; j < n; j += blockDim.x) xs[j] = x[j];
	__syncthreads();
	long long pair = (long long) blockIdx.x * blockDim.x + threadIdx.x;
	long long npairs = (long long) n * (n + 1) / 2;
	if (pair >= npairs) return;
	int i, j;
	unrank_upper(pair, n, i, j);
	double fij;
	if (i == j) {
		// XdXij[i] = (X[i] + dX[i]) + dX[i]   (Source/PNOL_Objective.cpp:61-62 with i == j)
		PerturbAcc acc{xs, i, (xs[i] + dx[i]) + dx[i]};
		fij = F::eval(P, acc, n);
	} else {
		Perturb2Acc acc{xs, i, xs[i] + dx[i], j, xs[j] + dx[j]};
		fij = F::eval(P, acc, n);
	}
	double b = (fij - fdx[i] - fdx[j] + *f0) / (dx[i] * dx[j]);
	Bout[(long long) i * n + j] = b;
	Bout[(long long) j * n + i] = b;
}


template <class F>
int fd_hessian(const pnol_launch_env * env, const FunctorParams & P, const double * x, const double * dx, int n,
               const double * fdx, const double * f0, double * B)
{
	size_t smem = (size_t) n * sizeof(double);
	PNOL_DEV_REQUIRE(env, smem <= env->smem_optin, "fd hessian: n = %d does not fit in shared memory", n);
	auto kern = fd_hessian_kernel<F>;
	PNOL_DEV_CUDA(env, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
	long long npairs = (long long) n * (n + 1) / 2;
	PNOL_DEV_LAUNCH(env, kern, (unsigned) ((npairs + kFdThreads - 1) / kFdThreads), kFdThreads, smem, P, x, dx, n, fdx, f0, B);
	return PNOL_OK;
}

// ---------------------------------------------------------------------------------------------------
// a6, analytic: H[i][j] = F::partial2(x, i, j) of a scalar functor that defines partial2 (functors.hpp: has_partial2), n x n row-major.
// The upper triangle is cut into 32 x 32 tiles (bi, bj), bi <= bj, numbered row-major and unranked as fd_hessian_kernel unranks its
// pairs. A tile is 8 warps, each warp one row of 32 columns at a time, so that every store is one coalesced 256-byte row segment:
//   - off-diagonal tile: partial2 of its 32 x 32 pairs, stored to rows i / columns j, and parked in a shared tile of odd pitch (33: the
//     transposed read below is free of bank conflicts), from which the block stores the transpose to rows j / columns i;
//   - diagonal tile: partial2 for r <= c only; r > c is filled from the shared tile, so each unordered pair is evaluated exactly once
//     and H[j][i] has the bits of H[i][j].
// Edge tiles mask rows and columns >= n. For a locally coupled objective partial2 is a few compares, so the kernel is bound by the n^2
// store. The point is staged in shared memory once per BLOCK with coalesced loads, and a block then walks tiles blockIdx.x,
// blockIdx.x + gridDim.x, ... (the grid is one wave): staging it once per tile would read n * 8 bytes from L2 for every 16 KB of
// output, as much as the tile writes at n = 2048 and twice as much at n = 4096. 256 threads a block: 1024 (one tile row per warp, 32
// warps between two barriers) measured 5-6 % faster at n >= 16384 but 37 % slower a call at n = 4096 (NVIDIA B200, DESIGN 4.3).
// n range: x and the tile both fit in the opt-in shared memory, n <= (smem_optin - 32 * 33 * 8) / 8 (28000 on a B200).
// ---------------------------------------------------------------------------------------------------
constexpr int kHessTile = 32;
constexpr int kHessPitch = kHessTile + 1;
constexpr int kHessThreads = 256;

template <class F>
__global__ void __launch_bounds__(kHessThreads)
hessian_kernel(FunctorParams P, const double * __restrict__ x, int n, double * __restrict__ H)
{
	extern __shared__ double sm[];
	double * tile = sm;                          // kHessTile x kHessPitch
	double * xs = sm + kHessTile * kHessPitch;   // n
#pragma unroll 4
	for (int j = threadIdx.x; j < n; j += blockDim.x) xs[j] = x[j];
	__syncthreads();
	const PtrAcc acc{xs};
	const int tx = threadIdx.x & (kHessTile - 1), ty = threadIdx.x / kHessTile;
	constexpr int kRowStep = kHessThreads / kHessTile;
	const int T = (n + kHessTile - 1) / kHessTile;
	const long long ntiles = (long long) T * (T + 1) / 2;
	for (long long t = blockIdx.x; t < ntiles; t += gridDim.x) {
		int bi, bj;
		unrank_upper(t, T, bi, bj);
		const int r0 = bi * kHessTile, c0 = bj * kHessTile;
		const bool diag = bi == bj;
		const int j = c0 + tx;
#pragma unroll 4
		for (int r = ty; r < kHessTile; r += kRowStep) {
			const int i = r0 + r;
			const bool in = i < n && j < n;
			double v = 0.0;
			if (in && (!diag || r <= tx)) v = F::partial2(P, acc, n, i, j);
			if (in && !diag) H[(long long) i * n + j] = v;
			tile[r * kHessPitch + tx] = v;
		}
		__syncthreads();
		// diagonal tile: row r0 + r, column c0 + tx;  off-diagonal: the transpose, row c0 + r, column r0 + tx
#pragma unroll 4
		for (int r = ty; r < kHessTile; r += kRowStep) {
			const int i = (diag ? r0 : c0) + r, jj = (diag ? c0 : r0) + tx;
			if (i < n && jj < n) H[(long long) i * n + jj] = diag && r <= tx ? tile[r * kHessPitch + tx] : tile[tx * kHessPitch + r];
		}
		__syncthreads();
	}
}

template <class F>
int hessian(const pnol_launch_env * env, const FunctorParams & P, const double * x, int n, double * H)
{
	const size_t smem = ((size_t) kHessTile * kHessPitch + (size_t) n) * sizeof(double);
	PNOL_DEV_REQUIRE(env, n >= 1 && smem <= env->smem_optin, "hessian: n = %d is outside 1 .. %d (the point and one %d x %d tile must fit "
	                 "in shared memory)", n, (int) ((env->smem_optin / sizeof(double)) - kHessTile * kHessPitch), kHessTile, kHessTile);
	auto kern = hessian_kernel<F>;
	PNOL_DEV_CUDA(env, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
	int per_sm = 1;
	PNOL_DEV_CUDA(env, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kHessThreads, smem));
	if (per_sm < 1) per_sm = 1;
	const long long T = (n + kHessTile - 1) / kHessTile;
	const long long ntiles = T * (T + 1) / 2;
	const long long cap = (long long) env->sm_count * per_sm;
	PNOL_DEV_LAUNCH(env, kern, (unsigned) (ntiles < cap ? ntiles : cap), kHessThreads, smem, P, x, n, H);
	return PNOL_OK;
}

// ---------------------------------------------------------------------------------------------------
// a13: alpha pool. Point k evaluates phi = f(x + alpha_k p) and (optionally) the forward-difference slope
// (f(x + (alpha_k + dalpha) p) - phi) / dalpha. Mirrors lineSearchObj / lineSearchFDDerivative
// (Source/BFGS_bnd_linesearch_MPI_SW.cpp:703-734: Xtemp[i] = X[i] + alpha*p[i], no contraction) and the
// NaN/inf -> 1e10 sentinel of evaluateAlphaPoolAndDerivatives (:657-668).
// ---------------------------------------------------------------------------------------------------
struct LineAcc {
	const double * x; const double * p; const unsigned char * is_const; double alpha;
	__device__ __forceinline__ double operator[](int j) const
	{
		if (is_const && is_const[j]) return x[j];
		return x[j] + alpha * p[j];
	}
};

template <class F>
__global__ void __launch_bounds__(32)
alpha_pool_kernel(FunctorParams P, const double * __restrict__ xfull, const double * __restrict__ pfull,
                  const unsigned char * __restrict__ is_const, int nfull, const double * __restrict__ alpha, int npool,
                  double dalpha, const unsigned char * __restrict__ eval_ind, double * __restrict__ vals /* 2*npool */)
{
	extern __shared__ double sm[];
	double * xs = sm;
	double * ps = sm + nfull;
	unsigned char * cs = reinterpret_cast<unsigned char *>(sm + 2 * nfull);
	for (int j = threadIdx.x; j < nfull; j += blockDim.x) {
		xs[j] = xfull[j]; ps[j] = pfull[j];
		cs[j] = is_const ? is_const[j] : 0;
	}
	__syncthreads();
	int t = blockIdx.x;   // one point per block (t < npool: phi, t >= npool: shifted point); the warp stages, lane 0 evaluates
	if (threadIdx.x != 0 || t >= 2 * npool) return;
	int k = t < npool ? t : t - npool;
	if (eval_ind && !eval_ind[k]) return;
	double a = t < npool ? alpha[k] : alpha[k] + dalpha;
	LineAcc acc{xs, ps, is_const ? cs : nullptr, a};
	vals[t] = F::eval(P, acc, nfull);
}


/* vals[t], t < npool: f(x + alpha_t p); vals[npool + t]: f(x + (alpha_t + dalpha) p) when want_shifted (the library turns them into
 * phi / dphi and applies the 1e10 sentinel) */
template <class F>
int alpha_pool(const pnol_launch_env * env, const FunctorParams & P, const double * xfull, const double * pfull,
               const unsigned char * is_const, int nfull, const double * alpha, int npool, double dalpha,
               const unsigned char * eval_ind, int want_shifted, double * vals)
{
	size_t smem = (size_t) nfull * (2 * sizeof(double) + 1) + 16;
	PNOL_DEV_REQUIRE(env, smem <= env->smem_optin, "alpha pool: n = %d does not fit in shared memory", nfull);
	auto kern = alpha_pool_kernel<F>;
	PNOL_DEV_CUDA(env, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
	int npts = want_shifted ? 2 * npool : npool;
	// one point per block of one warp: the pool is tiny and each point is a long dependent chain
	PNOL_DEV_LAUNCH(env, kern, (unsigned) npts, 32, smem, P, xfull, pfull, is_const, nfull, alpha, npool, dalpha, eval_ind, vals);
	return PNOL_OK;
}

// ---------------------------------------------------------------------------------------------------
// a13, analytic slope: point k gives phi = f(x + alpha_k p) and phi' = sum_r p_r * df/dx_{pos[r]}(x + alpha_k p) of a scalar functor that
// defines partial (functors.hpp: has_partial), in place of alpha_pool's forward-difference slope (pnol_alpha_pool_analytic).
// One block per pool entry. The block stages the trial point xa[j] = is_const[j] ? x[j] : x[j] + alpha_k p[j] in shared memory once --
// LineAcc's expression, so phi has the bits of alpha_pool's phi. Right after that barrier lane 0 of warp 0 starts the block's long chain,
// F::eval on xa, while the other warps form prod[r] = g_r * p_r for the reduced coordinates, g_r = F::partial(xa, pos[r]) (pos ==
// nullptr: r itself; pos[r] < 0, a reduced entry without a slot: 0, as gradient_kernel gives, so that entry contributes 0 * p_r). Those
// warps then meet on a named barrier of their own, and lane 0 of warp 1 sums the products sequentially in r order, s = 0;
// s = s + prod[0]; ... That is dotProd's order (include/pnol/UtilityFunctions.hpp), so at alpha = 0 the slope is bit for bit
// dotProd(pnol_gradient_recur(x), p), the host's dphi0dalpha, and the strong-Wolfe tests compare like with like. A tree reduction
// would be shorter but would lose that equality; the products and their sequential sum run beside the eval chain and are no longer
// than it. Starting the eval before the partials rather than after one common barrier measured 54.6 instead of 60.8 us a pool of 9 for
// Rosenbrock at n = 4096 (NVIDIA B200, DESIGN 4.4).
// Raw values out, as alpha_pool: vals[k] = phi, vals[npool + k] = phi' (the library applies the 1e10 sentinel to phi only).
// n range: xa (nfull doubles) and prod (n <= nfull doubles) in shared memory, 16 nfull bytes, less than alpha_pool's 17 nfull + 16.
// ---------------------------------------------------------------------------------------------------
constexpr int kSlopeThreads = 256;

template <class F>
__global__ void __launch_bounds__(kSlopeThreads)
alpha_slope_kernel(FunctorParams P, const double * __restrict__ xfull, const double * __restrict__ pfull,
                   const unsigned char * __restrict__ is_const, int nfull, const int * __restrict__ pos, const double * __restrict__ p,
                   int n, const double * __restrict__ alpha, int npool, const unsigned char * __restrict__ eval_ind,
                   double * __restrict__ vals /* 2*npool */)
{
	const int k = blockIdx.x;
	if (eval_ind && !eval_ind[k]) return;
	extern __shared__ double sm[];
	double * xa = sm;              // nfull
	double * prod = sm + nfull;    // n
	const double a = alpha[k];
	for (int j = threadIdx.x; j < nfull; j += blockDim.x) xa[j] = is_const && is_const[j] ? xfull[j] : xfull[j] + a * pfull[j];
	__syncthreads();
	const PtrAcc acc{xa};
	if (threadIdx.x < 32) {
		if (threadIdx.x == 0) vals[k] = F::eval(P, acc, nfull);
		return;
	}
	for (int r = threadIdx.x - 32; r < n; r += kSlopeThreads - 32) {
		const int pr = pos ? pos[r] : r;
		const double g = pr >= 0 ? F::partial(P, acc, nfull, pr) : 0.0;
		prod[r] = g * p[r];
	}
	asm volatile("bar.sync 1, %0;" :: "n"(kSlopeThreads - 32) : "memory");    // the product warps only: warp 0 is in the eval chain
	if (threadIdx.x == 32) {
		double s = 0.0;
		for (int r = 0; r < n; r++) s = s + prod[r];
		vals[npool + k] = s;
	}
}

/* vals[k] = f(x + alpha_k p), vals[npool + k] = its analytic slope along p (raw: the library applies the sentinel to phi) */
template <class F>
int alpha_slope(const pnol_launch_env * env, const FunctorParams & P, const double * xfull, const double * pfull, const unsigned char * is_const,
                int nfull, const int * pos, const double * p, int n, const double * alpha, int npool, const unsigned char * eval_ind,
                double * vals)
{
	const size_t smem = ((size_t) nfull + (size_t) n) * sizeof(double);
	PNOL_DEV_REQUIRE(env, n >= 1 && n <= nfull && smem <= env->smem_optin, "alpha slope: n = %d, nfull = %d: needs 1 <= n <= nfull and the "
	                 "trial point and the products, (nfull + n) * 8 bytes, within %zu bytes of shared memory", n, nfull, env->smem_optin);
	if (npool <= 0) return PNOL_OK;
	auto kern = alpha_slope_kernel<F>;
	PNOL_DEV_CUDA(env, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
	PNOL_DEV_LAUNCH(env, kern, (unsigned) npool, kSlopeThreads, smem, P, xfull, pfull, is_const, nfull, pos, p, n, alpha, npool, eval_ind, vals);
	return PNOL_OK;
}

// ---------------------------------------------------------------------------------------------------
// generic residual evaluation: F[i] = r_i(x)        (MultiObjective::objEval, Source/PNOL_Objective.hpp:57)
// ---------------------------------------------------------------------------------------------------
template <class R>
__global__ void __launch_bounds__(256)
residual_kernel(FunctorParams P, const double * __restrict__ x, int n, double * __restrict__ F)
{
	extern __shared__ double xs[];
	for (int j = threadIdx.x; j < n; j += blockDim.x) xs[j] = x[j];
	__syncthreads();
	PtrAcc acc{xs};
	for (long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x; i < P.m; i += (long long) gridDim.x * blockDim.x)
		F[i] = R::residual(P, acc, n, i);
}


template <class R>
int residual(const pnol_launch_env * env, const FunctorParams & P, const double * x, int n, double * F)
{
	const long long m = P.m;
	size_t smem = (size_t) n * sizeof(double);
	PNOL_DEV_REQUIRE(env, smem <= env->smem_optin, "residual: n = %d does not fit in shared memory", n);
	auto kern = residual_kernel<R>;
	PNOL_DEV_CUDA(env, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
	long long blocks = (m + 255) / 256;
	long long grid = blocks < (long long) env->sm_count * 8 ? blocks : (long long) env->sm_count * 8;
	if (grid < 1) grid = 1;
	PNOL_DEV_LAUNCH(env, kern, (unsigned) grid, 256, smem, P, x, n, F);
	return PNOL_OK;
}

// ---------------------------------------------------------------------------------------------------
// black-box forward-difference Jacobian  (MultiObjective::gradientApproximation, Source/PNOL_Objective.cpp:165-197)
//   J[i][j] = (F_i(x + dx_j e_j) - F_i(x)) / dx_j
// ---------------------------------------------------------------------------------------------------
constexpr int kBbRows = 128;      // rows per block (one per thread)
constexpr int kBbCols = 32;       // J columns staged per pass

template <class R>
__global__ void __launch_bounds__(kBbRows)
fd_jacobian_blackbox_kernel(FunctorParams P, const double * __restrict__ x, const double * __restrict__ dx, int n,
                            double * __restrict__ J, double * __restrict__ F)
{
	extern __shared__ double sm[];
	double * xs = sm;                       // n
	double * dxs = sm + n;                  // n
	double * rdx = sm + 2 * n;              // n   RN(1/dx) or 0 (exact_div.cuh)
	double * tile = sm + 3 * n;             // kBbRows x (kBbCols + 1)
	constexpr int pitch = kBbCols + 1;
	for (int j = threadIdx.x; j < n; j += blockDim.x) { xs[j] = x[j]; dxs[j] = dx[j]; rdx[j] = make_recip(dx[j]).r; }
	__syncthreads();
	for (long long row0 = (long long) blockIdx.x * kBbRows; row0 < P.m; row0 += (long long) gridDim.x * kBbRows) {
		const long long i = row0 + threadIdx.x;
		const bool live = i < P.m;
		const int rows = (int) min((long long) kBbRows, P.m - row0);
		double r0 = 0;
		if (live) {
			PtrAcc acc{xs};
			r0 = R::residual(P, acc, n, i);
			if (F) F[i] = r0;
		}
		for (int c0 = 0; c0 < n; c0 += kBbCols) {
			const int cols = min(kBbCols, n - c0);
			if (live) {
				for (int c = 0; c < cols; c++) {
					const int j = c0 + c;
					PerturbAcc acc{xs, j, xs[j] + dxs[j]};       // XdX[j] = XdX[j] + dX[j]   (PNOL_Objective.cpp:186)
					double rj = R::residual(P, acc, n, i);
					RecipDiv rd; rd.d = dxs[j]; rd.r = rdx[j];
					tile[threadIdx.x * pitch + c] = div_exact(rj - r0, rd);   // (FdX[i] - F[i])/dX[j]  (:192)
				}
			}
			__syncthreads();
			// coalesced write: consecutive threads write consecutive columns of one row
			for (int e = threadIdx.x; e < rows * cols; e += kBbRows) {
				int r = e / cols, c = e - r * cols;
				J[(row0 + r) * n + c0 + c] = tile[r * pitch + c];
			}
			__syncthreads();
		}
	}
}


template <class R>
int fd_jacobian(const pnol_launch_env * env, const FunctorParams & P, const double * x, const double * dx, int n, double * J, double * F)
{
	const long long m = P.m;
	size_t smem = ((size_t) 3 * n + (size_t) kBbRows * (kBbCols + 1)) * sizeof(double);
	PNOL_DEV_REQUIRE(env, smem <= env->smem_optin, "fd jacobian: n = %d does not fit in shared memory", n);
	auto kern = fd_jacobian_blackbox_kernel<R>;
	PNOL_DEV_CUDA(env, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
	long long blocks = (m + kBbRows - 1) / kBbRows;
	long long grid = blocks < (long long) env->sm_count * 4 ? blocks : (long long) env->sm_count * 4;
	if (grid < 1) grid = 1;
	PNOL_DEV_LAUNCH(env, kern, (unsigned) grid, kBbRows, smem, P, x, dx, n, J, F);
	return PNOL_OK;
}

// ---------------------------------------------------------------------------------------------------
// analytic Jacobian (PNOL_JAC_ANALYTIC) of a residual functor that defines R::jacobian (functors.hpp: has_jacobian)
//   J[i][j] = d r_i / d x_j
// One row per thread: R::jacobian writes the thread's row into a shared-memory tile (odd pitch: the threads' rows fall in different
// banks), the block then writes its rows out with coalesced stores -- the rows of a block are one contiguous range of J. Rows too
// wide for a tile of kJacRowsMin rows are written by R::jacobian straight to global memory. F (optional) from R::residual.
// ---------------------------------------------------------------------------------------------------
constexpr int kJacRows = 128;        // rows per block when the tile fits
constexpr int kJacRowsMin = 32;      // smallest tile

template <class R>
__global__ void __launch_bounds__(kJacRows)
jacobian_kernel(FunctorParams P, const double * __restrict__ x, int n, double * __restrict__ J, double * __restrict__ F, int tiled)
{
	extern __shared__ double sm[];
	double * xs = sm;                       // n
	double * tile = sm + n;                 // blockDim.x x (n | 1), when tiled
	const int pitch = n | 1;
	for (int j = threadIdx.x; j < n; j += blockDim.x) xs[j] = x[j];
	__syncthreads();
	const PtrAcc acc{xs};
	for (long long row0 = (long long) blockIdx.x * blockDim.x; row0 < P.m; row0 += (long long) gridDim.x * blockDim.x) {
		const long long i = row0 + threadIdx.x;
		const bool live = i < P.m;
		if (live && F) F[i] = R::residual(P, acc, n, i);
		if (!tiled) {
			if (live) R::jacobian(P, acc, n, i, J + i * n);
			continue;
		}
		if (live) R::jacobian(P, acc, n, i, tile + threadIdx.x * pitch);
		__syncthreads();
		const int rows = (int) min((long long) blockDim.x, P.m - row0);
		double * dst = J + row0 * n;
		for (int e = threadIdx.x; e < rows * n; e += blockDim.x) {
			const int r = e / n;
			dst[e] = tile[r * pitch + (e - r * n)];
		}
		__syncthreads();
	}
}

template <class R>
int jacobian(const pnol_launch_env * env, const FunctorParams & P, const double * x, int n, double * J, double * F)
{
	const long long m = P.m;
	if (m <= 0) return PNOL_OK;
	const size_t xbytes = (size_t) n * sizeof(double);
	const size_t row_bytes = (size_t) (n | 1) * sizeof(double);
	PNOL_DEV_REQUIRE(env, xbytes <= env->smem_optin, "analytic jacobian: n = %d does not fit in shared memory", n);
	int threads = kJacRows;
	while (threads > kJacRowsMin && xbytes + threads * row_bytes > env->smem_optin) threads /= 2;
	const int tiled = xbytes + threads * row_bytes <= env->smem_optin;
	if (!tiled) threads = kJacRows;
	const size_t smem = xbytes + (tiled ? threads * row_bytes : 0);
	auto kern = jacobian_kernel<R>;
	PNOL_DEV_CUDA(env, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
	int per_sm = 1;
	PNOL_DEV_CUDA(env, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem));
	if (per_sm < 1) per_sm = 1;
	const long long blocks = (m + threads - 1) / threads;
	const long long cap = (long long) env->sm_count * per_sm;
	const long long grid = blocks < cap ? blocks : cap;
	PNOL_DEV_LAUNCH(env, kern, (unsigned) grid, threads, smem, P, x, n, J, F, tiled);
	return PNOL_OK;
}

// ---------------------------------------------------------------------------------------------------
// batched Levenberg-Marquardt (pnol_lm_batch): problem b owns rows [row_off[b], row_off[b+1]) of the functor and row b of X (B x n).
// One CTA runs one problem's whole LevMarq::findMin (Source/LevenbergMarquardtMPI.cpp:12-173), operation for operation oracle_lm
// (oracle/pnol_oracle.cpp) restricted to the problem's rows, so every problem returns the bits the reference returns on it alone:
//   - chi^2 = r * r, r = sqrt(s), s = s + F_k F_k over the rows in ascending order (pow(vector2Norm(F), 2)): thread 0 walks the tile.
//   - J pass, per tile of TR rows: r0 (column n of the tile) by R::residual; the forward difference (r_i(X + dx_j e_j) - r0) / dx_j with
//     the IEEE quotient (div_exact) over (row, column) items, or the row of R::jacobian. The owners then add the tile's rows in row
//     order to their sums, held in registers: pair (i, j <= i) is JTJ[i][j], pair (i, n) is (J^T F)_i, each from 0, never fused.
//   - A = JTJ (mirrored) with A_ii = (1 + lambda) JTJ_ii, rhs = -(J^T F); the shim's LU with partial pivoting (whole-row swaps, first
//     largest |entry|, a zero pivot left to IEEE arithmetic) in shared memory: the pivot search, the substitutions and every sequential
//     sum by thread 0, the row swap and the elimination over the block (each entry still sees its updates in k order).
//   - X + sigma, its chi^2, the accept / reject rule, the stop ||sigma||_2 < x_min_diff after an accepted step.
// After a rejected step X is restored, so J, J^T J and J^T F are what they were: the sums are kept (the reference recomputes the
// same values). No global scratch: the residuals at X are recomputed in each J pass, as gradientApproximation recomputes F.
// A problem's bits depend on nothing but its own rows, X row, dx and the scalars: not on B, its position or the other problems.
// Configurations by n (threads, sums per owner thread, tile rows): n <= 8: 32/2/32, <= 16: 64/3/32, <= 32: 128/5/64, <= 64: 256/9/64.
// ---------------------------------------------------------------------------------------------------
constexpr int kLmBatchMaxN = 64;

// In-place LU with partial pivoting of the n x n matrix A (row pitch ap) in shared memory by a block of T threads, the shim's luSolve
// factorisation (oracle/shim/shim_impl.cpp:63-80): whole-row swaps, the first largest |entry| as pivot, a zero pivot left to IEEE
// arithmetic. The pivot search is thread 0's (piv, which must hold the identity on entry, records the row order; slot is one int of
// shared memory for the broadcast), the row swap, the column scaling and the elimination are spread over the block -- each entry still
// sees its updates in k order, so the factors have the bits of the sequential loop. Used by lm_batch_kernel and bfgs_batch_kernel.
template <int T>
__device__ __forceinline__ void block_lu_factor(double * A, int ap, int n, int * piv, int * slot)
{
	const int tid = threadIdx.x;
	for (int k = 0; k < n; k++) {
		if (tid == 0) {
			int p = k;
			double best = fabs(A[k * ap + k]);
			for (int i = k + 1; i < n; i++)
				if (fabs(A[i * ap + k]) > best) { best = fabs(A[i * ap + k]); p = i; }
			if (p != k) { const int t = piv[p]; piv[p] = piv[k]; piv[k] = t; }
			slot[0] = p;
		}
		__syncthreads();
		const int p = slot[0];
		if (p != k)
			for (int j = tid; j < n; j += T) { const double t = A[p * ap + j]; A[p * ap + j] = A[k * ap + j]; A[k * ap + j] = t; }
		__syncthreads();
		for (int i = k + 1 + tid; i < n; i += T) A[i * ap + k] = A[i * ap + k] / A[k * ap + k];
		__syncthreads();
		const int w = n - k - 1;
		for (int e = tid; e < w * w; e += T) {
			const int i = k + 1 + e / w, j = k + 1 + e % w;
			A[i * ap + j] = A[i * ap + j] - A[i * ap + k] * A[k * ap + j];
		}
		__syncthreads();
	}
}

__host__ __device__ inline int lm_batch_pitch(int n) { return (n + 1) | 1; }
__host__ __device__ inline int lm_batch_nsums(int n) { return n * (n + 1) / 2 + n; }
// shared memory of one problem: xs, xt, dx, 1/dx, sigma, y (6n), the sums, A (n x (n+1)), the tile, 2 broadcast slots; then n ints
__host__ __device__ inline size_t lm_batch_smem(int n, int tile_rows)
{
	return ((size_t) 6 * n + lm_batch_nsums(n) + (size_t) n * (n + 1) + (size_t) tile_rows * lm_batch_pitch(n) + 2) * sizeof(double) +
	       (size_t) n * sizeof(int);
}

template <class R, bool kAnalytic, int T, int OWN, int TR>
__global__ void __launch_bounds__(T)
lm_batch_kernel(FunctorParams P, const long long * __restrict__ row_off, int n, double * __restrict__ X, const double * __restrict__ dx,
                double lambda0, double lambda_factor, double x_min_diff, int max_iter, double * __restrict__ chisq_out,
                double * __restrict__ lambda_out, int * __restrict__ iters_out, int * __restrict__ stopped_out, double * __restrict__ F_out)
{
	extern __shared__ double sm[];
	const int tid = threadIdx.x;
	const long long b = blockIdx.x;
	const long long base = row_off[b];
	const long long mb = row_off[b + 1] - base;
	const int pitch = lm_batch_pitch(n);
	const int NL = n * (n + 1) / 2, NS = NL + n;
	const int ap = n + 1;
	double * xs = sm;                 // X
	double * xt = xs + n;             // trial X
	double * dxs = xt + n;
	double * rdx = dxs + n;           // RN(1/dx) or 0 (exact_div.cuh)
	double * sig = rdx + n;           // sigma
	double * yv = sig + n;            // forward substitution
	double * G = yv + n;              // the NS sums of the last J pass
	double * A = G + NS;              // n x ap
	double * tile = A + (size_t) n * ap;   // TR x pitch
	double * bc = tile + (size_t) TR * pitch;   // broadcast slots
	int * piv = reinterpret_cast<int *>(bc + 2);

	for (int j = tid; j < n; j += T) {
		xs[j] = X[b * n + j];
		if (!kAnalytic) { dxs[j] = dx[j]; rdx[j] = make_recip(dx[j]).r; }
	}
	// the pairs this thread owns: slot s < NL is (i, j <= i) of the lower triangle row by row, slot NL + i is (i, n)
	int pa[OWN], pb[OWN];
#pragma unroll
	for (int q = 0; q < OWN; q++) {
		const int s = tid + q * T;
		pa[q] = -1; pb[q] = 0;
		if (s < NL) {
			int i = 0;
			while ((i + 1) * (i + 2) / 2 <= s) i++;
			pa[q] = i; pb[q] = s - i * (i + 1) / 2;
		} else if (s < NS) {
			pa[q] = s - NL; pb[q] = n;
		}
	}
	__syncthreads();

	// chi^2 at x: tiles of residuals, thread 0 adds their squares in row order
	auto chisq_at = [&](const double * x) -> double {
		const PtrAcc acc{x};
		double s = 0.0;
		for (long long row0 = 0; row0 < mb; row0 += TR) {
			const int rows = (int) min((long long) TR, mb - row0);
			if (tid < rows) tile[tid] = R::residual(P, acc, n, base + row0 + tid);
			__syncthreads();
			if (tid == 0)
				for (int r = 0; r < rows; r++) s = s + tile[r] * tile[r];
			__syncthreads();
		}
		if (tid == 0) { const double root = sqrt(s); bc[0] = root * root; }
		__syncthreads();
		const double c = bc[0];
		__syncthreads();
		return c;
	};

	double lambda = lambda0;
	double chi = chisq_at(xs);
	int iter = 0, stopped = 0;
	bool fresh = false;            // G holds the sums at the current X
	while (iter < max_iter) {
		if (!fresh) {
			double acc[OWN];
#pragma unroll
			for (int q = 0; q < OWN; q++) acc[q] = 0.0;
			const PtrAcc ax{xs};
			for (long long row0 = 0; row0 < mb; row0 += TR) {
				const int rows = (int) min((long long) TR, mb - row0);
				if (tid < rows) {
					const long long i = base + row0 + tid;
					tile[tid * pitch + n] = R::residual(P, ax, n, i);
					if constexpr (kAnalytic) R::jacobian(P, ax, n, i, tile + tid * pitch);
				}
				if constexpr (!kAnalytic) {
					__syncthreads();
					for (int e = tid; e < rows * n; e += T) {
						const int j = e / rows, r = e - j * rows;
						const PerturbAcc acc1{xs, j, xs[j] + dxs[j]};       // XdX[j] = XdX[j] + dX[j]   (PNOL_Objective.cpp:186)
						const double rj = R::residual(P, acc1, n, base + row0 + r);
						RecipDiv rd; rd.d = dxs[j]; rd.r = rdx[j];
						tile[r * pitch + j] = div_exact(rj - tile[r * pitch + n], rd);   // (FdX[i] - F[i]) / dX[j]   (:192)
					}
				}
				__syncthreads();
#pragma unroll
				for (int q = 0; q < OWN; q++) {
					if (pa[q] < 0) continue;
					const double * ci = tile + pa[q];
					const double * cj = tile + pb[q];
					double a = acc[q];
					for (int r = 0; r < rows; r++) a = a + ci[r * pitch] * cj[r * pitch];
					acc[q] = a;
				}
				__syncthreads();
			}
#pragma unroll
			for (int q = 0; q < OWN; q++)
				if (pa[q] >= 0) G[tid + q * T] = acc[q];
			fresh = true;
		}
		__syncthreads();
		// damped normal matrix (Source/LevenbergMarquardtMPI.cpp:64-85); piv = identity
		for (int e = tid; e < n * n; e += T) {
			const int i = e / n, j = e - i * n;
			const double s = i >= j ? G[i * (i + 1) / 2 + j] : G[j * (j + 1) / 2 + i];
			A[i * ap + j] = i == j ? (1 + lambda) * s : s;
		}
		for (int i = tid; i < n; i += T) piv[i] = i;
		__syncthreads();
		block_lu_factor<T>(A, ap, n, piv, reinterpret_cast<int *>(bc));
		// substitutions (shim_impl.cpp:82-98) with rhs = -(J^T F)
		if (tid == 0) {
			for (int i = 0; i < n; i++) {
				double s = -G[NL + piv[i]];
				for (int k = 0; k < i; k++) s = s - A[i * ap + k] * yv[k];
				yv[i] = s;
			}
			for (int i = n - 1; i >= 0; i--) {
				double s = yv[i];
				for (int k = i + 1; k < n; k++) s = s - A[i * ap + k] * sig[k];
				sig[i] = s / A[i * ap + i];
			}
		}
		__syncthreads();
		for (int j = tid; j < n; j += T) xt[j] = xs[j] + sig[j];   // (:97-100)
		__syncthreads();
		const double chi_t = chisq_at(xt);                           // (:103-108)
		if (chi_t >= chi || chi_t != chi_t) {                        // (:110-129)
			lambda = lambda * lambda_factor;
		} else {                                                     // (:132-141)
			lambda = lambda / lambda_factor;
			chi = chi_t;
			for (int j = tid; j < n; j += T) xs[j] = xt[j];
			fresh = false;
			double s2 = 0.0;
			for (int j = 0; j < n; j++) s2 = s2 + sig[j] * sig[j];
			__syncthreads();
			if (sqrt(s2) < x_min_diff) { stopped = 1; break; }
		}
		iter++;
	}
	for (int j = tid; j < n; j += T) X[b * n + j] = xs[j];
	if (tid == 0) {
		chisq_out[b] = chi;
		lambda_out[b] = lambda;
		iters_out[b] = iter;
		stopped_out[b] = stopped;
	}
	if (F_out) {
		const PtrAcc acc{xs};
		for (long long r = tid; r < mb; r += T) F_out[base + r] = R::residual(P, acc, n, base + r);
	}
}

template <class R, bool kAnalytic, int T, int OWN, int TR>
int lm_batch_launch(const pnol_launch_env * env, const FunctorParams & P, const long long * row_off, long long B, int n, double * X,
                    const double * dx, double lambda0, double lambda_factor, double x_min_diff, int max_iter, double * chisq_out,
                    double * lambda_out, int * iters_out, int * stopped_out, double * F_out)
{
	const size_t smem = lm_batch_smem(n, TR);
	PNOL_DEV_REQUIRE(env, lm_batch_nsums(n) <= OWN * T && smem <= env->smem_optin, "lm batch: n = %d needs %zu bytes of shared memory", n, smem);
	auto kern = lm_batch_kernel<R, kAnalytic, T, OWN, TR>;
	PNOL_DEV_CUDA(env, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
	PNOL_DEV_LAUNCH(env, kern, (unsigned) B, T, smem, P, row_off, n, X, dx, lambda0, lambda_factor, x_min_diff, max_iter, chisq_out,
	                lambda_out, iters_out, stopped_out, F_out);
	return PNOL_OK;
}

template <class R, bool kAnalytic>
int lm_batch_mode(const pnol_launch_env * env, const FunctorParams & P, const long long * row_off, long long B, int n, double * X,
                  const double * dx, double lambda0, double lambda_factor, double x_min_diff, int max_iter, double * chisq_out,
                  double * lambda_out, int * iters_out, int * stopped_out, double * F_out)
{
#define PNOL_LM_BATCH_CFG(T, OWN, TR) \
	lm_batch_launch<R, kAnalytic, T, OWN, TR>(env, P, row_off, B, n, X, dx, lambda0, lambda_factor, x_min_diff, max_iter, chisq_out, \
	                                          lambda_out, iters_out, stopped_out, F_out)
	if (n <= 8) return PNOL_LM_BATCH_CFG(32, 2, 32);
	if (n <= 16) return PNOL_LM_BATCH_CFG(64, 3, 32);
	if (n <= 32) return PNOL_LM_BATCH_CFG(128, 5, 64);
	return PNOL_LM_BATCH_CFG(256, 9, 64);
#undef PNOL_LM_BATCH_CFG
}

/* pnol_lm_batch on device pointers: row_off (B + 1), X (B x n, in/out), dx (n; unused with PNOL_JAC_ANALYTIC), the four per-problem
 * outputs (B), F_out (rows, may be NULL). The caller has checked row_off. n in 1 .. 64; PNOL_JAC_ANALYTIC needs R::jacobian. */
template <class R>
int lm_batch(const pnol_launch_env * env, const FunctorParams & P, const long long * row_off, long long B, int n, double * X, const double * dx,
             double lambda0, double lambda_factor, double x_min_diff, int max_iter, int jac_mode, double * chisq_out, double * lambda_out,
             int * iters_out, int * stopped_out, double * F_out)
{
	PNOL_DEV_REQUIRE(env, n >= 1 && n <= kLmBatchMaxN, "lm batch: n = %d is outside 1 .. %d", n, kLmBatchMaxN);
	PNOL_DEV_REQUIRE(env, B >= 0 && B <= 0x7fffffffLL, "lm batch: B = %lld is outside 0 .. 2^31 - 1", B);
	if (B == 0) return PNOL_OK;
	if (jac_mode == PNOL_JAC_ANALYTIC) {
		if constexpr (has_jacobian<R>::value)
			return lm_batch_mode<R, true>(env, P, row_off, B, n, X, dx, lambda0, lambda_factor, x_min_diff, max_iter, chisq_out, lambda_out,
			                              iters_out, stopped_out, F_out);
		PNOL_DEV_ERR(env, "lm batch: the residual model has no analytic Jacobian (jacobian()): PNOL_JAC_ANALYTIC refused");
		return PNOL_ERR_NO_FUNCTOR;
	}
	PNOL_DEV_REQUIRE(env, dx != nullptr, "lm batch: dx is required for a forward-difference Jacobian");
	return lm_batch_mode<R, false>(env, P, row_off, B, n, X, dx, lambda0, lambda_factor, x_min_diff, max_iter, chisq_out, lambda_out,
	                               iters_out, stopped_out, F_out);
}

// ---------------------------------------------------------------------------------------------------
// batched BFGS (pnol_bfgs_batch): problem b starts from row b of X (B x n) and minimises the functor's objective. One CTA runs one
// problem's whole BFGS::findMin (Source/BFGS_with_linesearch.cpp:12-139) -- the strong-Wolfe line search with its zoom and
// cubicInterpMin (:177-385) and the literal updateHessianInv (:389-432) included -- operation for operation what the unmodified host
// BFGS controller computes on the C-ABI's CPU stand-in (oracle/host_logic_device.cpp, whose dense helpers are the reference's
// sequential ones), so every problem returns the bits the reference returns on that start alone:
//   - D: the identity, or (init_hess_fd) the inverse of the Hessian at X: B by the forward difference (n + 1 stencil values, then one
//     thread per pair i <= j with (f_ij - f_i - f_j + f) / (dx dx), the diagonal point (x_i + dx) + dx) or by F::partial2, mirrored;
//     then matrixInverse as the stand-in computes it, one LU with partial pivoting (block_lu_factor) and one pair of substitutions
//     with b = e_j per column j, each column one thread.
//   - gradient: n + 1 stencil points, one thread each (PerturbAcc: fd_points' bits), and the IEEE quotient; or n F::partial calls.
//   - p = -D g, one row per thread, each a sequential k sum.
//   - line search: every thread runs the same scalar control (Wolfe tests, zoom, cubicInterpMin with pow(d1, 2) as d1 * d1 and the
//     reference's sign(), the `iter > 1` of the sufficient-decrease test) on values broadcast through shared memory, so the control
//     flow is uniform and needs no extra barrier. A point is phi(alpha) and phi(alpha + dalpha) on lanes 0 and 1 (LineAcc: unfused
//     x + alpha p), slope (phi2 - phi) / dalpha; or, analytic slope, phi on thread 0 while the threads of the other warps (lanes 1 ..
//     n of a single-warp block) form p_r * df/dx_r at the staged point, summed in r order as alpha_slope_kernel sums them. Values are
//     raw: the serial class has no 1e10 sentinel. An exhausted search leaves alpha = 0 and Fopt = F (and then rho = 1/0: D turns NaN,
//     as in the reference).
//   - update: A = M1 D, then D = A M2 + M3, each entry one thread's sequential k sum, M1 / M2 / M3 formed on the fly with
//     oracle_update_hinv's expressions (never the RANK2 form, whose bits differ).
//   - stop: sum |X - Xprev| and ||g||_2 sequentially; stop code 0 / 1 / 2 for the first false conjunct of the loop condition.
// Scalar sums every thread needs (p . g, y . s, the stop norms) are computed by every thread from shared memory: same operations in the
// same order, hence the same bits everywhere. Two shared buffers alternate for the line-search values so that a point's writes never
// race the previous point's readers. A problem's bits depend on nothing but its start, the functor and the parameters.
// Configurations by n (threads): n <= 8: 32, <= 16: 64, <= 32: 128, <= 64: 256.
// ---------------------------------------------------------------------------------------------------
constexpr int kBfgsBatchMaxN = 64;

// D and the update / LU scratch A (n x (n + 1) each), twelve n-vectors, four line-search values and four broadcast slots; n + 1 ints
__host__ __device__ inline size_t bfgs_batch_smem(int n)
{
	return ((size_t) 2 * n * (n + 1) + (size_t) 12 * n + 8) * sizeof(double) + (size_t) (n + 1) * sizeof(int);
}

// the reference's sign() and cubicInterpMin (Source/BFGS_with_linesearch.cpp:359-385); pow(d1, 2) is d1 * d1 there (a literal square,
// folded by the compiler)
__device__ __forceinline__ double bfgs_sign(double x) { if (x > 0) return 1.0; if (x < 0) return -1.0; return 0.0; }
__device__ __forceinline__ double bfgs_cubic_interp_min(double alo, double ahi, double plo, double phh, double dlo, double dhh)
{
	const double d1 = dlo + dhh - 3 * (plo - phh) / (alo - ahi);
	const double d2 = bfgs_sign(ahi - alo) * sqrt(d1 * d1 - dlo * dhh);
	double a = ahi - (ahi - alo) * (dhh + d2 - d1) / (dhh - dlo + 2 * d2);
	if (alo < ahi) {
		if (a < alo) a = (ahi + alo) / 2;
	} else {
		if (a < ahi) a = (ahi + alo) / 2;
	}
	return a;
}

template <class F, int T>
__global__ void __launch_bounds__(T)
bfgs_batch_kernel(FunctorParams P, int n, double * __restrict__ X, pnol_bfgs_params prm, int flags, double * __restrict__ f0_out,
                  double * __restrict__ fopt_out, int * __restrict__ iters_out, int * __restrict__ stop_out)
{
	extern __shared__ double sm[];
	const int tid = threadIdx.x;
	const long long b = blockIdx.x;
	const int ap = n + 1;
	double * D = sm;                       // inverse Hessian, n x ap
	double * A = D + (size_t) n * ap;      // M1 D, or the Hessian and its LU factors
	double * xs = A + (size_t) n * ap;     // X
	double * ps = xs + n;                  // p
	double * g = ps + n;                   // dFdX
	double * gp = g + n;                   // dFdX_prev
	double * sv = gp + n;                  // s = alpha p
	double * yv = sv + n;                  // g = dFdX - dFdX_prev (the reference's name for it)
	double * rg = yv + n;                  // rho * yv
	double * ad = rg + n;                  // |X - Xprev|
	double * fdx = ad + n;                 // stencil values
	double * xa = fdx + n;                 // staged trial point (analytic slope)
	double * prod = xa + n;                // 2 x n slope products
	double * vals = prod + 2 * n;          // 2 x 2 line-search values
	double * bc = vals + 4;                // broadcast slots: [0] f(X) of the gradient, [1] f(X) of the FD Hessian
	int * piv = reinterpret_cast<int *>(bc + 4);   // n pivots, then the LU's broadcast slot

	bool agrad = false, aslope = false;
	if constexpr (has_partial<F>::value) {
		agrad = (flags & PNOL_BFGS_ANALYTIC_GRADIENT) != 0;
		aslope = (flags & PNOL_BFGS_ANALYTIC_SLOPE) != 0;
	}
	const int max_ls = prm.max_iter_ls;
	const double c1 = prm.c1, c2 = prm.c2;

	for (int j = tid; j < n; j += T) xs[j] = X[b * n + j];
	__syncthreads();

	// ---- D (:35-57) ----
	const int npairs = n * (n + 1) / 2;
	auto unrank = [](int e, int & i, int & j) {      // pair e of the lower triangle row by row -> (i <= j)
		int r = 0;
		while ((r + 1) * (r + 2) / 2 <= e) r++;
		i = e - r * (r + 1) / 2; j = r;
	};
	if (prm.init_hess_fd) {
		bool analytic_b = false;
		if constexpr (has_partial2<F>::value) {
			if (flags & PNOL_BFGS_ANALYTIC_HESSIAN) {
				analytic_b = true;
				const PtrAcc ax{xs};
				for (int e = tid; e < npairs; e += T) {
					int i, j;
					unrank(e, i, j);
					const double v = F::partial2(P, ax, n, i, j);
					A[i * ap + j] = v;
					A[j * ap + i] = v;
				}
			}
		}
		if (!analytic_b) {
			// Objective::hessianApproximation (Source/PNOL_Objective.cpp:38-85), f(X + dx e_i) computed once per i
			const double dxh = prm.dx_hess;
			for (int i = tid; i <= n; i += T) {
				if (i < n) {
					const PerturbAcc acc{xs, i, xs[i] + dxh};
					fdx[i] = F::eval(P, acc, n);
				} else {
					const PtrAcc ax{xs};
					bc[1] = F::eval(P, ax, n);
				}
			}
			__syncthreads();
			const double f = bc[1];
			for (int e = tid; e < npairs; e += T) {
				int i, j;
				unrank(e, i, j);
				double fij;
				if (i == j) {
					const PerturbAcc acc{xs, i, (xs[i] + dxh) + dxh};
					fij = F::eval(P, acc, n);
				} else {
					const Perturb2Acc acc{xs, i, xs[i] + dxh, j, xs[j] + dxh};
					fij = F::eval(P, acc, n);
				}
				const double v = (fij - fdx[i] - fdx[j] + f) / (dxh * dxh);
				A[i * ap + j] = v;
				A[j * ap + i] = v;
			}
		}
		for (int i = tid; i < n; i += T) piv[i] = i;
		__syncthreads();
		block_lu_factor<T>(A, ap, n, piv, piv + n);
		// matrixInverse: column j solves with b = e_j (oracle_lu_solve's substitutions), in place in column j of D
		for (int j = tid; j < n; j += T) {
			for (int i = 0; i < n; i++) {
				double s = piv[i] == j ? 1.0 : 0.0;
				for (int k = 0; k < i; k++) s = s - A[i * ap + k] * D[k * ap + j];
				D[i * ap + j] = s;
			}
			for (int i = n - 1; i >= 0; i--) {
				double s = D[i * ap + j];
				for (int k = i + 1; k < n; k++) s = s - A[i * ap + k] * D[k * ap + j];
				D[i * ap + j] = s / A[i * ap + i];
			}
		}
	} else {
		for (int e = tid; e < n * n; e += T) {
			const int i = e / n, j = e - i * n;
			D[i * ap + j] = i == j ? 1.0 : 0.0;
		}
	}
	__syncthreads();

	// ---- gradient at xs into g; with_f: bc[0] = f(xs) as well (the forward difference always evaluates it, for its quotient) ----
	auto gradient_at_x = [&](bool with_f) {
		const PtrAcc ax{xs};
		if constexpr (has_partial<F>::value) {
			if (agrad) {
				for (int i = tid; i < n; i += T) g[i] = F::partial(P, ax, n, i);
				if (with_f && tid == n) bc[0] = F::eval(P, ax, n);
				__syncthreads();
				return;
			}
		}
		const double dxg = prm.dx_grad;
		for (int i = tid; i <= n; i += T) {
			if (i < n) {
				const PerturbAcc acc{xs, i, xs[i] + dxg};      // XdX[i] = XdX[i] + dX[i]  (Source/PNOL_Objective.cpp:27)
				fdx[i] = F::eval(P, acc, n);
			} else {
				bc[0] = F::eval(P, ax, n);
			}
		}
		__syncthreads();
		const double f = bc[0];
		for (int i = tid; i < n; i += T) g[i] = (fdx[i] - f) / dxg;
		__syncthreads();
	};

	// ---- phi(a) and its slope; every thread gets both ----
	int parity = 0;
	const int pofs = T > 32 ? 32 : 1;      // first product thread: the second warp, or lane 1 of a single-warp block
	auto eval_phi = [&](double a, double & phi, double & dphi) {
		double * v = vals + 2 * parity;
		if constexpr (has_partial<F>::value) {
			if (aslope) {
				double * pr = prod + n * parity;
				for (int j = tid; j < n; j += T) xa[j] = xs[j] + a * ps[j];
				__syncthreads();
				const PtrAcc acc{xa};
				if (tid == 0) {
					v[0] = F::eval(P, acc, n);
				} else if (tid >= pofs && tid < pofs + n) {
					const int r = tid - pofs;
					pr[r] = F::partial(P, acc, n, r) * ps[r];
				}
				__syncthreads();
				phi = v[0];
				double s = 0.0;
				for (int r = 0; r < n; r++) s = s + pr[r];
				dphi = s;
				parity ^= 1;
				return;
			}
		}
		if (tid < 2) {
			// lineSearchObj / lineSearchFDDerivative (:144-172): X[i] + alpha*p[i], X[i] + (alpha+dalpha)*p[i]
			const LineAcc acc{xs, ps, nullptr, tid == 0 ? a : a + prm.dalpha};
			v[tid] = F::eval(P, acc, n);
		}
		__syncthreads();
		phi = v[0];
		dphi = (v[1] - v[0]) / prm.dalpha;
		parity ^= 1;
	};

	// ---- lineSearchZoom (:296-356) ----
	auto zoom = [&](double alo, double ahi, double plo, double phh, double dlo, double dhh, double phi0, double dphi0, double & aopt,
	                double & fopt) {
		for (int it = 0; it < max_ls; it++) {
			const double aj = bfgs_cubic_interp_min(alo, ahi, plo, phh, dlo, dhh);
			double pj, dj;
			eval_phi(aj, pj, dj);
			if (pj > phi0 + c1 * aj * dphi0 || pj >= plo) {
				ahi = aj; phh = pj; dhh = dj;
			} else {
				if (fabs(dj) <= fabs(c2 * dphi0)) { aopt = aj; fopt = pj; break; }
				if (dj * (ahi - alo) >= 0) { ahi = alo; phh = plo; dhh = dlo; }
				alo = aj; plo = pj; dlo = dj;
			}
		}
	};

	// ---- findMin (:62-139) ----
	gradient_at_x(true);
	double Fc = bc[0];
	const double f0 = Fc;
	const int max_iter = prm.max_iter;
	const double xmin = prm.x_min_diff, gmin = prm.min_grad_2norm;
	int iter = 0;
	double xdiff = xmin * 2;
	double g2 = 2 * gmin;
	while (iter < max_iter && xdiff > xmin && g2 > gmin) {
		for (int i = tid; i < n; i += T) {                             // p = -D dFdX (:78-79)
			double s = 0;
			for (int k = 0; k < n; k++) s = s + D[i * ap + k] * g[k];
			ps[i] = -s;
			gp[i] = g[i];
		}
		__syncthreads();
		// cubicInterpolationLineSearch (:177-291)
		double alpha = 0, Fopt = Fc;
		const double phi0 = Fc;
		double dphi0 = 0;
		for (int k = 0; k < n; k++) dphi0 = dphi0 + g[k] * ps[k];      // dotProd(dFdX, p)
		double am1 = 0, phim1 = phi0, dm1 = dphi0;
		double ai = prm.alpha_guess;
		for (int it = 0; it < max_ls; it++) {
			double phii, dphii;
			eval_phi(ai, phii, dphii);
			if ((phii > phi0 + c1 * ai * dphi0) || (phii >= phim1 && it > 1)) {
				zoom(am1, ai, phim1, phii, dm1, dphii, phi0, dphi0, alpha, Fopt);
				break;
			}
			if (fabs(dphii) <= fabs(c2 * dphi0)) { alpha = ai; Fopt = phii; break; }
			if (dphii >= 0) {
				zoom(ai, am1, phii, phim1, dphii, dm1, phi0, dphi0, alpha, Fopt);
				break;
			}
			am1 = ai; phim1 = phii; dm1 = dphii;
			ai = 2 * ai;
		}
		for (int i = tid; i < n; i += T) {                             // (:88-93), s (:100-105)
			const double xo = xs[i];
			const double xn = xo + alpha * ps[i];
			xs[i] = xn;
			sv[i] = alpha * ps[i];
			ad[i] = fabs(xn - xo);
		}
		Fc = Fopt;
		__syncthreads();
		gradient_at_x(false);                                          // (:97)
		for (int i = tid; i < n; i += T) yv[i] = g[i] - gp[i];
		__syncthreads();
		// updateHessianInv (:389-432): A = M1 D, D = A M2 + M3
		double ys = 0;
		for (int k = 0; k < n; k++) ys = ys + yv[k] * sv[k];
		const double rho = 1 / ys;
		for (int e = tid; e < n * n; e += T) {
			const int i = e / n, j = e - i * n;
			const double rs = rho * sv[i];
			double acc = 0;
			for (int k = 0; k < n; k++) {
				const double m1 = (i == k ? 1.0 : 0.0) - rs * yv[k];
				acc = acc + m1 * D[k * ap + j];
			}
			A[i * ap + j] = acc;
		}
		for (int i = tid; i < n; i += T) rg[i] = rho * yv[i];
		__syncthreads();
		for (int e = tid; e < n * n; e += T) {
			const int i = e / n, j = e - i * n;
			double acc = 0;
			for (int k = 0; k < n; k++) {
				const double m2 = (k == j ? 1.0 : 0.0) - rg[k] * sv[j];
				acc = acc + A[i * ap + k] * m2;
			}
			D[i * ap + j] = acc + (rho * sv[i]) * sv[j];
		}
		xdiff = 0;
		for (int i = 0; i < n; i++) xdiff = xdiff + ad[i];            // (:111-113)
		double s2 = 0;
		for (int i = 0; i < n; i++) s2 = s2 + g[i] * g[i];
		g2 = sqrt(s2);                                                 // vector2Norm(dFdX)
		__syncthreads();
		iter = iter + 1;
	}
	for (int j = tid; j < n; j += T) X[b * n + j] = xs[j];
	if (tid == 0) {
		f0_out[b] = f0;
		fopt_out[b] = Fc;
		iters_out[b] = iter;
		stop_out[b] = !(iter < max_iter) ? 0 : (!(xdiff > xmin) ? 1 : 2);
	}
}

template <class F, int T>
int bfgs_batch_launch(const pnol_launch_env * env, const FunctorParams & P, long long B, int n, double * X, const pnol_bfgs_params & prm,
                      int flags, double * f0_out, double * fopt_out, int * iters_out, int * stop_out)
{
	const size_t smem = bfgs_batch_smem(n);
	PNOL_DEV_REQUIRE(env, smem <= env->smem_optin, "bfgs batch: n = %d needs %zu bytes of shared memory", n, smem);
	auto kern = bfgs_batch_kernel<F, T>;
	PNOL_DEV_CUDA(env, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
	PNOL_DEV_LAUNCH(env, kern, (unsigned) B, T, smem, P, n, X, prm, flags, f0_out, fopt_out, iters_out, stop_out);
	return PNOL_OK;
}

/* pnol_bfgs_batch on device pointers: X (B x n, in/out), the four per-problem outputs (B). n in 1 .. 64. The analytic gradient and
 * slope flags need F::partial, the analytic Hessian flag with init_hess_fd F::partial2 (PNOL_ERR_NO_FUNCTOR otherwise). */
template <class F>
int bfgs_batch(const pnol_launch_env * env, const FunctorParams & P, long long B, int n, double * X, const pnol_bfgs_params * prm, int flags,
               double * f0_out, double * fopt_out, int * iters_out, int * stop_out)
{
	PNOL_DEV_REQUIRE(env, n >= 1 && n <= kBfgsBatchMaxN, "bfgs batch: n = %d is outside 1 .. %d", n, kBfgsBatchMaxN);
	PNOL_DEV_REQUIRE(env, B >= 0 && B <= 0x7fffffffLL, "bfgs batch: B = %lld is outside 0 .. 2^31 - 1", B);
	PNOL_DEV_REQUIRE(env, prm != nullptr, "bfgs batch: the parameters are required");
	if (B == 0) return PNOL_OK;
	if (!has_partial<F>::value && (flags & (PNOL_BFGS_ANALYTIC_GRADIENT | PNOL_BFGS_ANALYTIC_SLOPE))) {
		PNOL_DEV_ERR(env, "bfgs batch: the objective has no analytic gradient (partial()): the analytic gradient / slope flags are refused");
		return PNOL_ERR_NO_FUNCTOR;
	}
	if (!has_partial2<F>::value && (flags & PNOL_BFGS_ANALYTIC_HESSIAN) && prm->init_hess_fd) {
		PNOL_DEV_ERR(env, "bfgs batch: the objective has no analytic Hessian (partial2()): the analytic Hessian flag is refused");
		return PNOL_ERR_NO_FUNCTOR;
	}
#define PNOL_BFGS_BATCH_CFG(T) bfgs_batch_launch<F, T>(env, P, B, n, X, *prm, flags, f0_out, fopt_out, iters_out, stop_out)
	if (n <= 8) return PNOL_BFGS_BATCH_CFG(32);
	if (n <= 16) return PNOL_BFGS_BATCH_CFG(64);
	if (n <= 32) return PNOL_BFGS_BATCH_CFG(128);
	return PNOL_BFGS_BATCH_CFG(256);
#undef PNOL_BFGS_BATCH_CFG
}

// ---------------------------------------------------------------------------------------------------
// batched simplex search (pnol_simplex_batch): start b starts from row b of X (B x n) and runs SimplexSearch::findMin
// (host/SimplexSearch.cpp, Source/SimplexSearch.cpp:13-349) on the functor's objective, operation for operation what the unmodified
// host controller computes on the C-ABI's CPU stand-in, so every start returns the bits the reference returns on it alone:
//   - start simplex: vertex 0 is the start, vertex i = 1 .. n is x0[j] + initRandMax*(u - 0.5)*2.0 with u the stream's value at
//     stream_offset + b n^2 + (i - 1) n + j;
//   - centroid: xbar[i] = xbar[i] + x[k][i]/n over the n best vertices in sorted order from k = 0, each term divided (x (1/n) when n is
//     a power of two, else the IEEE quotient of div_exact: the divisor is loop-invariant); never a running centroid;
//   - reflection xbar + alpha*(xbar - w), expansion xbar + gamma*(xbar - w), contraction xbar + rho*(w - xbar), shrink
//     x0 + sigma*(xk - x0), all unfused, with the reference's accept rules; a shrink evaluates all n + 1 vertices, vertex 0 included
//     (a sentinel of the sort can sit in f[0]);
//   - simplexSort's permutation with both of its quirks (simplex_sort.hpp), and simplexDiff as a max with `>` (NaN skipped).
// Mapping: one group of G lanes per start (G from n: 4, 8, 16 or 32), 32 * kSimplexBatchWarps / G starts per CTA, a start's state in
// shared memory: the n + 1 vertex rows (physical storage), f and the sorted f, xbar, the candidate values, and idx (logical vertex k
// lives in row idx[k]) with the sort's scratch. A sort permutes idx, not the rows. Outside simplexSort's regime a pass can take an
// entry twice; the reference's rows are copies then, so the repeated entry gets the storage of the lost row and a copy of its content.
// Every iteration lanes 0, 1 and 2 evaluate the reflection, the expansion and the contraction in one F::eval instruction stream
// (SimplexCandAcc forms the coordinates on the fly), so that an iteration costs one evaluation latency; only the evaluations the
// reference makes are counted (evals_out). The groups of a warp run independently: every barrier is the group's __syncwarp, every
// reduction its shuffles, and a group that stopped idles until its warp ends.
// ---------------------------------------------------------------------------------------------------
constexpr int kSimplexBatchMaxN = 64;
constexpr int kSimplexBatchWarps = 4;

__host__ __device__ inline int simplex_batch_group(int n) { return n <= 4 ? 4 : (n <= 8 ? 8 : (n <= 16 ? 16 : 32)); }
// shared memory of one start in doubles: the (n + 1) x n vertex rows, f and the sorted f (n + 1 each), xbar (n), the candidate values
// (4), then five (n + 1)-int arrays (idx, the new idx, the pass order, the taken marks, the copy sources)
__host__ __device__ inline int simplex_batch_stride(int n)
{
	const int N = n + 1;
	return N * n + 2 * N + n + 4 + (5 * N + 1) / 2;
}

// a candidate from the centroid and the worst vertex w, formed on the fly: toward == 0 gives xbar + c*(xbar - w) (reflection,
// expansion), toward == 1 xbar + c*(w - xbar) (contraction)
struct SimplexCandAcc {
	const double * xbar; const double * w; double c; int toward;
	__device__ __forceinline__ double operator[](int j) const
	{
		const double xb = xbar[j], wj = w[j];
		return xb + c * (toward ? wj - xb : xb - wj);
	}
};

template <int G>
__device__ __forceinline__ SimplexSortStats simplex_group_stats(const double * f, int N, int lane, unsigned gmask)
{
	SimplexSortStats s = simplex_stats_partial(f, N, lane, G);
#pragma unroll
	for (int o = G / 2; o > 0; o >>= 1) {
		SimplexSortStats t;
		t.M = __shfl_xor_sync(gmask, s.M, o, G);
		t.m = __shfl_xor_sync(gmask, s.m, o, G);
		t.iM = __shfl_xor_sync(gmask, s.iM, o, G);
		t.im = __shfl_xor_sync(gmask, s.im, o, G);
		t.nan = __shfl_xor_sync(gmask, s.nan, o, G);
		s = simplex_stats_combine(s, t);
	}
	return s;
}

template <class F, int G>
__global__ void __launch_bounds__(32 * kSimplexBatchWarps)
simplex_batch_kernel(FunctorParams P, long long B, int n, double * __restrict__ X, pnol_simplex_params prm, StreamDev st,
                     unsigned long long offset, double * __restrict__ f0_out, double * __restrict__ fopt_out, int * __restrict__ iters_out,
                     int * __restrict__ stop_out, long long * __restrict__ evals_out)
{
	extern __shared__ double sm[];
	constexpr int kGroups = 32 * kSimplexBatchWarps / G;
	const int lane = threadIdx.x & (G - 1);
	const int grp = threadIdx.x / G;
	const long long b = (long long) blockIdx.x * kGroups + grp;
	if (b >= B) return;
	const unsigned gmask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << (threadIdx.x & 31 & ~(G - 1)));
	const int N = n + 1;
	double * V = sm + (size_t) grp * simplex_batch_stride(n);      // row r: V + r n
	double * fv = V + N * n;                                        // f of logical vertex k
	double * ft = fv + N;
	double * xbar = ft + N;
	double * cand = xbar + n;                                       // f of the reflection, expansion, contraction
	int * idx = reinterpret_cast<int *>(cand + 4);
	int * nidx = idx + N;
	int * perm = nidx + N;
	int * mark = perm + N;
	int * csrc = mark + N;

	// ---- simplexSort (:272-326): fv and idx in sorted order ----
	auto sort = [&]() {
		const SimplexSortStats s = simplex_group_stats<G>(fv, N, lane, gmask);
		if (simplex_in_regime(fv, s)) {
			const bool one_first = fv[1] == s.m;
			for (int i = lane; i < N; i += G) {
				const int r = simplex_rank(fv, N, i, one_first);
				nidx[r] = idx[i];
				ft[r] = fv[i];
			}
			__syncwarp(gmask);
			for (int k = lane; k < N; k += G) { idx[k] = nidx[k]; fv[k] = ft[k]; }
			__syncwarp(gmask);
			return;
		}
		// the literal N passes, each a group argmin
		const double S = 2 * simplex_first_max(fv, s);
		int c = 1;
		for (int k = 0; k < N; k++) {
			const SimplexSortStats t = simplex_group_stats<G>(fv, N, lane, gmask);
			c = simplex_pass_take(fv, c, t);
			__syncwarp(gmask);
			if (lane == 0) { perm[k] = c; ft[k] = fv[c]; fv[c] = S; }
			__syncwarp(gmask);
		}
		// a repeated entry gets the storage of a lost one (exactly as many are lost as repeated) and a copy of its row
		if (lane == 0) {
			for (int l = 0; l < N; l++) mark[l] = 0;
			for (int k = 0; k < N; k++) {
				const int e = perm[k];
				if (!mark[e]) { mark[e] = 1; nidx[k] = idx[e]; csrc[k] = -1; }
				else { nidx[k] = -1; csrc[k] = idx[e]; }
			}
			int l = 0;
			for (int k = 0; k < N; k++) {
				if (nidx[k] >= 0) continue;
				while (mark[l]) l++;
				nidx[k] = idx[l++];
			}
		}
		__syncwarp(gmask);
		for (int k = 0; k < N; k++)
			if (csrc[k] >= 0)
				for (int j = lane; j < n; j += G) V[nidx[k] * n + j] = V[csrc[k] * n + j];
		__syncwarp(gmask);
		for (int k = lane; k < N; k += G) { idx[k] = nidx[k]; fv[k] = ft[k]; }
		__syncwarp(gmask);
	};

	// ---- start simplex, its evaluation and sort (:47-73) ----
	const unsigned long long base = offset + (unsigned long long) b * (unsigned long long) (n * n);
	for (int e = lane; e < N * n; e += G) {
		const int i = e / n, j = e - i * n;
		double v = X[b * n + j];
		if (i > 0) v = v + prm.init_rand_max * (st.u(base + (unsigned long long) (e - n)) - 0.5) * 2.0;
		V[e] = v;
	}
	for (int k = lane; k < N; k += G) idx[k] = k;
	__syncwarp(gmask);
	for (int k = lane; k < N; k += G) {
		const PtrAcc a{V + k * n};
		fv[k] = F::eval(P, a, n);
	}
	__syncwarp(gmask);
	const double f0 = fv[0];
	long long evals = N;
	sort();

	const RecipDiv rd = make_recip((double) n);
	const bool pow2 = (n & (n - 1)) == 0;
	const bool three = recip_three_ok(rd) != 0;
	const double rn = 1.0 / (double) n;
	int iter = 0;
	double xdiff = prm.x_min_diff * 2;
	while (iter < prm.max_iter && xdiff > prm.x_min_diff) {
		// centroid of the n best vertices (:86-98)
		for (int i = lane; i < n; i += G) {
			double s = 0.0;
			for (int k = 0; k < n; k++) {
				const double x = V[idx[k] * n + i];
				double q;
				if (pow2) q = x * rn;
				else if (three && div_exact_x_ok_pz(x)) q = div_exact3_core(x, rd);
				else q = div_exact(x, rd);
				s = s + q;
			}
			xbar[i] = s;
		}
		__syncwarp(gmask);
		// the three candidates at once (:100-172)
		double * w = V + idx[n] * n;
		if (lane < 3) {
			const SimplexCandAcc acc{xbar, w, lane == 0 ? prm.alpha : (lane == 1 ? prm.gamma : prm.rho), lane == 2};
			cand[lane] = F::eval(P, acc, n);
		}
		__syncwarp(gmask);
		const double fr = cand[0], fe = cand[1], fc = cand[2];
		int take;                                                   // 0 reflection, 1 expansion, 2 contraction, 3 shrink
		evals += 1;
		if (fr >= fv[0] && fr < fv[n - 1]) {
			take = 0;
		} else if (fr < fv[0]) {
			evals += 1;
			take = fe < fr ? 1 : 0;
		} else {
			evals += 1;
			take = fc < fv[n] ? 2 : 3;
		}
		if (take < 3) {
			const double c = take == 0 ? prm.alpha : (take == 1 ? prm.gamma : prm.rho);
			for (int j = lane; j < n; j += G) {
				const double xb = xbar[j], wj = w[j];
				w[j] = xb + c * (take == 2 ? wj - xb : xb - wj);
			}
			__syncwarp(gmask);
			if (lane == 0) fv[n] = take == 0 ? fr : (take == 1 ? fe : fc);
		} else {
			// shrink towards the best vertex, then evaluate all n + 1 vertices (:175-189)
			const double * x0 = V + idx[0] * n;
			for (int e = lane; e < n * n; e += G) {
				const int k = 1 + e / n, j = e - (k - 1) * n;
				double * xk = V + idx[k] * n;
				xk[j] = x0[j] + prm.sigma * (xk[j] - x0[j]);
			}
			__syncwarp(gmask);
			for (int k = lane; k < N; k += G) {
				const PtrAcc a{V + idx[k] * n};
				fv[k] = F::eval(P, a, n);
			}
			evals += N;
		}
		__syncwarp(gmask);
		sort();
		// simplexDiff (:330-349): the largest |x0[j] - xk[j]| found with `>`, NaN skipped
		const double * x0 = V + idx[0] * n;
		double mx = 0;
		for (int e = lane; e < n * n; e += G) {
			const int k = 1 + e / n, j = e - (k - 1) * n;
			const double d = fabs(x0[j] - V[idx[k] * n + j]);
			if (d > mx) mx = d;
		}
#pragma unroll
		for (int o = G / 2; o > 0; o >>= 1) {
			const double t = __shfl_xor_sync(gmask, mx, o, G);
			if (t > mx) mx = t;
		}
		xdiff = mx;
		iter = iter + 1;
	}
	for (int j = lane; j < n; j += G) X[b * n + j] = V[idx[0] * n + j];
	if (lane == 0) {
		f0_out[b] = f0;
		fopt_out[b] = fv[0];
		iters_out[b] = iter;
		stop_out[b] = !(iter < prm.max_iter) ? 0 : 1;
		if (evals_out) evals_out[b] = evals;
	}
}

template <class F, int G>
int simplex_batch_launch(const pnol_launch_env * env, const FunctorParams & P, long long B, int n, double * X, const pnol_simplex_params & prm,
                         const StreamDev & st, unsigned long long offset, double * f0_out, double * fopt_out, int * iters_out, int * stop_out,
                         long long * evals_out)
{
	constexpr int kGroups = 32 * kSimplexBatchWarps / G;
	const size_t smem = (size_t) kGroups * simplex_batch_stride(n) * sizeof(double);
	PNOL_DEV_REQUIRE(env, smem <= env->smem_optin, "simplex batch: n = %d needs %zu bytes of shared memory", n, smem);
	auto kern = simplex_batch_kernel<F, G>;
	PNOL_DEV_CUDA(env, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
	const long long grid = (B + kGroups - 1) / kGroups;
	PNOL_DEV_LAUNCH(env, kern, (unsigned) grid, 32 * kSimplexBatchWarps, smem, P, B, n, X, prm, st, offset, f0_out, fopt_out, iters_out,
	                stop_out, evals_out);
	return PNOL_OK;
}

/* pnol_simplex_batch on device pointers: X (B x n, in/out), the per-start outputs (B; evals_out may be NULL), stream->values (when set)
 * a device array whose value at position p is values[p]. n in 1 .. 64. */
template <class F>
int simplex_batch(const pnol_launch_env * env, const FunctorParams & P, long long B, int n, double * X, const pnol_simplex_params * prm,
                  const pnol_stream_desc * stream, uint64_t stream_offset, double * f0_out, double * fopt_out, int * iters_out, int * stop_out,
                  long long * evals_out)
{
	PNOL_DEV_REQUIRE(env, n >= 1 && n <= kSimplexBatchMaxN, "simplex batch: n = %d is outside 1 .. %d", n, kSimplexBatchMaxN);
	PNOL_DEV_REQUIRE(env, B >= 0 && B <= 0x7fffffffLL, "simplex batch: B = %lld is outside 0 .. 2^31 - 1", B);
	PNOL_DEV_REQUIRE(env, prm != nullptr && stream != nullptr, "simplex batch: the parameters and the stream are required");
	if (B == 0) return PNOL_OK;
	StreamDev st;
	st.values = stream->values; st.n_values = stream->n_values; st.seed = stream->seed; st.scale = stream->scale;
#define PNOL_SIMPLEX_BATCH_CFG(G) \
	simplex_batch_launch<F, G>(env, P, B, n, X, *prm, st, stream_offset, f0_out, fopt_out, iters_out, stop_out, evals_out)
	switch (simplex_batch_group(n)) {
		case 4: return PNOL_SIMPLEX_BATCH_CFG(4);
		case 8: return PNOL_SIMPLEX_BATCH_CFG(8);
		case 16: return PNOL_SIMPLEX_BATCH_CFG(16);
		default: return PNOL_SIMPLEX_BATCH_CFG(32);
	}
#undef PNOL_SIMPLEX_BATCH_CFG
}

/* ---- launch tables (pnol_functor_vtable) of a functor type ---- */
template <class F> struct ScalarTable {
	static int eval_batch_(const pnol_launch_env * env, const pnol_functor_params * P, const double * pts, long long B, int n, long long ld,
	                       const unsigned char * ind, double * f_out) { return eval_batch<F>(env, *P, pts, B, n, ld, ind, f_out); }
	static int fd_points_(const pnol_launch_env * env, const pnol_functor_params * P, const double * xfull, int nfull, const int * pos,
	                      const double * dx, int i0, int i1, double * fdx, double * f0) { return fd_points<F>(env, *P, xfull, nfull, pos, dx, i0, i1, fdx, f0); }
	static int fd_hessian_(const pnol_launch_env * env, const pnol_functor_params * P, const double * x, const double * dx, int n,
	                       const double * fdx, const double * f0, double * B) { return fd_hessian<F>(env, *P, x, dx, n, fdx, f0, B); }
	static int alpha_pool_(const pnol_launch_env * env, const pnol_functor_params * P, const double * xfull, const double * pfull,
	                       const unsigned char * is_const, int nfull, const double * alpha, int npool, double dalpha,
	                       const unsigned char * eval_ind, int want_shifted, double * vals)
	{ return alpha_pool<F>(env, *P, xfull, pfull, is_const, nfull, alpha, npool, dalpha, eval_ind, want_shifted, vals); }
	static int gradient_(const pnol_launch_env * env, const pnol_functor_params * P, const double * xfull, int nfull, const int * pos, int i0,
	                     int i1, double * g, double * f0) { return gradient<F>(env, *P, xfull, nfull, pos, i0, i1, g, f0); }
	static int hessian_(const pnol_launch_env * env, const pnol_functor_params * P, const double * x, int n, double * H)
	{ return hessian<F>(env, *P, x, n, H); }
	static int alpha_slope_(const pnol_launch_env * env, const pnol_functor_params * P, const double * xfull, const double * pfull,
	                        const unsigned char * is_const, int nfull, const int * pos, const double * p, int n, const double * alpha, int npool,
	                        const unsigned char * eval_ind, double * vals)
	{ return alpha_slope<F>(env, *P, xfull, pfull, is_const, nfull, pos, p, n, alpha, npool, eval_ind, vals); }
	static int bfgs_batch_(const pnol_launch_env * env, const pnol_functor_params * P, long long B, int n, double * X, const pnol_bfgs_params * prm,
	                       int flags, double * f0_out, double * fopt_out, int * iters_out, int * stop_out)
	{ return bfgs_batch<F>(env, *P, B, n, X, prm, flags, f0_out, fopt_out, iters_out, stop_out); }
	static int simplex_batch_(const pnol_launch_env * env, const pnol_functor_params * P, long long B, int n, double * X,
	                          const pnol_simplex_params * prm, const pnol_stream_desc * stream, uint64_t stream_offset, double * f0_out,
	                          double * fopt_out, int * iters_out, int * stop_out, long long * evals_out)
	{ return simplex_batch<F>(env, *P, B, n, X, prm, stream, stream_offset, f0_out, fopt_out, iters_out, stop_out, evals_out); }
	static pnol_functor_vtable make(int n_columns)
	{
		pnol_functor_vtable vt = {};
		vt.abi_version = PNOL_FUNCTOR_ABI;
		vt.n_columns = n_columns;
		vt.eval_batch = eval_batch_;
		vt.fd_points = fd_points_;
		vt.fd_hessian = fd_hessian_;
		vt.alpha_pool = alpha_pool_;
		return vt;
	}
	/* registers the table, then its batched BFGS and simplex launchers, (F defines partial) its gradient and line-search slope launchers
	 * and (F defines partial2) its Hessian launcher, in this order: a launcher attaches to the registered table */
	static int register_as(int kind, const pnol_functor_vtable * vt)
	{
		int st = pnol_register_functor(kind, vt);
		if (st == PNOL_OK) st = pnol_register_functor_bfgs_batch(kind, bfgs_batch_);
		if (st == PNOL_OK) st = pnol_register_functor_simplex_batch(kind, simplex_batch_);
		if constexpr (has_partial<F>::value) {
			if (st == PNOL_OK) st = pnol_register_functor_gradient(kind, gradient_);
			if (st == PNOL_OK) st = pnol_register_functor_slope(kind, alpha_slope_);
		}
		if constexpr (has_partial2<F>::value) {
			if (st == PNOL_OK) st = pnol_register_functor_hessian(kind, hessian_);
		}
		return st;
	}
};
template <class R> struct ResidualTable {
	static int residual_(const pnol_launch_env * env, const pnol_functor_params * P, const double * x, int n, double * F) { return residual<R>(env, *P, x, n, F); }
	static int fd_jacobian_(const pnol_launch_env * env, const pnol_functor_params * P, const double * x, const double * dx, int n, double * J,
	                        double * F) { return fd_jacobian<R>(env, *P, x, dx, n, J, F); }
	static int jacobian_(const pnol_launch_env * env, const pnol_functor_params * P, const double * x, int n, double * J, double * F)
	{ return jacobian<R>(env, *P, x, n, J, F); }
	static int lm_batch_(const pnol_launch_env * env, const pnol_functor_params * P, const long long * row_off, long long B, int n, double * X,
	                     const double * dx, double lambda0, double lambda_factor, double x_min_diff, int max_iter, int jac_mode,
	                     double * chisq_out, double * lambda_out, int * iters_out, int * stopped_out, double * F_out)
	{
		return lm_batch<R>(env, *P, row_off, B, n, X, dx, lambda0, lambda_factor, x_min_diff, max_iter, jac_mode, chisq_out, lambda_out,
		                   iters_out, stopped_out, F_out);
	}
	static pnol_functor_vtable make(int n_columns)
	{
		pnol_functor_vtable vt = {};
		vt.abi_version = PNOL_FUNCTOR_ABI;
		vt.n_columns = n_columns;
		vt.residual = residual_;
		vt.fd_jacobian = fd_jacobian_;
		if constexpr (has_jacobian<R>::value) vt.jacobian = jacobian_;      // NULL otherwise: PNOL_JAC_ANALYTIC is refused
		return vt;
	}
	/* registers the table, then attaches its batched LM launcher (it serves PNOL_JAC_ANALYTIC only when R defines jacobian()) */
	static int register_as(int kind, const pnol_functor_vtable * vt)
	{
		int st = pnol_register_functor(kind, vt);
		if (st == PNOL_OK) st = pnol_register_functor_lm_batch(kind, lm_batch_);
		return st;
	}
};

} // namespace dev
} // namespace pnol

/* Registration at load time of the translation unit (one per functor). KIND: an integer constant in the user ranges of pnol_b200.h. */
#define PNOL_REGISTER_SCALAR_FUNCTOR(KIND, F, NCOLS)                                                              \
	static const pnol_functor_vtable pnol_vt_##F = pnol::dev::ScalarTable<F>::make(NCOLS);                        \
	static const int pnol_reg_##F = pnol::dev::ScalarTable<F>::register_as((KIND), &pnol_vt_##F);
#define PNOL_REGISTER_RESIDUAL_FUNCTOR(KIND, R, NCOLS)                                                            \
	static const pnol_functor_vtable pnol_vt_##R = pnol::dev::ResidualTable<R>::make(NCOLS);                      \
	static const int pnol_reg_##R = pnol::dev::ResidualTable<R>::register_as((KIND), &pnol_vt_##R);

#endif /* PNOL_DEVICE_FUNCTOR_KERNELS_CUH_ */
