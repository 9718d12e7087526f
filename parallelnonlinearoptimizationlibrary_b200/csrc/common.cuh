// common.cuh -- context, error handling, host/device pointer staging, launch accounting.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <map>
#include <string>
#include <thread>
#include <vector>

#include "pnol_b200.h"
#include "pnol/functors.hpp"

struct ncclComm;
namespace pnol { struct PnolPeer; }

struct PnolTimerEntry {
	double total_ms = 0;
	long long count = 0;
	std::vector<std::pair<cudaEvent_t, cudaEvent_t> > pending;
};

struct pnol_ctx {
	int device = 0;
	cudaStream_t stream = nullptr;
	int sm_count = 0;
	size_t smem_optin = 0;
	std::string err;
	char errbuf[512] = {0};        // text written by the header launchers (pnol_launch_env::err); pnol_last_error reads it when err is empty
	uint64_t launches = 0;

	// grow-only scratch buffers (device)
	void * ws[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
	size_t ws_bytes[5] = {0, 0, 0, 0, 0};
	// pinned staging for small scalar read-backs
	double * pinned = nullptr;
	size_t pinned_doubles = 0;
	// pinned staging + copy streams of the threaded host <-> device copy of large pageable buffers (capi.cu: staged_copy)
	void * stage_pinned = nullptr;
	cudaStream_t stage_streams[8] = {};
	cudaEvent_t stage_events[16] = {};

	std::thread * bg_copy = nullptr;       // pnol_copy_start: the worker of a device -> host copy in flight (one at a time)
	int bg_copy_status = 0;

	// SYRK work plan of the last (m, n) shape (device copy of the descriptor tables; see launch_syrk)
	void * syrk_plan = nullptr;
	size_t syrk_plan_bytes = 0;
	long long syrk_plan_m = -1;
	int syrk_plan_n = -1;
	int syrk_plan_kind = -1;       // 0: one role per CTA (LDGSTS kernel), 1 / 2: stream-K segments (TMA kernel) without / with J^T F

	// communicator
	ncclComm * comm = nullptr;
	int rank = 0;
	int nranks = 1;
	// local (non-collective) mode, pnol_comm_set_local: rank / nranks read 0 / 1 while it is on, the real values wait here
	bool local = false;
	int comm_rank = 0;
	int comm_nranks = 1;

	// what the last pnol_lm_iterate left behind (pnol_lm_last_run)
	int lm_last_stopped = 0;
	double lm_last_xdiff = 0.0;

	int ga_sharding = 0;           // pnol_ga_set_sharding: 0 auto, 1 rows, 2 sweep
	pnol::PnolPeer * peer = nullptr;   // NVLink peer-memory exchange of the sharded LM step (peer.cu)

	// timers
	int timers_on = 0;             // pnol_timer_enable: 0 off, 1 every scope, 2 the heavy kernels only (syrk, fd_jacobian, residual)
	std::map<std::string, PnolTimerEntry> timers;
};

struct pnol_functor {
	pnol_ctx * ctx;
	int kind;
	pnol::FunctorParams params;       // device-side view (column pointers are device pointers)
	void * owned[PNOL_MAX_COLUMNS];   // device columns we allocated (nullptr when borrowed)
	int n_columns;
};

#define PNOL_SET_ERR(ctx, ...)                                    \
	do {                                                          \
		char _buf[512];                                           \
		snprintf(_buf, sizeof _buf, __VA_ARGS__);                 \
		if (ctx) { (ctx)->err = _buf; (ctx)->errbuf[0] = 0; }     \
	} while (0)

#define PNOL_CUDA(ctx, call)                                                                       \
	do {                                                                                           \
		cudaError_t _e = (call);                                                                   \
		if (_e != cudaSuccess) {                                                                   \
			PNOL_SET_ERR(ctx, "%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
			return PNOL_ERR_CUDA;                                                                  \
		}                                                                                          \
	} while (0)

#define PNOL_CHECK(call)                     \
	do {                                     \
		int _s = (call);                     \
		if (_s != PNOL_OK) return _s;        \
	} while (0)

#define PNOL_REQUIRE(ctx, cond, ...)             \
	do {                                         \
		if (!(cond)) {                           \
			PNOL_SET_ERR(ctx, __VA_ARGS__);      \
			return PNOL_ERR_INVALID;             \
		}                                        \
	} while (0)

// every kernel launch of the library goes through this macro so that pnol_ctx_launches() is exact
#define PNOL_LAUNCH(ctx, kernel, grid, block, smem, ...)                                   \
	do {                                                                                   \
		kernel<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);                   \
		(ctx)->launches++;                                                                 \
		cudaError_t _e = cudaGetLastError();                                               \
		if (_e != cudaSuccess) {                                                           \
			PNOL_SET_ERR(ctx, "%s:%d: launch %s -> %s", __FILE__, __LINE__, #kernel, cudaGetErrorString(_e)); \
			return PNOL_ERR_CUDA;                                                          \
		}                                                                                  \
	} while (0)

namespace pnol {

inline bool is_device_ptr(const void * p)
{
	if (!p) return false;
	cudaPointerAttributes a;
	cudaError_t e = cudaPointerGetAttributes(&a, p);
	if (e != cudaSuccess) { cudaGetLastError(); return false; }
	return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

int ws_reserve(pnol_ctx * ctx, int slot, size_t bytes);
int pinned_reserve(pnol_ctx * ctx, size_t doubles);

// Input array that may live on the host: gives a device pointer valid until the object dies.
template <typename T> class DevIn {
  public:
	DevIn() {}
	~DevIn() { if (tmp_) cudaFreeAsync(tmp_, ctx_->stream); }
	int init(pnol_ctx * ctx, const T * p, size_t count)
	{
		ctx_ = ctx;
		if (!p || count == 0) { ptr_ = nullptr; return PNOL_OK; }
		if (is_device_ptr(p)) { ptr_ = p; return PNOL_OK; }
		PNOL_CUDA(ctx, cudaMallocAsync(&tmp_, count * sizeof(T), ctx->stream));
		PNOL_CUDA(ctx, cudaMemcpyAsync(tmp_, p, count * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
		ptr_ = (const T *) tmp_;
		return PNOL_OK;
	}
	const T * get() const { return ptr_; }
  private:
	pnol_ctx * ctx_ = nullptr;
	const T * ptr_ = nullptr;
	void * tmp_ = nullptr;
};

// Output (or in/out) array that may live on the host: commit() copies back and synchronises.
template <typename T> class DevOut {
  public:
	DevOut() {}
	~DevOut() { if (tmp_) cudaFreeAsync(tmp_, ctx_->stream); }
	int init(pnol_ctx * ctx, T * p, size_t count, bool copy_in = false)
	{
		ctx_ = ctx; host_ = nullptr; count_ = count;
		if (!p || count == 0) { ptr_ = nullptr; return PNOL_OK; }
		if (is_device_ptr(p)) { ptr_ = p; return PNOL_OK; }
		PNOL_CUDA(ctx, cudaMallocAsync(&tmp_, count * sizeof(T), ctx->stream));
		if (copy_in) PNOL_CUDA(ctx, cudaMemcpyAsync(tmp_, p, count * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
		ptr_ = (T *) tmp_; host_ = p;
		return PNOL_OK;
	}
	T * get() const { return ptr_; }
	bool staged() const { return host_ != nullptr; }
	// issue the copy back (no sync); caller must pnol::finish() afterwards
	int commit()
	{
		if (host_) PNOL_CUDA(ctx_, cudaMemcpyAsync(host_, tmp_, count_ * sizeof(T), cudaMemcpyDeviceToHost, ctx_->stream));
		return PNOL_OK;
	}
  private:
	pnol_ctx * ctx_ = nullptr;
	T * ptr_ = nullptr;
	T * host_ = nullptr;
	void * tmp_ = nullptr;
	size_t count_ = 0;
};

inline int finish(pnol_ctx * ctx)
{
	PNOL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	return PNOL_OK;
}

// RAII scope timer (CUDA events on the context's stream); a no-op unless pnol_timer_enable(ctx, 1)
class TimerScope {
  public:
	TimerScope(pnol_ctx * ctx, const char * name) : ctx_(ctx)
	{
		if (!ctx->timers_on) return;
		// mode 2: only the kernels that carry the step (an event pair costs about 5 us of stream time: seven scopes per LM iteration
		// are 2 % of an iteration at 8 GPUs)
		if (ctx->timers_on == 2 && strcmp(name, "syrk") != 0 && strcmp(name, "fd_jacobian") != 0 && strcmp(name, "residual") != 0) return;
		cudaEventCreate(&a_); cudaEventCreate(&b_);
		cudaEventRecord(a_, ctx->stream);
		name_ = name; on_ = true;
	}
	~TimerScope()
	{
		if (!on_) return;
		cudaEventRecord(b_, ctx_->stream);
		ctx_->timers[name_].pending.push_back(std::make_pair(a_, b_));
	}
  private:
	pnol_ctx * ctx_;
	bool on_ = false;
	const char * name_ = nullptr;
	cudaEvent_t a_ = nullptr, b_ = nullptr;
};

// ---- functor kinds: everything the library can launch for one kind ----
struct KindTable {
	pnol_functor_vtable vt;               // the family's launchers, n_columns and (residual models, may be null) jacobian
	pnol_gradient_launcher gradient;      // scalar objectives, may be null: pnol_gradient[_recur]
	pnol_hessian_launcher hessian;        // scalar objectives, may be null: pnol_hessian
	pnol_slope_launcher slope;            // scalar objectives, may be null: pnol_alpha_pool_analytic
	pnol_lm_batch_launcher lm_batch;      // residual models, may be null: pnol_lm_batch
	pnol_bfgs_batch_launcher bfgs_batch;  // scalar objectives, may be null: pnol_bfgs_batch
	pnol_simplex_batch_launcher simplex_batch;  // scalar objectives, may be null: pnol_simplex_batch
};
// copies out the record of a built-in or registered kind (capi.cu); false for any other kind. A copy, so that re-registering a kind
// while a launch runs is safe.
bool kind_table(int kind, KindTable * out);
const KindTable * builtin_kind_table(int kind);      // builtin_functors.cu: nullptr unless the kind is built in
inline bool is_user_kind(int kind) { return kind >= PNOL_F_USER_SCALAR_BASE && kind < PNOL_F_USER_RESIDUAL_BASE + 1000; }
inline bool is_residual_kind(int kind) { return (kind >= 100 && kind < PNOL_F_USER_SCALAR_BASE) || (kind >= PNOL_F_USER_RESIDUAL_BASE && kind < PNOL_F_USER_RESIDUAL_BASE + 1000); }
// a functor of the other family (family: "scalar objective" or "residual model"). The status differs by origin, as it always has:
// PNOL_ERR_NO_FUNCTOR for a built-in kind, PNOL_ERR_INVALID for a user kind.
inline int wrong_family(pnol_ctx * ctx, int kind, const char * family)
{
	PNOL_SET_ERR(ctx, "functor kind %d is not a %s", kind, family);
	return is_user_kind(kind) ? PNOL_ERR_INVALID : PNOL_ERR_NO_FUNCTOR;
}
inline pnol_launch_env make_env(pnol_ctx * ctx)
{
	pnol_launch_env env;
	env.stream = (void *) ctx->stream;
	env.sm_count = ctx->sm_count;
	env.smem_optin = ctx->smem_optin;
	env.launches = (unsigned long long *) &ctx->launches;
	env.err = ctx->errbuf;
	env.err_len = sizeof ctx->errbuf;
	return env;
}

// ---- internal entry points implemented across the .cu files (device pointers only) ----
int launch_eval_batch(pnol_ctx * ctx, const pnol_functor * f, const double * pts, long long B, int n, long long ld,
                      const unsigned char * indicator, double * f_out);
int launch_fd_points(pnol_ctx * ctx, const pnol_functor * f, const double * xfull, int nfull, const int * pos,
                     const double * dx, int i0, int i1, double * fdx_out, double * f0_out);
int launch_fd_quotient(pnol_ctx * ctx, const double * fdx, const double * f0, const double * dx, int n, double * g);
int launch_gradient(pnol_ctx * ctx, const pnol_functor * f, const double * xfull, int nfull, const int * pos, int i0, int i1,
                    double * g_out, double * f0_out);
int launch_assemble_recur(pnol_ctx * ctx, const double * xr, int nr, const double * const_x,
                          const unsigned char * const_ind, int nfull, double * xfull, int * pos, int * nr_found);
int launch_fd_hessian(pnol_ctx * ctx, const pnol_functor * f, const double * x, const double * dx, int n,
                      const double * fdx, const double * f0, double * B);
int launch_hessian(pnol_ctx * ctx, const pnol_functor * f, const double * x, int n, double * H);
int launch_alpha_pool(pnol_ctx * ctx, const pnol_functor * f, const double * xfull, const double * pfull,
                      const unsigned char * is_const, int nfull, const double * alpha, int npool, double dalpha,
                      const unsigned char * eval_ind, double * phi, double * dphi, int * bad_dev);
int launch_alpha_slope(pnol_ctx * ctx, const pnol_functor * f, const double * xfull, const double * pfull,
                       const unsigned char * is_const, int nfull, const int * pos, const double * p, int n, const double * alpha,
                       int npool, const unsigned char * eval_ind, double * phi, double * dphi, int * bad_dev);

// sum of squares: deterministic, fixed 4096-row blocks -> partials -> one 1024-thread block (sumsq_final_sum). partials_out / np_out
// (both): only the partials are produced and handed back, the caller's own kernel finishes with sumsq_final_sum
int launch_residual(pnol_ctx * ctx, const pnol_functor * f, const double * x, int n, double * F, double * sumsq_dev,
                    const double ** partials_out = nullptr, int * np_out = nullptr);

// the final stage of the sum of squares, for a block of 1024 threads (red: 1024 doubles of shared memory); the result is returned
// to every thread. One definition, so that every kernel that finishes the sum produces the same bits.
__device__ __forceinline__ double sumsq_final_sum(const double * __restrict__ partials, int np, double * red)
{
	double s = 0;
	for (int e = threadIdx.x; e < np; e += 1024) s = s + partials[e];
	red[threadIdx.x] = s;
	__syncthreads();
	for (int o = 512; o > 0; o >>= 1) {
		if (threadIdx.x < o) red[threadIdx.x] = red[threadIdx.x] + red[threadIdx.x + o];
		__syncthreads();
	}
	return red[0];
}
// PNOL_ERR_INVALID unless n = 2 * 2^j for the sum-of-Lorentzians model (its balanced tree); PNOL_OK for every other kind
int lorentz_shape_ok(pnol_ctx * ctx, const pnol_functor * f, int n);
int launch_fd_jacobian(pnol_ctx * ctx, const pnol_functor * f, const double * x, const double * dx, int n, double * J,
                       double * F, int mode, const double * Fw = nullptr, double * jtf_out = nullptr, bool * jtf_done = nullptr);

// rhs_src (device, n; only looked at when F == nullptr): J^T F already summed by the caller -- copied behind J^T J by the finish kernel
int launch_syrk(pnol_ctx * ctx, const double * J, const double * F, long long m, int n, double * packed /* n*n + n */,
                const double * rhs_src = nullptr);
int syrk_plan_selftest(long long m, int n, int sm_count, int with_f);
int launch_lm_damp(pnol_ctx * ctx, const double * packed, int n, double lambda, double * JTJ, double * A, double * rhs,
                   const double * lambda_dev = nullptr, bool rhs_behind_jtj = false /* JTJ holds n*n + n: -J^T F goes behind J^T J */);
int launch_dgemm_nn(pnol_ctx * ctx, const double * A, const double * B, double * C, int M, int N, int K);
// xbase / xtrial / step_out (all three or none): the kernel also writes step = x (NaN after a non-positive pivot) and xtrial = xbase + step
int launch_spd_solve(pnol_ctx * ctx, const double * A, const double * rhs, int n, double * x, int * info_dev,
                     const double * xbase = nullptr, double * xtrial = nullptr, double * step_out = nullptr);
int launch_lu_inverse(pnol_ctx * ctx, const double * A, int n, double * Ainv, int * info_dev);
int launch_matvec_neg(pnol_ctx * ctx, const double * D, const double * g, int n, double * p);
int launch_hinv_rank2(pnol_ctx * ctx, double * D, const double * g, const double * s, int n);
int launch_hinv_literal(pnol_ctx * ctx, double * D, const double * g, const double * s, int n);

int comm_allreduce_dev(pnol_ctx * ctx, double * dev_buf, size_t count);
int comm_allgather_dev(pnol_ctx * ctx, const double * send, double * recv, size_t count_per_rank);
int comm_broadcast_dev(pnol_ctx * ctx, double * buf, size_t count, int root);

// peer.cu: the sharded LM step's exchange over NVLink peer memory (fused all-reduce + damping); collective set-up, NCCL fallback
bool peer_ensure(pnol_ctx * ctx, size_t count);
double * peer_partial_slot(pnol_ctx * ctx);
int launch_peer_reduce_damp(pnol_ctx * ctx, int n, double lambda, const double * lambda_dev, double * JTJ, double * A, double * rhs);
int launch_peer_scalar_sum(pnol_ctx * ctx, double * ss);
int peer_check(pnol_ctx * ctx);
void peer_destroy(pnol_ctx * ctx);

} // namespace pnol
