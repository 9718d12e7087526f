// capi.cu -- extern "C" glue of include/pnol_b200.h: context, memory, functors, and the evaluation / LM / BFGS
// entry points (the GA entry points live in ga.cu, the communicator in comm.cu).
#include "common.cuh"
#include "peer.cuh"

#include <mutex>
#include <vector>
#include <thread>
#include "exact_div.cuh"

#include <math.h>

namespace pnol {

void comm_destroy(pnol_ctx * ctx);

int ws_reserve(pnol_ctx * ctx, int slot, size_t bytes)
{
	if (bytes <= ctx->ws_bytes[slot]) return PNOL_OK;
	if (ctx->ws[slot]) {
		PNOL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
		PNOL_CUDA(ctx, cudaFree(ctx->ws[slot]));
		ctx->ws[slot] = nullptr; ctx->ws_bytes[slot] = 0;
	}
	size_t cap = bytes + bytes / 4 + 256;
	PNOL_CUDA(ctx, cudaMalloc(&ctx->ws[slot], cap));
	ctx->ws_bytes[slot] = cap;
	return PNOL_OK;
}

int pinned_reserve(pnol_ctx * ctx, size_t doubles)
{
	if (doubles <= ctx->pinned_doubles) return PNOL_OK;
	if (ctx->pinned) { cudaStreamSynchronize(ctx->stream); cudaFreeHost(ctx->pinned); ctx->pinned = nullptr; }
	size_t cap = doubles < 64 ? 64 : doubles * 2;
	PNOL_CUDA(ctx, cudaMallocHost((void **) &ctx->pinned, cap * sizeof(double)));
	ctx->pinned_doubles = cap;
	return PNOL_OK;
}

static void timers_collect(pnol_ctx * ctx)
{
	for (auto & kv : ctx->timers) {
		for (auto & ev : kv.second.pending) {
			cudaEventSynchronize(ev.second);
			float ms = 0;
			if (cudaEventElapsedTime(&ms, ev.first, ev.second) == cudaSuccess) { kv.second.total_ms += ms; kv.second.count++; }
			cudaEventDestroy(ev.first); cudaEventDestroy(ev.second);
		}
		kv.second.pending.clear();
	}
}

} // namespace pnol

using namespace pnol;

// ---------------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------------
extern "C" const char * pnol_version(void) { return "pnol_b200 0.1 (sm_100a)"; }

extern "C" int pnol_ctx_create(pnol_ctx ** out, int device)
{
	if (!out) return PNOL_ERR_INVALID;
	*out = nullptr;
	int ndev = 0;
	if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { cudaGetLastError(); return PNOL_ERR_CUDA; }
	if (device < 0 || device >= ndev) return PNOL_ERR_INVALID;
	pnol_ctx * ctx = new pnol_ctx();
	ctx->device = device;
	if (cudaSetDevice(device) != cudaSuccess) { delete ctx; return PNOL_ERR_CUDA; }
	cudaDeviceProp prop;
	if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete ctx; return PNOL_ERR_CUDA; }
	ctx->sm_count = prop.multiProcessorCount;
	ctx->smem_optin = prop.sharedMemPerBlockOptin;
	if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return PNOL_ERR_CUDA; }
	// staging buffers come from the stream-ordered pool: keep freed blocks cached across synchronisations
	cudaMemPool_t pool;
	if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
		uint64_t keep = UINT64_MAX;
		cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
	}
	*out = ctx;
	return PNOL_OK;
}

static int bg_copy_join(pnol_ctx * ctx);

extern "C" void pnol_ctx_destroy(pnol_ctx * ctx)
{
	if (!ctx) return;
	cudaSetDevice(ctx->device);
	bg_copy_join(ctx);
	cudaStreamSynchronize(ctx->stream);
	timers_collect(ctx);
	comm_destroy(ctx);
	for (int s = 0; s < 5; s++) if (ctx->ws[s]) cudaFree(ctx->ws[s]);
	if (ctx->stage_pinned) cudaFreeHost(ctx->stage_pinned);
	for (int t = 0; t < 8; t++) if (ctx->stage_streams[t]) cudaStreamDestroy(ctx->stage_streams[t]);
	for (int e = 0; e < 16; e++) if (ctx->stage_events[e]) cudaEventDestroy(ctx->stage_events[e]);
	if (ctx->syrk_plan) cudaFree(ctx->syrk_plan);
	if (ctx->pinned) cudaFreeHost(ctx->pinned);
	cudaStreamSynchronize(ctx->stream);
	cudaMemPool_t pool;
	if (cudaDeviceGetDefaultMemPool(&pool, ctx->device) == cudaSuccess) cudaMemPoolTrimTo(pool, 0);
	cudaStreamDestroy(ctx->stream);
	delete ctx;
}

extern "C" const char * pnol_last_error(pnol_ctx * ctx)
{
	if (!ctx) return "null context";
	if (ctx->errbuf[0]) { ctx->err = ctx->errbuf; ctx->errbuf[0] = 0; }      // text of a launcher from include/pnol/device (newer than err)
	return ctx->err.c_str();
}
extern "C" int pnol_ctx_device(pnol_ctx * ctx) { return ctx ? ctx->device : -1; }
extern "C" void * pnol_ctx_stream(pnol_ctx * ctx) { return ctx ? (void *) ctx->stream : nullptr; }
extern "C" int pnol_ctx_sm_count(pnol_ctx * ctx) { return ctx ? ctx->sm_count : 0; }
extern "C" uint64_t pnol_ctx_launches(pnol_ctx * ctx) { return ctx ? ctx->launches : 0; }
extern "C" int pnol_ctx_sync(pnol_ctx * ctx)
{
	if (!ctx) return PNOL_ERR_INVALID;
	return finish(ctx);
}

extern "C" int pnol_malloc(pnol_ctx * ctx, void ** dev_ptr, size_t bytes)
{
	if (!ctx || !dev_ptr) return PNOL_ERR_INVALID;
	// stream-ordered pool with an unlimited release threshold (pnol_ctx_create): a freed block is reused by the next
	// request of that size without going back to the driver -- findMin allocates and frees its J / F work space per call
	PNOL_CUDA(ctx, cudaSetDevice(ctx->device));
	PNOL_CUDA(ctx, cudaMallocAsync(dev_ptr, bytes ? bytes : 1, ctx->stream));
	return PNOL_OK;
}
extern "C" int pnol_free(pnol_ctx * ctx, void * dev_ptr)
{
	if (!ctx) return PNOL_ERR_INVALID;
	if (!dev_ptr) return PNOL_OK;
	PNOL_CUDA(ctx, cudaFreeAsync(dev_ptr, ctx->stream));
	return PNOL_OK;
}
// ---------------------------------------------------------------------------------------------------
// Large copies between PAGEABLE host memory and the device. cudaMemcpy stages such a copy through the driver's pinned buffers with
// one host thread (~10 GB/s here), which made the host-vector API (LevMarq::findMin: data columns up, F0 / FOpt down, 128 MB per
// call at m = 4M) cost 0.9 ms per LM iteration. Here four threads each move every fourth 4 MB chunk through their own pair of
// pinned buffers and their own stream, so the host-side memcpy of one chunk overlaps the DMA of the others.
// ---------------------------------------------------------------------------------------------------
constexpr size_t kStageChunk = (size_t) 4 << 20;
constexpr int kStageThreads = 4;
// copies from 1 MB on take this path; below 8 chunks of 4 MB the chunk shrinks so that every thread still gets two chunks to overlap
// (a rank's data column at 8 GPUs is 4 MB: one chunk would be one thread's plain staged copy again)
constexpr size_t kStageMinBytes = (size_t) 1 << 20;

static bool is_pageable_host(const void * p)
{
	cudaPointerAttributes a;
	cudaError_t e = cudaPointerGetAttributes(&a, p);
	if (e != cudaSuccess) { cudaGetLastError(); return true; }
	return a.type == cudaMemoryTypeUnregistered;
}

static int stage_init(pnol_ctx * ctx)
{
	if (ctx->stage_pinned) return PNOL_OK;
	PNOL_CUDA(ctx, cudaHostAlloc(&ctx->stage_pinned, kStageChunk * 2 * kStageThreads, cudaHostAllocDefault));
	for (int t = 0; t < kStageThreads; t++) PNOL_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->stage_streams[t], cudaStreamNonBlocking));
	for (int e = 0; e < 2 * kStageThreads; e++) PNOL_CUDA(ctx, cudaEventCreateWithFlags(&ctx->stage_events[e], cudaEventDisableTiming));
	return PNOL_OK;
}

// dst / src: one of them pageable host memory, the other device memory; the context's stream is idle (the caller synchronised)
static int staged_copy(pnol_ctx * ctx, void * dst, const void * src, size_t bytes, bool h2d)
{
	PNOL_CHECK(stage_init(ctx));
	cudaError_t errs[kStageThreads];
	size_t chunk = (bytes + 2 * (size_t) kStageThreads - 1) / (2 * (size_t) kStageThreads);
	chunk = (chunk + 65535) & ~(size_t) 65535;
	if (chunk > kStageChunk) chunk = kStageChunk;
	auto worker = [&, chunk](int t) {
		cudaError_t e = cudaSetDevice(ctx->device);
		unsigned char * pin = (unsigned char *) ctx->stage_pinned + (size_t) t * 2 * kStageChunk;
		cudaStream_t st = ctx->stage_streams[t];
		cudaEvent_t * ev = &ctx->stage_events[2 * t];
		size_t prev_off = 0, prev_len = 0;
		for (size_t i = 0; e == cudaSuccess; i++) {
			const size_t off = ((size_t) t + i * kStageThreads) * chunk;
			const bool have = off < bytes;
			const size_t len = have ? (bytes - off < chunk ? bytes - off : chunk) : 0;
			const int b = (int) (i & 1);
			unsigned char * buf = pin + (size_t) b * kStageChunk;
			if (h2d) {
				if (!have) break;
				if (i >= 2) e = cudaEventSynchronize(ev[b]);      // the DMA out of this buffer two chunks ago
				memcpy(buf, (const unsigned char *) src + off, len);
				if (e == cudaSuccess) e = cudaMemcpyAsync((unsigned char *) dst + off, buf, len, cudaMemcpyHostToDevice, st);
				if (e == cudaSuccess) e = cudaEventRecord(ev[b], st);
			} else {
				if (have) {
					e = cudaMemcpyAsync(buf, (const unsigned char *) src + off, len, cudaMemcpyDeviceToHost, st);
					if (e == cudaSuccess) e = cudaEventRecord(ev[b], st);
				}
				if (i >= 1 && prev_len && e == cudaSuccess) {       // the previous chunk has landed in the other buffer
					e = cudaEventSynchronize(ev[b ^ 1]);
					memcpy((unsigned char *) dst + prev_off, pin + (size_t) (b ^ 1) * kStageChunk, prev_len);
				}
				prev_off = off; prev_len = len;
				if (!have) break;
			}
		}
		if (e == cudaSuccess) e = cudaStreamSynchronize(st);
		errs[t] = e;
	};
	std::thread th[kStageThreads];
	for (int t = 1; t < kStageThreads; t++) th[t - 1] = std::thread(worker, t);
	worker(0);
	for (int t = 1; t < kStageThreads; t++) th[t - 1].join();
	for (int t = 0; t < kStageThreads; t++)
		if (errs[t] != cudaSuccess) { PNOL_SET_ERR(ctx, "staged copy: %s", cudaGetErrorString(errs[t])); return PNOL_ERR_CUDA; }
	return PNOL_OK;
}

// ---- a device -> host copy that runs BESIDE the context's stream (pnol_copy_start / pnol_copy_wait): a worker thread drives the
// staged path above on the copy streams. The staging buffers have one user at a time: every other copy joins the worker first.
int copy_now(pnol_ctx * ctx, void * dst, const void * src, size_t bytes);
static int bg_copy_join(pnol_ctx * ctx)
{
	if (!ctx->bg_copy) return PNOL_OK;
	ctx->bg_copy->join();
	delete ctx->bg_copy;
	ctx->bg_copy = nullptr;
	const int st = ctx->bg_copy_status;
	ctx->bg_copy_status = PNOL_OK;
	return st;
}

extern "C" int pnol_copy_start(pnol_ctx * ctx, void * host_dst, const void * dev_src, size_t bytes)
{
	if (!ctx) return PNOL_ERR_INVALID;
	PNOL_CHECK(bg_copy_join(ctx));
	if (!bytes) return PNOL_OK;
	PNOL_REQUIRE(ctx, host_dst && dev_src && is_device_ptr(dev_src) && !is_device_ptr(host_dst), "copy_start: device source and host destination expected");
	if (bytes < kStageMinBytes || !is_pageable_host(host_dst)) return copy_now(ctx, host_dst, dev_src, bytes);
	PNOL_CHECK(stage_init(ctx));
	ctx->bg_copy_status = PNOL_OK;
	ctx->bg_copy = new std::thread([ctx, host_dst, dev_src, bytes] {
		cudaSetDevice(ctx->device);
		ctx->bg_copy_status = staged_copy(ctx, host_dst, dev_src, bytes, false);
	});
	return PNOL_OK;
}
extern "C" int pnol_copy_wait(pnol_ctx * ctx)
{
	if (!ctx) return PNOL_ERR_INVALID;
	return bg_copy_join(ctx);
}

// host <-> device copy that is complete on return (any pointer kinds)
int copy_now(pnol_ctx * ctx, void * dst, const void * src, size_t bytes)
{
	if (!bytes) return PNOL_OK;
	PNOL_CHECK(bg_copy_join(ctx));
	if (bytes >= kStageMinBytes) {
		const bool dst_dev = is_device_ptr(dst), src_dev = is_device_ptr(src);
		if (dst_dev != src_dev && is_pageable_host(dst_dev ? src : dst)) {
			PNOL_CHECK(finish(ctx));                             // whatever produced / still uses the device side
			return staged_copy(ctx, dst, src, bytes, dst_dev);
		}
	}
	PNOL_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, ctx->stream));
	return finish(ctx);
}

extern "C" int pnol_memcpy(pnol_ctx * ctx, void * dst, const void * src, size_t bytes)
{
	if (!ctx) return PNOL_ERR_INVALID;
	return copy_now(ctx, dst, src, bytes);
}
extern "C" int pnol_memset(pnol_ctx * ctx, void * dev_ptr, int value, size_t bytes)
{
	if (!ctx) return PNOL_ERR_INVALID;
	PNOL_CUDA(ctx, cudaMemsetAsync(dev_ptr, value, bytes, ctx->stream));
	return PNOL_OK;
}
extern "C" int pnol_host_alloc(void ** host_ptr, size_t bytes)
{
	if (!host_ptr) return PNOL_ERR_INVALID;
	return cudaMallocHost(host_ptr, bytes ? bytes : 1) == cudaSuccess ? PNOL_OK : PNOL_ERR_CUDA;
}
extern "C" int pnol_host_free(void * host_ptr)
{
	return cudaFreeHost(host_ptr) == cudaSuccess ? PNOL_OK : PNOL_ERR_CUDA;
}

extern "C" int pnol_timer_enable(pnol_ctx * ctx, int on)
{
	if (!ctx) return PNOL_ERR_INVALID;
	ctx->timers_on = on == 2 ? 2 : (on != 0 ? 1 : 0);
	return PNOL_OK;
}
extern "C" int pnol_timer_get(pnol_ctx * ctx, const char * name, double * total_ms, long long * count)
{
	if (!ctx || !name) return PNOL_ERR_INVALID;
	PNOL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	timers_collect(ctx);
	auto it = ctx->timers.find(name);
	if (total_ms) *total_ms = it == ctx->timers.end() ? 0.0 : it->second.total_ms;
	if (count) *count = it == ctx->timers.end() ? 0 : it->second.count;
	return PNOL_OK;
}
extern "C" int pnol_timer_reset(pnol_ctx * ctx)
{
	if (!ctx) return PNOL_ERR_INVALID;
	cudaStreamSynchronize(ctx->stream);
	timers_collect(ctx);
	ctx->timers.clear();
	return PNOL_OK;
}

// ---------------------------------------------------------------------------------------------------
// functors
// ---------------------------------------------------------------------------------------------------
// ---- open functor table (include/pnol_b200.h: pnol_register_functor) ----
namespace {
// the records of the registered user kinds: the library's own copy of each table and the side launchers attached to it
struct FunctorRegistry {
	std::mutex mu;
	std::map<int, KindTable> kinds;
};
FunctorRegistry & registry()
{
	static FunctorRegistry * r = new FunctorRegistry();      // never destroyed: registrations come from static initialisers of other modules
	return *r;
}

// pnol_register_functor_*: attaches fn as member `slot` of the record registered for a user kind of the family (residual or scalar)
template <class L> int attach(int kind, bool residual, L KindTable::*slot, L fn)
{
	if (!fn || !pnol::is_user_kind(kind) || pnol::is_residual_kind(kind) != residual) return PNOL_ERR_INVALID;
	FunctorRegistry & r = registry();
	std::lock_guard<std::mutex> lock(r.mu);
	auto it = r.kinds.find(kind);
	if (it == r.kinds.end()) return PNOL_ERR_INVALID;
	it->second.*slot = fn;
	return PNOL_OK;
}
} // namespace

bool pnol::kind_table(int kind, KindTable * out)
{
	if (const KindTable * b = builtin_kind_table(kind)) { *out = *b; return true; }
	if (!is_user_kind(kind)) return false;
	FunctorRegistry & r = registry();
	std::lock_guard<std::mutex> lock(r.mu);
	auto it = r.kinds.find(kind);
	if (it == r.kinds.end()) return false;
	*out = it->second;
	return true;
}

extern "C" int pnol_register_functor(int kind, const pnol_functor_vtable * vt)
{
	if (!vt || !pnol::is_user_kind(kind)) return PNOL_ERR_INVALID;
	// abi_version leads every version of the table; a version-1 table ends before `jacobian`, so only that prefix may be read
	const int abi = vt->abi_version;
	if (abi != 1 && abi != PNOL_FUNCTOR_ABI) return PNOL_ERR_INVALID;
	KindTable k = {};
	memcpy(&k.vt, vt, abi == 1 ? offsetof(pnol_functor_vtable, jacobian) : sizeof(pnol_functor_vtable));
	const pnol_functor_vtable * c = &k.vt;
	if (c->n_columns < 0 || c->n_columns > PNOL_MAX_COLUMNS) return PNOL_ERR_INVALID;
	const bool residual = pnol::is_residual_kind(kind);
	if (residual ? !(c->residual && c->fd_jacobian) : !(c->eval_batch && c->fd_points && c->fd_hessian && c->alpha_pool)) return PNOL_ERR_INVALID;
	if (!residual && c->jacobian) return PNOL_ERR_INVALID;      // an analytic Jacobian belongs to a residual model
	FunctorRegistry & r = registry();
	std::lock_guard<std::mutex> lock(r.mu);
	r.kinds[kind] = k;      // a new record: launchers attached to the replaced table do not carry over
	return PNOL_OK;
}

extern "C" int pnol_register_functor_gradient(int kind, pnol_gradient_launcher fn) { return attach(kind, false, &KindTable::gradient, fn); }
extern "C" int pnol_register_functor_hessian(int kind, pnol_hessian_launcher fn) { return attach(kind, false, &KindTable::hessian, fn); }
extern "C" int pnol_register_functor_slope(int kind, pnol_slope_launcher fn) { return attach(kind, false, &KindTable::slope, fn); }
extern "C" int pnol_register_functor_lm_batch(int kind, pnol_lm_batch_launcher fn) { return attach(kind, true, &KindTable::lm_batch, fn); }
extern "C" int pnol_register_functor_bfgs_batch(int kind, pnol_bfgs_batch_launcher fn) { return attach(kind, false, &KindTable::bfgs_batch, fn); }
extern "C" int pnol_register_functor_simplex_batch(int kind, pnol_simplex_batch_launcher fn)
{
	return attach(kind, false, &KindTable::simplex_batch, fn);
}

extern "C" int pnol_functor_registered(int kind)
{
	KindTable k;
	return pnol::kind_table(kind, &k);
}
extern "C" int pnol_functor_has_gradient(int kind)
{
	KindTable k;
	return pnol::kind_table(kind, &k) && k.gradient;
}
extern "C" int pnol_functor_has_hessian(int kind)
{
	KindTable k;
	return pnol::kind_table(kind, &k) && k.hessian;
}
extern "C" int pnol_functor_has_slope(int kind)
{
	KindTable k;
	return pnol::kind_table(kind, &k) && k.slope;
}
extern "C" int pnol_functor_has_lm_batch(int kind)
{
	KindTable k;
	return pnol::kind_table(kind, &k) && k.lm_batch;
}
extern "C" int pnol_functor_has_bfgs_batch(int kind)
{
	KindTable k;
	return pnol::kind_table(kind, &k) && k.bfgs_batch;
}
extern "C" int pnol_functor_has_simplex_batch(int kind)
{
	KindTable k;
	return pnol::kind_table(kind, &k) && k.simplex_batch;
}

extern "C" int pnol_functor_create(pnol_ctx * ctx, const pnol_functor_desc * desc, pnol_functor ** out)
{
	if (!ctx || !desc || !out) return PNOL_ERR_INVALID;
	*out = nullptr;
	PNOL_REQUIRE(ctx, desc->n_columns >= 0 && desc->n_columns <= PNOL_MAX_COLUMNS, "functor: bad column count %d", desc->n_columns);
	KindTable kt;
	if (!kind_table(desc->kind, &kt)) {
		PNOL_SET_ERR(ctx, "unknown functor kind %d (user kinds must be registered first: pnol_register_functor)", desc->kind);
		return PNOL_ERR_NO_FUNCTOR;
	}
	const int need_cols = kt.vt.n_columns;
	PNOL_REQUIRE(ctx, desc->n_columns == need_cols, "functor kind %d needs %d data columns, got %d", desc->kind, need_cols, desc->n_columns);
	PNOL_REQUIRE(ctx, need_cols == 0 || desc->m >= 0, "functor: bad row count");
	pnol_functor * f = new pnol_functor();
	f->ctx = ctx; f->kind = desc->kind; f->n_columns = desc->n_columns;
	memset(&f->params, 0, sizeof f->params);
	memset(f->owned, 0, sizeof f->owned);
	memcpy(f->params.scalars, desc->scalars, sizeof desc->scalars);
	memcpy(f->params.ints, desc->ints, sizeof desc->ints);
	f->params.m = need_cols ? desc->m : 0;
	for (int c = 0; c < desc->n_columns; c++) {
		if (is_device_ptr(desc->columns[c])) { f->params.col[c] = desc->columns[c]; continue; }
		void * d = nullptr;
		size_t bytes = (size_t) (desc->m > 0 ? desc->m : 1) * sizeof(double);
		cudaError_t e = cudaMallocAsync(&d, bytes, ctx->stream);
		if (e == cudaSuccess && desc->m > 0 && copy_now(ctx, d, desc->columns[c], (size_t) desc->m * sizeof(double)) != PNOL_OK) e = cudaErrorUnknown;
		if (e != cudaSuccess) {
			PNOL_SET_ERR(ctx, "functor column upload: %s", cudaGetErrorString(e));
			pnol_functor_destroy(f);
			return PNOL_ERR_CUDA;
		}
		f->owned[c] = d;
		f->params.col[c] = (const double *) d;
	}
	int st = finish(ctx);
	if (st != PNOL_OK) { pnol_functor_destroy(f); return st; }
	*out = f;
	return PNOL_OK;
}

extern "C" void pnol_functor_destroy(pnol_functor * f)
{
	if (!f) return;
	for (int c = 0; c < PNOL_MAX_COLUMNS; c++) if (f->owned[c]) cudaFreeAsync(f->owned[c], f->ctx->stream);
	delete f;
}

extern "C" int pnol_functor_is_residual(const pnol_functor * f) { return f && is_residual_kind(f->kind); }
extern "C" long long pnol_functor_rows(const pnol_functor * f) { return f && is_residual_kind(f->kind) ? f->params.m : 0; }

// ---------------------------------------------------------------------------------------------------
// scalar-objective entry points
// ---------------------------------------------------------------------------------------------------
extern "C" int pnol_eval_batch(pnol_ctx * ctx, const pnol_functor * f, const double * pts, long long B, int n, long long ld,
                               const unsigned char * indicator, double * f_out)
{
	if (!ctx || !f) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, pts && f_out && B >= 0 && n >= 1 && ld >= n, "eval_batch: bad arguments");
	if (B == 0) return PNOL_OK;
	DevIn<double> dp; DevIn<unsigned char> di; DevOut<double> df;
	PNOL_CHECK(dp.init(ctx, pts, (size_t) ((B - 1) * ld + n)));
	PNOL_CHECK(di.init(ctx, indicator, (size_t) B));
	PNOL_CHECK(df.init(ctx, f_out, (size_t) B, indicator != nullptr));
	PNOL_CHECK(launch_eval_batch(ctx, f, dp.get(), B, n, ld, di.get(), df.get()));
	PNOL_CHECK(df.commit());
	return finish(ctx);
}

// shared tail of the gradient entry points: coordinates [i0, i1) of this rank, gathered across ranks. Forward difference (dx_dev):
// stencil points (+ base), then the quotient. Analytic (dx_dev == nullptr): the functor's partials, written straight to the output
// on one rank, through the gather buffer on several; the base value only when f0_out asks for it.
static int gradient_common(pnol_ctx * ctx, const pnol_functor * f, const double * xfull_dev, int nfull, const int * pos_dev,
                           const double * dx_dev, int nvar, double * g_out, double * f0_out)
{
	const bool analytic = dx_dev == nullptr;
	// scratch: fdx[nvar_padded] (analytic: the gathered partials) | f0 | g
	const int R = ctx->nranks;
	const int per = (nvar + R - 1) / R;            // coordinates per rank (contiguous column blocks)
	const int padded = per * R;
	PNOL_CHECK(ws_reserve(ctx, 2, ((size_t) 2 * padded + 8) * sizeof(double)));
	double * fdx = (double *) ctx->ws[2];
	double * f0 = fdx + padded;
	double * gtmp = f0 + 1;
	int i0 = ctx->rank * per, i1 = i0 + per;
	if (i0 > nvar) i0 = nvar;
	if (i1 > nvar) i1 = nvar;
	DevOut<double> dg;
	if (analytic) {
		PNOL_CHECK(dg.init(ctx, g_out, (size_t) nvar));
		double * g = dg.get() ? dg.get() : gtmp;
		PNOL_CHECK(launch_gradient(ctx, f, xfull_dev, nfull, pos_dev, i0, i1, R > 1 ? fdx : g, f0_out ? f0 : nullptr));
		if (R > 1) {
			PNOL_CHECK(comm_allgather_dev(ctx, fdx + (size_t) ctx->rank * per, fdx, (size_t) per));
			PNOL_CUDA(ctx, cudaMemcpyAsync(g, fdx, (size_t) nvar * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
		}
	} else {
		// every rank also evaluates the base point (the reference gives it to one rank and sums; SURVEY 3.4)
		PNOL_CHECK(launch_fd_points(ctx, f, xfull_dev, nfull, pos_dev, dx_dev, i0, i1, fdx, f0));
		if (R > 1) PNOL_CHECK(comm_allgather_dev(ctx, fdx + (size_t) ctx->rank * per, fdx, (size_t) per));
		PNOL_CHECK(dg.init(ctx, g_out, (size_t) nvar));
		PNOL_CHECK(launch_fd_quotient(ctx, fdx, f0, dx_dev, nvar, dg.get() ? dg.get() : gtmp));
	}
	PNOL_CHECK(dg.commit());
	if (f0_out) PNOL_CUDA(ctx, cudaMemcpyAsync(f0_out, f0, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
	return finish(ctx);
}

extern "C" int pnol_fd_gradient(pnol_ctx * ctx, const pnol_functor * f, const double * x, const double * dx, int n,
                                double * g_out, double * f0_out)
{
	if (!ctx || !f) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, x && dx && g_out && n >= 1, "fd_gradient: bad arguments");
	DevIn<double> dxp, ddx;
	PNOL_CHECK(dxp.init(ctx, x, n));
	PNOL_CHECK(ddx.init(ctx, dx, n));
	return gradient_common(ctx, f, dxp.get(), n, nullptr, ddx.get(), n, g_out, f0_out);
}

extern "C" int pnol_gradient(pnol_ctx * ctx, const pnol_functor * f, const double * x, int n, double * g_out, double * f0_out)
{
	if (!ctx || !f) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, x && g_out && n >= 1, "gradient: bad arguments");
	DevIn<double> dxp;
	PNOL_CHECK(dxp.init(ctx, x, n));
	return gradient_common(ctx, f, dxp.get(), n, nullptr, nullptr, n, g_out, f0_out);
}

static int recur_assemble(pnol_ctx * ctx, const double * xr, int nr, const double * const_x, const unsigned char * const_ind,
                          int nfull, DevIn<double> & dxr, DevIn<double> & dcx, DevIn<unsigned char> & dci, double ** xfull,
                          int ** pos)
{
	PNOL_CHECK(dxr.init(ctx, xr, nr));
	PNOL_CHECK(dcx.init(ctx, const_x, nfull));
	PNOL_CHECK(dci.init(ctx, const_ind, nfull));
	PNOL_CHECK(ws_reserve(ctx, 1, (size_t) nfull * (sizeof(double) + sizeof(int)) + 64));
	*xfull = (double *) ctx->ws[1];
	*pos = (int *) (*xfull + nfull);
	int * found = *pos + nfull;
	// -1 = "no slot": a caller may pass more reduced entries than const_ind leaves free (BFGSBnd_MPI keeps iterating on the full
	// vector after every variable has been frozen, Source/BFGS_with_bnd_linsearch_MPI.cpp:808-810)
	PNOL_CUDA(ctx, cudaMemsetAsync(*pos, 0xFF, (size_t) nfull * sizeof(int), ctx->stream));
	PNOL_CHECK(launch_assemble_recur(ctx, dxr.get(), nr, dcx.get(), dci.get(), nfull, *xfull, *pos, found));
	return PNOL_OK;
}

extern "C" int pnol_eval_recur(pnol_ctx * ctx, const pnol_functor * f, const double * xr, int nr, const double * const_x,
                               const unsigned char * const_ind, int nfull, double * f_out)
{
	if (!ctx || !f) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, const_x && const_ind && f_out && nfull >= 1 && nr >= 0 && nr <= nfull, "eval_recur: bad arguments");
	DevIn<double> dxr, dcx; DevIn<unsigned char> dci;
	double * xfull; int * pos;
	PNOL_CHECK(recur_assemble(ctx, xr, nr, const_x, const_ind, nfull, dxr, dcx, dci, &xfull, &pos));
	PNOL_CHECK(ws_reserve(ctx, 2, 64));
	double * f0 = (double *) ctx->ws[2];
	PNOL_CHECK(launch_fd_points(ctx, f, xfull, nfull, nullptr, nullptr, 0, 0, nullptr, f0));
	PNOL_CUDA(ctx, cudaMemcpyAsync(f_out, f0, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
	return finish(ctx);
}

extern "C" int pnol_fd_gradient_recur(pnol_ctx * ctx, const pnol_functor * f, const double * xr, const double * dxr, int nr,
                                      const double * const_x, const unsigned char * const_ind, int nfull, double * g_out,
                                      double * f0_out)
{
	if (!ctx || !f) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, xr && dxr && const_x && const_ind && g_out && nfull >= 1 && nr >= 1 && nr <= nfull, "fd_gradient_recur: bad arguments");
	DevIn<double> dx_r, dcx, ddx; DevIn<unsigned char> dci;
	double * xfull; int * pos;
	PNOL_CHECK(recur_assemble(ctx, xr, nr, const_x, const_ind, nfull, dx_r, dcx, dci, &xfull, &pos));
	PNOL_CHECK(ddx.init(ctx, dxr, nr));
	return gradient_common(ctx, f, xfull, nfull, pos, ddx.get(), nr, g_out, f0_out);
}

extern "C" int pnol_gradient_recur(pnol_ctx * ctx, const pnol_functor * f, const double * xr, int nr, const double * const_x,
                                   const unsigned char * const_ind, int nfull, double * g_out, double * f0_out)
{
	if (!ctx || !f) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, xr && const_x && const_ind && g_out && nfull >= 1 && nr >= 1 && nr <= nfull, "gradient_recur: bad arguments");
	DevIn<double> dx_r, dcx; DevIn<unsigned char> dci;
	double * xfull; int * pos;
	PNOL_CHECK(recur_assemble(ctx, xr, nr, const_x, const_ind, nfull, dx_r, dcx, dci, &xfull, &pos));
	return gradient_common(ctx, f, xfull, nfull, pos, nullptr, nr, g_out, f0_out);
}

extern "C" int pnol_fd_hessian(pnol_ctx * ctx, const pnol_functor * f, const double * x, const double * dx, int n, double * B_out)
{
	if (!ctx || !f) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, x && dx && B_out && n >= 1, "fd_hessian: bad arguments");
	DevIn<double> dxp, ddx; DevOut<double> dB;
	PNOL_CHECK(dxp.init(ctx, x, n));
	PNOL_CHECK(ddx.init(ctx, dx, n));
	PNOL_CHECK(dB.init(ctx, B_out, (size_t) n * n));
	PNOL_CHECK(ws_reserve(ctx, 2, ((size_t) n + 8) * sizeof(double)));
	double * fdx = (double *) ctx->ws[2];
	double * f0 = fdx + n;
	PNOL_CHECK(launch_fd_points(ctx, f, dxp.get(), n, nullptr, ddx.get(), 0, n, fdx, f0));
	PNOL_CHECK(launch_fd_hessian(ctx, f, dxp.get(), ddx.get(), n, fdx, f0, dB.get()));
	PNOL_CHECK(dB.commit());
	return finish(ctx);
}

extern "C" int pnol_hessian(pnol_ctx * ctx, const pnol_functor * f, const double * x, int n, double * H_out)
{
	if (!ctx || !f) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, x && H_out && n >= 1, "hessian: bad arguments");
	DevIn<double> dxp; DevOut<double> dH;
	PNOL_CHECK(dxp.init(ctx, x, n));
	PNOL_CHECK(dH.init(ctx, H_out, (size_t) n * n));
	PNOL_CHECK(launch_hessian(ctx, f, dxp.get(), n, dH.get()));
	PNOL_CHECK(dH.commit());
	return finish(ctx);
}

// The points of a pool in the full space. With an active set (const_ind != NULL) x and p are expanded as objEvalRecur scatters them
// (p = 0 on constants; the kernels never add alpha*p there) and pos[i] is the slot of reduced entry i; without one they are x and p
// themselves and pos is NULL.
struct PoolPoints {
	DevIn<double> dx, dp, dcx; DevIn<unsigned char> dci;
	const double * xfull = nullptr; const double * pfull = nullptr; const unsigned char * is_const = nullptr; const int * pos = nullptr;
};
static int pool_points(pnol_ctx * ctx, const double * x, const double * p, int n, const double * const_x, const unsigned char * const_ind,
                       int nfull, PoolPoints & pp)
{
	if (!const_ind) {
		PNOL_CHECK(pp.dx.init(ctx, x, n));
		PNOL_CHECK(pp.dp.init(ctx, p, n));
		pp.xfull = pp.dx.get(); pp.pfull = pp.dp.get();
		return PNOL_OK;
	}
	PNOL_REQUIRE(ctx, const_x != nullptr, "alpha_pool: const_x missing");
	double * xf; int * pos;
	PNOL_CHECK(recur_assemble(ctx, x, n, const_x, const_ind, nfull, pp.dx, pp.dcx, pp.dci, &xf, &pos));
	// second assembly for p (constants -> 0): reuse the kernel with const_x := zeros
	PNOL_CHECK(ws_reserve(ctx, 0, (size_t) 2 * nfull * sizeof(double) + 64));
	double * zeros = (double *) ctx->ws[0];
	double * pf = zeros + nfull;
	PNOL_CUDA(ctx, cudaMemsetAsync(zeros, 0, (size_t) nfull * sizeof(double), ctx->stream));
	PNOL_CHECK(pp.dp.init(ctx, p, n));
	PNOL_CHECK(launch_assemble_recur(ctx, pp.dp.get(), n, zeros, pp.dci.get(), nfull, pf, nullptr, nullptr));
	pp.xfull = xf; pp.pfull = pf; pp.is_const = pp.dci.get(); pp.pos = pos;
	return PNOL_OK;
}

// the pool's evaluation: the forward-difference slope (dalpha) or, analytic, the functor's own slope (dalpha unused)
static int alpha_pool_common(pnol_ctx * ctx, const pnol_functor * f, const double * x, const double * p, int n, const double * alpha,
                             int npool, double dalpha, bool analytic, const unsigned char * eval_ind, const double * const_x,
                             const unsigned char * const_ind, int nfull, double * phi, double * dphi, int * bad_out)
{
	const bool recur = const_ind != nullptr;
	if (!recur) nfull = n;
	PNOL_REQUIRE(ctx, nfull >= n, "alpha_pool: nfull < n");
	DevIn<double> da_; DevIn<unsigned char> de_;
	DevOut<double> dphi_o, dph_o;
	PNOL_CHECK(da_.init(ctx, alpha, npool));
	PNOL_CHECK(de_.init(ctx, eval_ind, npool));
	PNOL_CHECK(dph_o.init(ctx, phi, npool, eval_ind != nullptr));
	PNOL_CHECK(dphi_o.init(ctx, dphi, npool, eval_ind != nullptr));
	PNOL_CHECK(ws_reserve(ctx, 2, 64));
	int * bad_dev = (int *) ctx->ws[2];
	PNOL_CUDA(ctx, cudaMemsetAsync(bad_dev, 0, sizeof(int), ctx->stream));
	PoolPoints pp;
	PNOL_CHECK(pool_points(ctx, x, p, n, const_x, const_ind, nfull, pp));
	if (analytic)
		PNOL_CHECK(launch_alpha_slope(ctx, f, pp.xfull, pp.pfull, pp.is_const, nfull, pp.pos, pp.dp.get(), n, da_.get(), npool, de_.get(),
		                              dph_o.get(), dphi_o.get(), bad_dev));
	else
		PNOL_CHECK(launch_alpha_pool(ctx, f, pp.xfull, pp.pfull, pp.is_const, nfull, da_.get(), npool, dalpha, de_.get(), dph_o.get(),
		                             dphi_o.get(), bad_dev));
	PNOL_CHECK(dph_o.commit());
	PNOL_CHECK(dphi_o.commit());
	int bad = 0;
	PNOL_CUDA(ctx, cudaMemcpyAsync(&bad, bad_dev, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
	PNOL_CHECK(finish(ctx));
	if (bad_out) *bad_out = bad;
	return PNOL_OK;
}

extern "C" int pnol_alpha_pool(pnol_ctx * ctx, const pnol_functor * f, const double * x, const double * p, int n,
                               const double * alpha, int npool, double dalpha, const unsigned char * eval_ind,
                               const double * const_x, const unsigned char * const_ind, int nfull,
                               double * phi, double * dphi, int * bad_out)
{
	if (!ctx || !f) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, x && p && alpha && phi && n >= 1 && npool >= 1, "alpha_pool: bad arguments");
	return alpha_pool_common(ctx, f, x, p, n, alpha, npool, dalpha, false, eval_ind, const_x, const_ind, nfull, phi, dphi, bad_out);
}

extern "C" int pnol_alpha_pool_analytic(pnol_ctx * ctx, const pnol_functor * f, const double * x, const double * p, int n,
                                        const double * alpha, int npool, const unsigned char * eval_ind,
                                        const double * const_x, const unsigned char * const_ind, int nfull,
                                        double * phi, double * dphi, int * bad_out)
{
	if (!ctx || !f) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, x && p && alpha && phi && dphi && n >= 1 && npool >= 1, "alpha_pool_analytic: bad arguments");
	return alpha_pool_common(ctx, f, x, p, n, alpha, npool, 0.0, true, eval_ind, const_x, const_ind, nfull, phi, dphi, bad_out);
}

// ---------------------------------------------------------------------------------------------------
// residual-model entry points
// ---------------------------------------------------------------------------------------------------
extern "C" int pnol_residual_eval(pnol_ctx * ctx, const pnol_functor * f, const double * x, int n, double * F, double * sumsq_out)
{
	if (!ctx || !f) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, x && F && n >= 1, "residual_eval: bad arguments");
	const long long m = f->params.m;
	DevIn<double> dx_; DevOut<double> dF;
	PNOL_CHECK(dx_.init(ctx, x, n));
	PNOL_CHECK(dF.init(ctx, F, (size_t) m));
	double * ss = nullptr;
	if (sumsq_out) { PNOL_CHECK(ws_reserve(ctx, 3, 64)); ss = (double *) ctx->ws[3]; }
	PNOL_CHECK(launch_residual(ctx, f, dx_.get(), n, dF.get(), ss));
	if (ss && ctx->nranks > 1) PNOL_CHECK(comm_allreduce_dev(ctx, ss, 1));
	PNOL_CHECK(dF.commit());
	if (ss) PNOL_CUDA(ctx, cudaMemcpyAsync(sumsq_out, ss, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
	return finish(ctx);
}

extern "C" int pnol_fd_jacobian(pnol_ctx * ctx, const pnol_functor * f, const double * x, const double * dx, int n,
                                double * J, double * F, int mode)
{
	if (!ctx || !f) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, x && (dx || mode == PNOL_JAC_ANALYTIC) && J && n >= 1, "fd_jacobian: bad arguments");
	const long long m = f->params.m;
	DevIn<double> dx_, ddx; DevOut<double> dJ, dF;
	PNOL_CHECK(dx_.init(ctx, x, n));
	PNOL_CHECK(ddx.init(ctx, dx, n));
	PNOL_CHECK(dJ.init(ctx, J, (size_t) m * n));
	PNOL_CHECK(dF.init(ctx, F, (size_t) m));
	PNOL_CHECK(launch_fd_jacobian(ctx, f, dx_.get(), ddx.get(), n, dJ.get(), dF.get(), mode));
	PNOL_CHECK(dJ.commit());
	PNOL_CHECK(dF.commit());
	if (dJ.staged() || dF.staged()) return finish(ctx);
	return PNOL_OK;
}

extern "C" int pnol_lm_normal_eq(pnol_ctx * ctx, const double * J, const double * F, long long m, int n, double lambda,
                                 double * JTJ, double * A, double * rhs)
{
	if (!ctx) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, J && m >= 0 && n >= 1, "lm_normal_eq: bad arguments");
	DevIn<double> dJ, dF; DevOut<double> oJTJ, oA, orhs;
	PNOL_CHECK(dJ.init(ctx, J, (size_t) m * n));
	PNOL_CHECK(dF.init(ctx, F, (size_t) m));
	PNOL_CHECK(oJTJ.init(ctx, JTJ, (size_t) n * n));
	PNOL_CHECK(oA.init(ctx, A, (size_t) n * n));
	PNOL_CHECK(orhs.init(ctx, rhs, (size_t) n));
	size_t packed_count = (size_t) n * n + n;
	PNOL_CHECK(ws_reserve(ctx, 1, packed_count * sizeof(double)));
	double * packed = (double *) ctx->ws[1];
	PNOL_CHECK(launch_syrk(ctx, dJ.get(), dF.get(), m, n, packed));
	if (ctx->nranks > 1) PNOL_CHECK(comm_allreduce_dev(ctx, packed, packed_count));
	PNOL_CHECK(launch_lm_damp(ctx, packed, n, lambda, oJTJ.get(), oA.get(), orhs.get()));
	PNOL_CHECK(oJTJ.commit());
	PNOL_CHECK(oA.commit());
	PNOL_CHECK(orhs.commit());
	if (oJTJ.staged() || oA.staged() || orhs.staged()) return finish(ctx);
	return PNOL_OK;
}

__global__ void redamp_kernel(const double * __restrict__ JTJ, int n, double lambda, double * __restrict__ A)
{
	long long idx = (long long) blockIdx.x * blockDim.x + threadIdx.x;
	if (idx >= (long long) n * n) return;
	int i = (int) (idx / n), j = (int) (idx - (long long) i * n);
	double v = JTJ[idx];
	A[idx] = (i == j) ? (1 + lambda) * v : v;
}

extern "C" int pnol_lm_damp(pnol_ctx * ctx, const double * JTJ, int n, double lambda, double * A)
{
	if (!ctx) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, JTJ && A && n >= 1, "lm_damp: bad arguments");
	DevIn<double> d; DevOut<double> o;
	PNOL_CHECK(d.init(ctx, JTJ, (size_t) n * n));
	PNOL_CHECK(o.init(ctx, A, (size_t) n * n));
	long long total = (long long) n * n;
	PNOL_LAUNCH(ctx, redamp_kernel, (unsigned) ((total + 255) / 256), 256, 0, d.get(), n, lambda, o.get());
	PNOL_CHECK(o.commit());
	if (o.staged()) return finish(ctx);
	return PNOL_OK;
}

// ---------------------------------------------------------------------------------------------------
// One Levenberg-Marquardt iteration's device work behind ONE call and ONE host synchronisation
// (Source/LevenbergMarquardtMPI.cpp:60-108): FD Jacobian at x -> J^T J | J^T F (+ all-reduce) -> damping -> Cholesky solve ->
// x_trial = x + sigma -> residuals at x_trial and their sum of squares (+ all-reduce). The accept / reject decision stays with the
// caller, exactly as in the reference. The five separate entry points above cost two synchronisations and five boundary
// crossings per iteration, which is what is left of an iteration at 8 GPUs.
// ---------------------------------------------------------------------------------------------------
static int normal_eq_blocks(pnol_ctx * ctx, const pnol_functor * f, const double * x_dev, const double * dx_dev, int n, int jac_mode,
                            const double * F_known, double * F_out, double * total);

// device scratch of one LM step (workspace slot 3): A (n*n) | rhs (n) | sigma (n) | xt (n) | sigma_final (n) | sumsq (2) | info (2) |
// packed J^T J|J^T F (n*n + n)
struct LmScratch {
	double * A, * rhs, * sig, * xt, * sigf, * ss, * packed;
	int * info;
};
static int lm_scratch(pnol_ctx * ctx, int n, LmScratch & W)
{
	const size_t nn = (size_t) n * n;
	PNOL_CHECK(ws_reserve(ctx, 3, (2 * nn + 5 * (size_t) n + 16) * sizeof(double)));
	W.A = (double *) ctx->ws[3];
	W.rhs = W.A + nn; W.sig = W.rhs + n; W.xt = W.sig + n; W.sigf = W.xt + n; W.ss = W.sigf + n;
	W.info = (int *) (W.ss + 2);
	W.packed = W.ss + 4;
	return PNOL_OK;
}

// enqueue the device work of one LM step (no synchronisation): x_dev / dx_dev device pointers; lambda from the host scalar or, when
// lambda_dev != nullptr, from device memory. Results stay in the scratch block: xt (trial point), sigf (step), ss (sum Ftrial^2), info.
// tail != nullptr (pnol_lm_iterate): on one rank, or with the peer exchange, the trial sum of squares is left as block partials for
// the caller's lm_tail_kernel (final sum + exchange + accept / reject in one launch); tail->deferred says whether that happened.
struct LmTail {
	const double * partials = nullptr;
	int np = 0;
	bool deferred = false, peer = false;
};
static int lm_step_enqueue(pnol_ctx * ctx, const pnol_functor * f, const double * x_dev, const double * dx_dev, int n, double * J,
                           const double * F, double * Ftrial, double lambda, const double * lambda_dev, int jac_mode, int reuse_jtj,
                           double * JTJ, const LmScratch & W, LmTail * tail = nullptr)
{
	const long long m = f->params.m;
	const size_t nn = (size_t) n * n;
	const size_t packed_count = nn + n;
	// several ranks: the partial sums are exchanged over NVLink peer memory when every rank could map every other's buffer (peer.cu:
	// all-reduce and damping in one kernel, the chi^2 sum in another), through NCCL otherwise. Collective decision, taken once.
	const bool peer = ctx->nranks > 1 && peer_ensure(ctx, packed_count);
	if (!reuse_jtj) {
		double * packed = peer ? peer_partial_slot(ctx) : W.packed;
		// J^T F: summed by the structured Jacobian kernel while it holds the rows of J (cheap there); the black-box kernel leaves
		// it to the SYRK (extra tensor tiles). Either way it ends behind J^T J in `packed`, before the all-reduce.
		if (!J) {
			// no J buffer given: the normal equations are summed over row blocks, J is never stored (normal_eq_blocks)
			PNOL_CHECK(normal_eq_blocks(ctx, f, x_dev, dx_dev, n, jac_mode, F, nullptr, packed));
		} else {
			bool jtf_done = false;
			double * jtf = W.sig;      // free until the solve
			PNOL_CHECK(launch_fd_jacobian(ctx, f, x_dev, dx_dev, n, J, nullptr, jac_mode, F, jtf, &jtf_done));
			PNOL_CHECK(launch_syrk(ctx, J, jtf_done ? nullptr : F, m, n, packed, jtf_done ? jtf : nullptr));      // the finish kernel puts jtf behind J^T J
		}
		if (peer) {
			PNOL_CHECK(launch_peer_reduce_damp(ctx, n, lambda, lambda_dev, JTJ, W.A, W.rhs));      // JTJ + nn takes the right-hand side as well
		} else {
			if (ctx->nranks > 1) PNOL_CHECK(comm_allreduce_dev(ctx, W.packed, packed_count));
			// the right-hand side is kept behind J^T J in the caller's buffer so that a re-damped step can reuse it
			PNOL_CHECK(launch_lm_damp(ctx, W.packed, n, lambda, JTJ, W.A, W.rhs, lambda_dev, true));
		}
	} else {
		PNOL_CHECK(launch_lm_damp(ctx, JTJ, n, lambda, nullptr, W.A, nullptr, lambda_dev));
		PNOL_CUDA(ctx, cudaMemcpyAsync(W.rhs, JTJ + nn, (size_t) n * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
	}
	// solve, and with it the trial point: sigf = sigma (NaN after a non-positive pivot), xt = x + sigf  (:88, :97-100)
	PNOL_CHECK(launch_spd_solve(ctx, W.A, W.rhs, n, W.sig, W.info, x_dev, W.xt, W.sigf));
	if (tail && (ctx->nranks == 1 || peer)) {
		PNOL_CHECK(launch_residual(ctx, f, W.xt, n, Ftrial, nullptr, &tail->partials, &tail->np));
		tail->deferred = true;
		tail->peer = peer;
		return PNOL_OK;
	}
	PNOL_CHECK(launch_residual(ctx, f, W.xt, n, Ftrial, W.ss));
	if (peer) PNOL_CHECK(launch_peer_scalar_sum(ctx, W.ss));
	else if (ctx->nranks > 1) PNOL_CHECK(comm_allreduce_dev(ctx, W.ss, 1));
	return PNOL_OK;
}

extern "C" int pnol_lm_step(pnol_ctx * ctx, const pnol_functor * f, const double * x, const double * dx, int n, double * J, const double * F,
                            double * Ftrial, double lambda, int jac_mode, int reuse_jtj, double * JTJ, double * sigma_out, double * x_trial_out,
                            double * sumsq_trial_out, int * spd_info_out)
{
	if (!ctx || !f) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, x && (dx || jac_mode == PNOL_JAC_ANALYTIC) && F && Ftrial && JTJ && n >= 1, "lm_step: bad arguments");
	PNOL_REQUIRE(ctx, (!J || is_device_ptr(J)) && is_device_ptr(F) && is_device_ptr(Ftrial) && is_device_ptr(JTJ), "lm_step: J, F, Ftrial and JTJ must be device memory");
	PNOL_REQUIRE(ctx, is_residual_kind(f->kind), "lm_step: the functor is not a residual model");
	DevIn<double> dx_, ddx;
	PNOL_CHECK(dx_.init(ctx, x, n));
	PNOL_CHECK(ddx.init(ctx, dx, n));
	// scratch, all in workspace slot 3 (slot 0: SYRK partial tiles, slot 1: the solve's factor, slot 2: sum-of-squares partials,
	// slot 4: the Jacobian kernel's J^T F block partials)
	LmScratch W;
	PNOL_CHECK(lm_scratch(ctx, n, W));
	PNOL_CHECK(lm_step_enqueue(ctx, f, dx_.get(), ddx.get(), n, J, F, Ftrial, lambda, nullptr, jac_mode, reuse_jtj, JTJ, W));
	// one pinned read-back of the contiguous scratch [x_trial | sigma | sumsq (2) | info (2)]
	PNOL_CHECK(pinned_reserve(ctx, 2 * (size_t) n + 4));
	double * pin = ctx->pinned;
	PNOL_CUDA(ctx, cudaMemcpyAsync(pin, W.xt, (2 * (size_t) n + 4) * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
	PNOL_CHECK(finish(ctx));
	PNOL_CHECK(peer_check(ctx));
	if (x_trial_out) memcpy(x_trial_out, pin, (size_t) n * sizeof(double));
	if (sigma_out) memcpy(sigma_out, pin + n, (size_t) n * sizeof(double));
	if (sumsq_trial_out) *sumsq_trial_out = pin[2 * n];
	int inf = 0;
	memcpy(&inf, pin + 2 * n + 2, sizeof(int));
	if (spd_info_out) *spd_info_out = inf;
	return PNOL_OK;
}

// ---------------------------------------------------------------------------------------------------
// A run of LM iterations on device-resident state with the accept / reject rule of Source/LevenbergMarquardtMPI.cpp:107-141 ON THE
// DEVICE: chi^2 test, lambda update, X and F committed by two small kernels behind every step, so the host enqueues a batch of
// iterations and synchronises once per batch (with the decision on the host every iteration paid a device -> host -> device round
// trip and the launch gaps behind it: 0.17 ms, 9 % of an iteration at 8 GPUs). Same arithmetic as the host rule: chi^2 =
// sqrt(sum)^2 with the IEEE square root, ||sigma||_2 as one sequential sum. An accepted step copies Ftrial into F (the host rule
// swapped pointers; kernels enqueued ahead cannot follow a pointer that is only known later).
// ---------------------------------------------------------------------------------------------------
struct LmDevState {
	double lambda, chisq, xdiff;      // xdiff: ||sigma||_2 of the last accepted step
	int accepted, rejected, stopped, last_accept;
};
constexpr int kLmStateDoubles = (int) (sizeof(LmDevState) / sizeof(double));
static_assert(sizeof(LmDevState) % sizeof(double) == 0, "LmDevState travels as doubles behind x");

// the rule itself, one thread: returns 1 when the step is accepted. `sum` = sum of the squared trial residuals over all rows
__device__ __forceinline__ int lm_decide_one(LmDevState * st, double sum, const double * sig_sm, int n, double factor, double x_min_diff)
{
	st->last_accept = 0;
	if (st->stopped) return 0;
	const double root = sqrt(sum);
	const double chi = root * root;                              // pow(vector2Norm(F),2)  (:108)
	if (chi >= st->chisq || chi != chi) {                        // (:110) X and F stay, lambda grows (:118-129)
		st->lambda = st->lambda * factor;
		st->rejected++;
		return 0;
	}
	st->lambda = st->lambda / factor;                            // (:132-141)
	st->chisq = chi;
	st->accepted++;
	st->last_accept = 1;
	double s2 = 0;
	for (int i = 0; i < n; i++) s2 = s2 + sig_sm[i] * sig_sm[i];          // vector2Norm: one sequential sum
	const double xd = sqrt(s2);
	st->xdiff = xd;
	if (x_min_diff > 0 && xd < x_min_diff) st->stopped = 1;              // (:138-140)
	return 1;
}

// one block: thread 0 takes the decision, all threads move x (one thread walking n global-memory entries twice took 13 us at n = 256)
__global__ void __launch_bounds__(256)
lm_decide_kernel(LmDevState * __restrict__ st, double * __restrict__ x, const double * __restrict__ xt,
                 const double * __restrict__ sigma, const double * __restrict__ ss, int n, double factor, double x_min_diff)
{
	extern __shared__ double sig_sm[];
	__shared__ int s_accept;
	for (int i = threadIdx.x; i < n; i += blockDim.x) sig_sm[i] = sigma[i];
	__syncthreads();
	if (threadIdx.x == 0) s_accept = lm_decide_one(st, ss[0], sig_sm, n, factor, x_min_diff);
	__syncthreads();
	if (s_accept) for (int i = threadIdx.x; i < n; i += blockDim.x) x[i] = xt[i];
}

// The end of a device-resident iteration in ONE launch (one block of 1024 threads): final stage of the trial sum of squares
// (sumsq_final_sum: the bits of sumsq_final_kernel), its sum over the ranks through peer memory (peer_scalar_exchange_warp: the bits
// of peer_scalar_sum_kernel; P.R <= 1: no exchange), the accept / reject rule and the move of x. Replaces three launches.
__global__ void __launch_bounds__(1024)
lm_tail_kernel(const double * __restrict__ partials, int np, const PeerScalarArgs P, LmDevState * __restrict__ st, double * __restrict__ x,
               const double * __restrict__ xt, const double * __restrict__ sigma, double * __restrict__ ss, int n, double factor, double x_min_diff)
{
	extern __shared__ double sig_sm[];
	__shared__ double red[1024];
	__shared__ int s_accept;
	for (int i = threadIdx.x; i < n; i += blockDim.x) sig_sm[i] = sigma[i];
	const double mine = sumsq_final_sum(partials, np, red);      // (ends in a barrier: sig_sm is complete as well)
	if (threadIdx.x < 32) {
		const double total = P.R > 1 ? peer_scalar_exchange_warp(P, mine) : mine;
		if (threadIdx.x == 0) {
			ss[0] = total;
			s_accept = lm_decide_one(st, total, sig_sm, n, factor, x_min_diff);
		}
	}
	__syncthreads();
	if (s_accept) for (int i = threadIdx.x; i < n; i += blockDim.x) x[i] = xt[i];
}

// the trial residuals become F after an accepted step (the copy at :91-94 of the reference, done after the decision)
__global__ void __launch_bounds__(256)
lm_commit_kernel(const LmDevState * __restrict__ st, double * __restrict__ F, const double * __restrict__ Ftrial, long long m)
{
	if (!st->last_accept) return;
	const long long m2 = m / 2;
	for (long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x; i < m2; i += (long long) gridDim.x * blockDim.x)
		reinterpret_cast<double2 *>(F)[i] = reinterpret_cast<const double2 *>(Ftrial)[i];
	if ((m & 1) && blockIdx.x == 0 && threadIdx.x == 0) F[m - 1] = Ftrial[m - 1];
}

extern "C" int pnol_lm_iterate(pnol_ctx * ctx, const pnol_functor * f, double * x, const double * dx, int n, double * J, double * F,
                               double * Ftrial, double * JTJ, double * lambda_inout, double * chisq_inout, double lambda_factor,
                               double x_min_diff, int iterations, int jac_mode, int * accepted_out, int * rejected_out,
                               int * swapped_out)
{
	if (!ctx || !f) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, x && (dx || jac_mode == PNOL_JAC_ANALYTIC) && lambda_inout && chisq_inout && iterations >= 0 && n >= 1,
	             "lm_iterate: bad arguments");
	PNOL_REQUIRE(ctx, !is_device_ptr(x), "lm_iterate: x is the host's in/out parameter vector");
	PNOL_REQUIRE(ctx, F && Ftrial && JTJ && (!J || is_device_ptr(J)) && is_device_ptr(F) && is_device_ptr(Ftrial) && is_device_ptr(JTJ),
	             "lm_iterate: J, F, Ftrial and JTJ must be device memory");
	PNOL_REQUIRE(ctx, is_residual_kind(f->kind), "lm_iterate: the functor is not a residual model");
	PNOL_REQUIRE(ctx, ((((size_t) F) | ((size_t) Ftrial)) & 15) == 0, "lm_iterate: F and Ftrial must be 16-byte aligned");
	const long long m = f->params.m;
	DevIn<double> ddx;
	PNOL_CHECK(ddx.init(ctx, dx, n));
	LmScratch W;
	PNOL_CHECK(lm_scratch(ctx, n, W));
	// device state: [LmDevState | x (n)] in workspace slot 2's tail is taken by the sum-of-squares partials, so a slot of its own
	double * xs = nullptr;
	LmDevState * st = nullptr;
	PNOL_CUDA(ctx, cudaMallocAsync((void **) &xs, ((size_t) n + 8) * sizeof(double), ctx->stream));
	static_assert(kLmStateDoubles <= 8, "state block behind x");
	st = (LmDevState *) (xs + n);
	PNOL_CHECK(pinned_reserve(ctx, (size_t) n + 8));
	LmDevState h0;
	h0.lambda = *lambda_inout; h0.chisq = *chisq_inout; h0.xdiff = 0.0; h0.accepted = 0; h0.rejected = 0; h0.stopped = 0; h0.last_accept = 0;
	int status = PNOL_OK;
	auto body = [&]() -> int {
		memcpy(ctx->pinned, x, (size_t) n * sizeof(double));
		memcpy(ctx->pinned + n, &h0, sizeof h0);
		PNOL_CUDA(ctx, cudaMemcpyAsync(xs, ctx->pinned, ((size_t) n + kLmStateDoubles) * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
		// without a stopping rule the whole run is enqueued at once; with one, in batches of four (a stop in the middle of a batch
		// turns the rest of the batch into no-ops for X, F, lambda and chi^2)
		const int batch = x_min_diff > 0 ? 4 : 64;
		int done = 0;
		LmDevState h = h0;
		const int copy_grid = ctx->sm_count * 4;
		while (done < iterations && !h.stopped) {
			const int k = iterations - done < batch ? iterations - done : batch;
			for (int it = 0; it < k; it++) {
				LmTail tail;
				PNOL_CHECK(lm_step_enqueue(ctx, f, xs, ddx.get(), n, J, F, Ftrial, 0.0, &st->lambda, jac_mode, 0, JTJ, W, &tail));
				if (tail.deferred) {
					PeerScalarArgs pa;
					if (tail.peer) pa = peer_scalar_next(ctx);
					else { memset(&pa, 0, sizeof pa); }
					PNOL_LAUNCH(ctx, lm_tail_kernel, 1, 1024, (size_t) n * sizeof(double), tail.partials, tail.np, pa, st, xs, W.xt, W.sigf, W.ss, n,
					            lambda_factor, x_min_diff);
				} else {
					PNOL_LAUNCH(ctx, lm_decide_kernel, 1, 256, (size_t) n * sizeof(double), st, xs, W.xt, W.sigf, W.ss, n, lambda_factor, x_min_diff);
				}
				PNOL_LAUNCH(ctx, lm_commit_kernel, copy_grid, 256, 0, st, F, Ftrial, m);
			}
			PNOL_CUDA(ctx, cudaMemcpyAsync(ctx->pinned, xs, ((size_t) n + kLmStateDoubles) * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
			PNOL_CHECK(finish(ctx));
			PNOL_CHECK(peer_check(ctx));
			memcpy(&h, ctx->pinned + n, sizeof h);
			done += k;
		}
		memcpy(x, ctx->pinned, (size_t) n * sizeof(double));
		*lambda_inout = h.lambda;
		*chisq_inout = h.chisq;
		if (accepted_out) *accepted_out = h.accepted;
		if (rejected_out) *rejected_out = h.rejected;
		if (swapped_out) *swapped_out = 0;                           // accepted residuals are copied into F: they never end in Ftrial
		ctx->lm_last_stopped = h.stopped;
		ctx->lm_last_xdiff = h.xdiff;
		return PNOL_OK;
	};
	ctx->lm_last_stopped = 0;
	ctx->lm_last_xdiff = 0.0;
	if (iterations > 0) status = body();
	else { if (accepted_out) *accepted_out = 0; if (rejected_out) *rejected_out = 0; if (swapped_out) *swapped_out = 0; }
	cudaFreeAsync(xs, ctx->stream);
	return status;
}

extern "C" int pnol_lm_last_run(pnol_ctx * ctx, int * stopped_out, double * xdiff_out)
{
	if (!ctx) return PNOL_ERR_INVALID;
	if (stopped_out) *stopped_out = ctx->lm_last_stopped;
	if (xdiff_out) *xdiff_out = ctx->lm_last_xdiff;
	return PNOL_OK;
}

// host-only: invariants of the SYRK's stream-K work plan for a shape (no device needed; see syrk_plan_selftest in dmma.cu)
extern "C" int pnol_selftest_syrk_plan(long long m, int n, int sm_count, int with_f)
{
	return syrk_plan_selftest(m, n, sm_count, with_f);
}

__global__ void packed_accumulate_kernel(double * __restrict__ acc, const double * __restrict__ add, long long count)
{
	long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x;
	if (i < count) acc[i] = acc[i] + add[i];
}

// SURVEY.md 8(f) item 2: the normal equations without J in HBM. The rows are walked in blocks: the Jacobian kernel writes a block
// of J (512 MB by default, PNOL_FUSED_MB overrides) into a scratch buffer, the SYRK reads it back, the block's J^T J | J^T F is
// added to the running sum: work space 512 MB instead of m*n*8 bytes (8.19 GB at m = 4M, n = 256), so m is no longer limited by
// the 180 GB of HBM. It is the memory-footprint mode, not a faster one: both kernels are bound by the FP64 unit, not by HBM
// (DESIGN.md section 5.1), and every block pays the SYRK's ramp-up and reduction. Measured at m = 4M, n = 256
// (profiles/r01_fused_sweep.txt): 35.6 / 21.9 / 15.2 / 13.2 / 12.1 / 11.5 / 10.9 ms per call with 16 / 32 / 64 / 128 / 256 / 512 /
// 1024 MB blocks against 10.56 ms for the stored-J path -- blocks small enough to stay in the L2 are the slowest.
// The block sums are added in row order, so the result is deterministic; it differs from the stored-J path in summation order only.
//   F_known (device, m) != nullptr: the residuals at x are known (LM step): J^T F comes from the structured Jacobian kernel when it
//                                   can provide it, else from the SYRK, as in pnol_lm_step;
//   F_known == nullptr:             the residuals are computed with the Jacobian and written to F_out (device, m) when wanted.
// `total` (device, n*n + n) receives J^T J followed by J^T F of this rank's rows (no all-reduce here).
static int normal_eq_blocks(pnol_ctx * ctx, const pnol_functor * f, const double * x_dev, const double * dx_dev, int n, int jac_mode,
                            const double * F_known, double * F_out, double * total)
{
	const long long m = f->params.m;
	const char * env_mb = getenv("PNOL_FUSED_MB");       // read per call: tests walk several block sizes in one process
	double block_mb = env_mb ? atof(env_mb) : 512.0;    // fractions allowed (tests: 0.1 MB -> the 1024-row minimum)
	if (!(block_mb > 0.0)) block_mb = 512.0;
	long long rows = (long long) (block_mb * 1048576.0) / ((long long) n * (long long) sizeof(double));
	rows = rows / 1024 * 1024;                      // keeps every block of J and F 8 KB-aligned (TMA, double2 stores)
	if (rows < 1024) rows = 1024;
	if (rows > m) rows = m > 0 ? m : 1;
	const size_t nn = (size_t) n * n, packed_count = nn + n;
	// scratch (stream-ordered pool): block of J | residuals of the block | block sum | J^T F of the block
	const size_t j_count = (size_t) rows * n;
	double * scratch = nullptr;
	PNOL_CUDA(ctx, cudaMallocAsync(&scratch, (j_count + (size_t) rows + packed_count + (size_t) n + 64) * sizeof(double), ctx->stream));
	double * Jb = scratch, * Fb = Jb + j_count, * part = Fb + rows, * jtf = part + packed_count;
	int st = PNOL_OK;
	if (cudaMemsetAsync(total, 0, packed_count * sizeof(double), ctx->stream) != cudaSuccess) st = PNOL_ERR_CUDA;
	for (long long r0 = 0; r0 < m && st == PNOL_OK; r0 += rows) {
		const long long nr = (m - r0 < rows) ? (m - r0) : rows;
		pnol_functor view = *f;                     // the same model on rows [r0, r0 + nr): data columns advanced, row count cut
		for (int c = 0; c < f->n_columns && c < PNOL_MAX_COLUMNS; c++)
			if (view.params.col[c]) view.params.col[c] = f->params.col[c] + r0;
		view.params.m = nr;
		if (F_known) {
			bool jtf_done = false;
			st = launch_fd_jacobian(ctx, &view, x_dev, dx_dev, n, Jb, nullptr, jac_mode, F_known + r0, jtf, &jtf_done);
			if (st == PNOL_OK) st = launch_syrk(ctx, Jb, jtf_done ? nullptr : F_known + r0, nr, n, part);
			if (st == PNOL_OK && jtf_done &&
			    cudaMemcpyAsync(part + nn, jtf, (size_t) n * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream) != cudaSuccess) st = PNOL_ERR_CUDA;
		} else {
			double * Fr = F_out ? F_out + r0 : Fb;
			st = launch_fd_jacobian(ctx, &view, x_dev, dx_dev, n, Jb, Fr, jac_mode);
			if (st == PNOL_OK) st = launch_syrk(ctx, Jb, Fr, nr, n, part);
		}
		if (st == PNOL_OK) {
			st = [&]() -> int {
				PNOL_LAUNCH(ctx, packed_accumulate_kernel, (unsigned) ((packed_count + 255) / 256), 256, 0, total, part, (long long) packed_count);
				return PNOL_OK;
			}();
		}
	}
	if (cudaFreeAsync(scratch, ctx->stream) != cudaSuccess && st == PNOL_OK) { PNOL_SET_ERR(ctx, "normal_eq_blocks: freeing the block scratch failed"); st = PNOL_ERR_CUDA; }
	if (st == PNOL_ERR_CUDA && ctx->err.empty()) PNOL_SET_ERR(ctx, "normal_eq_blocks: CUDA error in the block loop");
	return st;
}

extern "C" int pnol_lm_normal_eq_fused(pnol_ctx * ctx, const pnol_functor * f, const double * x, const double * dx, int n,
                                       double lambda, double * JTJ, double * A, double * rhs, double * F)
{
	if (!ctx || !f) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, x && dx && n >= 1, "lm_normal_eq_fused: bad arguments");
	PNOL_REQUIRE(ctx, is_residual_kind(f->kind), "lm_normal_eq_fused: the functor is not a residual model");
	const long long m = f->params.m;
	DevIn<double> dx_, ddx; DevOut<double> oJTJ, oA, orhs, oF;
	PNOL_CHECK(dx_.init(ctx, x, n));
	PNOL_CHECK(ddx.init(ctx, dx, n));
	PNOL_CHECK(oJTJ.init(ctx, JTJ, (size_t) n * n));
	PNOL_CHECK(oA.init(ctx, A, (size_t) n * n));
	PNOL_CHECK(orhs.init(ctx, rhs, (size_t) n));
	PNOL_CHECK(oF.init(ctx, F, (size_t) m));
	const size_t packed_count = (size_t) n * n + n;
	PNOL_CHECK(ws_reserve(ctx, 3, packed_count * sizeof(double)));
	double * total = (double *) ctx->ws[3];
	PNOL_CHECK(normal_eq_blocks(ctx, f, dx_.get(), ddx.get(), n, PNOL_JAC_AUTO, nullptr, oF.get(), total));
	if (ctx->nranks > 1) PNOL_CHECK(comm_allreduce_dev(ctx, total, packed_count));
	PNOL_CHECK(launch_lm_damp(ctx, total, n, lambda, oJTJ.get(), oA.get(), orhs.get()));
	PNOL_CHECK(oJTJ.commit());
	PNOL_CHECK(oA.commit());
	PNOL_CHECK(orhs.commit());
	PNOL_CHECK(oF.commit());
	return finish(ctx);
}

extern "C" int pnol_spd_solve(pnol_ctx * ctx, const double * A, const double * rhs, int n, double * x, int * info)
{
	if (!ctx) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, A && rhs && x && n >= 1, "spd_solve: bad arguments");
	DevIn<double> dA, db; DevOut<double> dx_;
	PNOL_CHECK(dA.init(ctx, A, (size_t) n * n));
	PNOL_CHECK(db.init(ctx, rhs, (size_t) n));
	PNOL_CHECK(dx_.init(ctx, x, (size_t) n));
	PNOL_CHECK(ws_reserve(ctx, 3, 64));
	int * info_dev = (int *) ctx->ws[3];
	PNOL_CHECK(launch_spd_solve(ctx, dA.get(), db.get(), n, dx_.get(), info_dev));
	PNOL_CHECK(dx_.commit());
	int inf = 0;
	PNOL_CUDA(ctx, cudaMemcpyAsync(&inf, info_dev, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
	PNOL_CHECK(finish(ctx));
	if (info) *info = inf;
	if (inf != 0) { PNOL_SET_ERR(ctx, "spd_solve: pivot %d is outside [2^-1022, 2^1000)", inf); return PNOL_ERR_NOT_SPD; }
	return PNOL_OK;
}

// general inverse (LU, partial pivoting): matrixInverse of the FD Hessian, Source/BFGS_bnd_linesearch_MPI_SW.cpp:51-59
extern "C" int pnol_lu_inverse(pnol_ctx * ctx, const double * A, int n, double * Ainv, int * info)
{
	if (!ctx) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, A && Ainv && n >= 1, "lu_inverse: bad arguments");
	DevIn<double> dA; DevOut<double> dI;
	PNOL_CHECK(dA.init(ctx, A, (size_t) n * n));
	PNOL_CHECK(dI.init(ctx, Ainv, (size_t) n * n));
	PNOL_CHECK(ws_reserve(ctx, 3, 64));
	int * info_dev = (int *) ctx->ws[3];
	PNOL_CHECK(launch_lu_inverse(ctx, dA.get(), n, dI.get(), info_dev));
	PNOL_CHECK(dI.commit());
	int inf = 0;
	PNOL_CUDA(ctx, cudaMemcpyAsync(&inf, info_dev, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
	PNOL_CHECK(finish(ctx));
	if (info) *info = inf;
	return PNOL_OK;
}

// ---------------------------------------------------------------------------------------------------
// BFGS dense pieces
// ---------------------------------------------------------------------------------------------------
extern "C" int pnol_matvec_neg(pnol_ctx * ctx, const double * D, const double * g, int n, double * p)
{
	if (!ctx) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, D && g && p && n >= 1, "matvec_neg: bad arguments");
	DevIn<double> dD, dg; DevOut<double> dp;
	PNOL_CHECK(dD.init(ctx, D, (size_t) n * n));
	PNOL_CHECK(dg.init(ctx, g, (size_t) n));
	PNOL_CHECK(dp.init(ctx, p, (size_t) n));
	PNOL_CHECK(launch_matvec_neg(ctx, dD.get(), dg.get(), n, dp.get()));
	PNOL_CHECK(dp.commit());
	if (dp.staged()) return finish(ctx);
	return PNOL_OK;
}

extern "C" int pnol_bfgs_update_hinv(pnol_ctx * ctx, double * D, const double * g, const double * s, int n, int mode)
{
	if (!ctx) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, D && g && s && n >= 1, "bfgs_update_hinv: bad arguments");
	PNOL_REQUIRE(ctx, mode == PNOL_HINV_LITERAL || mode == PNOL_HINV_RANK2, "bfgs_update_hinv: bad mode %d", mode);
	DevOut<double> dD; DevIn<double> dg, ds;
	PNOL_CHECK(dD.init(ctx, D, (size_t) n * n, true));
	PNOL_CHECK(dg.init(ctx, g, (size_t) n));
	PNOL_CHECK(ds.init(ctx, s, (size_t) n));
	if (mode == PNOL_HINV_LITERAL) PNOL_CHECK(launch_hinv_literal(ctx, dD.get(), dg.get(), ds.get(), n));
	else PNOL_CHECK(launch_hinv_rank2(ctx, dD.get(), dg.get(), ds.get(), n));
	PNOL_CHECK(dD.commit());
	if (dD.staged()) return finish(ctx);
	return PNOL_OK;
}

extern "C" int pnol_dgemm_nn(pnol_ctx * ctx, const double * A, const double * B, double * C, int M, int N, int K)
{
	if (!ctx) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, A && B && C, "dgemm: null argument");
	DevIn<double> dA, dB; DevOut<double> dC;
	PNOL_CHECK(dA.init(ctx, A, (size_t) M * K));
	PNOL_CHECK(dB.init(ctx, B, (size_t) K * N));
	PNOL_CHECK(dC.init(ctx, C, (size_t) M * N));
	PNOL_CHECK(launch_dgemm_nn(ctx, dA.get(), dB.get(), dC.get(), M, N, K));
	PNOL_CHECK(dC.commit());
	if (dC.staged()) return finish(ctx);
	return PNOL_OK;
}

// ---------------------------------------------------------------------------------------------------
// box-bound helpers (host arithmetic)
// ---------------------------------------------------------------------------------------------------
// checkBoxBounds (Source/Box_boundary_functions.cpp:11-40): a start value outside the box by more than
// |bound|/1000 is replaced by the box midpoint.
extern "C" int pnol_check_box_bounds(double * x, const double * xlb, const double * xub, int n, int * n_replaced)
{
	if (!x || !xlb || !xub || n < 0) return PNOL_ERR_INVALID;
	int cnt = 0;
	for (int i = 0; i < n; i++) {
		if (x[i] - xlb[i] < -fabs(xlb[i]) / 1000 || x[i] - xub[i] > fabs(xub[i]) / 1000) {
			x[i] = (xlb[i] + xub[i]) / 2.0;
			cnt++;
		}
	}
	if (n_replaced) *n_replaced = cnt;
	return PNOL_OK;
}

// computeAlphaBnd (Source/BFGS_with_bnd_linsearch_MPI.cpp:665-708): largest feasible step along p
extern "C" double pnol_compute_alpha_bnd(const double * x, const double * xlb, const double * xub, const double * p, int n)
{
	double alphaBnd = 0;
	for (int i = 0; i < n; i++) {
		double a1 = (xub[i] - x[i]) / p[i];
		double a2 = (xlb[i] - x[i]) / p[i];
		double ai;
		if (a1 > 0) ai = a1;
		else if (a2 > 0) ai = a2;
		else ai = 0;
		if (i == 0) alphaBnd = ai;
		if (alphaBnd > ai) alphaBnd = ai;
	}
	return alphaBnd;
}

// counter-based uniform stream (host side of the generator the GA kernels use)
extern "C" double pnol_stream_uniform(uint64_t seed, uint64_t k, double scale)
{
	uint64_t z = seed + (k + 1ULL) * 0x9E3779B97F4A7C15ULL;
	z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
	z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
	z = z ^ (z >> 31);
	return ((double) (z >> 11) * (1.0 / 9007199254740992.0)) * scale;
}

// ---------------------------------------------------------------------------------------------------
// copy-bandwidth probe (HBM roofline cross-check)
// ---------------------------------------------------------------------------------------------------
__global__ void copy_kernel(const double2 * __restrict__ a, double2 * __restrict__ b, long long n2)
{
	for (long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (long long) gridDim.x * blockDim.x) b[i] = a[i];
}

extern "C" int pnol_measure_copy_bandwidth(pnol_ctx * ctx, double * gbs_out)
{
	if (!ctx || !gbs_out) return PNOL_ERR_INVALID;
	const long long n2 = (long long) 1 << 26;     // 2^26 double2 = 1 GiB per buffer
	void * a = nullptr; void * b = nullptr;
	PNOL_CUDA(ctx, cudaMalloc(&a, n2 * 16));
	PNOL_CUDA(ctx, cudaMalloc(&b, n2 * 16));
	PNOL_CUDA(ctx, cudaMemsetAsync(a, 1, n2 * 16, ctx->stream));
	cudaEvent_t e0, e1;
	cudaEventCreate(&e0); cudaEventCreate(&e1);
	double best = 0;
	for (int rep = 0; rep < 6; rep++) {
		cudaEventRecord(e0, ctx->stream);
		PNOL_LAUNCH(ctx, copy_kernel, ctx->sm_count * 16, 512, 0, (const double2 *) a, (double2 *) b, n2);
		cudaEventRecord(e1, ctx->stream);
		cudaEventSynchronize(e1);
		float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
		double gbs = 2.0 * n2 * 16 / (ms * 1e-3) / 1e9;
		if (rep > 0 && gbs > best) best = gbs;
	}
	cudaEventDestroy(e0); cudaEventDestroy(e1);
	cudaFree(a); cudaFree(b);
	*gbs_out = best;
	return PNOL_OK;
}

// ---------------------------------------------------------------------------------------------------
// self test of exact_div.cuh: counts pairs where div_exact(x, d) differs from x / d (must be 0)
// ---------------------------------------------------------------------------------------------------
__global__ void exact_div_selftest_kernel(unsigned long long seed, long long per_thread, unsigned long long * __restrict__ bad)
{
	unsigned long long s = seed + 0x9E3779B97F4A7C15ULL * (1 + (unsigned long long) blockIdx.x * blockDim.x + threadIdx.x);
	unsigned long long nbad = 0;
	for (long long i = 0; i < per_thread; i++) {
		s ^= s << 13; s ^= s >> 7; s ^= s << 17;
		unsigned long long md = s;
		s ^= s << 13; s ^= s >> 7; s ^= s << 17;
		unsigned long long mx = s;
		s ^= s << 13; s ^= s >> 7; s ^= s << 17;
		const int mode = (int) (i & 7);
		if (mode == 1) md |= 0xFFFFFFFFFF000ULL;
		if (mode == 2) md &= 0xFFFULL;
		if (mode == 3) mx |= 0xFFFFFFFFFFFF0ULL;
		if (mode == 4) mx &= 0xFFULL;
		if (mode == 5) md = 0xFFFFFFFFFFFFFULL - (s & 0xF);
		int ed = (int) ((s >> 8) % 60) - 40, exx = (int) ((s >> 20) % 80) - 40;
		if (mode == 6) exx = (int) ((s >> 20) % 2040) - 1020;      // whole exponent range incl. subnormal-ish, inf/nan
		double d = __longlong_as_double((long long) (((unsigned long long) (ed + 1023) << 52) | (md & 0xFFFFFFFFFFFFFULL)));
		double x = __longlong_as_double((long long) (((unsigned long long) (exx + 1023) << 52) | (mx & 0xFFFFFFFFFFFFFULL)));
		if (mode == 7 && (i & 8)) x = 0.0;
		if (s & 1) x = -x;
		if (s & 2) d = -d;
		pnol::RecipDiv rd = pnol::make_recip(d);
		double got = pnol::div_exact(x, rd);
		double want = x / d;
		if (__double_as_longlong(got) != __double_as_longlong(want) && !(got != got && want != want)) nbad++;
	}
	if (nbad) atomicAdd(bad, nbad);
}

extern "C" int pnol_selftest_exact_div(pnol_ctx * ctx, long long pairs, unsigned long long seed, unsigned long long * mismatches)
{
	if (!ctx || !mismatches) return PNOL_ERR_INVALID;
	PNOL_CHECK(ws_reserve(ctx, 3, 64));
	unsigned long long * bad = (unsigned long long *) ctx->ws[3];
	PNOL_CUDA(ctx, cudaMemsetAsync(bad, 0, sizeof(unsigned long long), ctx->stream));
	const int blocks = ctx->sm_count * 8, threads = 256;
	long long per_thread = (pairs + (long long) blocks * threads - 1) / ((long long) blocks * threads);
	PNOL_LAUNCH(ctx, exact_div_selftest_kernel, blocks, threads, 0, seed, per_thread, bad);
	PNOL_CUDA(ctx, cudaMemcpyAsync(mismatches, bad, sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
	return finish(ctx);
}

// self test of the branch-free division cores: pairs (a, b) inside the validity predicates for which div_core(a, b) differs
// from a / b, plus pairs (x, d) with div_exact_x_ok(x) for which div_exact_core differs from x / d (must be 0)
__global__ void fast_div_selftest_kernel(unsigned long long seed, long long per_thread, unsigned long long * __restrict__ bad)
{
	unsigned long long s = seed + 0x9E3779B97F4A7C15ULL * (1 + (unsigned long long) blockIdx.x * blockDim.x + threadIdx.x);
	unsigned long long nbad = 0;
	for (long long i = 0; i < per_thread; i++) {
		s ^= s << 13; s ^= s >> 7; s ^= s << 17;
		unsigned long long mb = s;
		s ^= s << 13; s ^= s >> 7; s ^= s << 17;
		unsigned long long ma = s;
		s ^= s << 13; s ^= s >> 7; s ^= s << 17;
		const int mode = (int) (i & 7);
		if (mode == 1) mb |= 0xFFFFFFFFFF000ULL;
		if (mode == 2) mb &= 0xFFFULL;
		if (mode == 3) ma |= 0xFFFFFFFFFFFF0ULL;
		if (mode == 4) ma &= 0xFFULL;
		if (mode == 5) mb = 0xFFFFFFFFFFFFFULL - (s & 0xF);
		int eb = (int) ((s >> 8) % 60) - 30, ea = (int) ((s >> 20) % 80) - 40;
		if (mode == 6) { eb = (int) ((s >> 8) % 798) - 399; ea = (int) ((s >> 20) % 798) - 399; }     // the whole validity range
		double b = __longlong_as_double((long long) (((unsigned long long) (eb + 1023) << 52) | (mb & 0xFFFFFFFFFFFFFULL)));
		double a = __longlong_as_double((long long) (((unsigned long long) (ea + 1023) << 52) | (ma & 0xFFFFFFFFFFFFFULL)));
		if (mode == 7 && (i & 8)) a = (i & 16) ? 0.0 : -0.0;
		if (s & 1) a = -a;
		if (s & 2) b = -b;
		if (pnol::div_den_ok(b) && pnol::div_num_ok(a)) {
			double got = pnol::div_core(a, b), want = a / b;
			if (__double_as_longlong(got) != __double_as_longlong(want)) nbad++;
		}
		pnol::RecipDiv rd = pnol::make_recip(b);
		if (rd.r != 0.0 && pnol::div_exact_x_ok(a)) {
			double got = pnol::div_exact_core(a, rd), want = a / b;
			if (__double_as_longlong(got) != __double_as_longlong(want)) nbad++;
		}
		// the three-operation quotient for the divisors with a good rounded reciprocal (about half of them), x = -0 excluded as in the row
		if (pnol::recip_three_ok(rd) && pnol::div_exact_x_ok_pz(a)) {
			double got = pnol::div_exact3_core(a, rd), want = a / b;
			if (__double_as_longlong(got) != __double_as_longlong(want)) nbad++;
		}
		// ... and with the quotient next to a floating-point number or a midpoint: x = RN(b q + k b ulp(q) / 2) for a random q, k = -1 .. 2
		if (pnol::recip_three_ok(rd) && (mode == 0 || mode == 2)) {
			const double q = __longlong_as_double((long long) (((unsigned long long) (ea + 1023) << 52) | (ma & 0xFFFFFFFFFFFFFULL)));
			const double u = __longlong_as_double(__double_as_longlong(q) + 1) - q;
			const double xq = fma(b, q, 0.5 * (double) ((int) (s >> 40 & 3) - 1) * (b * u));
			if (pnol::div_exact_x_ok_pz(xq)) {
				double got = pnol::div_exact3_core(xq, rd), want = xq / b;
				if (__double_as_longlong(got) != __double_as_longlong(want)) nbad++;
			}
		}
	}
	if (nbad) atomicAdd(bad, nbad);
}

extern "C" int pnol_selftest_fast_div(pnol_ctx * ctx, long long pairs, unsigned long long seed, unsigned long long * mismatches)
{
	if (!ctx || !mismatches) return PNOL_ERR_INVALID;
	PNOL_CHECK(ws_reserve(ctx, 3, 64));
	unsigned long long * bad = (unsigned long long *) ctx->ws[3];
	PNOL_CUDA(ctx, cudaMemsetAsync(bad, 0, sizeof(unsigned long long), ctx->stream));
	const int blocks = ctx->sm_count * 8, threads = 256;
	long long per_thread = (pairs + (long long) blocks * threads - 1) / ((long long) blocks * threads);
	PNOL_LAUNCH(ctx, fast_div_selftest_kernel, blocks, threads, 0, seed, per_thread, bad);
	PNOL_CUDA(ctx, cudaMemcpyAsync(mismatches, bad, sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
	return finish(ctx);
}
