// ga.cu -- genetic algorithm on the device (a15 / a16): the C-ABI layer. The state object of GeneticAlgorithmMPI::findMinBnd
// (Source/GeneticAlgorithmMPI.cpp:12-276) and its initial population (:55-81), and the free functions popSort /
// checkIndenticalChildAndReplace / checkPopulationBoundsAndReplace (Source/GeneticAlgorithm.cpp:313-412) as stand-alone stages.
// Everything after the start population runs on the generation's stages in ga_pipeline.cu: pnol_ga_init is a generation whose
// children are the start population, and the stand-alone calls run the same stage functions on the caller's rows.
#include "ga_common.cuh"

#include <math.h>

namespace pnol {

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
	GA_TRY(ga_alloc(ga, &ga->Xnew, NN));
	GA_TRY(ga_alloc(ga, &ga->fitness, Npop));
	GA_TRY(ga_alloc(ga, &ga->lb, n));
	GA_TRY(ga_alloc(ga, &ga->ub, n));
	GA_TRY(ga_alloc(ga, &ga->x0, n));
	GA_TRY(ga_alloc(ga, &ga->cross_idx, (size_t) ncross * n));
	GA_TRY(ga_alloc(ga, &ga->mut_idx, nrand));
	GA_TRY(ga_alloc(ga, &ga->mut_pos, nrand));
	GA_TRY(ga_alloc(ga, &ga->elite_idx, (size_t) nelmut * n));
	if (stream->values && stream->n_values) {
		GA_TRY(ga_alloc(ga, &ga->stream_values, stream->n_values));
		cudaError_t e = cudaMemcpyAsync(ga->stream_values, stream->values, stream->n_values * sizeof(double), cudaMemcpyDefault, ctx->stream);
		if (e != cudaSuccess) { PNOL_SET_ERR(ctx, "ga: stream upload: %s", cudaGetErrorString(e)); pnol_ga_destroy(ga); return PNOL_ERR_CUDA; }
	}
	cudaMemcpyAsync(ga->lb, xlb, n * sizeof(double), cudaMemcpyDefault, ctx->stream);
	cudaMemcpyAsync(ga->ub, xub, n * sizeof(double), cudaMemcpyDefault, ctx->stream);
	GA_TRY(finish(ctx));
	GA_TRY(ga_pipe_create(ga));
#undef GA_TRY
	*out = ga;
	return PNOL_OK;
}

// Source/GeneticAlgorithmMPI.cpp:55-81
extern "C" int pnol_ga_init(pnol_ga * ga, const double * x0, double * f0_out)
{
	if (!ga || !x0) return PNOL_ERR_INVALID;
	pnol_ctx * ctx = ga->ctx;
	const long long Npop = ga->prm.npop;
	const int n = ga->n;
	ga->pos = 0; ga->generation = 0; ga->n_static = 0; ga->stopped = 0;
	PNOL_CUDA(ctx, cudaMemcpyAsync(ga->x0, x0, n * sizeof(double), cudaMemcpyDefault, ctx->stream));
	PNOL_LAUNCH(ctx, ga_init_pop_kernel, (unsigned) ((Npop * n + 255) / 256), 256, 0, ga->Xnew, Npop, n, ga->x0, ga->lb, ga->ub, ga_stream(ga),
	            (unsigned long long) ga->pos);
	ga->pos += (uint64_t) (Npop - 1) * n;
	// The reference then checks the all-zero XpopNew for identical children (:71, sic). Row i is only compared with later rows, and
	// those are untouched zeros: every row but the last is replaced once, n draws each, and the replaced rows are never read again.
	// So the check only advances the stream by (Npop - 1) n.
	ga->pos += (uint64_t) (Npop - 1) * n;
	return ga_pipe_init(ga, f0_out);
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
extern "C" int pnol_ga_pop_sort(pnol_ctx * ctx, double * xpop, double * F, long long npop, int n)
{
	if (!ctx) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, xpop && F && npop >= 1 && n >= 1, "ga_pop_sort: bad arguments");
	PNOL_REQUIRE(ctx, npop <= (1LL << 32), "ga_pop_sort: npop = %lld, at most 2^32 (32-bit row numbers)", npop);
	DevOut<double> dX, dF;
	PNOL_CHECK(dX.init(ctx, xpop, (size_t) npop * n, true));
	PNOL_CHECK(dF.init(ctx, F, (size_t) npop, true));
	PNOL_CHECK(ga_stage_pop_sort(ctx, dX.get(), dF.get(), npop, n));
	PNOL_CHECK(dX.commit());
	PNOL_CHECK(dF.commit());
	return finish(ctx);
}

static int ga_stage_call(pnol_ctx * ctx, bool identical, double * xpop, long long npop, int n, const double * xlb, const double * xub,
                         unsigned char * indicator, const pnol_stream_desc * stream, uint64_t * stream_pos)
{
	PNOL_REQUIRE(ctx, xpop && xlb && xub && stream && stream_pos && npop >= 1 && n >= 1, "ga stage: bad arguments");
	// the packed stream offsets of the generation's stage 5 count replaced rows in 24 bits and repaired genes in 40
	if (identical) PNOL_REQUIRE(ctx, npop <= (1LL << 24), "ga_check_identical: npop = %lld, at most 2^24", npop);
	else PNOL_REQUIRE(ctx, npop < (1LL << 40) / n, "ga_check_bounds: npop x n = %lld x %d, below 2^40", npop, n);
	DevOut<double> dX; DevIn<double> dlb, dub, dvalues; DevOut<unsigned char> dind;
	PNOL_CHECK(dX.init(ctx, xpop, (size_t) npop * n, true));
	PNOL_CHECK(dlb.init(ctx, xlb, n));
	PNOL_CHECK(dub.init(ctx, xub, n));
	PNOL_CHECK(dind.init(ctx, indicator, (size_t) npop, true));
	PNOL_CHECK(dvalues.init(ctx, stream->values, stream->n_values));
	StreamDev st;
	st.values = dvalues.get(); st.n_values = stream->n_values; st.seed = stream->seed; st.scale = stream->scale;
	unsigned long long pos_end = 0;
	PNOL_CHECK(ga_stage_repair(ctx, identical, dX.get(), npop, n, dlb.get(), dub.get(), dind.get(), st, *stream_pos, &pos_end));
	PNOL_CHECK(dX.commit());
	PNOL_CHECK(dind.commit());
	PNOL_CHECK(finish(ctx));
	*stream_pos = pos_end;
	// the stage reads the draws [pos, pos_end); reads past the end of an explicit stream gave 0.0
	if (st.values && pos_end > stream->n_values) { PNOL_SET_ERR(ctx, "ga: the explicit random stream is exhausted"); return PNOL_ERR_STREAM; }
	return PNOL_OK;
}

extern "C" int pnol_ga_check_bounds(pnol_ctx * ctx, double * xpop, long long npop, int n, const double * xlb, const double * xub,
                                    unsigned char * indicator, const pnol_stream_desc * stream, uint64_t * stream_pos)
{
	if (!ctx) return PNOL_ERR_INVALID;
	return ga_stage_call(ctx, false, xpop, npop, n, xlb, xub, indicator, stream, stream_pos);
}

extern "C" int pnol_ga_check_identical(pnol_ctx * ctx, double * xpop, long long npop, int n, const double * xlb, const double * xub,
                                       unsigned char * indicator, const pnol_stream_desc * stream, uint64_t * stream_pos)
{
	if (!ctx) return PNOL_ERR_INVALID;
	return ga_stage_call(ctx, true, xpop, npop, n, xlb, xub, indicator, stream, stream_pos);
}
