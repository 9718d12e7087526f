// simplex_batch.cu -- pnol_simplex_batch: many independent Nelder-Mead minimisations of one scalar objective (multiple starts) in one
// kernel launch, each start bit for bit the reference's SimplexSearch::findMin on that start alone. The kernel (simplex_batch_kernel)
// is the header template of include/pnol/device/functor_kernels.cuh; the launcher comes from the record of the functor's kind
// (kind_table): builtin_simplex_batch.cu instantiates it for the six built-in scalar objectives, a user scalar kind attaches its own
// with pnol_register_functor_simplex_batch.
#include "common.cuh"
#include "pnol/device/functor_kernels.cuh"

using namespace pnol;

extern "C" int pnol_simplex_batch(pnol_ctx * ctx, const pnol_functor * f, long long B, int n, double * X, const pnol_simplex_params * prm,
                                  const pnol_stream_desc * stream, uint64_t stream_offset, double * f0_out, double * fopt_out, int * iters_out,
                                  int * stop_out, long long * evals_out)
{
	if (!ctx || !f) return PNOL_ERR_INVALID;
	KindTable kt;
	if (!kind_table(f->kind, &kt) || !kt.vt.eval_batch) return wrong_family(ctx, f->kind, "scalar objective");
	PNOL_REQUIRE(ctx, n >= 1 && n <= dev::kSimplexBatchMaxN, "simplex_batch: n = %d is outside 1 .. %d (larger problems: the SimplexSearch class)",
	             n, dev::kSimplexBatchMaxN);
	PNOL_REQUIRE(ctx, B >= 0 && B <= 0x7fffffffLL, "simplex_batch: B = %lld is outside 0 .. 2^31 - 1", B);
	PNOL_REQUIRE(ctx, prm, "simplex_batch: the parameters (prm) are required");
	PNOL_REQUIRE(ctx, stream, "simplex_batch: the random stream is required");
	if (B == 0) return PNOL_OK;
	PNOL_REQUIRE(ctx, X && f0_out && fopt_out && iters_out && stop_out, "simplex_batch: X and the four per-start outputs are required");
	// every draw precedes the first evaluation, so a short stream is refused before anything runs
	const uint64_t draws = (uint64_t) B * (uint64_t) n * (uint64_t) n;
	if (stream->values && (stream_offset > stream->n_values || stream->n_values - stream_offset < draws)) {
		PNOL_SET_ERR(ctx, "simplex_batch: the explicit random stream has %llu values, the batch needs %llu from position %llu",
		             (unsigned long long) stream->n_values, (unsigned long long) draws, (unsigned long long) stream_offset);
		return PNOL_ERR_STREAM;
	}
	if (!kt.simplex_batch) {
		PNOL_SET_ERR(ctx, "functor kind %d has no batched simplex launcher (pnol_register_functor_simplex_batch)", f->kind);
		return PNOL_ERR_NO_FUNCTOR;
	}

	TimerScope ts(ctx, "simplex_batch");
	// the launcher reads an explicit stream from the device, its own slice from index 0
	pnol_stream_desc sd = *stream;
	DevOut<double> dvals;
	if (stream->values) {
		PNOL_CHECK(dvals.init(ctx, const_cast<double *>(stream->values) + stream_offset, (size_t) draws, true));
		sd.values = dvals.get();
		sd.n_values = draws;
		stream_offset = 0;
	}
	DevOut<double> dX, df0, dfopt;
	DevOut<int> dit, dstop;
	DevOut<long long> devals;
	PNOL_CHECK(dX.init(ctx, X, (size_t) B * n, true));
	PNOL_CHECK(df0.init(ctx, f0_out, (size_t) B));
	PNOL_CHECK(dfopt.init(ctx, fopt_out, (size_t) B));
	PNOL_CHECK(dit.init(ctx, iters_out, (size_t) B));
	PNOL_CHECK(dstop.init(ctx, stop_out, (size_t) B));
	PNOL_CHECK(devals.init(ctx, evals_out, (size_t) B));
	const pnol_launch_env env = make_env(ctx);
	PNOL_CHECK(kt.simplex_batch(&env, &f->params, B, n, dX.get(), prm, &sd, stream_offset, df0.get(), dfopt.get(), dit.get(), dstop.get(),
	                            devals.get()));
	PNOL_CHECK(dX.commit());
	PNOL_CHECK(df0.commit());
	PNOL_CHECK(dfopt.commit());
	PNOL_CHECK(dit.commit());
	PNOL_CHECK(dstop.commit());
	PNOL_CHECK(devals.commit());
	return finish(ctx);
}
