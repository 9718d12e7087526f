// lm_batch.cu -- pnol_lm_batch: many small independent Levenberg-Marquardt fits in one kernel launch, each problem bit for bit the
// reference's LevMarq::findMin on its own rows. The kernel (lm_batch_kernel) is the header template of include/pnol/device/
// functor_kernels.cuh; the launcher comes from the record of the functor's kind (kind_table): builtin_residual_functors.cu instantiates
// it for the three built-in residual models, a user residual kind attaches its own with pnol_register_functor_lm_batch.
#include "common.cuh"
#include "pnol/device/functor_kernels.cuh"

#include <vector>

using namespace pnol;

extern "C" int pnol_lm_batch(pnol_ctx * ctx, const pnol_functor * f, const long long * row_off, long long B, int n, double * X,
                             const double * dx, double lambda0, double lambda_factor, double x_min_diff, int max_iter, int jac_mode,
                             double * chisq_out, double * lambda_out, int * iters_out, int * stopped_out, double * F_out)
{
	if (!ctx || !f) return PNOL_ERR_INVALID;
	PNOL_REQUIRE(ctx, is_residual_kind(f->kind), "lm_batch: functor kind %d is not a residual model", f->kind);
	PNOL_REQUIRE(ctx, n >= 1 && n <= dev::kLmBatchMaxN, "lm_batch: n = %d is outside 1 .. %d (larger problems: pnol_lm_iterate)", n,
	             dev::kLmBatchMaxN);
	PNOL_REQUIRE(ctx, B >= 0 && B <= 0x7fffffffLL, "lm_batch: B = %lld is outside 0 .. 2^31 - 1", B);
	if (B == 0) return PNOL_OK;
	PNOL_REQUIRE(ctx, row_off && X && chisq_out && lambda_out && iters_out && stopped_out, "lm_batch: row_off, X and the four per-problem "
	             "outputs are required");
	const bool analytic = jac_mode == PNOL_JAC_ANALYTIC;
	PNOL_REQUIRE(ctx, analytic || dx, "lm_batch: dx is required for a forward-difference Jacobian");
	PNOL_CHECK(lorentz_shape_ok(ctx, f, n));
	KindTable kt;
	if (!kind_table(f->kind, &kt) || !kt.vt.residual) return wrong_family(ctx, f->kind, "residual model");
	if (!kt.lm_batch) {
		PNOL_SET_ERR(ctx, "functor kind %d has no batched LM launcher (pnol_register_functor_lm_batch)", f->kind);
		return PNOL_ERR_NO_FUNCTOR;
	}
	// row_off: B + 1 non-decreasing offsets within [0, m] (read on the host: a device array is copied back first)
	const long long m = f->params.m;
	std::vector<long long> ro_host;
	const long long * ro = row_off;
	if (is_device_ptr(row_off)) {
		ro_host.resize((size_t) B + 1);
		PNOL_CUDA(ctx, cudaMemcpyAsync(ro_host.data(), row_off, ((size_t) B + 1) * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
		PNOL_CHECK(finish(ctx));
		ro = ro_host.data();
	}
	PNOL_REQUIRE(ctx, ro[0] >= 0 && ro[B] <= m, "lm_batch: row_off[0] = %lld and row_off[B] = %lld must lie within [0, m = %lld]", ro[0], ro[B], m);
	for (long long b = 0; b < B; b++)
		PNOL_REQUIRE(ctx, ro[b] <= ro[b + 1], "lm_batch: row_off decreases at problem %lld (%lld > %lld)", b, ro[b], ro[b + 1]);

	TimerScope ts(ctx, "lm_batch");
	DevIn<long long> dro; DevIn<double> ddx;
	DevOut<double> dX, dchi, dlam, dF; DevOut<int> dit, dstop;
	PNOL_CHECK(dro.init(ctx, row_off, (size_t) B + 1));
	if (!analytic) PNOL_CHECK(ddx.init(ctx, dx, (size_t) n));
	PNOL_CHECK(dX.init(ctx, X, (size_t) B * n, true));
	PNOL_CHECK(dchi.init(ctx, chisq_out, (size_t) B));
	PNOL_CHECK(dlam.init(ctx, lambda_out, (size_t) B));
	PNOL_CHECK(dit.init(ctx, iters_out, (size_t) B));
	PNOL_CHECK(dstop.init(ctx, stopped_out, (size_t) B));
	if (F_out) PNOL_CHECK(dF.init(ctx, F_out, (size_t) m, true));      // rows outside every problem keep what they held
	const pnol_launch_env env = make_env(ctx);
	PNOL_CHECK(kt.lm_batch(&env, &f->params, dro.get(), B, n, dX.get(), ddx.get(), lambda0, lambda_factor, x_min_diff, max_iter, jac_mode,
	                       dchi.get(), dlam.get(), dit.get(), dstop.get(), dF.get()));
	PNOL_CHECK(dX.commit());
	PNOL_CHECK(dchi.commit());
	PNOL_CHECK(dlam.commit());
	PNOL_CHECK(dit.commit());
	PNOL_CHECK(dstop.commit());
	PNOL_CHECK(dF.commit());
	return finish(ctx);
}
