// bfgs_batch.cu -- pnol_bfgs_batch: many independent BFGS minimisations of one scalar objective (multiple starts) in one kernel launch,
// each start bit for bit the reference's BFGS::findMin on that start alone. The kernel (bfgs_batch_kernel) is the header template of
// include/pnol/device/functor_kernels.cuh; the launcher comes from the record of the functor's kind (kind_table): builtin_bfgs_batch.cu
// instantiates it for the six built-in scalar objectives, a user scalar kind attaches its own with pnol_register_functor_bfgs_batch.
#include "common.cuh"
#include "pnol/device/functor_kernels.cuh"

using namespace pnol;

extern "C" int pnol_bfgs_batch(pnol_ctx * ctx, const pnol_functor * f, long long B, int n, double * X, const pnol_bfgs_params * prm,
                               int deriv_flags, double * f0_out, double * fopt_out, int * iters_out, int * stop_out)
{
	if (!ctx || !f) return PNOL_ERR_INVALID;
	KindTable kt;
	if (!kind_table(f->kind, &kt) || !kt.vt.eval_batch) return wrong_family(ctx, f->kind, "scalar objective");
	PNOL_REQUIRE(ctx, n >= 1 && n <= dev::kBfgsBatchMaxN, "bfgs_batch: n = %d is outside 1 .. %d (larger problems: the BFGS class)", n,
	             dev::kBfgsBatchMaxN);
	PNOL_REQUIRE(ctx, B >= 0 && B <= 0x7fffffffLL, "bfgs_batch: B = %lld is outside 0 .. 2^31 - 1", B);
	PNOL_REQUIRE(ctx, prm, "bfgs_batch: the parameters (prm) are required");
	if (B == 0) return PNOL_OK;
	PNOL_REQUIRE(ctx, X && f0_out && fopt_out && iters_out && stop_out, "bfgs_batch: X and the four per-problem outputs are required");
	if ((deriv_flags & PNOL_BFGS_ANALYTIC_GRADIENT) && !kt.gradient) {
		PNOL_SET_ERR(ctx, "functor kind %d has no analytic gradient: its functor defines no partial() (PNOL_BFGS_ANALYTIC_GRADIENT)", f->kind);
		return PNOL_ERR_NO_FUNCTOR;
	}
	if ((deriv_flags & PNOL_BFGS_ANALYTIC_SLOPE) && !kt.slope) {
		PNOL_SET_ERR(ctx, "functor kind %d has no analytic line-search slope: its functor defines no partial() (PNOL_BFGS_ANALYTIC_SLOPE)",
		             f->kind);
		return PNOL_ERR_NO_FUNCTOR;
	}
	if ((deriv_flags & PNOL_BFGS_ANALYTIC_HESSIAN) && prm->init_hess_fd && !kt.hessian) {
		PNOL_SET_ERR(ctx, "functor kind %d has no analytic Hessian: its functor defines no partial2() (PNOL_BFGS_ANALYTIC_HESSIAN)", f->kind);
		return PNOL_ERR_NO_FUNCTOR;
	}
	if (!kt.bfgs_batch) {
		PNOL_SET_ERR(ctx, "functor kind %d has no batched BFGS launcher (pnol_register_functor_bfgs_batch)", f->kind);
		return PNOL_ERR_NO_FUNCTOR;
	}

	TimerScope ts(ctx, "bfgs_batch");
	DevOut<double> dX, df0, dfopt;
	DevOut<int> dit, dstop;
	PNOL_CHECK(dX.init(ctx, X, (size_t) B * n, true));
	PNOL_CHECK(df0.init(ctx, f0_out, (size_t) B));
	PNOL_CHECK(dfopt.init(ctx, fopt_out, (size_t) B));
	PNOL_CHECK(dit.init(ctx, iters_out, (size_t) B));
	PNOL_CHECK(dstop.init(ctx, stop_out, (size_t) B));
	const pnol_launch_env env = make_env(ctx);
	PNOL_CHECK(kt.bfgs_batch(&env, &f->params, B, n, dX.get(), prm, deriv_flags, df0.get(), dfopt.get(), dit.get(), dstop.get()));
	PNOL_CHECK(dX.commit());
	PNOL_CHECK(df0.commit());
	PNOL_CHECK(dfopt.commit());
	PNOL_CHECK(dit.commit());
	PNOL_CHECK(dstop.commit());
	return finish(ctx);
}
