// eval_kernels.cu -- scalar-objective launchers: population / batch sweep, forward-difference point evaluation (gradient, Recur
// gradient, Hessian), the analytic gradient and Hessian, and the alpha-pool evaluation of the pooled line searches (forward-difference
// or analytic slopes).
//
// The kernels themselves are templates over the device functor in include/pnol/device/functor_kernels.cuh -- the SAME templates an
// out-of-tree objective instantiates (open functor table, pnol_register_functor). Every launcher here calls the record of the functor's
// kind (kind_table): builtin_functors.cu instantiates the templates for the built-in objectives, a user kind brings its own.
//
// Mapping (north_star): one evaluation point per THREAD, the shared base point staged in shared memory;
// population tiles are read from HBM with coalesced 16-byte loads and parked in shared memory with an odd row
// pitch so that thread r walking row r is bank-conflict free. Functor code is compiled with -fmad=false.
#include "common.cuh"

namespace pnol {

// a1 / a15: batch sweep. Replaces GeneticAlgorithmMPI::evaluatePopulationParallel (Source/GeneticAlgorithmMPI.cpp:283-414)
int launch_eval_batch(pnol_ctx * ctx, const pnol_functor * f, const double * pts, long long B, int n, long long ld,
                      const unsigned char * indicator, double * f_out)
{
	if (B <= 0) return PNOL_OK;
	TimerScope ts(ctx, "eval_batch");
	KindTable kt;
	if (!kind_table(f->kind, &kt) || !kt.vt.eval_batch) return wrong_family(ctx, f->kind, "scalar objective");
	const pnol_launch_env env = make_env(ctx);
	return kt.vt.eval_batch(&env, &f->params, pts, B, n, ld, indicator, f_out);
}

// a3 / a4 / a5: forward-difference stencil points (Source/PNOL_Objective.cpp:19-32, 125-145; Recur: :345-358, :399-420)
int launch_fd_points(pnol_ctx * ctx, const pnol_functor * f, const double * xfull, int nfull, const int * pos,
                     const double * dx, int i0, int i1, double * fdx_out, double * f0_out)
{
	TimerScope ts(ctx, "fd_points");
	KindTable kt;
	if (!kind_table(f->kind, &kt) || !kt.vt.fd_points) return wrong_family(ctx, f->kind, "scalar objective");
	const pnol_launch_env env = make_env(ctx);
	return kt.vt.fd_points(&env, &f->params, xfull, nfull, pos, dx, i0, i1, fdx_out, f0_out);
}

// a3 / a4 / a5, analytic: the functor's partial derivatives, one coordinate per thread (pnol_gradient[_recur])
int launch_gradient(pnol_ctx * ctx, const pnol_functor * f, const double * xfull, int nfull, const int * pos, int i0, int i1,
                    double * g_out, double * f0_out)
{
	TimerScope ts(ctx, "gradient");
	KindTable kt;
	if (!kind_table(f->kind, &kt) || !kt.vt.fd_points) return wrong_family(ctx, f->kind, "scalar objective");
	if (!kt.gradient) {
		PNOL_SET_ERR(ctx, "functor kind %d has no analytic gradient: its functor defines no partial() (pnol_register_functor_gradient)", f->kind);
		return PNOL_ERR_NO_FUNCTOR;
	}
	const pnol_launch_env env = make_env(ctx);
	return kt.gradient(&env, &f->params, xfull, nfull, pos, i0, i1, g_out, f0_out);
}

// g[i] = (fdx[i] - f0) / dx[i]     (Source/PNOL_Objective.cpp:31, :150-153, :451-454)
__global__ void fd_quotient_kernel(const double * __restrict__ fdx, const double * __restrict__ f0,
                                   const double * __restrict__ dx, int n, double * __restrict__ g)
{
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n) g[i] = (fdx[i] - *f0) / dx[i];
}

int launch_fd_quotient(pnol_ctx * ctx, const double * fdx, const double * f0, const double * dx, int n, double * g)
{
	if (n <= 0) return PNOL_OK;
	PNOL_LAUNCH(ctx, fd_quotient_kernel, (n + 255) / 256, 256, 0, fdx, f0, dx, n, g);
	return PNOL_OK;
}

// Active-set assembly (Objective::objEvalRecur, Source/PNOL_Objective.cpp:303-323): the full point takes
// const_x[j] where const_ind[j], else the next reduced variable. Also emits pos[i] (full index of reduced
// variable i; the caller presets pos to -1, which stays for reduced entries beyond the number of free variables). Single block; a serial scan over chunks of blockDim entries.
__global__ void assemble_recur_kernel(const double * __restrict__ xr, int nr,
                                      const double * __restrict__ const_x, const unsigned char * __restrict__ const_ind,
                                      int nfull, double * __restrict__ xfull, int * __restrict__ pos,
                                      int * __restrict__ nr_found)
{
	__shared__ int warp_tot[32];
	__shared__ int base;
	if (threadIdx.x == 0) base = 0;
	__syncthreads();
	const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
	for (int j0 = 0; j0 < nfull; j0 += blockDim.x) {
		int j = j0 + threadIdx.x;
		int freev = (j < nfull && !(const_ind && const_ind[j])) ? 1 : 0;
		int incl = freev;
		for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
		if (lane == 31) warp_tot[wid] = incl;
		__syncthreads();
		int woff = 0;
		for (int w = 0; w < wid; w++) woff += warp_tot[w];
		int tot = 0;
		for (int w = 0; w < nw; w++) tot += warp_tot[w];
		int idx = base + woff + incl - freev;   // exclusive rank among free variables
		if (j < nfull) {
			if (freev) {
				double v = idx < nr ? xr[idx] : 0.0;
				xfull[j] = v;
				if (idx < nr && pos) pos[idx] = j;
			} else {
				xfull[j] = const_x[j];
			}
		}
		__syncthreads();
		if (threadIdx.x == 0) base += tot;
		__syncthreads();
	}
	if (threadIdx.x == 0 && nr_found) *nr_found = base;
}

int launch_assemble_recur(pnol_ctx * ctx, const double * xr, int nr, const double * const_x,
                          const unsigned char * const_ind, int nfull, double * xfull, int * pos, int * nr_found)
{
	PNOL_LAUNCH(ctx, assemble_recur_kernel, 1, 256, 0, xr, nr, const_x, const_ind, nfull, xfull, pos, nr_found);
	return PNOL_OK;
}

// a6: forward-difference Hessian (Objective::hessianApproximation, Source/PNOL_Objective.cpp:38-85)
int launch_fd_hessian(pnol_ctx * ctx, const pnol_functor * f, const double * x, const double * dx, int n,
                      const double * fdx, const double * f0, double * B)
{
	TimerScope ts(ctx, "fd_hessian");
	KindTable kt;
	if (!kind_table(f->kind, &kt) || !kt.vt.fd_hessian) return wrong_family(ctx, f->kind, "scalar objective");
	const pnol_launch_env env = make_env(ctx);
	return kt.vt.fd_hessian(&env, &f->params, x, dx, n, fdx, f0, B);
}

// a6, analytic: the functor's second derivatives, one 32 x 32 tile of the upper triangle at a time, mirrored (pnol_hessian)
int launch_hessian(pnol_ctx * ctx, const pnol_functor * f, const double * x, int n, double * H)
{
	TimerScope ts(ctx, "hessian");
	KindTable kt;
	if (!kind_table(f->kind, &kt) || !kt.vt.fd_hessian) return wrong_family(ctx, f->kind, "scalar objective");
	if (!kt.hessian) {
		PNOL_SET_ERR(ctx, "functor kind %d has no analytic Hessian: its functor defines no partial2() (pnol_register_functor_hessian)", f->kind);
		return PNOL_ERR_NO_FUNCTOR;
	}
	const pnol_launch_env env = make_env(ctx);
	return kt.hessian(&env, &f->params, x, n, H);
}

// a13: alpha pool: phi, the forward-difference slope and the NaN/inf -> 1e10 sentinel of evaluateAlphaPoolAndDerivatives
// (Source/BFGS_bnd_linesearch_MPI_SW.cpp:657-668) from the raw values the functor's kernel produced
__global__ void alpha_pool_finish_kernel(const double * __restrict__ vals, int npool, double dalpha,
                                         const unsigned char * __restrict__ eval_ind, bool want_dphi,
                                         double * __restrict__ phi, double * __restrict__ dphi, int * __restrict__ bad)
{
	int k = blockIdx.x * blockDim.x + threadIdx.x;
	if (k >= npool) return;
	if (eval_ind && !eval_ind[k]) return;
	double ph = vals[k];
	int nbad = 0;
	if (want_dphi) dphi[k] = (vals[npool + k] - ph) / dalpha;   // slope keeps NaN/inf: the reference only guards phi
	if (ph != ph || isinf(ph)) { ph = 1e10; nbad++; }
	phi[k] = ph;
	if (nbad) atomicAdd(bad, nbad);
}

int launch_alpha_pool(pnol_ctx * ctx, const pnol_functor * f, const double * xfull, const double * pfull,
                      const unsigned char * is_const, int nfull, const double * alpha, int npool, double dalpha,
                      const unsigned char * eval_ind, double * phi, double * dphi, int * bad_dev)
{
	TimerScope ts(ctx, "alpha_pool");
	PNOL_CHECK(ws_reserve(ctx, 3, (size_t) 2 * npool * sizeof(double)));
	double * vals = (double *) ctx->ws[3];
	KindTable kt;
	if (!kind_table(f->kind, &kt) || !kt.vt.alpha_pool) return wrong_family(ctx, f->kind, "scalar objective");
	const pnol_launch_env env = make_env(ctx);
	PNOL_CHECK(kt.vt.alpha_pool(&env, &f->params, xfull, pfull, is_const, nfull, alpha, npool, dalpha, eval_ind, dphi != nullptr, vals));
	PNOL_LAUNCH(ctx, alpha_pool_finish_kernel, (npool + 63) / 64, 64, 0, vals, npool, dalpha, eval_ind, dphi != nullptr, phi, dphi, bad_dev);
	return PNOL_OK;
}

// a13, analytic slope: the sentinel on phi only, the slope copied raw (as alpha_pool_finish_kernel leaves the forward difference raw).
// A kernel of its own so that alpha_pool_finish_kernel's code stays as it is.
__global__ void alpha_slope_finish_kernel(const double * __restrict__ vals, int npool, const unsigned char * __restrict__ eval_ind,
                                          double * __restrict__ phi, double * __restrict__ dphi, int * __restrict__ bad)
{
	int k = blockIdx.x * blockDim.x + threadIdx.x;
	if (k >= npool) return;
	if (eval_ind && !eval_ind[k]) return;
	double ph = vals[k];
	dphi[k] = vals[npool + k];
	if (ph != ph || isinf(ph)) { ph = 1e10; atomicAdd(bad, 1); }
	phi[k] = ph;
}

// a13, analytic slope: phi and sum_r p_r df/dx_{pos[r]} at each trial point, one block per pool entry (pnol_alpha_pool_analytic)
int launch_alpha_slope(pnol_ctx * ctx, const pnol_functor * f, const double * xfull, const double * pfull,
                       const unsigned char * is_const, int nfull, const int * pos, const double * p, int n, const double * alpha,
                       int npool, const unsigned char * eval_ind, double * phi, double * dphi, int * bad_dev)
{
	TimerScope ts(ctx, "alpha_slope");
	PNOL_CHECK(ws_reserve(ctx, 3, (size_t) 2 * npool * sizeof(double)));
	double * vals = (double *) ctx->ws[3];
	KindTable kt;
	if (!kind_table(f->kind, &kt) || !kt.vt.alpha_pool) return wrong_family(ctx, f->kind, "scalar objective");
	if (!kt.slope) {
		PNOL_SET_ERR(ctx, "functor kind %d has no analytic line-search slope: its functor defines no partial() (pnol_register_functor_slope)", f->kind);
		return PNOL_ERR_NO_FUNCTOR;
	}
	const pnol_launch_env env = make_env(ctx);
	PNOL_CHECK(kt.slope(&env, &f->params, xfull, pfull, is_const, nfull, pos, p, n, alpha, npool, eval_ind, vals));
	PNOL_LAUNCH(ctx, alpha_slope_finish_kernel, (npool + 63) / 64, 64, 0, vals, npool, eval_ind, phi, dphi, bad_dev);
	return PNOL_OK;
}

} // namespace pnol
