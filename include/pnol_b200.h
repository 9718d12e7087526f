/*
 * pnol_b200.h -- C-ABI of the B200-native (sm_100a) evaluation-and-derivative hot path of PNOL.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++ or torch types. The C++ plugin API of the
 * reference (include/pnol/PNOL_Objective.hpp, PNOL_Algorithm.hpp and the algorithm classes) is implemented
 * in host C++ ABOVE these entry points; the CUDA kernels live BELOW them in libpnol_b200.so.
 * There is no CPU fallback: every function that computes launches CUDA kernels on the context's device and
 * returns PNOL_ERR_CUDA if that is impossible.
 *
 * Conventions
 *   - every function returns an int status (PNOL_OK == 0); pnol_last_error() gives the text. Nothing calls
 *     exit() (the reference does: Source/GeneticAlgorithmMPI.cpp:40-44).
 *   - array arguments may be HOST or DEVICE pointers; the library detects which (cudaPointerGetAttributes)
 *     and stages host arrays through the context's stream. Scalar outputs (double*, int*) are host pointers.
 *   - matrices are dense row-major FP64; J is m x n (row = residual), JTJ/A/D are n x n.
 *   - one context drives one GPU; multi-GPU runs use one process (or thread) per GPU and a communicator
 *     attached with pnol_comm_init(). A context must not be used from two host threads at once.
 *   - reference citations are path:line under /root/reference/.
 *
 * Environment switches read by the library (tuning / A-B timing runs; the defaults are the product path). Read once per
 * process unless stated:
 *   PNOL_SYRK_NO_PAIR=1   J^T J with the stream-K TMA kernel instead of the CTA-pair kernel (n = 256, no F)
 *   PNOL_SYRK_LEGACY=1    J^T J with the LDGSTS-ring kernel (one tile role per CTA)
 *   PNOL_SYRK_WDIAG=w     cost of a diagonal tile's chunk in the stream-K work plan
 *   PNOL_SYRK_NOF=1       J^T J without J^T F (timing only: results lack the right-hand side)
 *   PNOL_SWEEP_DEEP=0     fitness sweep with one load ahead instead of four; PNOL_SWEEP_G / PNOL_SWEEP_WAVES: sweep tile shapes
 *   PNOL_COPY_THREADS=k   host threads of the staged pageable <-> device copies (1..8, default 4)
 *   PNOL_FUSED_MB=x       MB of J per row block of pnol_lm_normal_eq_fused / J == NULL steps (read per call, default 512)
 *   PNOL_GA_LEGACY=1      genetic algorithm with the stage-by-stage generation of round 1 instead of the fused pipeline
 *   PNOL_GA_SHARD=rows|sweep|none   overrides pnol_ga_set_sharding
 *   PNOL_GA_NO_IPC=1      several GPUs: population replicas + all-gather instead of peer mappings (A/B runs, boxes without IPC)
 *   PNOL_GA_SORT=radix    GA popSort with the cooperative radix kernel only (default: splitter buckets in front of it; read per pnol_ga_create)
 *   PNOL_LM_PEER=0        several GPUs: the LM step's two sums through NCCL instead of the fused peer-memory kernels (csrc/peer.cu)
 *   PNOL_LORENTZ_ROWWISE=0  trial residuals of the sum-of-Lorentzians model with the row-per-warp kernel (default: one row per thread)
 * and by the host classes (include/pnol/Runtime.hpp): PNOL_DEVICE, PNOL_POOL_WIDTH, PNOL_LM_JACOBIAN_CACHE.
 */
#ifndef PNOL_B200_H_
#define PNOL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pnol_ctx pnol_ctx;
typedef struct pnol_functor pnol_functor;
typedef struct pnol_ga pnol_ga;

enum {
	PNOL_OK = 0,
	PNOL_ERR_INVALID = 1,      /* bad argument */
	PNOL_ERR_CUDA = 2,         /* CUDA runtime error / no device */
	PNOL_ERR_NO_FUNCTOR = 3,   /* functor kind does not implement the requested operation */
	PNOL_ERR_NONFINITE = 4,    /* NaN/inf met where the reference would have printed and gone on */
	PNOL_ERR_NOT_SPD = 5,      /* damped normal matrix not positive definite */
	PNOL_ERR_COMM = 6,         /* NCCL error / communicator missing */
	PNOL_ERR_STREAM = 7        /* random stream exhausted */
};

/* ---------------------------------------------------------------------------------------------------
 * context
 * ------------------------------------------------------------------------------------------------- */
int pnol_ctx_create(pnol_ctx ** ctx, int device);
void pnol_ctx_destroy(pnol_ctx * ctx);
const char * pnol_last_error(pnol_ctx * ctx);
int pnol_ctx_device(pnol_ctx * ctx);
void * pnol_ctx_stream(pnol_ctx * ctx);            /* cudaStream_t all kernels of this context run on */
int pnol_ctx_sync(pnol_ctx * ctx);
int pnol_ctx_sm_count(pnol_ctx * ctx);
uint64_t pnol_ctx_launches(pnol_ctx * ctx);        /* number of kernels this context has launched */
const char * pnol_version(void);

/* device memory owned by the caller (cudaMallocAsync on the context's stream) */
int pnol_malloc(pnol_ctx * ctx, void ** dev_ptr, size_t bytes);
int pnol_free(pnol_ctx * ctx, void * dev_ptr);
int pnol_memcpy(pnol_ctx * ctx, void * dst, const void * src, size_t bytes);   /* any direction, stream ordered + sync */
int pnol_memset(pnol_ctx * ctx, void * dev_ptr, int value, size_t bytes);
/* A device -> host copy that runs BESIDE the work enqueued on the context's stream (copy streams of its own, driven by a worker
 * thread): findMin reads F0 back while the iterations already run. dev_src must be complete when the call is made (synchronise
 * first) and must not change, host_dst must not be touched, until pnol_copy_wait returns. One copy in flight per context (a second
 * start, pnol_memcpy and pnol_ctx_destroy wait for it); small or pinned destinations are copied at once. */
int pnol_copy_start(pnol_ctx * ctx, void * host_dst, const void * dev_src, size_t bytes);
int pnol_copy_wait(pnol_ctx * ctx);
int pnol_host_alloc(void ** host_ptr, size_t bytes);                          /* pinned host memory */
int pnol_host_free(void * host_ptr);

/* ---------------------------------------------------------------------------------------------------
 * multi-GPU communicator (NCCL; replaces the reference's MPI_COMM_WORLD collectives, SURVEY.md 2.4)
 * ------------------------------------------------------------------------------------------------- */
#define PNOL_COMM_ID_BYTES 128
int pnol_comm_unique_id(char id[PNOL_COMM_ID_BYTES]);                 /* rank 0 calls, launcher distributes */
int pnol_comm_init(pnol_ctx * ctx, const char id[PNOL_COMM_ID_BYTES], int nranks, int rank);
int pnol_comm_rank(pnol_ctx * ctx);                                   /* 0 when no communicator */
int pnol_comm_size(pnol_ctx * ctx);                                   /* 1 when no communicator */
/* local (non-collective) mode: while on, the context behaves like a single-GPU context -- no entry point issues a collective and
 * pnol_comm_rank / pnol_comm_size answer 0 / 1. The serial plugin classes (BFGS, BFGS_Bnd, LevMarq, GeneticAlgorithm, SimplexSearch,
 * Objective::gradientApproximation) run under it, as the reference's serial classes never touch MPI. Returns the previous setting. */
int pnol_comm_set_local(pnol_ctx * ctx, int on);
int pnol_comm_allreduce_sum(pnol_ctx * ctx, double * buf, size_t count);   /* in place, host or device buf */
int pnol_comm_allgather(pnol_ctx * ctx, const double * send, double * recv, size_t count_per_rank);
int pnol_comm_broadcast(pnol_ctx * ctx, double * buf, size_t count, int root);

/* ---------------------------------------------------------------------------------------------------
 * device functors: the device twin of a PNOL Objective / MultiObjective
 * (Source/PNOL_Objective.hpp:25-62; fixtures Source/ExampleObjectives.hpp)
 * ------------------------------------------------------------------------------------------------- */
enum {
	/* scalar objectives f(x) -> double                      (Objective::objEval, PNOL_Objective.hpp:29) */
	PNOL_F_ROSENBROCK = 1,      /* ExampleObjectives.hpp:87-103 */
	PNOL_F_POWER = 2,           /* ExampleObjectives.hpp:214-224; ints[0] = power (repeated multiplication) */
	PNOL_F_BOOTH = 3,           /* ExampleObjectives.hpp:58-69 */
	PNOL_F_GOLDSTEIN = 4,       /* ExampleObjectives.hpp:27-39 */
	PNOL_F_RASTRIGIN = 5,       /* ours (BASELINE.json config 4): 10 n + sum x^2 - 10 cos2pi(x), shared polynomial cos */
	PNOL_F_EXPCURVE_SINGLE = 6, /* ExampleObjectives.hpp:287-298 with pnol_exp; columns {x, y} */
	/* residual models F(x) -> R^m                            (MultiObjective::objEval, PNOL_Objective.hpp:57) */
	PNOL_F_EXPCURVE = 101,      /* ExampleObjectives.hpp:123-132 with pnol_exp; columns {x, y} */
	PNOL_F_CUBIC = 102,         /* ExampleObjectives.hpp:170-179; columns {x^3 (host libm pow), x, y} */
	PNOL_F_LORENTZ_SUM = 103    /* ours (configs 2 and 5): y - tree-sum_k a_k/(1 + w (t - c_k)^2); n = 2K, K a power
	                               of two; scalars[0] = w; columns {t, y} */
};

#define PNOL_MAX_SCALARS 8
#define PNOL_MAX_INTS 4
#define PNOL_MAX_COLUMNS 8

typedef struct {
	int kind;                                    /* PNOL_F_* */
	double scalars[PNOL_MAX_SCALARS];
	long long ints[PNOL_MAX_INTS];
	int n_columns;                               /* data columns, each of length m */
	const double * columns[PNOL_MAX_COLUMNS];    /* host pointers are copied to the device; device pointers are borrowed */
	long long m;                                 /* number of data rows held by THIS context (its shard) */
} pnol_functor_desc;

/* ---- open functor table: objectives that are not built in (Source/PNOL_Objective.hpp:29, :57 let a user plug in any objEval) ----
 * A user objective brings its own instantiations of the library's kernel templates (include/pnol/device/functor_kernels.cuh, compiled
 * out of tree by the user's nvcc) and registers their launchers under a kind of its choice:
 *     kinds [PNOL_F_USER_SCALAR_BASE, +1000)   scalar objectives  (eval_batch, fd_points, fd_hessian, alpha_pool)
 *     kinds [PNOL_F_USER_RESIDUAL_BASE, +1000) residual models    (residual, fd_jacobian)
 * pnol_functor_create and every entry point that takes a functor then work for that kind as for the built-ins; libpnol_b200.so is not
 * rebuilt. PNOL_REGISTER_SCALAR_FUNCTOR / PNOL_REGISTER_RESIDUAL_FUNCTOR in that header fill the table and call pnol_register_functor
 * at load time. INTEGRATION.md section A shows the whole recipe; tests/test_gpu_user_functor.py does it end to end. */
#define PNOL_F_USER_SCALAR_BASE 1000
#define PNOL_F_USER_RESIDUAL_BASE 2000
#define PNOL_FUNCTOR_ABI 1

/* parameters of a functor as the kernels see them (POD, passed by value as a kernel argument; pnol::FunctorParams) */
typedef struct pnol_functor_params {
	double scalars[PNOL_MAX_SCALARS];
	long long ints[PNOL_MAX_INTS];
	const double * col[PNOL_MAX_COLUMNS];        /* data columns (device pointers) */
	long long m;
} pnol_functor_params;

/* what a launcher needs from the calling context */
typedef struct pnol_launch_env {
	void * stream;                               /* cudaStream_t of the context: launch here */
	int sm_count;
	size_t smem_optin;                           /* opt-in shared memory per block */
	unsigned long long * launches;               /* ++ per kernel launch (pnol_ctx_launches) */
	char * err;                                  /* error text buffer (pnol_last_error) */
	size_t err_len;
} pnol_launch_env;

/* launch table of one functor kind; every pointer argument is a DEVICE pointer, every call only enqueues on env->stream */
typedef struct pnol_functor_vtable {
	int abi_version;                             /* PNOL_FUNCTOR_ABI */
	int n_columns;                               /* data columns the functor expects in pnol_functor_desc */
	int (*eval_batch)(const pnol_launch_env *, const pnol_functor_params *, const double * pts, long long B, int n, long long ld,
	                  const unsigned char * indicator, double * f_out);
	int (*fd_points)(const pnol_launch_env *, const pnol_functor_params *, const double * xfull, int nfull, const int * pos,
	                 const double * dx, int i0, int i1, double * fdx_out, double * f0_out);
	int (*fd_hessian)(const pnol_launch_env *, const pnol_functor_params *, const double * x, const double * dx, int n,
	                  const double * fdx, const double * f0, double * B);
	int (*alpha_pool)(const pnol_launch_env *, const pnol_functor_params *, const double * xfull, const double * pfull,
	                  const unsigned char * is_const, int nfull, const double * alpha, int npool, double dalpha,
	                  const unsigned char * eval_ind, int want_shifted, double * vals /* 2 * npool */);
	int (*residual)(const pnol_launch_env *, const pnol_functor_params *, const double * x, int n, double * F);
	int (*fd_jacobian)(const pnol_launch_env *, const pnol_functor_params *, const double * x, const double * dx, int n, double * J,
	                   double * F /* may be NULL */);
} pnol_functor_vtable;

/* registers (or replaces) the launch table of a user kind; the table must outlive its use. Thread-safe; callable before any context
 * exists (static initialisers). Returns PNOL_OK, or PNOL_ERR_INVALID for a kind outside the user ranges, a missing launcher or another ABI. */
int pnol_register_functor(int kind, const pnol_functor_vtable * vt);
int pnol_functor_registered(int kind);                     /* 1 for built-in and registered kinds */

int pnol_functor_create(pnol_ctx * ctx, const pnol_functor_desc * desc, pnol_functor ** out);
void pnol_functor_destroy(pnol_functor * f);
int pnol_functor_is_residual(const pnol_functor * f);     /* 1 for the built-in kinds >= 100 and the user residual range */
long long pnol_functor_rows(const pnol_functor * f);      /* m of a residual functor, 0 otherwise */

/* ---------------------------------------------------------------------------------------------------
 * a1 / a15: batched objective evaluation.  f_out[b] = f(pts[b*ld .. b*ld+n))  for rows with
 * indicator[b] != 0 (indicator == NULL: all rows). Rows that are skipped keep f_out[b].
 * Replaces GeneticAlgorithmMPI::evaluatePopulationParallel (Source/GeneticAlgorithmMPI.cpp:283-414) and
 * GeneticAlgorithm::evaluatePopulation (Source/GeneticAlgorithm.cpp:301-311).
 * ------------------------------------------------------------------------------------------------- */
int pnol_eval_batch(pnol_ctx * ctx, const pnol_functor * f, const double * pts, long long B, int n, long long ld,
                    const unsigned char * indicator, double * f_out);

/* ---------------------------------------------------------------------------------------------------
 * a3 / a4: forward-difference gradient  g[i] = (f(x + dx[i] e_i) - f(x)) / dx[i]
 * Replaces Objective::gradientApproximation[MPI] (Source/PNOL_Objective.cpp:12-34, 88-159).
 * With a communicator the coordinates are split by contiguous column blocks and all-gathered.
 * f0_out (optional) receives f(x).
 * ------------------------------------------------------------------------------------------------- */
int pnol_fd_gradient(pnol_ctx * ctx, const pnol_functor * f, const double * x, const double * dx, int n,
                     double * g_out, double * f0_out);

/* a5: active-set ("Recur") variants (Source/PNOL_Objective.cpp:303-333, 337-360, 366-459).
 * The full point has nfull entries: const_x[j] where const_ind[j] != 0, else the next entry of xr. */
int pnol_eval_recur(pnol_ctx * ctx, const pnol_functor * f, const double * xr, int nr, const double * const_x,
                    const unsigned char * const_ind, int nfull, double * f_out);
int pnol_fd_gradient_recur(pnol_ctx * ctx, const pnol_functor * f, const double * xr, const double * dxr, int nr,
                           const double * const_x, const unsigned char * const_ind, int nfull, double * g_out,
                           double * f0_out);

/* a6: forward-difference Hessian, upper triangle computed and mirrored
 * (Objective::hessianApproximation, Source/PNOL_Objective.cpp:38-85). B_out is n x n. */
int pnol_fd_hessian(pnol_ctx * ctx, const pnol_functor * f, const double * x, const double * dx, int n, double * B_out);

/* a13: alpha-pool evaluation for the pooled line searches. For k < npool with eval_ind[k] != 0
 * (eval_ind == NULL: all):  phi[k] = f(x + alpha[k] p)  and, when dphi != NULL,
 * dphi[k] = (f(x + (alpha[k] + dalpha) p) - phi[k]) / dalpha.  NaN/inf values of phi are replaced by the 1e10
 * sentinel (the slope is computed from the raw phi and left as is) and *bad_out is set to the number of sentinels (Source/BFGS_bnd_linesearch_MPI_SW.cpp:599-699,
 * 703-734; Source/BFGS_with_linesearch_MPI.cpp:163-223). const_x/const_ind may be NULL (no active set). */
int pnol_alpha_pool(pnol_ctx * ctx, const pnol_functor * f, const double * x, const double * p, int n,
                    const double * alpha, int npool, double dalpha, const unsigned char * eval_ind,
                    const double * const_x, const unsigned char * const_ind, int nfull,
                    double * phi, double * dphi, int * bad_out);

/* ---------------------------------------------------------------------------------------------------
 * a2 / a10: residual evaluation F = F(x) over this context's rows; sumsq_out (optional) receives the
 * sequentially-ordered-per-block sum of F^2 over ALL ranks (MultiObjective::objEval + vector2Norm^2,
 * Source/LevenbergMarquardtMPI.cpp:103-108). F is required (host or device, m doubles).
 * ------------------------------------------------------------------------------------------------- */
int pnol_residual_eval(pnol_ctx * ctx, const pnol_functor * f, const double * x, int n, double * F, double * sumsq_out);

/* a7 / a8: forward-difference Jacobian J[i][j] = (F_i(x + dx[j] e_j) - F_i(x)) / dx[j], J is m x n row-major,
 * F (optional) receives F(x). Replaces MultiObjective::gradientApproximation[MPI]
 * (Source/PNOL_Objective.cpp:165-197, 202-299). mode: PNOL_JAC_AUTO picks the structured kernel when the
 * functor has one; PNOL_JAC_BLACKBOX forces n+1 full model evaluations per row. Results are bit-identical. */
enum { PNOL_JAC_AUTO = 0, PNOL_JAC_BLACKBOX = 1, PNOL_JAC_STRUCTURED = 2 };
int pnol_fd_jacobian(pnol_ctx * ctx, const pnol_functor * f, const double * x, const double * dx, int n,
                     double * J, double * F, int mode);

/* a9: Levenberg-Marquardt normal equations (Source/LevenbergMarquardtMPI.cpp:64-88):
 *   JTJ = J^T J (FP64 tensor-core DMMA, lower triangle computed and mirrored), A = JTJ with
 *   A_ii = (1 + lambda) JTJ_ii, rhs = -J^T F. With a communicator J/F are this rank's row block and
 *   JTJ/rhs are all-reduced (packed, one collective). Any of JTJ, A, rhs may be NULL.
 *   m is the LOCAL row count. */
int pnol_lm_normal_eq(pnol_ctx * ctx, const double * J, const double * F, long long m, int n, double lambda,
                      double * JTJ, double * A, double * rhs);
/* re-damp only: A = JTJ with A_ii = (1 + lambda) JTJ_ii (J unchanged after a rejected step) */
int pnol_lm_damp(pnol_ctx * ctx, const double * JTJ, int n, double lambda, double * A);

/* One LM iteration's device work behind one call and ONE host synchronisation (Source/LevenbergMarquardtMPI.cpp:60-108):
 * FD Jacobian at x -> J^T J | J^T F (+ all-reduce over the ranks) -> Marquardt damping -> Cholesky solve -> x_trial = x + sigma ->
 * Ftrial = F(x_trial) and its sum of squares (+ all-reduce). The accept / reject decision stays with the caller as in the reference.
 *   x, dx       host or device, n
 *   J           device, m x n work space (m = rows of the functor), or NULL: the normal equations are then summed over row blocks
 *               and J is never stored (see pnol_lm_normal_eq_fused); F device: residuals at x; Ftrial device: receives F(x_trial)
 *   JTJ         device, n*n + n doubles: receives J^T J followed by -J^T F. reuse_jtj != 0: J^T J / rhs are taken from it instead of
 *               being recomputed (x unchanged after a rejected step), only the damping is redone with the new lambda
 *   sigma_out, x_trial_out (host, n), sumsq_trial_out, spd_info_out (host): the step, the trial point, sum Ftrial^2 over all
 *               ranks and the Cholesky status (k > 0: pivot k rejected, see pnol_spd_solve; the step is then NaN, which the caller's
 *               chi^2 test rejects). n <= 704 (the solve's range) */
int pnol_lm_step(pnol_ctx * ctx, const pnol_functor * f, const double * x, const double * dx, int n, double * J, const double * F,
                 double * Ftrial, double lambda, int jac_mode, int reuse_jtj, double * JTJ, double * sigma_out, double * x_trial_out,
                 double * sumsq_trial_out, int * spd_info_out);

/* `iterations` LM iterations on device-resident state (J, F, Ftrial, JTJ as in pnol_lm_step) with the accept / reject decision of
 * Source/LevenbergMarquardtMPI.cpp:107-141 taken ON THE DEVICE by two small kernels behind every step, so that the host enqueues a
 * batch of iterations per synchronisation (all of them without a stopping rule, four at a time with one): chi^2 =
 * pow(sqrt(sum Ftrial^2), 2); chi^2 >= previous or NaN -> lambda *= factor, x and F stay; otherwise lambda /= factor, x = x_trial,
 * F = Ftrial (copied) and, with x_min_diff > 0, no further change once ||sigma||_2 < x_min_diff (:138-140). The arithmetic is the
 * host rule's (IEEE square root, sequential sum), so pnol_lm_step + the rule on the host gives the same bits. The Jacobian is
 * recomputed in every iteration as in the reference (:60).
 *   x (host, n) in/out; lambda_inout, chisq_inout in/out; swapped_out: always 0 (kept for callers written against the pointer-
 *   swapping host rule: the current residuals are in `F`) */
int pnol_lm_iterate(pnol_ctx * ctx, const pnol_functor * f, double * x, const double * dx, int n, double * J, double * F, double * Ftrial,
                    double * JTJ, double * lambda_inout, double * chisq_inout, double lambda_factor, double x_min_diff, int iterations,
                    int jac_mode, int * accepted_out, int * rejected_out, int * swapped_out);

/* Which way the sums of the row-sharded LM step (J^T J | J^T F and the trial chi^2, Source/LevenbergMarquardtMPI.cpp:60-108) travel on
 * this context: 0 one rank, 1 NVLink peer memory inside the step's own kernels (csrc/peer.cu), 2 NCCL all-reduce (a peer mapping
 * failed, or PNOL_LM_PEER=0), -1 not decided yet (the first sharded pnol_lm_step / pnol_lm_iterate decides, collectively). */
int pnol_lm_exchange_mode(pnol_ctx * ctx);

/* What the last pnol_lm_iterate of this context ended with: *stopped_out != 0 when the stopping rule ||sigma||_2 < x_min_diff fired
 * (Source/LevenbergMarquardtMPI.cpp:138-140 -- the reference leaves its loop there WITHOUT counting that pass in `iter`, so its
 * iteration count is accepted + rejected - 1 in that case), *xdiff_out = ||sigma||_2 of the last accepted step (0 when none was). */
int pnol_lm_last_run(pnol_ctx * ctx, int * stopped_out, double * xdiff_out);

/* SURVEY.md 8(f) item 2 -- the normal equations without J in HBM: the rows are walked in blocks (512 MB of J per block by default,
 * $PNOL_FUSED_MB), each block's Jacobian is written to a scratch buffer, read back by the SYRK and its J^T J | J^T F added to the
 * running sum in row order (deterministic; equal to pnol_fd_jacobian + pnol_lm_normal_eq up to summation order). Work space 512 MB
 * instead of m*n*8 bytes: the memory-footprint mode (9 % slower than the stored-J path at m = 4M, n = 256; both are FP64-bound). Any
 * residual functor (structured or black-box Jacobian). F (optional, host or device, m doubles) receives the residuals at x;
 * JTJ / A / rhs as in pnol_lm_normal_eq. Replaces Source/LevenbergMarquardtMPI.cpp:60-85 in one call. pnol_lm_step / pnol_lm_iterate
 * take the same path when their J argument is NULL. */
int pnol_lm_normal_eq_fused(pnol_ctx * ctx, const pnol_functor * f, const double * x, const double * dx, int n,
                            double lambda, double * JTJ, double * A, double * rhs, double * F);

/* a9: damped solve  A sigma = rhs  by Cholesky, 1 <= n <= 704 (PNOL_ERR_INVALID otherwise). A is symmetric positive definite;
 * only its lower triangle (diagonal included) is read, the strict upper triangle may hold anything, NaN included. Every pivot
 * (the Schur complement's diagonal entry d_k when column k is eliminated) must lie in [2^-1022, 2^1000): zero, negative, subnormal,
 * too large or NaN pivots are rejected. On success *info = 0 and x = sigma. On a rejected pivot the call returns PNOL_ERR_NOT_SPD
 * with *info = k > 0, the 1-based index of the first rejected pivot (named in pnol_last_error), and every entry of x is NaN.
 * Replaces luSolve (Source/LevenbergMarquardtMPI.cpp:88). */
int pnol_spd_solve(pnol_ctx * ctx, const double * A, const double * rhs, int n, double * x, int * info);

/* General inverse Ainv = A^-1 by LU with partial pivoting (first largest |entry| on ties) and one pair of substitutions per unit
 * vector: `matrixInverse` of the forward-difference Hessian when initHessFD is set (Source/BFGS_bnd_linesearch_MPI_SW.cpp:51-59,
 * Source/BFGS_with_linesearch.cpp:35-41). An indefinite A is inverted like any other, as the reference does; *info = k + 1 when
 * pivot k is exactly zero (the entries are then inf / NaN, as the reference's would be), else 0. Operation for operation the
 * oracle/shim definition of matrixInverse (the reference takes it from an un-vendored library), so results agree bit for bit. */
int pnol_lu_inverse(pnol_ctx * ctx, const double * A, int n, double * Ainv, int * info);

/* ---------------------------------------------------------------------------------------------------
 * a11 / a12: dense BFGS pieces
 * ------------------------------------------------------------------------------------------------- */
/* p = -D g   (Source/BFGS_bnd_linesearch_MPI_SW.cpp:143-144; BFGS_with_linesearch.cpp:78-79) */
int pnol_matvec_neg(pnol_ctx * ctx, const double * D, const double * g, int n, double * p);

/* updateHessianInv(D, g, s) (Source/BFGS_with_linesearch.cpp:389-432), D updated in place.
 *   PNOL_HINV_LITERAL: forms M1 = I - rho s g^T, M2 = I - rho g s^T and computes (M1 D) M2 + rho s s^T with two
 *                      n^3 DMMA GEMMs, as the reference does;
 *   PNOL_HINV_RANK2:   the algebraically equal O(n^2) update D - rho s (g^T D) - rho (D g) s^T
 *                      + (rho^2 g^T D g + rho) s s^T (HBM-bound). */
enum { PNOL_HINV_LITERAL = 0, PNOL_HINV_RANK2 = 1 };
int pnol_bfgs_update_hinv(pnol_ctx * ctx, double * D, const double * g, const double * s, int n, int mode);

/* general FP64 DMMA GEMM C = A B (all n x n row-major); exported because the literal update is built on it */
int pnol_dgemm_nn(pnol_ctx * ctx, const double * A, const double * B, double * C, int M, int N, int K);

/* ---------------------------------------------------------------------------------------------------
 * a14: box-bound helpers (host arithmetic, O(n); exported so bindings need not re-implement them)
 * (Source/Box_boundary_functions.cpp:11-40; Source/BFGS_with_bnd_linsearch_MPI.cpp:665-708)
 * ------------------------------------------------------------------------------------------------- */
int pnol_check_box_bounds(double * x, const double * xlb, const double * xub, int n, int * n_replaced);
double pnol_compute_alpha_bnd(const double * x, const double * xlb, const double * xub, const double * p, int n);

/* ---------------------------------------------------------------------------------------------------
 * random stream: "host-supplied" uniform stream u_0, u_1, ... consumed in the reference's sequential order
 * (every timeRand() call of Source/GeneticAlgorithmMPI.cpp / GeneticAlgorithm.cpp:313-365).
 * Either an explicit array, or the counter-based generator below (same values on host and device).
 * ------------------------------------------------------------------------------------------------- */
typedef struct {
	const double * values;      /* explicit stream (host pointer) or NULL */
	uint64_t n_values;
	uint64_t seed;              /* counter mode: u_k = pnol_stream_uniform(seed, k, scale) */
	double scale;               /* counter mode: values lie in [0, scale); use scale <= 1 - 0.5/Npop */
} pnol_stream_desc;
double pnol_stream_uniform(uint64_t seed, uint64_t k, double scale);

/* ---------------------------------------------------------------------------------------------------
 * a15 / a16: genetic algorithm state machine (Source/GeneticAlgorithmMPI.cpp:12-276)
 * ------------------------------------------------------------------------------------------------- */
typedef struct {
	int npop;
	int max_generations;
	double elite_frac, cross_frac, elite_mutation_frac;
	double mutation_size, elite_mutation_size;
	double n_static_generations;
} pnol_ga_params;

typedef struct {
	int generation;             /* generations completed */
	int n_static;
	int stopped;                /* 1 once the static-generation test fired */
	double f_best;
	uint64_t stream_pos;        /* draws consumed so far */
	int n_elite, n_elite_mut, n_cross, n_rand;
} pnol_ga_status;

int pnol_ga_create(pnol_ctx * ctx, const pnol_functor * f, const pnol_ga_params * params, int n,
                   const double * xlb, const double * xub, const pnol_stream_desc * stream, pnol_ga ** out);
void pnol_ga_destroy(pnol_ga * ga);
/* initial population, repair, evaluation and sort (GeneticAlgorithmMPI.cpp:55-81); f0_out = F of the start point */
int pnol_ga_init(pnol_ga * ga, const double * x0, double * f0_out);
/* one generation (GeneticAlgorithmMPI.cpp:87-249) */
int pnol_ga_generation(pnol_ga * ga);
int pnol_ga_status_get(pnol_ga * ga, pnol_ga_status * st);
/* How pnol_ga_create splits a generation over the ranks of the context's communicator (set before pnol_ga_create):
 *   PNOL_GA_SHARD_ROWS   rank r owns child rows [r per, (r+1) per): it creates, repairs and evaluates them; parents are read from
 *                        their owners over NVLink (CUDA IPC peer mappings; replicas refreshed by an all-gather when those are
 *                        unavailable); row hashes / box counts and objective values are all-gathered. Memory per GPU ~ 1 / ranks.
 *   PNOL_GA_SHARD_SWEEP  every rank keeps the population and makes all children; the fitness sweep is split and the objective values
 *                        are all-gathered (the reference's evaluatePopulationParallel, Source/GeneticAlgorithmMPI.cpp:283-414).
 *   PNOL_GA_SHARD_NONE   replicas: every rank keeps the population, makes all children and sweeps all of them -- no collective. For a
 *                        cheap objective the split sweep does not pay for its all-gather (1M x 32 Rastrigin: the whole sweep 0.057 ms,
 *                        the all-gather of the 8 MB of objective values 0.06 - 0.17 ms at 2 - 8 GPUs).
 *   PNOL_GA_SHARD_AUTO   (default) rows when the population does not fit one GPU comfortably; otherwise sweep when the share of the
 *                        sweep the other ranks take over costs more than the all-gather (always for user functors), else none.
 * Results are bit-identical in every mode and at every rank count. */
enum { PNOL_GA_SHARD_AUTO = 0, PNOL_GA_SHARD_ROWS = 1, PNOL_GA_SHARD_SWEEP = 2, PNOL_GA_SHARD_NONE = 3 };
int pnol_ga_set_sharding(pnol_ctx * ctx, int mode);
/* what a GA object does: 0 one rank (or the stage-by-stage generation), 1 rows sharded + peer mappings, 2 rows sharded + replicas
 * (peer mappings unavailable, or PNOL_GA_NO_IPC=1), 3 rows replicated + sweep sharded, 4 replicas (no collective) */
int pnol_ga_peer_mode(pnol_ga * ga);
/* sorted population (npop x n) and objective values; either may be NULL */
int pnol_ga_get_population(pnol_ga * ga, double * xpop, double * F);
/* parent indices chosen in the last generation: crossover (n_cross x n), mutation (n_rand), elite mutation
 * (n_elite_mut x n); any may be NULL. These are the "selection/crossover indices" of the parity bar. */
int pnol_ga_get_indices(pnol_ga * ga, int * cross_idx, int * mut_idx, int * elite_idx);

/* stand-alone GA stages on caller data (per-stage parity at full size) */
int pnol_ga_pop_sort(pnol_ctx * ctx, double * xpop, double * F, long long npop, int n);             /* GeneticAlgorithm.cpp:370-412 */
int pnol_ga_check_bounds(pnol_ctx * ctx, double * xpop, long long npop, int n, const double * xlb, const double * xub,
                         unsigned char * indicator, const pnol_stream_desc * stream, uint64_t * stream_pos); /* :347-365 */
int pnol_ga_check_identical(pnol_ctx * ctx, double * xpop, long long npop, int n, const double * xlb, const double * xub,
                            unsigned char * indicator, const pnol_stream_desc * stream, uint64_t * stream_pos); /* :313-344 */

/* ---------------------------------------------------------------------------------------------------
 * measurement helpers
 * ------------------------------------------------------------------------------------------------- */
/* register-resident FP64 DMMA microbenchmark: returns achieved TFLOP/s (the tensor roofline denominator) */
int pnol_measure_dmma_peak(pnol_ctx * ctx, double * tflops_out);
/* device-to-device copy bandwidth, GB/s (read + write bytes) */
int pnol_measure_copy_bandwidth(pnol_ctx * ctx, double * gbs_out);
/* per-kernel timing of the last call of a timed entry point (ms), name -> value; see DESIGN.md.
 * on: 0 off, 1 every scope, 2 only the kernels that carry an LM iteration ("syrk", "fd_jacobian", "residual": an event pair costs
 * about 5 us of stream time, which shows in a 1.5 ms iteration at 8 GPUs) */
int pnol_timer_enable(pnol_ctx * ctx, int on);
int pnol_timer_get(pnol_ctx * ctx, const char * name, double * total_ms, long long * count);
int pnol_timer_reset(pnol_ctx * ctx);
/* self test: number of (x, d) pairs out of `pairs` pseudo-random / adversarial ones for which the reciprocal-based
 * exact division of the Jacobian kernels (csrc/exact_div.cuh) differs from x / d. Must return 0 mismatches. */
/* host-only self-test of the J^T J kernel's stream-K work plan for m x n on sm_count CTAs (with_f: J^T F summed as well): 0 when
 * every K chunk of every tile role is covered exactly once, in order, with contiguous slots per role, at most 8 segments per CTA and
 * CTA shares within one chunk of the mean; otherwise the number of the violated rule. Needs no device. */
int pnol_selftest_syrk_plan(long long m, int n, int sm_count, int with_f);
int pnol_selftest_exact_div(pnol_ctx * ctx, long long pairs, unsigned long long seed, unsigned long long * mismatches);
/* the same for the branch-free cores the speculative row kernels use (div_core, div_exact_core), over their validity range */
int pnol_selftest_fast_div(pnol_ctx * ctx, long long pairs, unsigned long long seed, unsigned long long * mismatches);

#ifdef __cplusplus
}
#endif
#endif /* PNOL_B200_H_ */
