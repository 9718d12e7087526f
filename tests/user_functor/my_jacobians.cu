/* Residual models with analytic Jacobians, compiled out of tree like my_objectives.cu (tests/user_jacobian_lib.py):
 *   nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -Xcompiler -fPIC,-ffp-contract=off -I<repo>/include -shared \
 *        -o libmy_jacobians.so my_jacobians.cu -L<repo>/parallelnonlinearoptimizationlibrary_b200/lib -lpnol_b200 -lpnol_b200_host
 * PNOL_REGISTER_RESIDUAL_FUNCTOR fills the table's `jacobian` launcher for a functor that defines jacobian(), and leaves it NULL for
 * one that does not. One more table is written out by hand in the version-1 layout (without `jacobian`). */
#include "my_jacobians.hpp"

#include "pnol/device/functor_kernels.cuh"

PNOL_REGISTER_RESIDUAL_FUNCTOR(MYJ_F_LORENTZ, MyLorentzFunctor, 2)
PNOL_REGISTER_RESIDUAL_FUNCTOR(MYJ_F_GAUSS, MyGaussFunctor, 2)
PNOL_REGISTER_RESIDUAL_FUNCTOR(MYJ_F_GAUSS_NOJAC, MyGaussNoJacFunctor, 2)

/* the version-1 layout of pnol_functor_vtable: the table as a library built against ABI 1 lays it out */
struct my_vtable_v1 {
	int abi_version;
	int n_columns;
	int (*eval_batch)(const pnol_launch_env *, const pnol_functor_params *, const double *, long long, int, long long, const unsigned char *,
	                  double *);
	int (*fd_points)(const pnol_launch_env *, const pnol_functor_params *, const double *, int, const int *, const double *, int, int, double *,
	                 double *);
	int (*fd_hessian)(const pnol_launch_env *, const pnol_functor_params *, const double *, const double *, int, const double *, const double *,
	                  double *);
	int (*alpha_pool)(const pnol_launch_env *, const pnol_functor_params *, const double *, const double *, const unsigned char *, int,
	                  const double *, int, double, const unsigned char *, int, double *);
	int (*residual)(const pnol_launch_env *, const pnol_functor_params *, const double *, int, double *);
	int (*fd_jacobian)(const pnol_launch_env *, const pnol_functor_params *, const double *, const double *, int, double *, double *);
};

/* What follows the version-1 table in memory: a word where a version-2 table has `jacobian`. The library must not read it; if it
 * ever called it, the call would fail with this text instead of computing anything. */
static int my_not_a_launcher(const pnol_launch_env * env, const pnol_functor_params *, const double *, int, double *, double *)
{
	PNOL_DEV_ERR(env, "the word behind a version-1 table was called as a jacobian launcher");
	return PNOL_ERR_CUDA;
}
struct MyV1Block {
	my_vtable_v1 vt;
	int (*behind)(const pnol_launch_env *, const pnol_functor_params *, const double *, int, double *, double *);
};
static MyV1Block make_v1_block()
{
	MyV1Block b;
	memset(&b, 0, sizeof b);
	b.vt.abi_version = 1;
	b.vt.n_columns = 2;
	b.vt.residual = pnol::dev::ResidualTable<MyGaussFunctor>::residual_;
	b.vt.fd_jacobian = pnol::dev::ResidualTable<MyGaussFunctor>::fd_jacobian_;
	b.behind = my_not_a_launcher;
	return b;
}
static MyV1Block my_v1_block = make_v1_block();
static const int my_reg_v1 = pnol_register_functor(MYJ_F_GAUSS_V1, reinterpret_cast<const pnol_functor_vtable *>(&my_v1_block.vt));

/* ---- the plugin class of the Gaussian peak (reference-style user code) ---- */
#include "pnol/ExampleObjectives.hpp"
#include "pnol/LevenbergMarquardt.hpp"

class MyGaussObjective : public pnol::FunctorMultiObjective<MyGaussFunctor> {
  public:
	MyGaussObjective(const double * t, const double * y, long long m, double c0)
	{
		cols.resize(2);
		cols[0].assign(t, t + m);
		cols[1].assign(y, y + m);
		P.scalars[0] = c0;
		bindColumns();
	}
};

/* ---- C face for the tests (ctypes) ---- */
namespace {
template <class R> void host_rows(const pnol_functor_params * P, const double * x, int n, const long long * rows, long long nrows, double * J,
                                  double * F)
{
	const pnol::PtrAcc acc{x};
	for (long long r = 0; r < nrows; r++) {
		if (J) R::jacobian(*P, acc, n, rows[r], J + r * n);
		if (F) F[r] = R::residual(*P, acc, n, rows[r]);
	}
}
} // namespace

extern "C" {

int my_jacobians_registration_status(void)
{
	return pnol_reg_MyLorentzFunctor | pnol_reg_MyGaussFunctor | pnol_reg_MyGaussNoJacFunctor | my_reg_v1;
}

/* rows[r] of the analytic Jacobian (J, nrows x n) and of the residual (F, nrows) on the host, through the same __host__ __device__
 * definitions the kernels compile; kind: a built-in residual model or one of this file's. Returns 0, or -1 for an unknown kind. */
int my_host_jacobian_rows(int kind, const pnol_functor_params * P, const double * x, int n, const long long * rows, long long nrows, double * J,
                          double * F)
{
	switch (kind) {
		case PNOL_F_EXPCURVE: host_rows<pnol::ExpCurveFunctor>(P, x, n, rows, nrows, J, F); return 0;
		case PNOL_F_CUBIC: host_rows<pnol::CubicFunctor>(P, x, n, rows, nrows, J, F); return 0;
		case PNOL_F_LORENTZ_SUM: host_rows<pnol::LorentzSumFunctor>(P, x, n, rows, nrows, J, F); return 0;
		case MYJ_F_LORENTZ: host_rows<MyLorentzFunctor>(P, x, n, rows, nrows, J, F); return 0;
		case MYJ_F_GAUSS: host_rows<MyGaussFunctor>(P, x, n, rows, nrows, J, F); return 0;
		default: return -1;
	}
}

/* LevMarq::findMin on the Gaussian peak with the Jacobian mode of pnol::Runtime (hostapi.set_jac_mode) */
int my_lm_gauss(const double * t, const double * y, long long m, double c0, double * x, int maxiter)
{
	try {
		MyGaussObjective obj(t, y, m, c0);
		LevMarq lm;
		lm.setObjPtr(obj);
		lm.setParams(0.001, 10, 1e-7, maxiter, 1e-12, 0);
		std::vector<double> X(x, x + 3), F0((size_t) m), F((size_t) m);
		lm.findMin(X, F0, F);
		for (int i = 0; i < 3; i++) x[i] = X[(size_t) i];
		return 0;
	} catch (const std::exception & e) {
		fprintf(stderr, "my_lm_gauss: %s\n", e.what());
		return -1;
	}
}

}
