/* Scalar objectives with analytic Hessians, compiled out of tree like my_objectives.cu (tests/user_hessian_lib.py):
 *   nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -Xcompiler -fPIC,-ffp-contract=off -I<repo>/include -shared \
 *        -o libmy_hessians.so my_hessians.cu -L<repo>/parallelnonlinearoptimizationlibrary_b200/lib -lpnol_b200 -lpnol_b200_host
 * PNOL_REGISTER_SCALAR_FUNCTOR registers each table and, because both functors define partial2(), attaches its Hessian launcher. */
#include "my_hessians.hpp"

#include "pnol/device/functor_kernels.cuh"

PNOL_REGISTER_SCALAR_FUNCTOR(MYH_F_QUADFORM, MyQuadFormFunctor, 1)
PNOL_REGISTER_SCALAR_FUNCTOR(MYH_F_STYBLINSKI, MyHessStyblinskiFunctor, 0)

/* ---- C face for the tests (ctypes) ---- */
namespace {
template <class F> void host_partial2(const pnol_functor_params * P, const double * x, int n, const int * ii, const int * jj,
                                      long long npairs, double * out)
{
	const pnol::PtrAcc acc{x};
	if (!ii) {
		for (int i = 0; i < n; i++)
			for (int j = i; j < n; j++) out[(long long) i * n + j] = out[(long long) j * n + i] = F::partial2(*P, acc, n, i, j);
		return;
	}
	for (long long k = 0; k < npairs; k++) out[k] = F::partial2(*P, acc, n, ii[k], jj[k]);
}
} // namespace

extern "C" {

int my_hessians_registration_status(void) { return pnol_reg_MyQuadFormFunctor | pnol_reg_MyHessStyblinskiFunctor; }

/* partial2() on the host, through the same __host__ __device__ definition the kernels compile. ii == NULL: the whole n x n matrix into
 * out, upper triangle computed and mirrored as the kernel does; else out[k] = d2f/dx_ii[k] dx_jj[k] for k < npairs (ii[k] <= jj[k]).
 * kind: a built-in scalar objective or one of this file's. Returns 0, or -1 for a kind without partial2(). */
int my_host_partial2(int kind, const pnol_functor_params * P, const double * x, int n, const int * ii, const int * jj, long long npairs,
                     double * out)
{
	switch (kind) {
		case PNOL_F_ROSENBROCK: host_partial2<pnol::RosenbrockFunctor>(P, x, n, ii, jj, npairs, out); return 0;
		case PNOL_F_POWER: host_partial2<pnol::PowerFunctor>(P, x, n, ii, jj, npairs, out); return 0;
		case PNOL_F_BOOTH: host_partial2<pnol::BoothFunctor>(P, x, n, ii, jj, npairs, out); return 0;
		case PNOL_F_GOLDSTEIN: host_partial2<pnol::GoldsteinFunctor>(P, x, n, ii, jj, npairs, out); return 0;
		case PNOL_F_RASTRIGIN: host_partial2<pnol::RastriginFunctor>(P, x, n, ii, jj, npairs, out); return 0;
		case PNOL_F_EXPCURVE_SINGLE: host_partial2<pnol::ExpCurveSingleFunctor>(P, x, n, ii, jj, npairs, out); return 0;
		case MYH_F_QUADFORM: host_partial2<MyQuadFormFunctor>(P, x, n, ii, jj, npairs, out); return 0;
		case MYH_F_STYBLINSKI: host_partial2<MyHessStyblinskiFunctor>(P, x, n, ii, jj, npairs, out); return 0;
		default: return -1;
	}
}

}
