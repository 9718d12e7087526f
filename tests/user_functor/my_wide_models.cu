/* The wide residual model of my_wide_models.hpp, compiled out of tree like my_jacobians.cu (tests/user_wide_lib.py):
 *   nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -Xcompiler -fPIC,-ffp-contract=off -I<repo>/include -shared \
 *        -o libmy_wide_models.so my_wide_models.cu -L<repo>/parallelnonlinearoptimizationlibrary_b200/lib -lpnol_b200 -lpnol_b200_host
 * The host side runs the same __host__ __device__ definitions: the reference of the kernels' bits. */
#include "my_wide_models.hpp"

#include "pnol/device/functor_kernels.cuh"

PNOL_REGISTER_RESIDUAL_FUNCTOR(MYW_F_WIDE, MyWideFunctor, 3)

extern "C" {

int my_wide_registration_status(void) { return pnol_reg_MyWideFunctor; }

/* rows [i0, i1) of the analytic Jacobian (J, (i1 - i0) x n, when not NULL) and of the residual (F, i1 - i0) on the host */
void my_wide_host_rows(const pnol_functor_params * P, const double * x, int n, long long i0, long long i1, double * J, double * F)
{
	const pnol::PtrAcc acc{x};
	for (long long i = i0; i < i1; i++) {
		if (J) MyWideFunctor::jacobian(*P, acc, n, i, J + (i - i0) * n);
		F[i - i0] = MyWideFunctor::residual(*P, acc, n, i);
	}
}

/* the forward-difference stencil values on the host: Rp[i * n + j] = r_i(x with x_j replaced by x_j + dx_j), the point the black-box
 * kernel evaluates (PerturbAcc); the quotient is left to the caller */
void my_wide_host_stencils(const pnol_functor_params * P, const double * x, const double * dx, int n, long long m, double * Rp)
{
	for (long long i = 0; i < m; i++)
		for (int j = 0; j < n; j++) {
			const pnol::PerturbAcc acc{x, j, x[j] + dx[j]};
			Rp[i * n + j] = MyWideFunctor::residual(*P, acc, n, i);
		}
}

}
