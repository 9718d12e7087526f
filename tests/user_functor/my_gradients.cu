/* Scalar objectives with analytic gradients, compiled out of tree like my_objectives.cu (tests/user_gradient_lib.py):
 *   nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -Xcompiler -fPIC,-ffp-contract=off -I<repo>/include -shared \
 *        -o libmy_gradients.so my_gradients.cu -L<repo>/parallelnonlinearoptimizationlibrary_b200/lib -lpnol_b200 -lpnol_b200_host
 * PNOL_REGISTER_SCALAR_FUNCTOR registers each table and, because both functors define partial(), attaches its gradient launcher. */
#include "my_gradients.hpp"

#include "pnol/device/functor_kernels.cuh"

PNOL_REGISTER_SCALAR_FUNCTOR(MYG_F_TRID, MyTridFunctor, 0)
PNOL_REGISTER_SCALAR_FUNCTOR(MYG_F_STYBLINSKI, MyStyblinskiFunctor, 0)

/* ---- C face for the tests (ctypes) ---- */
namespace {
template <class F> void host_partials(const pnol_functor_params * P, const double * x, int n, const int * idx, int nidx, double * g)
{
	const pnol::PtrAcc acc{x};
	for (int k = 0; k < nidx; k++) g[k] = F::partial(*P, acc, n, idx ? idx[k] : k);
}
} // namespace

extern "C" {

int my_gradients_registration_status(void) { return pnol_reg_MyTridFunctor | pnol_reg_MyStyblinskiFunctor; }

/* g[k] = df/dx_{idx[k]} (idx NULL: k) on the host, through the same __host__ __device__ partial() the kernels compile; kind: a built-in
 * scalar objective or one of this file's. Returns 0, or -1 for a kind without partial(). */
int my_host_partials(int kind, const pnol_functor_params * P, const double * x, int n, const int * idx, int nidx, double * g)
{
	switch (kind) {
		case PNOL_F_ROSENBROCK: host_partials<pnol::RosenbrockFunctor>(P, x, n, idx, nidx, g); return 0;
		case PNOL_F_POWER: host_partials<pnol::PowerFunctor>(P, x, n, idx, nidx, g); return 0;
		case PNOL_F_BOOTH: host_partials<pnol::BoothFunctor>(P, x, n, idx, nidx, g); return 0;
		case PNOL_F_GOLDSTEIN: host_partials<pnol::GoldsteinFunctor>(P, x, n, idx, nidx, g); return 0;
		case PNOL_F_RASTRIGIN: host_partials<pnol::RastriginFunctor>(P, x, n, idx, nidx, g); return 0;
		case PNOL_F_EXPCURVE_SINGLE: host_partials<pnol::ExpCurveSingleFunctor>(P, x, n, idx, nidx, g); return 0;
		case MYG_F_TRID: host_partials<MyTridFunctor>(P, x, n, idx, nidx, g); return 0;
		case MYG_F_STYBLINSKI: host_partials<MyStyblinskiFunctor>(P, x, n, idx, nidx, g); return 0;
		default: return -1;
	}
}

/* the shared host/device math of include/pnol/pnol_math.h on the host: which = 0 sin2pi, 1 cos2pi, 2 exp_hd */
int my_host_math(int which, const double * x, long long n, double * out)
{
	for (long long k = 0; k < n; k++) {
		switch (which) {
			case 0: out[k] = pnol::sin2pi(x[k]); break;
			case 1: out[k] = pnol::cos2pi(x[k]); break;
			case 2: out[k] = pnol::exp_hd(x[k]); break;
			default: return -1;
		}
	}
	return 0;
}

}
