/* Registers the simplex test objectives of my_simplex_objectives.hpp with the library; compiled out of tree like my_objectives.cu:
 *   nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -Xcompiler -fPIC,-ffp-contract=off -I<repo>/include -shared \
 *        -o libmy_simplex_objectives.so my_simplex_objectives.cu -L<repo>/parallelnonlinearoptimizationlibrary_b200/lib -lpnol_b200 */
#include "my_simplex_objectives.hpp"

#include "pnol/device/functor_kernels.cuh"

PNOL_REGISTER_SCALAR_FUNCTOR(MYS_F_NEGATIVE, SimplexNegativeFunctor, 0)
PNOL_REGISTER_SCALAR_FUNCTOR(MYS_F_QUANTIZED, SimplexQuantizedFunctor, 0)
PNOL_REGISTER_SCALAR_FUNCTOR(MYS_F_SIGNED_ZERO, SimplexSignedZeroFunctor, 0)
PNOL_REGISTER_SCALAR_FUNCTOR(MYS_F_NAN_REGION, SimplexNanRegionFunctor, 0)

extern "C" int my_simplex_registration_status(void)
{
	return pnol_reg_SimplexNegativeFunctor | pnol_reg_SimplexQuantizedFunctor | pnol_reg_SimplexSignedZeroFunctor | pnol_reg_SimplexNanRegionFunctor;
}
