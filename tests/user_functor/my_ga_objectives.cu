/* Registers the GA test objectives of my_ga_objectives.hpp with the library; compiled out of tree like my_objectives.cu:
 *   nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -Xcompiler -fPIC,-ffp-contract=off -I<repo>/include -shared \
 *        -o libmy_ga_objectives.so my_ga_objectives.cu -L<repo>/parallelnonlinearoptimizationlibrary_b200/lib -lpnol_b200 */
#include "my_ga_objectives.hpp"

#include "pnol/device/functor_kernels.cuh"

PNOL_REGISTER_SCALAR_FUNCTOR(MY_F_QUANTIZED, QuantizedFunctor, 0)
PNOL_REGISTER_SCALAR_FUNCTOR(MY_F_SIGNED_ZERO, SignedZeroFunctor, 0)

extern "C" int my_ga_registration_status(void) { return pnol_reg_QuantizedFunctor | pnol_reg_SignedZeroFunctor; }
