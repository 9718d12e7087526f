"""What the library can launch for each functor kind, without a GPU: pnol_functor_registered and the four pnol_functor_has_* for every
kind from -1 to 3100, with the built-in objectives only and with the user functor libraries of tests/user_functor/ loaded. Each scan
runs in a process of its own: a registration cannot be undone, and other tests register kinds of their own in this one."""
import subprocess
import sys

import user_functor_lib as U
import user_gradient_lib as UG
import user_hessian_lib as UH
import user_jacobian_lib as UJ

_SCAN = r"""
import ctypes as C, sys
sys.path.insert(0, sys.argv[1])
from parallelnonlinearoptimizationlibrary_b200 import capi, hostapi
lib = capi.load_library()
hostapi.lib()
for so in sys.argv[2:]:
    C.CDLL(so, mode=C.RTLD_GLOBAL)
for kind in range(-1, 3101):
    row = [lib.pnol_functor_registered(kind), lib.pnol_functor_has_gradient(kind), lib.pnol_functor_has_hessian(kind),
           lib.pnol_functor_has_slope(kind), lib.pnol_functor_has_lm_batch(kind)]
    if any(row):
        print(kind, *row)
"""

# kind: (registered, has_gradient, has_hessian, has_slope, has_lm_batch); every kind not listed answers 0 to all five
SCALAR_ALL = (1, 1, 1, 1, 0)          # a built-in scalar objective: every one has partial() and partial2()
RESIDUAL_BATCH = (1, 0, 0, 0, 1)      # a residual model with a batched LM launcher
BUILTINS = {1: SCALAR_ALL, 2: SCALAR_ALL, 3: SCALAR_ALL, 4: SCALAR_ALL, 5: SCALAR_ALL, 6: SCALAR_ALL,
            101: RESIDUAL_BATCH, 102: RESIDUAL_BATCH, 103: RESIDUAL_BATCH}
USER = {
    U.MY_F_TRID: (1, 0, 0, 0, 0), U.MY_F_STYBLINSKI: (1, 0, 0, 0, 0),                 # no derivatives
    UG.MYG_F_TRID: (1, 1, 0, 1, 0), UG.MYG_F_STYBLINSKI: (1, 1, 0, 1, 0),             # partial(): gradient and slope
    UH.MYH_F_QUADFORM: (1, 0, 1, 0, 0), UH.MYH_F_STYBLINSKI: (1, 0, 1, 0, 0),         # partial2(): Hessian
    U.MY_F_GAUSSFIT: RESIDUAL_BATCH,
    UJ.MYJ_F_LORENTZ: RESIDUAL_BATCH, UJ.MYJ_F_GAUSS: RESIDUAL_BATCH, UJ.MYJ_F_GAUSS_NOJAC: RESIDUAL_BATCH,
    UJ.MYJ_F_GAUSS_V1: (1, 0, 0, 0, 0),                                               # a raw version-1 table, nothing attached
}


def _scan(libraries):
    r = subprocess.run([sys.executable, "-c", _SCAN, U.ROOT] + libraries, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    got = {}
    for line in r.stdout.split("\n"):
        if line.strip():
            kind, *row = map(int, line.split())
            got[kind] = tuple(row)
    return got


def test_builtin_kinds_only():
    assert _scan([]) == BUILTINS


def test_with_the_user_functor_libraries():
    libraries = [m.build_and_load()._name for m in (U, UG, UH, UJ)]
    assert _scan(libraries) == {**BUILTINS, **USER}
