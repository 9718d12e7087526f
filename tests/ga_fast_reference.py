"""TEST INFRASTRUCTURE: ctypes face of tests/ga_fast_reference.cpp, the O(Npop log Npop) restatement of oracle_ga. The library is
built with g++ into a temporary directory on first use and linked against oracle/libpnol_oracle.so (whose stream it draws from)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import oracle_lib as O

ROOT = O.ROOT
SRC = os.path.join(ROOT, "tests", "ga_fast_reference.cpp")
ORACLE_DIR = os.path.join(ROOT, "oracle")

# objective kinds of tests/user_functor/my_ga_objectives.hpp (PNOL_F_USER_SCALAR_BASE + 11, + 12)
MY_F_QUANTIZED, MY_F_SIGNED_ZERO = 1011, 1012
OBJ_FN = C.CFUNCTYPE(C.c_double, C.c_void_p, C.c_int)
GEN_CB = C.CFUNCTYPE(None, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64)
REFUSED = -3

_lib = None


def lib():
    global _lib
    if _lib is None:
        O.lib()                                                   # builds oracle/libpnol_oracle.so if needed
        d = tempfile.mkdtemp(prefix="pnol_ga_fast_ref_")
        out = os.path.join(d, "libga_fast_reference.so")
        cmd = ["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-I" + ORACLE_DIR, "-I" + os.path.join(ROOT, "include"),
               "-I" + os.path.join(ROOT, "tests", "user_functor"), "-o", out, SRC, "-L" + ORACLE_DIR, "-lpnol_oracle",
               "-Wl,-rpath," + ORACLE_DIR]
        subprocess.run(cmd, check=True, capture_output=True, text=True)
        _lib = C.CDLL(out)
        _lib.ga_fast_quantized.restype = C.c_double
        _lib.ga_fast_signed_zero.restype = C.c_double
    return _lib


def objective_fn(kind):
    """C function pointer of a test objective of my_ga_objectives.hpp (None: a built-in kind of the oracle)"""
    name = {MY_F_QUANTIZED: "ga_fast_quantized", MY_F_SIGNED_ZERO: "ga_fast_signed_zero"}.get(kind)
    return None if name is None else C.cast(getattr(lib(), name), C.c_void_p)


def set_faults(flip_ties=False, miss_duplicate=False):
    """deliberately wrong variants of the reference, for the sensitivity checks"""
    lib().ga_fast_set_faults(int(flip_ties), int(miss_duplicate))


def _run(entry, f, fn, x0, lb, ub, npop, maxgen, stream, elite_frac, cross_frac, elite_mut_frac, mut_size, elite_mut_size, nstatic,
         stop_after, extra=()):
    X = O.f64(x0).copy()
    n = X.size
    lb, ub = O.f64(lb), O.f64(ub)
    nelite = int(np.ceil(elite_frac * npop))
    nelmut = int(np.ceil(elite_mut_frac * npop))
    ncross = int(np.ceil(cross_frac * npop))
    nrand = npop - nelite - nelmut - ncross
    f0, fopt = C.c_double(), C.c_double()
    xpop, F = np.empty((npop, n)), np.empty(npop)
    cross = np.zeros((max(ncross, 1), n), dtype=np.int32)
    mut = np.zeros(max(nrand, 1), dtype=np.int32)
    elite = np.zeros((max(nelmut, 1), n), dtype=np.int32)
    pos = C.c_uint64()
    it = entry(*f.args(), fn if fn is not None else C.c_void_p(0), O._p(X), O._p(lb), O._p(ub), C.c_int(n), C.c_int(npop), C.c_int(maxgen), C.c_double(elite_frac),
               C.c_double(cross_frac), C.c_double(elite_mut_frac), C.c_double(mut_size), C.c_double(elite_mut_size), C.c_double(nstatic),
               C.c_int(stop_after), *O._stream_args(stream), C.byref(f0), C.byref(fopt), O._p(xpop), O._p(F), O._p(cross), O._p(mut),
               O._p(elite), C.byref(pos), *extra)
    return dict(iters=it, X=X, f0=f0.value, fOpt=fopt.value, xpop=xpop, F=F, cross_idx=cross, mut_idx=mut, elite_idx=elite,
                stream_pos=int(pos.value), sizes=(nelite, nelmut, ncross, nrand))


def ga(f, x0, lb, ub, npop, maxgen, stream, elite_frac=0.1, cross_frac=0.3, elite_mut_frac=0.2, mut_size=0.5, elite_mut_size=0.01,
       nstatic=50.0, stop_after=-1, fn=None, on_generation=None):
    """ga_fast: the outputs of oracle_lib.ga. fn: objective pointer (objective_fn), replaces f's kind. on_generation(g, X, F, cross,
    mut, elite, pos) is called with copies of the outputs of the start population (g = 0) and of every completed generation."""
    nelite = int(np.ceil(elite_frac * npop))
    nelmut = int(np.ceil(elite_mut_frac * npop))
    ncross = int(np.ceil(cross_frac * npop))
    nrand = npop - nelite - nelmut - ncross
    n = np.asarray(x0).size
    cb = None
    if on_generation is not None:
        def _cb(g, px, pf, pc, pm, pe, pos):
            arr = lambda p, shape, t: np.ctypeslib.as_array(C.cast(p, C.POINTER(t)), shape=shape).copy()
            on_generation(g, arr(px, (npop, n), C.c_double), arr(pf, (npop,), C.c_double), arr(pc, (ncross, n), C.c_int),
                          arr(pm, (nrand,), C.c_int), arr(pe, (nelmut, n), C.c_int), int(pos))
        cb = GEN_CB(_cb)
    return _run(lib().ga_fast, f, fn, x0, lb, ub, npop, maxgen, stream, elite_frac, cross_frac, elite_mut_frac, mut_size, elite_mut_size,
                nstatic, stop_after, extra=(cb if cb is not None else C.c_void_p(0),))


def oracle_ga(f, x0, lb, ub, npop, maxgen, stream, elite_frac=0.1, cross_frac=0.3, elite_mut_frac=0.2, mut_size=0.5, elite_mut_size=0.01,
              nstatic=50.0, stop_after=-1, fn=None):
    """the literal O(Npop^2 n) oracle_ga_fn (oracle/pnol_oracle.cpp) with the same arguments"""
    return _run(O.lib().oracle_ga_fn, f, fn, x0, lb, ub, npop, maxgen, stream, elite_frac, cross_frac, elite_mut_frac, mut_size,
                elite_mut_size, nstatic, stop_after)
