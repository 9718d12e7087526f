"""Shared cases of the batched simplex tests: the objectives and their dimensions (those of tests/bfgs_batch_cases.py), seeded starts,
parameters and streams, and the runners of the CPU stand-in (tests/host_logic_standin.cpp): oracle_simplex per start through
SimplexSearchBatch or the stand-in's C-ABI, and the unmodified host SimplexSearch controller per start on exactly that start's draws."""
import ctypes as C

import numpy as np

import bfgs_batch_cases as BC
from parallelnonlinearoptimizationlibrary_b200 import capi

OBJECTIVES = BC.OBJECTIVES
starts = BC.starts
same = BC.same
diff_report = BC.diff_report
ERR_STREAM = 7      # PNOL_ERR_STREAM
PRM = dict(alpha=1.0, gamma=2.0, rho=0.5, sigma=0.5, max_iter=150, init_rand_max=1.0, x_min_diff=1e-9)
KEYS = ("alpha", "gamma", "rho", "sigma", "max_iter", "init_rand_max", "x_min_diff")


def params(**kw):
    return dict(PRM, **kw)


def vec(prm):
    """the seven numbers of pnolhost_simplex / pnolhost_simplex_batch, in setSimplexParams' order"""
    return np.array([float(prm[k]) for k in KEYS], dtype=np.float64)


def c_params(prm):
    return capi.SimplexParams(*[int(prm[k]) if k == "max_iter" else float(prm[k]) for k in KEYS])


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def set_stream(lib, stream):
    """stream: ("seed", seed, scale) -- the counter stream -- or ("values", array)"""
    if stream[0] == "values":
        vals = np.ascontiguousarray(stream[1], dtype=np.float64)
        lib.pnolhost_set_stream(_p(vals), C.c_ulonglong(vals.size), C.c_ulonglong(0), C.c_double(1.0))
        return vals
    lib.pnolhost_set_stream(C.c_void_p(0), C.c_ulonglong(0), C.c_ulonglong(stream[1]), C.c_double(stream[2]))
    return None


def stream_desc(stream):
    """(StreamDesc, the array it points to, kept alive by the caller)"""
    if stream[0] == "values":
        vals = np.ascontiguousarray(stream[1], dtype=np.float64)
        return capi.StreamDesc(vals.ctypes.data, vals.size, 0, 1.0), vals
    return capi.StreamDesc(None, 0, int(stream[1]), float(stream[2])), None


def draws(lib, stream, pos, count):
    """the stream's values at positions pos .. pos + count - 1"""
    if stream[0] == "values":
        return np.ascontiguousarray(stream[1][pos:pos + count], dtype=np.float64)
    return np.array([lib.pnol_stream_uniform(int(stream[1]), pos + t, float(stream[2])) for t in range(count)])


def run_batch(lib, name, X, prm, stream):
    """SimplexSearchBatch::findMin(X, reports) through pnolhost_simplex_batch of a host library (stand-in or product)"""
    Xv = np.array(X, dtype=np.float64, order="C")
    B, n = Xv.shape
    f0, fopt = np.zeros(B), np.zeros(B)
    it, stop = np.zeros(B, dtype=np.int32), np.zeros(B, dtype=np.int32)
    ev = np.zeros(B, dtype=np.int64)
    rep = np.zeros(2)
    keep = set_stream(lib, stream)
    try:
        st = lib.pnolhost_simplex_batch(name.encode(), _p(Xv), C.c_longlong(B), int(n), _p(vec(prm)), 0, _p(f0), _p(fopt), _p(it), _p(stop),
                                        _p(ev), _p(rep))
    finally:
        lib.pnolhost_clear_stream()
    del keep
    return st, dict(X=Xv, f0=f0, fopt=fopt, iters=it, stop=stop, evals=ev, stream_pos=int(rep[1]), total_evals=int(lib.pnolhost_last_evaluations()))


def run_serial(lib, name, x0, prm, values):
    """the unmodified host SimplexSearch::findMin on one start (pnolhost_simplex) drawing from `values` alone"""
    Xv = np.array(x0, dtype=np.float64)
    f0, fopt = C.c_double(), C.c_double()
    rep = np.zeros(2)
    keep = set_stream(lib, ("values", values))
    try:
        st = lib.pnolhost_simplex(name.encode(), _p(Xv), Xv.size, _p(vec(prm)), 0, C.byref(f0), C.byref(fopt), _p(rep))
    finally:
        lib.pnolhost_clear_stream()
    del keep
    return st, dict(X=Xv, f0=f0.value, fopt=fopt.value, iters=int(rep[0]), stream_pos=int(rep[1]), evals=int(lib.pnolhost_last_evaluations()))


def run_standin_capi(lib, kind, X, prm, stream, offset=0, ints=(), scalars=()):
    """the stand-in's pnol_simplex_batch (oracle_simplex per start) on a functor of `kind`"""
    Xv = np.array(X, dtype=np.float64, order="C")
    B, n = Xv.shape
    f0, fopt = np.zeros(B), np.zeros(B)
    it, stop = np.zeros(B, dtype=np.int32), np.zeros(B, dtype=np.int32)
    ev = np.zeros(B, dtype=np.int64)
    sd, keep = stream_desc(stream)
    sc = np.zeros(8)
    sc[:len(scalars)] = scalars
    iv = np.zeros(4, dtype=np.int64)
    iv[:len(ints)] = ints
    p = c_params(prm)
    st = lib.standin_simplex_batch(int(kind), _p(sc), _p(iv), C.c_longlong(B), int(n), _p(Xv), C.byref(p), C.byref(sd), C.c_uint64(int(offset)),
                                   _p(f0), _p(fopt), _p(it), _p(stop), _p(ev))
    del keep
    return st, dict(X=Xv, f0=f0, fopt=fopt, iters=it, stop=stop, evals=ev)


def kind_of(name):
    """(kind, ints) of a host objective name"""
    return OBJECTIVES[name][0], OBJECTIVES[name][1]
