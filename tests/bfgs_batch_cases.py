"""Shared cases of the batched BFGS tests: the objectives, their dimensions, seeded starts and parameters, and the runners of the CPU
stand-in (tests/host_logic_standin.cpp): oracle_bfgs per start through BFGSBatch, and the unmodified host BFGS controller per start."""
import ctypes as C

import numpy as np

from parallelnonlinearoptimizationlibrary_b200 import capi

# host objective name -> (kind, ints, dimensions the objective allows, start box half-width)
OBJECTIVES = {
    "rosenbrock": (capi.F_ROSENBROCK, (), (2, 3, 8, 64), 2.0),
    "power:3": (capi.F_POWER, (3,), (1, 5, 16), 2.0),
    "booth": (capi.F_BOOTH, (), (2,), 10.0),
    "goldstein": (capi.F_GOLDSTEIN, (), (2,), 2.0),
    "rastrigin": (capi.F_RASTRIGIN, (), (1, 4, 16, 33), 5.12),
    "expsingle": (capi.F_EXPCURVE_SINGLE, (), (3,), 1.0),
}
FLAG_SETS = list(range(8))      # every combination of gradient (1), slope (2) and Hessian (4)
PRM = dict(c1=1e-4, c2=0.9, dalpha=1e-6, alpha_guess=1.0, max_iter_ls=40, dx_grad=1e-6, dx_hess=1e-3, max_iter=30, x_min_diff=1e-9,
           min_grad_2norm=1e-6, init_hess_fd=0)


def starts(name, n, B, seed):
    """B seeded starts in the objective's box; expsingle near its fit; the last rows are edges: a NaN start, an overflowing one, and
    the minimiser (or a point close to it)"""
    rng = np.random.default_rng(seed)
    w = OBJECTIVES[name][3]
    X = rng.uniform(-w, w, size=(B, n))
    if name == "expsingle":
        X = np.array([1.0, 0.5, 0.0]) + rng.uniform(-0.3, 0.3, size=(B, n))
    if B >= 6:
        X[-1] = np.nan
        X[-2] = 1e200
        X[-3] = {"rosenbrock": 1.0, "booth": 1.0, "rastrigin": 0.0, "power:3": 0.0, "goldstein": 0.0, "expsingle": 1.0}[name]
        if name == "booth":
            X[-3] = [1.0, 3.0]
        if name == "goldstein":
            X[-3] = [0.0, -1.0]
    return X


def params(**kw):
    return dict(PRM, **kw)


def vec(prm):
    from parallelnonlinearoptimizationlibrary_b200 import hostapi
    return hostapi.bfgs_params(**prm)


def _p(a):
    return C.c_void_p(a.ctypes.data)


def set_flags(lib, flags):
    lib.pnolhost_set_analytic_gradient(int(bool(flags & 1)))
    lib.pnolhost_set_analytic_slope(int(bool(flags & 2)))
    lib.pnolhost_set_analytic_hessian(int(bool(flags & 4)))


def run_batch(lib, name, X, prm, flags):
    """BFGSBatch::findMin(X, reports) through pnolhost_bfgs_batch of a host library (stand-in or product)"""
    Xv = np.array(X, dtype=np.float64, order="C")
    B, n = Xv.shape
    f0, fopt = np.zeros(B), np.zeros(B)
    it, stop = np.zeros(B, dtype=np.int32), np.zeros(B, dtype=np.int32)
    set_flags(lib, flags)
    try:
        st = lib.pnolhost_bfgs_batch(name.encode(), _p(Xv), C.c_longlong(B), int(n), _p(vec(prm)), 0, _p(f0), _p(fopt), _p(it), _p(stop))
    finally:
        set_flags(lib, 0)
    return st, dict(X=Xv, f0=f0, fopt=fopt, iters=it, stop=stop)


def run_serial(lib, name, x0, prm, flags):
    """the unmodified host BFGS::findMin on one start (pnolhost_bfgs("bfgs", ...))"""
    Xv = np.array(x0, dtype=np.float64)
    f0, fopt, it = C.c_double(), C.c_double(), C.c_int()
    set_flags(lib, flags)
    try:
        st = lib.pnolhost_bfgs(b"bfgs", name.encode(), _p(Xv), Xv.size, _p(vec(prm)), None, None, 0, 0, C.byref(f0), C.byref(fopt), C.byref(it))
    finally:
        set_flags(lib, 0)
    return st, dict(X=Xv, f0=f0.value, fopt=fopt.value, iters=it.value)


def same(a, b):
    """bit for bit, except that any NaN equals any NaN: the sign and payload of a NaN that an invalid operation (inf - inf, 0 * inf)
    creates, and how a sign operation treats it, are the hardware's own (x86 and the GPU differ, e.g. 0xfff8000000000000 against
    0x7ff8000000000000 for the same entry), so a start that turns NaN is NaN at the same entries on both, not always in the same
    encoding. Every other value is compared by its bits."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    if a.shape != b.shape:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint64), b[~nb].view(np.uint64))


def diff_report(a, b, limit=6):
    """the first entries whose bits differ, as hex, for an assertion message"""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    if a.shape != b.shape:
        return "shapes %s and %s" % (a.shape, b.shape)
    idx = np.argwhere(a.view(np.uint64) != b.view(np.uint64))[:limit]
    return "; ".join("%s: %016x vs %016x" % (tuple(int(v) for v in i), a[tuple(i)].view(np.uint64), b[tuple(i)].view(np.uint64)) for i in idx)

