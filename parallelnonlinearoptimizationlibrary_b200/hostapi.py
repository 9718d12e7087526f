"""ctypes binding of lib/libpnol_b200_host.so: the host C++ mirror of the reference's plugin API (include/pnol/*.hpp --
LevMarq[MPI], BFGS, BFGS_MPI, BFGS_Bnd, BFGS_Bnd_MPI_SW, BFGSBnd_MPI, GeneticAlgorithm[MPI], SimplexSearch, Objective /
MultiObjective stencils) driven through
the small C face of host/host_capi.cpp. Tests and bench.py use it to call exactly what a C++ user of the reference API
calls (`alg.setObjPtr(obj); alg.setParams(...); alg.findMin(...)`). No CPU fallback: every call ends in CUDA kernels."""
import ctypes as C
import os

import numpy as np

from . import capi

_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    capi.load_library()          # libpnol_b200.so first (RTLD_GLOBAL), the host library links against it
    if not os.path.exists(capi.HOST_LIB_PATH):
        raise capi.PnolError("libpnol_b200_host.so is missing (%s): run `make`" % capi.HOST_LIB_PATH)
    h = C.CDLL(capi.HOST_LIB_PATH, mode=C.RTLD_GLOBAL)
    h.pnolhost_last_error.restype = C.c_char_p
    h.pnolhost_obj_eval.restype = C.c_double
    h.pnolhost_compute_alpha_bnd.restype = C.c_double
    h.pnolhost_attach.argtypes = [C.c_void_p]
    h.pnolhost_lm_problem_create.restype = C.c_void_p
    h.pnolhost_lm_problem_destroy.argtypes = [C.c_void_p]
    h.pnolhost_lm_problem_destroy.restype = None
    _lib = h
    return h


def _check(st):
    if st != 0:
        raise capi.PnolError("%s: %s" % (capi.ERR_NAMES.get(st, st), lib().pnolhost_last_error().decode()))


def _p(a):
    if a is None:
        return C.c_void_p(0)
    if isinstance(a, (int, np.integer)):
        return C.c_void_p(int(a))
    assert a.flags["C_CONTIGUOUS"]
    return C.c_void_p(a.ctypes.data)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def attach(ctx):
    """Make the plugin classes run on this capi.Context (pnol::Runtime::attach)."""
    _check(lib().pnolhost_attach(ctx.h))


def detach():
    _check(lib().pnolhost_detach())


def set_pool_width(w):
    lib().pnolhost_set_pool_width(int(w))


def set_hinv_mode(mode):
    lib().pnolhost_set_hinv_mode(int(mode))


def set_jac_mode(mode):
    lib().pnolhost_set_jac_mode(int(mode))


def set_analytic_gradient(on):
    """True: the plugin classes' gradients (Objective::gradientApproximation*, hence the BFGS family) come from the objective's own
    derivative (pnol_gradient[_recur]) instead of the forward difference (pnol::Runtime::setAnalyticGradient)"""
    lib().pnolhost_set_analytic_gradient(int(bool(on)))


def set_analytic_hessian(on):
    """True: the plugin classes' Hessians (Objective::hessianApproximation, hence initHessFD of the BFGS family) come from the
    objective's own second derivative (pnol_hessian) instead of the forward difference (pnol::Runtime::setAnalyticHessian)"""
    lib().pnolhost_set_analytic_hessian(int(bool(on)))


def set_analytic_slope(on):
    """True: the line-search slopes of BFGS, BFGS_Bnd and BFGS_Bnd_MPI_SW come from the objective's own derivative
    (pnol_alpha_pool_analytic) instead of the forward difference with their dalpha (pnol::Runtime::setAnalyticSlope); meant to be used
    together with set_analytic_gradient(True)"""
    lib().pnolhost_set_analytic_slope(int(bool(on)))


def set_jacobian_cache(on):
    lib().pnolhost_set_jacobian_cache(int(bool(on)))


def set_store_jacobian(on):
    """False: LM never stores J (normal equations summed over row blocks, pnol::Runtime::setStoreJacobian)"""
    lib().pnolhost_set_store_jacobian(int(bool(on)))


_stream_keep = None


def set_stream(values=None, seed=0, scale=1.0):
    global _stream_keep
    if values is not None:
        _stream_keep = _f64(values)
        lib().pnolhost_set_stream(_p(_stream_keep), C.c_ulonglong(_stream_keep.size), C.c_ulonglong(seed), C.c_double(scale))
    else:
        _stream_keep = None
        lib().pnolhost_set_stream(C.c_void_p(0), C.c_ulonglong(0), C.c_ulonglong(seed), C.c_double(scale))


def clear_stream():
    """forget the explicit stream: the algorithms fall back to the clock-seeded default stream (seed drawn on rank 0, broadcast)"""
    global _stream_keep
    _stream_keep = None
    lib().pnolhost_clear_stream()


def lm_lorentz(t, y, w, x0, lambda0=0.001, factor=10.0, dxgrad=1e-7, maxiter=10, xmindiff=0.0, serial=False, X=None, F0=None,
               F=None):
    """LevMarqMPI::findMin (LevMarq when serial) on LorentzSumObjective(t, y, w). t/y/F0/F may be numpy arrays or raw host
    pointers (ints, e.g. pinned buffers) -- then pass m=... through t.size of a numpy view."""
    t, y = _f64(t), _f64(y)
    m = t.size
    Xv = _f64(x0).copy() if X is None else X
    n = Xv.size
    F0 = np.empty(m) if F0 is None else F0
    F = np.empty(m) if F is None else F
    rep = np.zeros(6)
    _check(lib().pnolhost_lm_lorentz(_p(t), _p(y), C.c_longlong(m), C.c_double(w), _p(Xv), n, C.c_double(lambda0), C.c_double(factor),
                                     C.c_double(dxgrad), C.c_double(maxiter), C.c_double(xmindiff), int(bool(serial)), _p(F0), _p(F),
                                     _p(rep)))
    return dict(X=Xv, F0=F0, F=F, iterations=int(rep[0]), accepted=int(rep[1]), rejected=int(rep[2]), chiSq=rep[3], lam=rep[4],
                xdiff2Norm=rep[5])


def _model_args(kind, scalars, columns):
    sc = np.zeros(8)
    sc[:len(scalars)] = scalars
    cols = [_f64(c) for c in columns]
    ptrs = (C.c_void_p * len(cols))(*[c.ctypes.data for c in cols])
    return sc, cols, ptrs


def lm_batch_model(kind, scalars, columns, row_off, X, lambda0=0.001, factor=10.0, dxgrad=1e-7, maxiter=100, xmindiff=1e-7):
    """LevMarqBatch::findMin(rowOffsets, X, reports) on a built-in residual model (capi.F_EXPCURVE / F_CUBIC / F_LORENTZ_SUM) over the
    columns; X is B x n. The Jacobian mode is the one set with set_jac_mode. Returns dict(X, iters, stopped, chisq, lam)."""
    sc, cols, ptrs = _model_args(kind, scalars, columns)
    Xv = np.array(X, dtype=np.float64, order="C")
    B, n = Xv.shape
    ro = np.ascontiguousarray(row_off, dtype=np.int64)
    it, stp = np.zeros(B, dtype=np.int32), np.zeros(B, dtype=np.int32)
    chi, lam = np.zeros(B), np.zeros(B)
    _check(lib().pnolhost_lm_batch(int(kind), _p(sc), ptrs, len(cols), C.c_longlong(cols[0].size), _p(ro), C.c_longlong(B), _p(Xv), int(n),
                                   C.c_double(lambda0), C.c_double(factor), C.c_double(dxgrad), C.c_double(maxiter), C.c_double(xmindiff),
                                   _p(it), _p(stp), _p(chi), _p(lam)))
    return dict(X=Xv, iters=it, stopped=stp, chisq=chi, lam=lam)


def lm_batch_lorentz(t, y, w, row_off, X, **kw):
    """LevMarqBatch::findMin on LorentzSumObjective(t, y, w): every problem a spectrum of rows [row_off[b], row_off[b+1])"""
    return lm_batch_model(capi.F_LORENTZ_SUM, (w,), (t, y), row_off, X, **kw)


def lm_batch_single(kind, scalars, columns, x0, lambda0=0.001, factor=10.0, dxgrad=1e-7, maxiter=100, xmindiff=1e-7):
    """LevMarqBatch::findMin(X, F0, FOpt): all rows as one problem. Returns dict(X, F0, F)."""
    sc, cols, ptrs = _model_args(kind, scalars, columns)
    m = cols[0].size
    Xv = _f64(x0).copy()
    F0, F = np.empty(m), np.empty(m)
    _check(lib().pnolhost_lm_batch_single(int(kind), _p(sc), ptrs, len(cols), C.c_longlong(m), _p(Xv), int(Xv.size), C.c_double(lambda0),
                                          C.c_double(factor), C.c_double(dxgrad), C.c_double(maxiter), C.c_double(xmindiff), _p(F0), _p(F)))
    return dict(X=Xv, F0=F0, F=F)


class LMProblem:
    """A LorentzSumObjective held the way a C++ user holds it (built once from host data); run() is
    `LevMarqMPI lm; lm.setObjPtr(obj); lm.setParams(...); lm.findMin(X, F0, F)` on vectors that live with the problem."""

    def __init__(self, t, y, w):
        t, y = _f64(t), _f64(y)
        self.m = t.size
        self.h = lib().pnolhost_lm_problem_create(_p(t), _p(y), C.c_longlong(self.m), C.c_double(w))
        if not self.h:
            raise capi.PnolError("pnolhost_lm_problem_create failed: %s" % lib().pnolhost_last_error().decode())

    def run(self, x0, lambda0=0.001, factor=10.0, dxgrad=1e-7, maxiter=10, xmindiff=0.0, serial=False, fresh_device_twin=False):
        Xv = _f64(x0).copy()
        rep = np.zeros(6)
        pF0, pF = C.c_void_p(), C.c_void_p()
        _check(lib().pnolhost_lm_problem_run(C.c_void_p(self.h), _p(Xv), Xv.size, C.c_double(lambda0), C.c_double(factor), C.c_double(dxgrad),
                                             C.c_double(maxiter), C.c_double(xmindiff), int(bool(serial)), int(bool(fresh_device_twin)), _p(rep),
                                             C.byref(pF0), C.byref(pF)))
        view = lambda p: np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_double)), shape=(self.m,))   # noqa: E731
        return dict(X=Xv, F0=view(pF0), F=view(pF), iterations=int(rep[0]), accepted=int(rep[1]), rejected=int(rep[2]), chiSq=rep[3],
                    lam=rep[4], xdiff2Norm=rep[5])

    def close(self):
        if self.h:
            lib().pnolhost_lm_problem_destroy(C.c_void_p(self.h))
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def lm_example(name, x0, lambda0=0.001, factor=10.0, dxgrad=1e-6, maxiter=100, xmindiff=1e-6, m=100):
    Xv = _f64(x0).copy()
    F0, F, rep = np.empty(m), np.empty(m), np.zeros(6)
    _check(lib().pnolhost_lm_example(name.encode(), _p(Xv), Xv.size, C.c_double(lambda0), C.c_double(factor), C.c_double(dxgrad),
                                     C.c_double(maxiter), C.c_double(xmindiff), _p(F0), _p(F), _p(rep)))
    return dict(X=Xv, F0=F0, F=F, iterations=int(rep[0]), accepted=int(rep[1]), rejected=int(rep[2]), chiSq=rep[3])


def gradient(objective, x, dx, mpi=False):
    x, dx = _f64(x), _f64(dx)
    g = np.empty_like(x)
    _check(lib().pnolhost_gradient(objective.encode(), _p(x), _p(dx), x.size, int(bool(mpi)), _p(g)))
    return g


def gradient_recur(objective, xr, dxr, const_x, const_ind):
    xr, dxr, const_x = _f64(xr), _f64(dxr), _f64(const_x)
    ind = np.ascontiguousarray(const_ind, dtype=np.uint8)
    g = np.empty_like(xr)
    f = C.c_double()
    _check(lib().pnolhost_gradient_recur(objective.encode(), _p(xr), _p(dxr), xr.size, _p(const_x), _p(ind), const_x.size, _p(g),
                                         C.byref(f)))
    return g, f.value


def hessian(objective, x, dx):
    x, dx = _f64(x), _f64(dx)
    B = np.empty((x.size, x.size))
    _check(lib().pnolhost_hessian(objective.encode(), _p(x), _p(dx), x.size, _p(B)))
    return B


def obj_eval(objective, x):
    x = _f64(x)
    return lib().pnolhost_obj_eval(objective.encode(), _p(x), x.size)


def jacobian_example(name, x, dx, m=100):
    x, dx = _f64(x), _f64(dx)
    J, F = np.empty((m, x.size)), np.empty(m)
    _check(lib().pnolhost_jacobian_example(name.encode(), _p(x), _p(dx), x.size, _p(J), _p(F)))
    return J, F


def bfgs(variant, objective, x0, params, xlb=None, xub=None, pool_width=0, verbose=0):
    Xv = _f64(x0).copy()
    p = _f64(params)
    lb = None if xlb is None else _f64(xlb)
    ub = None if xub is None else _f64(xub)
    f0, fopt, it = C.c_double(), C.c_double(), C.c_int()
    _check(lib().pnolhost_bfgs(variant.encode(), objective.encode(), _p(Xv), Xv.size, _p(p), _p(lb), _p(ub), int(pool_width),
                               int(verbose), C.byref(f0), C.byref(fopt), C.byref(it)))
    return dict(X=Xv, f0=f0.value, fOpt=fopt.value, iterations=it.value)


BFGS_DEFAULTS = dict(c1=1e-4, c2=0.9, dalpha=1e-6, alpha_guess=1.0, max_iter_ls=1000, dx_grad=1e-6, dx_hess=1e-3, max_iter=10000,
                     x_min_diff=1e-5, min_grad_2norm=1e-5, init_hess_fd=0)


def bfgs_params(**kw):
    """BFGS::setParams' eleven numbers in order (pnolhost_bfgs("bfgs", ...) and bfgs_batch), BFGS's defaults for what kw leaves out"""
    unknown = set(kw) - set(BFGS_DEFAULTS)
    if unknown:
        raise TypeError("unknown BFGS parameters %s" % sorted(unknown))
    prm = dict(BFGS_DEFAULTS, **kw)
    return np.array([float(prm[k]) for k in BFGS_DEFAULTS], dtype=np.float64)


def bfgs_batch(objective, X, params=None, single=False):
    """BFGSBatch::findMin(X, reports) on an example objective ("rosenbrock", "booth", "goldstein", "rastrigin", "expsingle", "power:k"):
    X is B x n, one start per row; params: the eleven numbers of bfgs_params() (None: the defaults). The derivative modes are those set
    with set_analytic_gradient / set_analytic_slope / set_analytic_hessian. Returns dict(X, f0, fOpt, iterations, stop). single=True:
    the base class's findMin(X, f0, fOpt) on the one start of X (iterations and stop are then not reported: -1)."""
    Xv = np.array(X, dtype=np.float64, order="C")
    if Xv.ndim == 1:
        Xv = Xv.reshape(1, -1)
    B, n = Xv.shape
    p = bfgs_params() if params is None else _f64(params)
    f0, fopt = np.zeros(max(B, 1)), np.zeros(max(B, 1))
    it, stop = np.full(max(B, 1), -1, dtype=np.int32), np.full(max(B, 1), -1, dtype=np.int32)
    _check(lib().pnolhost_bfgs_batch(objective.encode(), _p(Xv), C.c_longlong(B), int(n), _p(p), int(bool(single)), _p(f0), _p(fopt), _p(it),
                                     _p(stop)))
    return dict(X=Xv, f0=f0[:B], fOpt=fopt[:B], iterations=it[:B], stop=stop[:B])


def ga(objective, x0, xlb, xub, npop, maxgen, elite_frac=0.1, cross_frac=0.3, elite_mut_frac=0.2, mut_size=0.5,
       elite_mut_size=0.01, nstatic=50.0, serial=False):
    Xv, lb, ub = _f64(x0).copy(), _f64(xlb), _f64(xub)
    f0, fopt = C.c_double(), C.c_double()
    rep = np.zeros(7)
    _check(lib().pnolhost_ga(objective.encode(), _p(Xv), Xv.size, _p(lb), _p(ub), int(npop), int(maxgen), C.c_double(elite_frac),
                             C.c_double(cross_frac), C.c_double(elite_mut_frac), C.c_double(mut_size), C.c_double(elite_mut_size),
                             C.c_double(nstatic), int(bool(serial)), C.byref(f0), C.byref(fopt), _p(rep)))
    return dict(X=Xv, f0=f0.value, fOpt=fopt.value, generations=int(rep[0]), stopped=int(rep[1]), stream_pos=int(rep[2]),
                sizes=tuple(int(v) for v in rep[3:7]))


def simplex(objective, x0, alpha=1.0, gamma=2.0, rho=0.5, sigma=0.5, maxiter=10000, init_rand_max=1.0, xmindiff=1e-7, verbose=0):
    """SimplexSearch::findMin on an example objective; the start simplex draws from the stream of set_stream()"""
    Xv = _f64(x0).copy()
    p = _f64([alpha, gamma, rho, sigma, maxiter, init_rand_max, xmindiff])
    f0, fopt = C.c_double(), C.c_double()
    rep = np.zeros(2)
    _check(lib().pnolhost_simplex(objective.encode(), _p(Xv), Xv.size, _p(p), int(verbose), C.byref(f0), C.byref(fopt), _p(rep)))
    return dict(X=Xv, f0=f0.value, fOpt=fopt.value, iterations=int(rep[0]), stream_pos=int(rep[1]))


def simplex_batch(objective, X, alpha=1.0, gamma=2.0, rho=0.5, sigma=0.5, maxiter=10000, init_rand_max=1.0, xmindiff=1e-7, single=False):
    """SimplexSearchBatch::findMin(X, reports) on an example objective ("rosenbrock", "booth", "goldstein", "rastrigin", "expsingle",
    "power:k"): X is B x n, one start per row; start b draws its start simplex from position b n^2 of the stream of set_stream().
    Returns dict(X, f0, fOpt, iterations, stop, evals, stream_pos). single=True: the base class's findMin(X, f0, fOpt) on the one start
    of X (iterations, stop and evals are then not reported: -1)."""
    Xv = np.array(X, dtype=np.float64, order="C")
    if Xv.ndim == 1:
        Xv = Xv.reshape(1, -1)
    B, n = Xv.shape
    p = _f64([alpha, gamma, rho, sigma, maxiter, init_rand_max, xmindiff])
    f0, fopt = np.zeros(max(B, 1)), np.zeros(max(B, 1))
    it, stop = np.full(max(B, 1), -1, dtype=np.int32), np.full(max(B, 1), -1, dtype=np.int32)
    ev = np.full(max(B, 1), -1, dtype=np.int64)
    rep = np.zeros(2)
    _check(lib().pnolhost_simplex_batch(objective.encode(), _p(Xv), C.c_longlong(B), int(n), _p(p), int(bool(single)), _p(f0), _p(fopt),
                                        _p(it), _p(stop), _p(ev), _p(rep)))
    return dict(X=Xv, f0=f0[:B], fOpt=fopt[:B], iterations=it[:B], stop=stop[:B], evals=ev[:B], stream_pos=int(rep[1]))


def check_box_bounds(x, xlb, xub):
    Xv, lb, ub = _f64(x).copy(), _f64(xlb), _f64(xub)
    _check(lib().pnolhost_check_box_bounds(_p(Xv), _p(lb), _p(ub), Xv.size))
    return Xv


def compute_alpha_bnd(x, xlb, xub, p):
    x, lb, ub, p = _f64(x), _f64(xlb), _f64(xub), _f64(p)
    return lib().pnolhost_compute_alpha_bnd(_p(x), _p(lb), _p(ub), _p(p), x.size)
