"""TEST INFRASTRUCTURE: ctypes face of oracle/libpnol_oracle.so (the CPU restatement) and a runner for
oracle/_ref/pnol_ref_cli (the verbatim reference compiled against oracle/shim). Never imported by the product."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_SO = os.path.join(ROOT, "oracle", "libpnol_oracle.so")
REF_CLI = os.path.join(ROOT, "oracle", "_ref", "pnol_ref_cli")

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(ORACLE_SO):
            subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "port"])
        _lib = C.CDLL(ORACLE_SO)
        _lib.oracle_obj_eval.restype = C.c_double
        _lib.oracle_eval_recur.restype = C.c_double
        _lib.oracle_compute_alpha_bnd.restype = C.c_double
        _lib.oracle_stream_uniform.restype = C.c_double
        _lib.oracle_stream_uniform.argtypes = [C.c_uint64, C.c_uint64, C.c_double]
        _lib.oracle_ga_check_bounds.restype = C.c_uint64
        _lib.oracle_ga_check_identical.restype = C.c_uint64
    return _lib


def have_ref():
    return os.path.exists(REF_CLI)


def _p(a):
    if a is None:
        return C.c_void_p(0)
    assert a.flags["C_CONTIGUOUS"]
    return C.c_void_p(a.ctypes.data)


def f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


class OFunctor:
    """kind + scalars + ints + data columns, in the layout every oracle_* entry point takes first."""

    def __init__(self, kind, scalars=(), ints=(), columns=(), m=0):
        self.kind = kind
        self.scalars = np.zeros(8)
        self.scalars[:len(scalars)] = scalars
        self.ints = np.zeros(4, dtype=np.int64)
        self.ints[:len(ints)] = ints
        self.columns = [f64(c) for c in columns]
        self.colptr = (C.c_void_p * 8)(*[c.ctypes.data for c in self.columns] + [0] * (8 - len(self.columns)))
        self.m = int(m)

    def args(self):
        return (C.c_int(self.kind), _p(self.scalars), _p(self.ints), C.cast(self.colptr, C.c_void_p), C.c_longlong(self.m))


def obj_eval(f, x):
    x = f64(x)
    return lib().oracle_obj_eval(*f.args(), _p(x), C.c_int(x.size))


def eval_batch(f, pts, indicator=None, f_out=None):
    pts = f64(pts)
    B, n = pts.shape
    out = np.zeros(B) if f_out is None else f_out
    ind = None if indicator is None else np.ascontiguousarray(indicator, dtype=np.uint8)
    lib().oracle_eval_batch(*f.args(), _p(pts), C.c_longlong(B), C.c_int(n), C.c_longlong(n), _p(ind), _p(out))
    return out


def residual(f, x):
    x = f64(x)
    F = np.empty(f.m)
    lib().oracle_residual(*f.args(), _p(x), C.c_int(x.size), _p(F))
    return F


def fd_gradient(f, x, dx):
    x, dx = f64(x), f64(dx)
    g = np.empty_like(x)
    f0 = C.c_double()
    lib().oracle_fd_gradient(*f.args(), _p(x), _p(dx), C.c_int(x.size), _p(g), C.byref(f0))
    return g, f0.value


def eval_recur(f, xr, const_x, ind):
    xr, const_x = f64(xr), f64(const_x)
    ind = np.ascontiguousarray(ind, dtype=np.uint8)
    return lib().oracle_eval_recur(*f.args(), _p(xr), C.c_int(xr.size), _p(const_x), _p(ind), C.c_int(const_x.size))


def fd_gradient_recur(f, xr, dxr, const_x, ind):
    xr, dxr, const_x = f64(xr), f64(dxr), f64(const_x)
    ind = np.ascontiguousarray(ind, dtype=np.uint8)
    g = np.empty_like(xr)
    f0 = C.c_double()
    lib().oracle_fd_gradient_recur(*f.args(), _p(xr), _p(dxr), C.c_int(xr.size), _p(const_x), _p(ind), C.c_int(const_x.size),
                                   _p(g), C.byref(f0))
    return g, f0.value


def fd_hessian(f, x, dx):
    x, dx = f64(x), f64(dx)
    B = np.empty((x.size, x.size))
    lib().oracle_fd_hessian(*f.args(), _p(x), _p(dx), C.c_int(x.size), _p(B))
    return B


def fd_jacobian(f, x, dx):
    x, dx = f64(x), f64(dx)
    J = np.empty((f.m, x.size))
    F = np.empty(f.m)
    lib().oracle_fd_jacobian(*f.args(), _p(x), _p(dx), C.c_int(x.size), _p(J), _p(F))
    return J, F


def lm_normal_eq(J, F, lam):
    J, F = f64(J), f64(F)
    m, n = J.shape
    JTJ, A, rhs = np.empty((n, n)), np.empty((n, n)), np.empty(n)
    lib().oracle_lm_normal_eq(_p(J), _p(F), C.c_longlong(m), C.c_int(n), C.c_double(lam), _p(JTJ), _p(A), _p(rhs))
    return JTJ, A, rhs


def lu_solve(A, b):
    A, b = f64(A), f64(b)
    x = np.empty_like(b)
    lib().oracle_lu_solve(_p(A), _p(b), C.c_int(b.size), _p(x))
    return x


def lm(f, x0, lambda0=0.001, factor=10.0, dxgrad=1e-6, maxiter=100, xmindiff=1e-6, want_trace=False):
    X = f64(x0).copy()
    n = X.size
    F0, F = np.empty(f.m), np.empty(f.m)
    chisq, lam = C.c_double(), C.c_double()
    trace = np.full((maxiter + 1, n + 2), np.nan) if want_trace else None
    it = lib().oracle_lm(*f.args(), _p(X), C.c_int(n), C.c_double(lambda0), C.c_double(factor), C.c_double(dxgrad),
                         C.c_int(maxiter), C.c_double(xmindiff), _p(F0), _p(F), C.byref(chisq), C.byref(lam), _p(trace))
    return dict(X=X, F0=F0, F=F, iters=it, chisq=chisq.value, lam=lam.value, trace=trace)


def lm_mt(f, x0, lambda0=0.001, factor=10.0, dxgrad=1e-6, maxiter=100, xmindiff=1e-6, want_trace=False, threads=None):
    """oracle_lm with the loops re-nested and dealt to host threads (oracle/pnol_oracle_mt.cpp): the same bits, at full BASELINE sizes"""
    X = f64(x0).copy()
    n = X.size
    F0, F = np.empty(f.m), np.empty(f.m)
    chisq, lam = C.c_double(), C.c_double()
    trace = np.full((maxiter + 1, n + 2), np.nan) if want_trace else None
    threads = threads or os.cpu_count() or 1
    it = lib().oracle_lm_mt(*f.args(), _p(X), C.c_int(n), C.c_double(lambda0), C.c_double(factor), C.c_double(dxgrad),
                            C.c_int(maxiter), C.c_double(xmindiff), _p(F0), _p(F), C.byref(chisq), C.byref(lam), _p(trace), C.c_int(threads))
    return dict(X=X, F0=F0, F=F, iters=it, chisq=chisq.value, lam=lam.value, trace=trace)


def update_hinv(D, g, s):
    D = f64(D).copy()
    g, s = f64(g), f64(s)
    lib().oracle_update_hinv(_p(D), _p(g), _p(s), C.c_int(g.size))
    return D


def matvec_neg(D, g):
    D, g = f64(D), f64(g)
    p = np.empty_like(g)
    lib().oracle_matvec_neg(_p(D), _p(g), C.c_int(g.size), _p(p))
    return p


def dgemm_nn(A, B):
    A, B = f64(A), f64(B)
    M, K = A.shape
    N = B.shape[1]
    Cm = np.empty((M, N))
    lib().oracle_dgemm_nn(_p(A), _p(B), _p(Cm), C.c_int(M), C.c_int(N), C.c_int(K))
    return Cm


def alpha_pool(f, x, p, alpha, dalpha, want_dphi=True, eval_ind=None, const_x=None, const_ind=None):
    x, p, alpha = f64(x), f64(p), f64(alpha)
    npool = alpha.size
    phi = np.zeros(npool)
    dphi = np.zeros(npool) if want_dphi else None
    bad = C.c_int()
    ei = None if eval_ind is None else np.ascontiguousarray(eval_ind, dtype=np.uint8)
    cx = None if const_x is None else f64(const_x)
    ci = None if const_ind is None else np.ascontiguousarray(const_ind, dtype=np.uint8)
    nfull = x.size if cx is None else cx.size
    lib().oracle_alpha_pool(*f.args(), _p(x), _p(p), C.c_int(x.size), _p(alpha), C.c_int(npool), C.c_double(dalpha), _p(ei),
                            _p(cx), _p(ci), C.c_int(nfull), _p(phi), _p(dphi), C.byref(bad))
    return phi, dphi, bad.value


def check_box_bounds(x, lb, ub):
    x = f64(x).copy()
    lb, ub = f64(lb), f64(ub)
    cnt = lib().oracle_check_box_bounds(_p(x), _p(lb), _p(ub), C.c_int(x.size))
    return x, cnt


def compute_alpha_bnd(x, lb, ub, p):
    x, lb, ub, p = f64(x), f64(lb), f64(ub), f64(p)
    return lib().oracle_compute_alpha_bnd(_p(x), _p(lb), _p(ub), _p(p), C.c_int(x.size))


def stream_uniform(seed, k, scale):
    return lib().oracle_stream_uniform(seed, k, scale)


def stream_array(seed, count, scale, start=0):
    return np.array([stream_uniform(seed, start + k, scale) for k in range(count)])


def ga_pop_sort(xpop, F):
    xpop, F = f64(xpop).copy(), f64(F).copy()
    lib().oracle_ga_pop_sort(_p(xpop), _p(F), C.c_longlong(xpop.shape[0]), C.c_int(xpop.shape[1]))
    return xpop, F


def _stream_args(stream):
    values = stream.get("values")
    if values is not None:
        values = f64(values)
        stream["_keep"] = values
    return (_p(values), C.c_uint64(0 if values is None else values.size), C.c_uint64(stream.get("seed", 0)),
            C.c_double(stream.get("scale", 1.0)))


def ga_check_bounds(xpop, lb, ub, stream, pos=0, ind=None):
    xpop = f64(xpop).copy()
    lb, ub = f64(lb), f64(ub)
    ind = np.zeros(xpop.shape[0], dtype=np.uint8) if ind is None else np.array(ind, dtype=np.uint8)
    newpos = lib().oracle_ga_check_bounds(_p(xpop), C.c_longlong(xpop.shape[0]), C.c_int(xpop.shape[1]), _p(lb), _p(ub), _p(ind),
                                          *_stream_args(stream), C.c_uint64(pos))
    return xpop, ind, int(newpos)


def ga_check_identical(xpop, lb, ub, stream, pos=0, ind=None):
    xpop = f64(xpop).copy()
    lb, ub = f64(lb), f64(ub)
    ind = np.zeros(xpop.shape[0], dtype=np.uint8) if ind is None else np.array(ind, dtype=np.uint8)
    newpos = lib().oracle_ga_check_identical(_p(xpop), C.c_longlong(xpop.shape[0]), C.c_int(xpop.shape[1]), _p(lb), _p(ub),
                                             _p(ind), *_stream_args(stream), C.c_uint64(pos))
    return xpop, ind, int(newpos)


def ga(f, x0, lb, ub, npop, maxgen, stream, elite_frac=0.1, cross_frac=0.3, elite_mut_frac=0.2, mut_size=0.5,
       elite_mut_size=0.01, nstatic=50.0, stop_after=-1):
    X = f64(x0).copy()
    n = X.size
    lb, ub = f64(lb), f64(ub)
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
    it = lib().oracle_ga(*f.args(), _p(X), _p(lb), _p(ub), C.c_int(n), C.c_int(npop), C.c_int(maxgen), C.c_double(elite_frac),
                         C.c_double(cross_frac), C.c_double(elite_mut_frac), C.c_double(mut_size), C.c_double(elite_mut_size),
                         C.c_double(nstatic), C.c_int(stop_after), *_stream_args(stream), C.byref(f0), C.byref(fopt), _p(xpop), _p(F), _p(cross),
                         _p(mut), _p(elite), C.byref(pos))
    return dict(iters=it, X=X, f0=f0.value, fOpt=fopt.value, xpop=xpop, F=F, cross_idx=cross, mut_idx=mut, elite_idx=elite,
                stream_pos=int(pos.value), sizes=(nelite, nelmut, ncross, nrand))


# ---- verbatim reference through the CLI -------------------------------------------------------------------
def ref_cli(cmd, arrays=None, nprocs=1, timeout=600, **kw):
    """Run oracle/_ref/pnol_ref_cli; `arrays` are written as raw f64 files and passed by path. Returns
    {name: ndarray} of every <out>.<name>.f64 produced, plus '_stdout'."""
    assert have_ref(), "oracle/_ref/pnol_ref_cli not built (make -C oracle ref needs /root/reference)"
    with tempfile.TemporaryDirectory() as td:
        args = [REF_CLI, cmd, "out=" + os.path.join(td, "o")]
        for k, a in (arrays or {}).items():
            path = os.path.join(td, "in_%s.f64" % k)
            f64(a).tofile(path)
            args.append("%s=%s" % (k, path))
        for k, v in kw.items():
            args.append("%s=%s" % (k, repr(float(v)) if isinstance(v, float) else v))
        env = dict(os.environ, PNOL_SHIM_NPROCS=str(nprocs))
        res = subprocess.run(args, env=env, capture_output=True, text=True, timeout=timeout)
        if res.returncode != 0:
            raise RuntimeError("ref_cli %s failed: %s\n%s" % (cmd, res.stdout[-2000:], res.stderr[-2000:]))
        out = {"_stdout": res.stdout}
        for fn in os.listdir(td):
            if fn.startswith("o.") and fn.endswith(".f64"):
                out[fn[2:-4]] = np.fromfile(os.path.join(td, fn), dtype=np.float64)
        return out
