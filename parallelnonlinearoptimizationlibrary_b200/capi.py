"""ctypes binding of the C-ABI declared in include/pnol_b200.h.

This is the thin Python face of libpnol_b200.so (hand-written sm_100a CUDA kernels behind `extern "C"`).
There is no CPU fallback: loading fails loudly if the library has not been built (`python -c "import
__graft_entry__ as g; g.build()"` or `make`), and every compute call fails with PnolError on a box without a GPU.
"""
import ctypes as C
import os
import weakref

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# PNOL_B200_LIB: a differently built libpnol_b200.so (kernel tuning runs, tools/build_variants.sh); the product path is lib/
LIB_PATH = os.environ.get("PNOL_B200_LIB") or os.path.join(_HERE, "lib", "libpnol_b200.so")
HOST_LIB_PATH = os.path.join(_HERE, "lib", "libpnol_b200_host.so")

PNOL_OK = 0
ERR_INVALID, ERR_CUDA, ERR_NO_FUNCTOR = 1, 2, 3
F_USER_SCALAR_BASE, F_USER_RESIDUAL_BASE = 1000, 2000      # open functor table (pnol_register_functor)
ERR_NAMES = {1: "INVALID", 2: "CUDA", 3: "NO_FUNCTOR", 4: "NONFINITE", 5: "NOT_SPD", 6: "COMM", 7: "STREAM"}

# functor kinds (include/pnol_b200.h)
F_ROSENBROCK, F_POWER, F_BOOTH, F_GOLDSTEIN, F_RASTRIGIN, F_EXPCURVE_SINGLE = 1, 2, 3, 4, 5, 6
F_EXPCURVE, F_CUBIC, F_LORENTZ_SUM = 101, 102, 103
JAC_AUTO, JAC_BLACKBOX, JAC_STRUCTURED, JAC_ANALYTIC = 0, 1, 2, 3      # JAC_ANALYTIC: the model's own derivative, dx may be None
HINV_LITERAL, HINV_RANK2 = 0, 1
BFGS_ANALYTIC_GRADIENT, BFGS_ANALYTIC_SLOPE, BFGS_ANALYTIC_HESSIAN = 1, 2, 4      # pnol_bfgs_batch deriv_flags
COMM_ID_BYTES = 128

c_double_p = C.POINTER(C.c_double)
c_ubyte_p = C.POINTER(C.c_ubyte)
c_int_p = C.POINTER(C.c_int)


class PnolError(RuntimeError):
    pass


class FunctorDesc(C.Structure):
    _fields_ = [
        ("kind", C.c_int),
        ("scalars", C.c_double * 8),
        ("ints", C.c_longlong * 4),
        ("n_columns", C.c_int),
        ("columns", C.c_void_p * 8),
        ("m", C.c_longlong),
    ]


class StreamDesc(C.Structure):
    _fields_ = [("values", C.c_void_p), ("n_values", C.c_uint64), ("seed", C.c_uint64), ("scale", C.c_double)]


class GaParams(C.Structure):
    _fields_ = [
        ("npop", C.c_int),
        ("max_generations", C.c_int),
        ("elite_frac", C.c_double),
        ("cross_frac", C.c_double),
        ("elite_mutation_frac", C.c_double),
        ("mutation_size", C.c_double),
        ("elite_mutation_size", C.c_double),
        ("n_static_generations", C.c_double),
    ]


class BfgsParams(C.Structure):
    """pnol_bfgs_params: BFGS::setParams' arguments in order"""
    _fields_ = [
        ("c1", C.c_double),
        ("c2", C.c_double),
        ("dalpha", C.c_double),
        ("alpha_guess", C.c_double),
        ("max_iter_ls", C.c_int),
        ("dx_grad", C.c_double),
        ("dx_hess", C.c_double),
        ("max_iter", C.c_int),
        ("x_min_diff", C.c_double),
        ("min_grad_2norm", C.c_double),
        ("init_hess_fd", C.c_int),
    ]


class SimplexParams(C.Structure):
    """pnol_simplex_params: SimplexSearch::setSimplexParams' arguments in order"""
    _fields_ = [
        ("alpha", C.c_double),
        ("gamma", C.c_double),
        ("rho", C.c_double),
        ("sigma", C.c_double),
        ("max_iter", C.c_int),
        ("init_rand_max", C.c_double),
        ("x_min_diff", C.c_double),
    ]


class GaStatus(C.Structure):
    _fields_ = [
        ("generation", C.c_int),
        ("n_static", C.c_int),
        ("stopped", C.c_int),
        ("f_best", C.c_double),
        ("stream_pos", C.c_uint64),
        ("n_elite", C.c_int),
        ("n_elite_mut", C.c_int),
        ("n_cross", C.c_int),
        ("n_rand", C.c_int),
    ]


# every symbol include/pnol_b200.h declares (tests/test_abi.py checks the header against this list and the .so)
EXPORTS = [
    "pnol_ctx_create", "pnol_ctx_destroy", "pnol_last_error", "pnol_ctx_device", "pnol_ctx_stream", "pnol_ctx_sync",
    "pnol_ctx_sm_count", "pnol_ctx_launches", "pnol_version", "pnol_malloc", "pnol_free", "pnol_memcpy", "pnol_copy_start", "pnol_copy_wait", "pnol_memset",
    "pnol_host_alloc", "pnol_host_free", "pnol_comm_unique_id", "pnol_comm_init", "pnol_comm_rank", "pnol_comm_size",
    "pnol_comm_set_local", "pnol_comm_allreduce_sum", "pnol_comm_allgather", "pnol_comm_broadcast", "pnol_register_functor", "pnol_functor_registered",
    "pnol_register_functor_gradient", "pnol_functor_has_gradient", "pnol_register_functor_hessian", "pnol_functor_has_hessian",
    "pnol_register_functor_slope", "pnol_functor_has_slope", "pnol_register_functor_lm_batch", "pnol_functor_has_lm_batch",
    "pnol_register_functor_bfgs_batch", "pnol_functor_has_bfgs_batch", "pnol_register_functor_simplex_batch", "pnol_functor_has_simplex_batch",
    "pnol_functor_create",
    "pnol_functor_destroy", "pnol_functor_is_residual", "pnol_functor_rows", "pnol_eval_batch", "pnol_fd_gradient",
    "pnol_eval_recur", "pnol_fd_gradient_recur", "pnol_gradient", "pnol_gradient_recur", "pnol_fd_hessian", "pnol_hessian", "pnol_alpha_pool",
    "pnol_alpha_pool_analytic", "pnol_residual_eval",
    "pnol_fd_jacobian", "pnol_lm_normal_eq", "pnol_lm_damp", "pnol_lm_step", "pnol_lm_iterate", "pnol_lm_last_run", "pnol_lm_exchange_mode", "pnol_lm_batch", "pnol_bfgs_batch", "pnol_simplex_batch", "pnol_lm_normal_eq_fused", "pnol_spd_solve", "pnol_lu_inverse",
    "pnol_matvec_neg", "pnol_bfgs_update_hinv", "pnol_dgemm_nn", "pnol_check_box_bounds", "pnol_compute_alpha_bnd",
    "pnol_stream_uniform", "pnol_ga_create", "pnol_ga_destroy", "pnol_ga_init", "pnol_ga_generation",
    "pnol_ga_status_get", "pnol_ga_set_sharding", "pnol_ga_peer_mode", "pnol_ga_get_population", "pnol_ga_get_indices", "pnol_ga_pop_sort", "pnol_ga_check_bounds",
    "pnol_ga_check_identical", "pnol_measure_dmma_peak", "pnol_measure_copy_bandwidth", "pnol_timer_enable",
    "pnol_timer_get", "pnol_timer_reset", "pnol_selftest_exact_div", "pnol_selftest_fast_div", "pnol_selftest_syrk_plan",
]

_lib = None


def load_library():
    """Load libpnol_b200.so (once). Raises PnolError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PnolError(
            "libpnol_b200.so is missing (%s): build it with `make` or __graft_entry__.build(); "
            "this package has no CPU fallback" % LIB_PATH)
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    lib.pnol_last_error.restype = C.c_char_p
    lib.pnol_version.restype = C.c_char_p
    lib.pnol_ctx_stream.restype = C.c_void_p
    lib.pnol_ctx_launches.restype = C.c_uint64
    lib.pnol_functor_rows.restype = C.c_longlong
    lib.pnol_compute_alpha_bnd.restype = C.c_double
    lib.pnol_stream_uniform.restype = C.c_double
    lib.pnol_stream_uniform.argtypes = [C.c_uint64, C.c_uint64, C.c_double]
    lib.pnol_ctx_create.argtypes = [C.POINTER(C.c_void_p), C.c_int]
    lib.pnol_ctx_destroy.argtypes = [C.c_void_p]
    lib.pnol_ctx_destroy.restype = None
    lib.pnol_functor_destroy.argtypes = [C.c_void_p]
    lib.pnol_functor_destroy.restype = None
    lib.pnol_ga_destroy.argtypes = [C.c_void_p]
    lib.pnol_ga_destroy.restype = None
    _lib = lib
    return lib


def _ptr(a):
    """void* of a numpy array, a raw int device pointer, a torch tensor, or None."""
    if a is None:
        return C.c_void_p(0)
    if isinstance(a, (int, np.integer)):
        return C.c_void_p(int(a))
    if isinstance(a, np.ndarray):
        assert a.flags["C_CONTIGUOUS"], "array must be C-contiguous"
        return C.c_void_p(a.ctypes.data)
    if hasattr(a, "data_ptr"):
        return C.c_void_p(a.data_ptr())
    raise TypeError("unsupported buffer %r" % type(a))


def _f64(a):
    """Host arrays are made contiguous float64; raw device pointers (int) and torch tensors pass through."""
    if a is None or isinstance(a, (int, np.integer)) or hasattr(a, "data_ptr"):
        return a
    return np.ascontiguousarray(a, dtype=np.float64)


def _len(a, n):
    if n is not None:
        return int(n)
    if isinstance(a, np.ndarray):
        return int(a.size)
    if hasattr(a, "numel"):
        return int(a.numel())
    raise TypeError("pass n= explicitly when the point is a raw device pointer")


class Functor:
    def __init__(self, ctx, handle, kind, m, keep):
        self.ctx, self.handle, self.kind, self.m, self._keep = ctx, handle, kind, m, keep
        ctx._children.add(self)

    def close(self):
        # a functor must die before its context (pnol_functor_destroy frees on the context's stream): Context.close()
        # closes its children first, and a functor that outlives a closed context only drops its handle
        if self.handle and self.ctx.h:
            self.ctx.lib.pnol_functor_destroy(self.handle)
        self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Context:
    """One pnol_ctx: one GPU, one stream."""

    def __init__(self, device=0):
        self.lib = load_library()
        h = C.c_void_p()
        st = self.lib.pnol_ctx_create(C.byref(h), int(device))
        if st != PNOL_OK:
            raise PnolError("pnol_ctx_create(device=%d) failed with %s: a CUDA device is required, there is no CPU "
                            "fallback" % (device, ERR_NAMES.get(st, st)))
        self.h = h
        self.device = device
        self._children = weakref.WeakSet()

    def close(self):
        if getattr(self, "h", None):
            for child in list(self._children):
                child.close()
            self.lib.pnol_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, st):
        if st != PNOL_OK:
            msg = self.lib.pnol_last_error(self.h)
            raise PnolError("%s: %s" % (ERR_NAMES.get(st, st), msg.decode() if msg else ""))

    # ---- plumbing ----
    @property
    def stream(self):
        return self.lib.pnol_ctx_stream(self.h)

    @property
    def sm_count(self):
        return self.lib.pnol_ctx_sm_count(self.h)

    def launches(self):
        return int(self.lib.pnol_ctx_launches(self.h))

    def sync(self):
        self.check(self.lib.pnol_ctx_sync(self.h))

    def malloc(self, nbytes):
        p = C.c_void_p()
        self.check(self.lib.pnol_malloc(self.h, C.byref(p), C.c_size_t(nbytes)))
        return p.value

    def free(self, p):
        self.check(self.lib.pnol_free(self.h, C.c_void_p(p)))

    def memcpy(self, dst, src, nbytes):
        self.check(self.lib.pnol_memcpy(self.h, _ptr(dst), _ptr(src), C.c_size_t(nbytes)))

    def copy_start(self, dst_host, src_dev, nbytes):
        """device -> host copy that runs beside the context's stream; dst_host must stay alive and untouched until copy_wait()"""
        self.check(self.lib.pnol_copy_start(self.h, _ptr(dst_host), _ptr(src_dev), C.c_size_t(nbytes)))

    def copy_wait(self):
        self.check(self.lib.pnol_copy_wait(self.h))

    def to_device(self, arr):
        arr = np.ascontiguousarray(arr)
        p = self.malloc(arr.nbytes)
        self.memcpy(p, arr, arr.nbytes)
        return p

    def to_host(self, p, shape, dtype=np.float64):
        out = np.empty(shape, dtype=dtype)
        self.memcpy(out, p, out.nbytes)
        return out

    def timer_enable(self, on=True):
        self.check(self.lib.pnol_timer_enable(self.h, int(on)))

    def timer_reset(self):
        self.check(self.lib.pnol_timer_reset(self.h))

    def timer_get(self, name):
        ms, cnt = C.c_double(), C.c_longlong()
        self.check(self.lib.pnol_timer_get(self.h, name.encode(), C.byref(ms), C.byref(cnt)))
        return ms.value, cnt.value

    def measure_dmma_peak(self):
        v = C.c_double()
        self.check(self.lib.pnol_measure_dmma_peak(self.h, C.byref(v)))
        return v.value

    def measure_copy_bandwidth(self):
        v = C.c_double()
        self.check(self.lib.pnol_measure_copy_bandwidth(self.h, C.byref(v)))
        return v.value

    def selftest_exact_div(self, pairs, seed=1):
        bad = C.c_ulonglong()
        self.check(self.lib.pnol_selftest_exact_div(self.h, C.c_longlong(pairs), C.c_ulonglong(seed), C.byref(bad)))
        return int(bad.value)

    def selftest_fast_div(self, pairs, seed=1):
        bad = C.c_ulonglong()
        self.check(self.lib.pnol_selftest_fast_div(self.h, C.c_longlong(pairs), C.c_ulonglong(seed), C.byref(bad)))
        return int(bad.value)

    # ---- communicator ----
    def comm_unique_id(self):
        buf = C.create_string_buffer(COMM_ID_BYTES)
        st = self.lib.pnol_comm_unique_id(buf)
        if st != PNOL_OK:
            raise PnolError("pnol_comm_unique_id failed (NCCL not loadable)")
        return buf.raw

    def comm_init(self, uid, nranks, rank):
        buf = C.create_string_buffer(bytes(uid), COMM_ID_BYTES)
        self.check(self.lib.pnol_comm_init(self.h, buf, int(nranks), int(rank)))

    def comm_size(self):
        return self.lib.pnol_comm_size(self.h)

    def comm_rank(self):
        return self.lib.pnol_comm_rank(self.h)

    def set_local(self, on):
        """local (non-collective) mode on / off; returns the previous setting"""
        return bool(self.lib.pnol_comm_set_local(self.h, int(bool(on))))

    def allreduce_sum(self, buf, count):
        self.check(self.lib.pnol_comm_allreduce_sum(self.h, _ptr(buf), C.c_size_t(count)))

    # ---- functors ----
    def functor(self, kind, scalars=(), ints=(), columns=(), m=0):
        d = FunctorDesc()
        d.kind = kind
        for i, v in enumerate(scalars):
            d.scalars[i] = float(v)
        for i, v in enumerate(ints):
            d.ints[i] = int(v)
        keep = []
        d.n_columns = len(columns)
        for i, col in enumerate(columns):
            if isinstance(col, np.ndarray):
                col = _f64(col)
                keep.append(col)
            d.columns[i] = _ptr(col).value
        d.m = int(m)
        h = C.c_void_p()
        self.check(self.lib.pnol_functor_create(self.h, C.byref(d), C.byref(h)))
        return Functor(self, h, kind, int(m), keep)

    # ---- scalar objectives ----
    def eval_batch(self, f, pts, B, n, ld=None, indicator=None, f_out=None):
        ld = n if ld is None else ld
        host_out = f_out is None
        if host_out:
            f_out = np.zeros(B, dtype=np.float64)
        self.check(self.lib.pnol_eval_batch(self.h, f.handle, _ptr(pts), C.c_longlong(B), int(n), C.c_longlong(ld),
                                            _ptr(indicator), _ptr(f_out)))
        return f_out

    def fd_gradient(self, f, x, dx):
        x, dx = _f64(x), _f64(dx)
        g = np.empty_like(x)
        f0 = C.c_double()
        self.check(self.lib.pnol_fd_gradient(self.h, f.handle, _ptr(x), _ptr(dx), x.size, _ptr(g), C.byref(f0)))
        return g, f0.value

    def eval_recur(self, f, xr, const_x, const_ind):
        xr, const_x = _f64(xr), _f64(const_x)
        ind = np.ascontiguousarray(const_ind, dtype=np.uint8)
        out = C.c_double()
        self.check(self.lib.pnol_eval_recur(self.h, f.handle, _ptr(xr), xr.size, _ptr(const_x), _ptr(ind), const_x.size,
                                            C.byref(out)))
        return out.value

    def fd_gradient_recur(self, f, xr, dxr, const_x, const_ind):
        xr, dxr, const_x = _f64(xr), _f64(dxr), _f64(const_x)
        ind = np.ascontiguousarray(const_ind, dtype=np.uint8)
        g = np.empty_like(xr)
        f0 = C.c_double()
        self.check(self.lib.pnol_fd_gradient_recur(self.h, f.handle, _ptr(xr), _ptr(dxr), xr.size, _ptr(const_x), _ptr(ind),
                                                   const_x.size, _ptr(g), C.byref(f0)))
        return g, f0.value

    def gradient(self, f, x, want_f0=False, g=None, n=None):
        """analytic gradient (pnol_gradient) from the functor's own derivative: returns (g, f0), f0 None unless want_f0. x and g may be
        numpy arrays or raw device pointers (then pass n=); g defaults to a new host array"""
        x = _f64(x)
        n = _len(x, n)
        if g is None:
            g = np.empty(n, dtype=np.float64)
        f0 = C.c_double()
        self.check(self.lib.pnol_gradient(self.h, f.handle, _ptr(x), n, _ptr(g), C.byref(f0) if want_f0 else None))
        return g, (f0.value if want_f0 else None)

    def gradient_recur(self, f, xr, const_x, const_ind, want_f0=False):
        """analytic gradient over the free variables (pnol_gradient_recur): returns (g, f0), f0 None unless want_f0"""
        xr, const_x = _f64(xr), _f64(const_x)
        ind = np.ascontiguousarray(const_ind, dtype=np.uint8)
        g = np.empty(xr.size, dtype=np.float64)
        f0 = C.c_double()
        self.check(self.lib.pnol_gradient_recur(self.h, f.handle, _ptr(xr), xr.size, _ptr(const_x), _ptr(ind), const_x.size, _ptr(g),
                                                C.byref(f0) if want_f0 else None))
        return g, (f0.value if want_f0 else None)

    def fd_hessian(self, f, x, dx):
        x, dx = _f64(x), _f64(dx)
        B = np.empty((x.size, x.size), dtype=np.float64)
        self.check(self.lib.pnol_fd_hessian(self.h, f.handle, _ptr(x), _ptr(dx), x.size, _ptr(B)))
        return B

    def hessian(self, f, x, H=None, n=None):
        """analytic Hessian (pnol_hessian) from the functor's own second derivative: returns H (n x n). x and H may be numpy arrays,
        torch tensors or raw device pointers (then pass n=); H defaults to a new host array"""
        x = _f64(x)
        n = _len(x, n)
        if H is None:
            H = np.empty((n, n), dtype=np.float64)
        self.check(self.lib.pnol_hessian(self.h, f.handle, _ptr(x), n, _ptr(H)))
        return H

    def alpha_pool(self, f, x, p, alpha, dalpha, want_dphi=True, eval_ind=None, const_x=None, const_ind=None):
        x, p, alpha = _f64(x), _f64(p), _f64(alpha)
        npool = alpha.size
        phi = np.zeros(npool)
        dphi = np.zeros(npool) if want_dphi else None
        bad = C.c_int()
        ei = None if eval_ind is None else np.ascontiguousarray(eval_ind, dtype=np.uint8)
        cx = None if const_x is None else _f64(const_x)
        ci = None if const_ind is None else np.ascontiguousarray(const_ind, dtype=np.uint8)
        nfull = x.size if cx is None else cx.size
        self.check(self.lib.pnol_alpha_pool(self.h, f.handle, _ptr(x), _ptr(p), x.size, _ptr(alpha), npool,
                                            C.c_double(dalpha), _ptr(ei), _ptr(cx), _ptr(ci), nfull, _ptr(phi), _ptr(dphi),
                                            C.byref(bad)))
        return phi, dphi, bad.value

    def alpha_pool_analytic(self, f, x, p, alpha, eval_ind=None, const_x=None, const_ind=None, phi=None, dphi=None, n=None, npool=None):
        """phi = f(x + alpha p) and the analytic slope dphi = p . grad f(x + alpha p) for a pool of step lengths
        (pnol_alpha_pool_analytic): returns (phi, dphi, bad). x, p, alpha, phi and dphi may be numpy arrays, torch tensors or raw device
        pointers (then pass n= and npool=); phi and dphi default to new host arrays, and entries with eval_ind == 0 keep what they
        held"""
        x, p, alpha = _f64(x), _f64(p), _f64(alpha)
        n = _len(x, n)
        npool = _len(alpha, npool)
        if phi is None:
            phi = np.zeros(npool)
        if dphi is None:
            dphi = np.zeros(npool)
        bad = C.c_int()
        ei = None if eval_ind is None else np.ascontiguousarray(eval_ind, dtype=np.uint8)
        cx = None if const_x is None else _f64(const_x)
        ci = None if const_ind is None else np.ascontiguousarray(const_ind, dtype=np.uint8)
        nfull = n if cx is None else cx.size
        self.check(self.lib.pnol_alpha_pool_analytic(self.h, f.handle, _ptr(x), _ptr(p), n, _ptr(alpha), npool, _ptr(ei), _ptr(cx),
                                                     _ptr(ci), nfull, _ptr(phi), _ptr(dphi), C.byref(bad)))
        return phi, dphi, bad.value

    # ---- residual models ----
    def residual_eval(self, f, x, F=None, want_sumsq=True, n=None):
        x = _f64(x)
        n = _len(x, n)
        host = F is None
        if host:
            F = np.empty(f.m, dtype=np.float64)
        ss = C.c_double()
        self.check(self.lib.pnol_residual_eval(self.h, f.handle, _ptr(x), n, _ptr(F),
                                               C.byref(ss) if want_sumsq else None))
        return F, ss.value

    def fd_jacobian(self, f, x, dx=None, J=None, F=None, mode=JAC_AUTO, n=None):
        """J (m x n) and F at x; mode=JAC_ANALYTIC: J from the model's analytic derivative, dx ignored (None allowed)"""
        x, dx = _f64(x), _f64(dx)
        n = _len(x, n)
        host = J is None
        if host:
            J = np.empty((f.m, n), dtype=np.float64)
            F = np.empty(f.m, dtype=np.float64)
        self.check(self.lib.pnol_fd_jacobian(self.h, f.handle, _ptr(x), _ptr(dx), n, _ptr(J), _ptr(F), int(mode)))
        return J, F

    def lm_normal_eq(self, J, F, m, n, lam, JTJ=None, A=None, rhs=None):
        host = JTJ is None and A is None and rhs is None
        if host:
            JTJ, A, rhs = np.empty((n, n)), np.empty((n, n)), np.empty(n)
        self.check(self.lib.pnol_lm_normal_eq(self.h, _ptr(J), _ptr(F), C.c_longlong(m), int(n), C.c_double(lam), _ptr(JTJ),
                                              _ptr(A), _ptr(rhs)))
        return JTJ, A, rhs

    def lm_normal_eq_fused(self, f, x, dx, n, lam, JTJ=None, A=None, rhs=None, F=None, want_F=True):
        """normal equations straight from the residual model, J never stored (walked in row blocks):
        returns (JTJ, A, rhs, F)"""
        x, dx = _f64(x), _f64(dx)
        if JTJ is None and A is None and rhs is None:
            JTJ, A, rhs = np.empty((n, n)), np.empty((n, n)), np.empty(n)
        if F is None and want_F:
            F = np.empty(f.m, dtype=np.float64)
        self.check(self.lib.pnol_lm_normal_eq_fused(self.h, f.handle, _ptr(x), _ptr(dx), int(n), C.c_double(lam), _ptr(JTJ), _ptr(A),
                                                    _ptr(rhs), _ptr(F)))
        return JTJ, A, rhs, F

    def lm_step(self, f, x, dx, n, J, F, Ftrial, lam, JTJ, jac_mode=JAC_AUTO, reuse_jtj=False):
        """one LM iteration's device work, one synchronisation: returns (sigma, x_trial, sumsq_trial, spd_info).
        dx may be None with jac_mode=JAC_ANALYTIC"""
        x, dx = _f64(x), _f64(dx)
        sigma, xt = np.empty(n), np.empty(n)
        ss, info = C.c_double(), C.c_int()
        self.check(self.lib.pnol_lm_step(self.h, f.handle, _ptr(x), _ptr(dx), int(n), _ptr(J), _ptr(F), _ptr(Ftrial), C.c_double(lam), int(jac_mode),
                                         int(bool(reuse_jtj)), _ptr(JTJ), _ptr(sigma), _ptr(xt), C.byref(ss), C.byref(info)))
        return sigma, xt, ss.value, info.value

    def lm_iterate(self, f, x, dx, n, J, F, Ftrial, JTJ, lam, chisq, factor, iterations, x_min_diff=0.0, jac_mode=JAC_AUTO):
        """`iterations` LM iterations on device-resident state, accept / reject on the host in C++:
        returns (x, lambda, chisq, accepted, rejected, swapped). dx may be None with jac_mode=JAC_ANALYTIC"""
        x, dx = np.array(x, dtype=np.float64), _f64(dx)
        lam_c, chi_c = C.c_double(lam), C.c_double(chisq)
        acc, rej, sw = C.c_int(), C.c_int(), C.c_int()
        self.check(self.lib.pnol_lm_iterate(self.h, f.handle, _ptr(x), _ptr(dx), int(n), _ptr(J), _ptr(F), _ptr(Ftrial), _ptr(JTJ),
                                            C.byref(lam_c), C.byref(chi_c), C.c_double(factor), C.c_double(x_min_diff), int(iterations),
                                            int(jac_mode), C.byref(acc), C.byref(rej), C.byref(sw)))
        return x, lam_c.value, chi_c.value, acc.value, rej.value, sw.value

    def lm_batch(self, f, row_off, X, dx=None, lambda0=0.001, factor=10.0, x_min_diff=1e-7, max_iter=100, jac_mode=JAC_AUTO,
                 want_F=False, n=None, B=None, out=None):
        """Batched LM (pnol_lm_batch): problem b owns rows [row_off[b], row_off[b+1]) of the functor and row b of X (B x n).
        Returns dict(X, chisq, lam, iters, stopped, F). X is fitted in place when it is a float64 numpy array, torch tensor or raw
        device pointer (then pass n= and B=); otherwise a fitted copy is returned. dx: n entries (None with jac_mode=JAC_ANALYTIC).
        out (optional): dict of preallocated outputs under the same names (host or device), e.g. prefilled arrays."""
        if isinstance(X, np.ndarray) and X.dtype == np.float64 and X.flags["C_CONTIGUOUS"]:
            Xa = X
        else:
            Xa = _f64(X) if not isinstance(X, np.ndarray) else np.array(X, dtype=np.float64)
        if isinstance(Xa, np.ndarray) and Xa.ndim == 2:
            B, n = Xa.shape if B is None or n is None else (B, n)
        ro = row_off if (isinstance(row_off, (int, np.integer)) or hasattr(row_off, "data_ptr")) else \
            np.ascontiguousarray(row_off, dtype=np.int64)
        if B is None:
            B = _len(ro, None) - 1
        if n is None:
            n = _len(Xa, None) // max(B, 1)
        dx = _f64(dx)
        out = dict(out or {})
        chisq = out.get("chisq", np.empty(B))
        lam = out.get("lam", np.empty(B))
        iters = out.get("iters", np.empty(B, dtype=np.int32))
        stopped = out.get("stopped", np.empty(B, dtype=np.int32))
        F = out.get("F", np.empty(f.m) if want_F else None)
        self.check(self.lib.pnol_lm_batch(self.h, f.handle, _ptr(ro), C.c_longlong(B), int(n), _ptr(Xa), _ptr(dx), C.c_double(lambda0),
                                          C.c_double(factor), C.c_double(x_min_diff), int(max_iter), int(jac_mode), _ptr(chisq),
                                          _ptr(lam), _ptr(iters), _ptr(stopped), _ptr(F)))
        return dict(X=Xa, chisq=chisq, lam=lam, iters=iters, stopped=stopped, F=F)

    def bfgs_batch(self, f, X, c1=1e-4, c2=0.9, dalpha=1e-6, alpha_guess=1.0, max_iter_ls=1000, dx_grad=1e-6, dx_hess=1e-3, max_iter=10000,
                   x_min_diff=1e-5, min_grad_2norm=1e-5, init_hess_fd=False, flags=0, n=None, B=None, out=None, prm=None):
        """Batched BFGS (pnol_bfgs_batch): start b is row b of X (B x n), every start minimises the scalar functor f. The keywords are
        BFGS::setParams' (BFGS's defaults); prm (optional) a ready BfgsParams or None to pass NULL. flags: BFGS_ANALYTIC_* bits.
        Returns dict(X, f0, fopt, iters, stop). X is minimised in place when it is a float64 numpy array, torch tensor or raw device
        pointer (then pass n= and B=); otherwise a copy is returned. out (optional): dict of preallocated outputs under the same names."""
        if isinstance(X, np.ndarray) and X.dtype == np.float64 and X.flags["C_CONTIGUOUS"]:
            Xa = X
        else:
            Xa = _f64(X) if not isinstance(X, np.ndarray) else np.array(X, dtype=np.float64)
        if B is None or n is None:
            shape = tuple(Xa.shape)
            B, n = (shape[0], shape[1]) if len(shape) == 2 else (1, shape[0])
        if prm is None:
            prm = BfgsParams(c1, c2, dalpha, alpha_guess, int(max_iter_ls), dx_grad, dx_hess, int(max_iter), x_min_diff, min_grad_2norm,
                             int(bool(init_hess_fd)))
        elif prm == "null":
            prm = None
        out = dict(out or {})
        nb = max(int(B), 0)              # a negative B is the library's to refuse
        f0 = out.get("f0", np.empty(nb))
        fopt = out.get("fopt", np.empty(nb))
        iters = out.get("iters", np.empty(nb, dtype=np.int32))
        stop = out.get("stop", np.empty(nb, dtype=np.int32))
        self.check(self.lib.pnol_bfgs_batch(self.h, f.handle, C.c_longlong(B), int(n), _ptr(Xa), C.byref(prm) if prm is not None else None,
                                            int(flags), _ptr(f0), _ptr(fopt), _ptr(iters), _ptr(stop)))
        return dict(X=Xa, f0=f0, fopt=fopt, iters=iters, stop=stop)

    def simplex_batch(self, f, X, alpha=1.0, gamma=2.0, rho=0.5, sigma=0.5, max_iter=10000, init_rand_max=1.0, x_min_diff=1e-7, stream=None,
                      stream_offset=0, n=None, B=None, out=None, prm=None, want_evals=True):
        """Batched simplex search (pnol_simplex_batch): start b is row b of X (B x n), every start minimises the scalar functor f. The
        keywords are SimplexSearch::setSimplexParams' (SimplexSearch's defaults); prm (optional) a ready SimplexParams, or "null" to pass
        NULL. stream: a StreamDesc, an array of explicit values (host or device), an int seed of the counter stream (scale 1), or "null";
        None is the counter stream with seed 0. Returns dict(X, f0, fopt, iters, stop, evals). X is minimised in place when it is a
        float64 numpy array, torch tensor or raw device pointer (then pass n= and B=); otherwise a copy is returned. out (optional): dict
        of preallocated outputs under the same names; want_evals=False passes NULL for evals."""
        if isinstance(X, np.ndarray) and X.dtype == np.float64 and X.flags["C_CONTIGUOUS"]:
            Xa = X
        else:
            Xa = _f64(X) if not isinstance(X, np.ndarray) else np.array(X, dtype=np.float64)
        if B is None or n is None:
            shape = tuple(Xa.shape)
            B, n = (shape[0], shape[1]) if len(shape) == 2 else (1, shape[0])
        if prm is None:
            prm = SimplexParams(alpha, gamma, rho, sigma, int(max_iter), init_rand_max, x_min_diff)
        elif prm == "null":
            prm = None
        keep = None
        if stream is None or isinstance(stream, (int, np.integer)):
            sd = StreamDesc(None, 0, int(stream or 0), 1.0)
        elif isinstance(stream, StreamDesc):
            sd = stream
        elif isinstance(stream, str) and stream == "null":
            sd = None
        else:
            keep = stream if hasattr(stream, "data_ptr") else np.ascontiguousarray(stream, dtype=np.float64)
            sd = StreamDesc(_ptr(keep).value, int(keep.numel() if hasattr(keep, "numel") else keep.size), 0, 1.0)
        out = dict(out or {})
        nb = max(int(B), 0)              # a negative B is the library's to refuse
        f0 = out.get("f0", np.empty(nb))
        fopt = out.get("fopt", np.empty(nb))
        iters = out.get("iters", np.empty(nb, dtype=np.int32))
        stop = out.get("stop", np.empty(nb, dtype=np.int32))
        evals = out.get("evals", np.empty(nb, dtype=np.int64)) if want_evals else None
        self.check(self.lib.pnol_simplex_batch(self.h, f.handle, C.c_longlong(B), int(n), _ptr(Xa), C.byref(prm) if prm is not None else None,
                                               C.byref(sd) if sd is not None else None, C.c_uint64(int(stream_offset)), _ptr(f0), _ptr(fopt),
                                               _ptr(iters), _ptr(stop), _ptr(evals)))
        del keep
        return dict(X=Xa, f0=f0, fopt=fopt, iters=iters, stop=stop, evals=evals)

    def lm_exchange_mode(self):
        """0 one rank, 1 NVLink peer memory, 2 NCCL, -1 not decided yet"""
        return int(self.lib.pnol_lm_exchange_mode(self.h))

    def lm_last_run(self):
        """(stopped, xdiff2norm) of the last lm_iterate"""
        st, xd = C.c_int(), C.c_double()
        self.check(self.lib.pnol_lm_last_run(self.h, C.byref(st), C.byref(xd)))
        return bool(st.value), xd.value

    def spd_solve(self, A, rhs, n, x=None):
        host = x is None
        if host:
            x = np.empty(n)
        info = C.c_int()
        self.check(self.lib.pnol_spd_solve(self.h, _ptr(A), _ptr(rhs), int(n), _ptr(x), C.byref(info)))
        return x

    def lu_inverse(self, A, n):
        """general inverse (LU, partial pivoting) -- matrixInverse of the FD Hessian; returns (Ainv, info)"""
        A = _f64(A)
        out = np.empty((n, n))
        info = C.c_int()
        self.check(self.lib.pnol_lu_inverse(self.h, _ptr(A), int(n), _ptr(out), C.byref(info)))
        return out, info.value

    # ---- BFGS dense pieces ----
    def matvec_neg(self, D, g, n, p=None):
        if p is None:
            p = np.empty(n)
        self.check(self.lib.pnol_matvec_neg(self.h, _ptr(D), _ptr(g), int(n), _ptr(p)))
        return p

    def bfgs_update_hinv(self, D, g, s, n, mode=HINV_RANK2):
        self.check(self.lib.pnol_bfgs_update_hinv(self.h, _ptr(D), _ptr(g), _ptr(s), int(n), int(mode)))
        return D

    def dgemm_nn(self, A, B, Cm, M, N, K):
        self.check(self.lib.pnol_dgemm_nn(self.h, _ptr(A), _ptr(B), _ptr(Cm), int(M), int(N), int(K)))
        return Cm


    # ---- genetic algorithm ----
    def _stream_desc(self, stream):
        d = StreamDesc()
        keep = None
        values = stream.get("values")
        if values is not None:
            keep = np.ascontiguousarray(values, dtype=np.float64)
            d.values = keep.ctypes.data
            d.n_values = keep.size
        d.seed = int(stream.get("seed", 0))
        d.scale = float(stream.get("scale", 1.0))
        return d, keep

    def ga_create(self, f, n, lb, ub, npop, maxgen, stream, elite_frac=0.1, cross_frac=0.3, elite_mut_frac=0.2, mut_size=0.5,
                  elite_mut_size=0.01, nstatic=50.0):
        prm = GaParams(int(npop), int(maxgen), elite_frac, cross_frac, elite_mut_frac, mut_size, elite_mut_size, float(nstatic))
        sd, keep = self._stream_desc(stream)
        lb, ub = _f64(lb), _f64(ub)
        h = C.c_void_p()
        self.check(self.lib.pnol_ga_create(self.h, f.handle, C.byref(prm), int(n), _ptr(lb), _ptr(ub), C.byref(sd), C.byref(h)))
        return GA(self, h, int(npop), int(n), keep, f)

    def ga_set_sharding(self, mode):
        """0 auto, 1 rows sharded over the ranks, 2 rows replicated + sweep sharded, 3 replicas: no collective (before ga_create)"""
        self.check(self.lib.pnol_ga_set_sharding(self.h, int(mode)))

    def ga_pop_sort(self, xpop, F):
        xpop, F = _f64(xpop).copy(), _f64(F).copy()
        self.check(self.lib.pnol_ga_pop_sort(self.h, _ptr(xpop), _ptr(F), C.c_longlong(xpop.shape[0]), int(xpop.shape[1])))
        return xpop, F

    def _ga_stage(self, fn, xpop, lb, ub, stream, pos, ind):
        xpop = _f64(xpop).copy()
        lb, ub = _f64(lb), _f64(ub)
        ind = np.zeros(xpop.shape[0], dtype=np.uint8) if ind is None else np.array(ind, dtype=np.uint8)
        sd, keep = self._stream_desc(stream)
        p = C.c_uint64(pos)
        self.check(fn(self.h, _ptr(xpop), C.c_longlong(xpop.shape[0]), int(xpop.shape[1]), _ptr(lb), _ptr(ub), _ptr(ind), C.byref(sd),
                      C.byref(p)))
        return xpop, ind, int(p.value)

    def ga_check_bounds(self, xpop, lb, ub, stream, pos=0, ind=None):
        """-> (population, evaluation flags, stream position). The flags start as ind (zeros when None); repaired rows are set to 1."""
        return self._ga_stage(self.lib.pnol_ga_check_bounds, xpop, lb, ub, stream, pos, ind)

    def ga_check_identical(self, xpop, lb, ub, stream, pos=0, ind=None):
        """-> (population, evaluation flags, stream position). The flags start as ind (zeros when None); replaced rows are set to 1."""
        return self._ga_stage(self.lib.pnol_ga_check_identical, xpop, lb, ub, stream, pos, ind)


class GA:
    """pnol_ga state machine (GeneticAlgorithmMPI::findMinBnd, one generation per call)."""

    def __init__(self, ctx, handle, npop, n, keep, functor):
        self.ctx, self.handle, self.npop, self.n, self._keep, self._f = ctx, handle, npop, n, keep, functor
        ctx._children.add(self)

    def close(self):
        if self.handle and self.ctx.h:
            self.ctx.lib.pnol_ga_destroy(self.handle)
        self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def init(self, x0):
        x0 = _f64(x0)
        f0 = C.c_double()
        self.ctx.check(self.ctx.lib.pnol_ga_init(self.handle, _ptr(x0), C.byref(f0)))
        return f0.value

    def generation(self):
        self.ctx.check(self.ctx.lib.pnol_ga_generation(self.handle))

    def status(self):
        s = GaStatus()
        self.ctx.check(self.ctx.lib.pnol_ga_status_get(self.handle, C.byref(s)))
        return s

    def peer_mode(self):
        """0: one rank; 1: rows read from their owners over NVLink (CUDA IPC); 2: replicas + all-gather"""
        return int(self.ctx.lib.pnol_ga_peer_mode(self.handle))

    def population(self):
        x = np.empty((self.npop, self.n))
        F = np.empty(self.npop)
        self.ctx.check(self.ctx.lib.pnol_ga_get_population(self.handle, _ptr(x), _ptr(F)))
        return x, F

    def indices(self):
        s = self.status()
        cross = np.zeros((max(s.n_cross, 1), self.n), dtype=np.int32)
        mut = np.zeros(max(s.n_rand, 1), dtype=np.int32)
        elite = np.zeros((max(s.n_elite_mut, 1), self.n), dtype=np.int32)
        self.ctx.check(self.ctx.lib.pnol_ga_get_indices(self.handle, _ptr(cross), _ptr(mut), _ptr(elite)))
        return cross, mut, elite

    def run(self, x0, max_generations):
        """findMinBnd: init + generations until the generation count or the static-generation stop."""
        f0 = self.init(x0)
        while True:
            s = self.status()
            if s.stopped or s.generation >= max_generations:
                break
            self.generation()
        return f0
