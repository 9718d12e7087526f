"""Batched BFGS without a GPU: oracle_bfgs (tests/host_logic_standin.cpp, the CPU stand-in's pnol_bfgs_batch, reached through
BFGSBatch) bit for bit against the unmodified host BFGS controller on the same stand-in, start by start, for the six built-in
objectives, every derivative-flag combination, both initial inverse Hessians and the edge parameters; the base-class findMin; the
refusal on a C-ABI without pnol_bfgs_batch; pnol_register_functor_bfgs_batch's rules and pnol_functor_has_bfgs_batch for every kind."""
import ctypes as C
import subprocess
import sys

import numpy as np
import pytest

import bfgs_batch_cases as BC
import host_standin
from parallelnonlinearoptimizationlibrary_b200 import capi


@pytest.fixture(scope="module")
def standin():
    hl = host_standin.load()
    if hl is None:
        pytest.skip("no g++ on this box")
    return hl


def check_against_serial(lib, name, X, prm, flags):
    st, got = BC.run_batch(lib, name, X, prm, flags)
    assert st == 0, lib.pnolhost_last_error()
    for b in range(X.shape[0]):
        st, want = BC.run_serial(lib, name, X[b], prm, flags)
        assert st == 0, lib.pnolhost_last_error()
        where = (name, X.shape[1], flags, prm["init_hess_fd"], b)
        assert BC.same(got["X"][b], want["X"]), where
        assert BC.same(got["f0"][b], want["f0"]) and BC.same(got["fopt"][b], want["fopt"]), where
        assert got["iters"][b] == want["iters"], where
    return got


@pytest.mark.parametrize("flags", BC.FLAG_SETS)
@pytest.mark.parametrize("name", sorted(BC.OBJECTIVES))
def test_each_start_is_the_host_bfgs_alone(standin, name, flags):
    for n in BC.OBJECTIVES[name][2]:
        for ih in (0, 1):
            prm = BC.params(init_hess_fd=ih)
            got = check_against_serial(standin, name, BC.starts(name, n, 8, seed=n + 17 * ih), prm, flags)
            assert set(got["stop"]) <= {0, 1, 2}
            # the stop code is the first false conjunct of the loop condition
            assert all((s == 0) == (it == prm["max_iter"]) for s, it in zip(got["stop"], got["iters"]))


@pytest.mark.parametrize("edge", ["max_iter_0", "max_iter_ls_0", "max_iter_ls_1", "no_tolerances"])
@pytest.mark.parametrize("name", ["rosenbrock", "rastrigin", "goldstein"])
def test_edge_parameters(standin, name, edge):
    kw = {"max_iter_0": dict(max_iter=0), "max_iter_ls_0": dict(max_iter_ls=0), "max_iter_ls_1": dict(max_iter_ls=1),
          "no_tolerances": dict(x_min_diff=0.0, min_grad_2norm=0.0, max_iter=12)}[edge]
    n = 2 if name == "goldstein" else 4
    for flags in (0, 7):
        for ih in (0, 1):
            prm = BC.params(init_hess_fd=ih, **kw)
            got = check_against_serial(standin, name, BC.starts(name, n, 7, seed=3), prm, flags)
            if edge == "max_iter_0":
                assert np.all(got["iters"] == 0) and np.all(got["stop"] == 0)
                assert BC.same(got["f0"], got["fopt"])


def test_exhausted_line_search_turns_d_nan_as_the_reference(standin):
    """max_iter_ls = 0: alpha = 0, s = 0, rho = 1/0 and D NaN; X stays, xdiff is 0 and the loop stops with code 1"""
    X = BC.starts("rosenbrock", 3, 5, seed=2)
    got = check_against_serial(standin, "rosenbrock", X, BC.params(max_iter_ls=0), 0)
    assert np.all(got["iters"][:-1] == 1) and np.all(got["stop"] == 1)


def test_base_class_find_min_is_one_start(standin):
    from parallelnonlinearoptimizationlibrary_b200 import hostapi
    x0 = np.array([-1.2, 1.0, 0.5])
    prm = BC.params(max_iter=100)
    Xv, f0, fopt = x0.copy(), np.zeros(1), np.zeros(1)
    p = lambda a: C.c_void_p(a.ctypes.data)
    assert standin.pnolhost_bfgs_batch(b"rosenbrock", p(Xv), C.c_longlong(1), 3, p(hostapi.bfgs_params(**prm)), 1, p(f0), p(fopt), None, None) == 0
    st, want = BC.run_serial(standin, "rosenbrock", x0, prm, 0)
    assert st == 0 and BC.same(Xv, want["X"]) and BC.same(f0[0], want["f0"]) and BC.same(fopt[0], want["fopt"])
    assert np.max(np.abs(Xv - 1.0)) < 1e-4


_REFUSAL = r"""
import ctypes as C, sys
import numpy as np
lib = C.CDLL(sys.argv[1], mode=C.RTLD_LOCAL)
lib.pnolhost_last_error.restype = C.c_char_p
p = lambda a: C.c_void_p(a.ctypes.data)
X = np.array([[-1.2, 1.0]]); prm = np.array([1e-4, 0.9, 1e-6, 1.0, 40, 1e-6, 1e-3, 10, 1e-9, 1e-6, 0.0])
f0, fopt = np.zeros(1), np.zeros(1); it, stop = np.zeros(1, dtype=np.int32), np.zeros(1, dtype=np.int32)
st = lib.pnolhost_bfgs_batch(b"rosenbrock", p(X), C.c_longlong(1), 2, p(prm), 0, p(f0), p(fopt), p(it), p(stop))
print(st, lib.pnolhost_last_error().decode())
"""


def test_bfgs_batch_on_a_c_abi_without_it_is_refused():
    """The host sources reference pnol_bfgs_batch weakly: linked against a C-ABI implementation without it (the unmodified stand-in) they
    still build and load, and BFGSBatch fails with PNOL_ERR_NO_FUNCTOR."""
    so = host_standin.base_path()
    if so is None:
        pytest.skip("no g++ on this box")
    r = subprocess.run([sys.executable, "-c", _REFUSAL, so], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    st, msg = r.stdout.strip().split(" ", 1)
    assert int(st) == capi.ERR_NO_FUNCTOR and "pnol_bfgs_batch" in msg and "not provided by the C-ABI implementation" in msg, r.stdout


def test_register_functor_bfgs_batch_rules():
    from test_user_gradient_cpu import _table
    lib = capi.load_library()
    fn = C.c_void_p(C.cast(lib.pnol_version, C.c_void_p).value)      # any non-NULL code address: registration never calls a launcher
    S, R = capi.F_USER_SCALAR_BASE + 760, capi.F_USER_RESIDUAL_BASE + 760
    keep = [_table(2, True), _table(1, False), _table(2, True), _table(2, True)]
    assert lib.pnol_register_functor(S, C.byref(keep[0])) == capi.PNOL_OK
    assert lib.pnol_register_functor(R, C.byref(keep[1])) == capi.PNOL_OK
    assert lib.pnol_register_functor(S + 1, C.byref(keep[2])) == capi.PNOL_OK
    for kind in (S, S + 1):
        assert lib.pnol_functor_has_bfgs_batch(kind) == 0
        assert lib.pnol_register_functor_bfgs_batch(kind, fn) == capi.PNOL_OK
        assert lib.pnol_functor_has_bfgs_batch(kind) == 1
    # a residual kind, a kind without a table, a built-in kind, a kind outside every range and NULL are refused
    assert lib.pnol_register_functor_bfgs_batch(R, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_bfgs_batch(S + 2, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_bfgs_batch(capi.F_ROSENBROCK, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_bfgs_batch(5000, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_bfgs_batch(S, None) == capi.ERR_INVALID
    assert lib.pnol_functor_has_bfgs_batch(R) == 0 and lib.pnol_functor_has_bfgs_batch(S + 2) == 0
    # replacing the table drops the launcher attached to the old one
    assert lib.pnol_register_functor(S, C.byref(keep[3])) == capi.PNOL_OK
    assert lib.pnol_functor_has_bfgs_batch(S) == 0 and lib.pnol_functor_registered(S) == 1 and lib.pnol_functor_has_bfgs_batch(S + 1) == 1


_SCAN = r"""
import ctypes as C, sys
sys.path.insert(0, sys.argv[1])
from parallelnonlinearoptimizationlibrary_b200 import capi, hostapi
lib = capi.load_library()
hostapi.lib()
for so in sys.argv[2:]:
    C.CDLL(so, mode=C.RTLD_GLOBAL)
print(" ".join(str(k) for k in range(-1, 3101) if lib.pnol_functor_has_bfgs_batch(k)))
"""


def _scan(libraries):
    r = subprocess.run([sys.executable, "-c", _SCAN, host_standin.ROOT] + libraries, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return [int(k) for k in r.stdout.split()]


def test_has_bfgs_batch_for_every_kind():
    """each scan in a fresh process: the six built-in scalar objectives; with the user libraries of tests/user_functor/ loaded also
    every user scalar kind registered with PNOL_REGISTER_SCALAR_FUNCTOR (with or without derivatives), never a residual model or a raw
    version-1 table"""
    import user_functor_lib as U
    import user_gradient_lib as UG
    import user_hessian_lib as UH
    import user_jacobian_lib as UJ
    assert _scan([]) == [1, 2, 3, 4, 5, 6]
    libraries = [m.build_and_load()._name for m in (U, UG, UH, UJ)]
    want = sorted([1, 2, 3, 4, 5, 6, U.MY_F_TRID, U.MY_F_STYBLINSKI, UG.MYG_F_TRID, UG.MYG_F_STYBLINSKI, UH.MYH_F_QUADFORM, UH.MYH_F_STYBLINSKI])
    assert _scan(libraries) == want
