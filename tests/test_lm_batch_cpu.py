"""Batched Levenberg-Marquardt without a GPU: LevMarqBatch (include/pnol/LevenbergMarquardtBatch.hpp) on the CPU stand-in extended by
pnol_lm_batch (tests/host_logic_standin.cpp: oracle_lm per problem on its sliced columns), each problem bit for bit oracle_lib.lm on
the problem alone; the refusal on a C-ABI implementation without pnol_lm_batch; and the registration rules of
pnol_register_functor_lm_batch in the product library."""
import ctypes as C
import subprocess
import sys

import numpy as np
import pytest

import host_standin
import lm_batch_cases as LC
from parallelnonlinearoptimizationlibrary_b200 import capi

PRM = dict(lambda0=1e-3, factor=10.0, dxgrad=1e-7, maxiter=40, xmindiff=1e-9)


@pytest.fixture(scope="module")
def standin():
    hl = host_standin.load()
    if hl is None:
        pytest.skip("no g++ on this box")
    return hl


def run_batch(lib, case, X=None, jac_mode=capi.JAC_AUTO, **kw):
    """LevMarqBatch::findMin(rowOffsets, X, reports) through pnolhost_lm_batch of a host library"""
    prm = dict(PRM, **kw)
    sc = np.zeros(8)
    sc[:len(case["scalars"])] = case["scalars"]
    cols = case["columns"]
    ptrs = (C.c_void_p * len(cols))(*[c.ctypes.data for c in cols])
    Xv = np.array(case["X0"] if X is None else X, dtype=np.float64, order="C")
    B, n = Xv.shape
    ro = np.ascontiguousarray(case["row_off"], dtype=np.int64)
    it, stp = np.zeros(B, dtype=np.int32), np.zeros(B, dtype=np.int32)
    chi, lam = np.zeros(B), np.zeros(B)
    p = lambda a: C.c_void_p(a.ctypes.data)
    lib.pnolhost_set_jac_mode(int(jac_mode))
    try:
        st = lib.pnolhost_lm_batch(int(case["kind"]), p(sc), ptrs, len(cols), C.c_longlong(cols[0].size), p(ro), C.c_longlong(B), p(Xv), int(n),
                                   C.c_double(prm["lambda0"]), C.c_double(prm["factor"]), C.c_double(prm["dxgrad"]), C.c_double(prm["maxiter"]),
                                   C.c_double(prm["xmindiff"]), p(it), p(stp), p(chi), p(lam))
    finally:
        lib.pnolhost_set_jac_mode(0)
    return st, dict(X=Xv, iters=it, stopped=stp, chisq=chi, lam=lam)


def _same(a, b):
    return np.array_equal(np.asarray(a).view(np.uint64), np.asarray(b).view(np.uint64))


CASES = [("expcurve", capi.F_EXPCURVE, 3), ("cubic", capi.F_CUBIC, 4), ("lorentz1", capi.F_LORENTZ_SUM, 2),
         ("lorentz2", capi.F_LORENTZ_SUM, 4), ("lorentz4", capi.F_LORENTZ_SUM, 8)]


@pytest.mark.parametrize("name,kind,n", CASES, ids=[c[0] for c in CASES])
def test_each_problem_is_the_oracle_alone(standin, name, kind, n):
    sizes = [64, 0, 1, n - 1, n, 200, 37]
    case = LC.make_batch(kind, n, sizes, seed=n)
    st, got = run_batch(standin, case)
    assert st == 0, standin.pnolhost_last_error()
    for b in range(len(sizes)):
        want = LC.oracle_problem(case, b, PRM["lambda0"], PRM["factor"], PRM["dxgrad"], PRM["maxiter"], PRM["xmindiff"])
        assert _same(got["X"][b], want["X"]), (name, b)
        assert _same(got["chisq"][b], want["chisq"]) and _same(got["lam"][b], want["lam"]), (name, b)
        assert got["iters"][b] == want["iters"] and got["stopped"][b] == want["stopped"], (name, b)


def test_fits_reach_the_true_parameters(standin):
    case = LC.make_batch(capi.F_LORENTZ_SUM, 4, [256] * 6, seed=3)
    for mode in (capi.JAC_AUTO, capi.JAC_ANALYTIC):
        st, got = run_batch(standin, case, jac_mode=mode, maxiter=100)
        assert st == 0, standin.pnolhost_last_error()
        assert np.max(np.abs(got["X"] - case["Xtrue"])) < 1e-2, (mode, got["X"] - case["Xtrue"])


def test_analytic_mode_is_the_python_restatement(standin):
    """the stand-in's analytic loop is oracle_lm with J from the model's derivative: restated in Python (ExpCurve: J written out)"""
    case = LC.make_batch(capi.F_CUBIC, 4, [50, 3, 120], seed=9)
    st, got = run_batch(standin, case, jac_mode=capi.JAC_ANALYTIC)
    assert st == 0, standin.pnolhost_last_error()
    import oracle_lib as O
    for b in range(3):
        cols, m = LC.problem_columns(case, b)
        of = O.OFunctor(capi.F_CUBIC, (), (), cols, m)
        J = np.stack([-cols[0], -(cols[1] * cols[1]), -cols[1], -np.ones(m)], axis=1)
        want = LC.py_lm(lambda x: O.residual(of, x), lambda x, F: J, case["X0"][b], PRM["lambda0"], PRM["factor"], PRM["maxiter"],
                        PRM["xmindiff"])
        assert _same(got["X"][b], want["X"]) and _same(got["chisq"][b], want["chisq"]) and got["iters"][b] == want["iters"], b


def test_max_iter_zero_and_empty_batch(standin):
    case = LC.make_batch(capi.F_EXPCURVE, 3, [30, 40], seed=1)
    st, got = run_batch(standin, case, maxiter=0)
    assert st == 0 and _same(got["X"], case["X0"]) and np.all(got["iters"] == 0) and np.all(got["lam"] == PRM["lambda0"])
    for b in range(2):
        want = LC.oracle_problem(case, b, PRM["lambda0"], PRM["factor"], PRM["dxgrad"], 0, PRM["xmindiff"])
        assert _same(got["chisq"][b], want["chisq"])
    empty = dict(case, row_off=np.zeros(1, dtype=np.int64), X0=np.zeros((0, 3)))
    st, got = run_batch(standin, empty)
    assert st == 0 and got["X"].shape == (0, 3)


_REFUSAL = r"""
import ctypes as C, sys
import numpy as np
lib = C.CDLL(sys.argv[1], mode=C.RTLD_LOCAL)
lib.pnolhost_last_error.restype = C.c_char_p
p = lambda a: C.c_void_p(a.ctypes.data)
t = np.linspace(0, 1, 20); y = 2 * np.exp(0.5 * t) + 0.1
sc = np.zeros(8); ptrs = (C.c_void_p * 2)(t.ctypes.data, y.ctypes.data)
ro = np.array([0, 20], dtype=np.int64); X = np.array([1.0, 0.4, 0.0])
it, stp = np.zeros(1, dtype=np.int32), np.zeros(1, dtype=np.int32); chi, lam = np.zeros(1), np.zeros(1)
st = lib.pnolhost_lm_batch(101, p(sc), ptrs, 2, C.c_longlong(20), p(ro), C.c_longlong(1), p(X), 3, C.c_double(1e-3), C.c_double(10.0),
                           C.c_double(1e-7), C.c_double(10.0), C.c_double(1e-9), p(it), p(stp), p(chi), p(lam))
print(st, lib.pnolhost_last_error().decode())
"""


def test_lm_batch_on_a_c_abi_without_it_is_refused():
    """The host sources reference pnol_lm_batch weakly: linked against a C-ABI implementation without it (the unmodified stand-in, in a
    process where no libpnol_b200.so is loaded) they still build and load, and LevMarqBatch fails with PNOL_ERR_NO_FUNCTOR."""
    so = host_standin.base_path()
    if so is None:
        pytest.skip("no g++ on this box")
    r = subprocess.run([sys.executable, "-c", _REFUSAL, so], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    st, msg = r.stdout.strip().split(" ", 1)
    assert int(st) == capi.ERR_NO_FUNCTOR and "pnol_lm_batch" in msg and "not provided by the C-ABI implementation" in msg, r.stdout


def test_register_functor_lm_batch_rules():
    from test_user_gradient_cpu import _table
    lib = capi.load_library()
    fn = C.c_void_p(C.cast(lib.pnol_version, C.c_void_p).value)      # any non-NULL code address: registration never calls a launcher
    S, R = capi.F_USER_SCALAR_BASE + 740, capi.F_USER_RESIDUAL_BASE + 740
    keep = [_table(2, True), _table(1, False), _table(2, False), _table(2, False)]
    assert lib.pnol_register_functor(S, C.byref(keep[0])) == capi.PNOL_OK
    assert lib.pnol_register_functor(R, C.byref(keep[1])) == capi.PNOL_OK          # ABI 1
    assert lib.pnol_register_functor(R + 1, C.byref(keep[2])) == capi.PNOL_OK      # ABI 2
    for kind in (R, R + 1):
        assert lib.pnol_functor_has_lm_batch(kind) == 0
        assert lib.pnol_register_functor_lm_batch(kind, fn) == capi.PNOL_OK
        assert lib.pnol_functor_has_lm_batch(kind) == 1
    # a scalar kind, a kind without a table, a built-in kind, a kind outside every range and NULL are refused
    assert lib.pnol_register_functor_lm_batch(S, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_lm_batch(R + 2, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_lm_batch(capi.F_EXPCURVE, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_lm_batch(5000, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_lm_batch(R, None) == capi.ERR_INVALID
    assert lib.pnol_functor_has_lm_batch(S) == 0 and lib.pnol_functor_has_lm_batch(R + 2) == 0 and lib.pnol_functor_has_lm_batch(R) == 1
    for kind in (capi.F_EXPCURVE, capi.F_CUBIC, capi.F_LORENTZ_SUM):
        assert lib.pnol_functor_has_lm_batch(kind) == 1
    assert lib.pnol_functor_has_lm_batch(capi.F_ROSENBROCK) == 0
    # replacing the table drops the launcher attached to the old one
    assert lib.pnol_register_functor(R, C.byref(keep[3])) == capi.PNOL_OK
    assert lib.pnol_functor_has_lm_batch(R) == 0 and lib.pnol_functor_registered(R) == 1 and lib.pnol_functor_has_lm_batch(R + 1) == 1
