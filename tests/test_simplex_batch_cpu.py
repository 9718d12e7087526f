"""Batched simplex search without a GPU: oracle_simplex (tests/host_logic_standin.cpp, the CPU stand-in's pnol_simplex_batch,
reached through SimplexSearchBatch or the stand-in's C-ABI) bit for bit against the unmodified host SimplexSearch controller on the same
stand-in, start by start, each start given exactly its slice of the stream, for the six built-in objectives, both stream kinds,
offsets, non-default and edge parameters, with the evaluation counts; simplex_sort_perm (include/pnol/device/simplex_sort.hpp, the
permutation logic the kernel runs) against the library's simplexSort on random arrays with ties, signed zeros, infinities and NaN; the
refusals; pnol_register_functor_simplex_batch's rules and pnol_functor_has_simplex_batch for every kind."""
import ctypes as C
import subprocess
import sys

import numpy as np
import pytest

import host_standin
import simplex_batch_cases as SC
from parallelnonlinearoptimizationlibrary_b200 import capi


@pytest.fixture(scope="module")
def standin():
    hl = host_standin.load()
    if hl is None:
        pytest.skip("no g++ on this box")
    return hl


def check_against_serial(lib, name, X, prm, stream, got, offset=0):
    B, n = X.shape
    for b in range(B):
        vals = SC.draws(lib, stream, offset + b * n * n, n * n)
        st, want = SC.run_serial(lib, name, X[b], prm, vals)
        assert st == 0, lib.pnolhost_last_error()
        where = (name, n, stream[0], offset, b)
        assert SC.same(got["X"][b], want["X"]), (where, SC.diff_report(got["X"][b], want["X"]))
        assert SC.same(got["f0"][b], want["f0"]) and SC.same(got["fopt"][b], want["fopt"]), where
        assert got["iters"][b] == want["iters"], where
        assert got["evals"][b] == want["evals"], where          # the Objective's own counter of the serial run
        assert want["stream_pos"] == n * n
        assert (got["stop"][b] == 0) == (got["iters"][b] == prm["max_iter"]) and got["stop"][b] in (0, 1), where


STREAMS = [("seed", 12345, 1.0), ("values", None)]


def _stream(kind, B, n, seed):
    if kind[0] == "seed":
        return kind
    return ("values", np.random.default_rng(seed).uniform(size=B * n * n))


STOPS = set()


@pytest.mark.parametrize("stream_kind", ["seed", "values"])
@pytest.mark.parametrize("name", sorted(SC.OBJECTIVES))
def test_each_start_is_the_host_simplex_alone(standin, name, stream_kind):
    for n in SC.OBJECTIVES[name][2]:
        B = 7 if n < 64 else 4
        X = SC.starts(name, n, B, seed=n + 3)
        stream = _stream(("seed", 1000 + n, 1.0) if stream_kind == "seed" else ("values",), B, n, n)
        prm = SC.params(max_iter=150 if n < 33 else 60)
        st, got = SC.run_batch(standin, name, X, prm, stream)
        assert st == 0, standin.pnolhost_last_error()
        assert got["stream_pos"] == B * n * n and got["total_evals"] == int(np.sum(got["evals"]))
        check_against_serial(standin, name, X, prm, stream, got)
        STOPS.update(int(s) for s in got["stop"])


@pytest.mark.parametrize("kw", [dict(alpha=1.3, gamma=2.7, rho=0.35, sigma=0.8), dict(alpha=0.7, gamma=1.5, rho=0.6, sigma=0.25, init_rand_max=3.0),
                                dict(max_iter=0), dict(max_iter=1), dict(x_min_diff=0.0, max_iter=90), dict(init_rand_max=0.0),
                                dict(x_min_diff=1e-3, max_iter=400)])
def test_parameters(standin, kw):
    for name, n in (("rosenbrock", 3), ("rastrigin", 4), ("goldstein", 2), ("power:3", 5)):
        X = SC.starts(name, n, 6, seed=11)
        stream = ("seed", 77, 0.75)
        prm = SC.params(**kw)
        st, got = SC.run_batch(standin, name, X, prm, stream)
        assert st == 0, standin.pnolhost_last_error()
        check_against_serial(standin, name, X, prm, stream, got)
        STOPS.update(int(s) for s in got["stop"])
        if kw.get("max_iter") == 0:
            # no iteration: the best vertex of the sorted start simplex, evaluated once per vertex
            assert np.all(got["iters"] == 0) and np.all(got["stop"] == 0) and np.all(got["evals"] == n + 1)
        if kw.get("init_rand_max") == 0.0:
            # every vertex is the start: xdiff is 0 after one iteration
            assert np.all(got["iters"] == 1) and np.all(got["stop"] == 1)


@pytest.mark.parametrize("offset", [0, 5, 1000])
def test_stream_offsets_of_the_c_abi(standin, offset):
    for name, n in (("rosenbrock", 8), ("booth", 2)):
        kind, ints = SC.kind_of(name)
        X = SC.starts(name, n, 5, seed=offset)
        prm = SC.params()
        for stream in (("seed", 9, 1.0), ("values", np.random.default_rng(offset).uniform(size=offset + 5 * n * n))):
            st, got = SC.run_standin_capi(standin, kind, X, prm, stream, offset=offset, ints=ints)
            assert st == 0
            check_against_serial(standin, name, X, prm, stream, got, offset=offset)


def test_both_stop_codes_occur():
    if not STOPS:
        pytest.skip("runs after the parity tests")
    assert STOPS == {0, 1}


def test_base_class_find_min_is_one_start(standin):
    x0 = np.array([-1.2, 1.0, 0.5])
    prm = SC.params(max_iter=2000)
    vals = np.random.default_rng(5).uniform(size=9)
    SC.set_stream(standin, ("values", vals))
    Xv, f0, fopt = x0.copy(), np.zeros(1), np.zeros(1)
    p = lambda a: C.c_void_p(a.ctypes.data)
    try:
        assert standin.pnolhost_simplex_batch(b"rosenbrock", p(Xv), C.c_longlong(1), 3, p(SC.vec(prm)), 1, p(f0), p(fopt), None, None, None, None) == 0
    finally:
        standin.pnolhost_clear_stream()
    st, want = SC.run_serial(standin, "rosenbrock", x0, prm, vals)
    assert st == 0 and SC.same(Xv, want["X"]) and SC.same(f0[0], want["f0"]) and SC.same(fopt[0], want["fopt"])
    assert np.max(np.abs(Xv - 1.0)) < 1e-3


def test_short_explicit_stream_is_refused_and_nothing_is_written(standin):
    X = SC.starts("rosenbrock", 3, 4, seed=1)
    prm = SC.params()
    for size, offset in ((4 * 9 - 1, 0), (4 * 9, 1), (10, 11)):
        st, got = SC.run_standin_capi(standin, capi.F_ROSENBROCK, X, prm, ("values", np.full(size, 0.5)), offset=offset)
        assert st == SC.ERR_STREAM
        assert SC.same(got["X"], X) and np.all(got["iters"] == 0)
    st, _ = SC.run_standin_capi(standin, capi.F_ROSENBROCK, X, prm, ("values", np.full(36, 0.5)))
    assert st == capi.PNOL_OK


def _random_fvec(rng, N):
    pools = [np.array([0.0, -0.0, 1.0, 2.0, -1.0, np.inf, -np.inf, np.nan, 0.5]), np.array([1.0, 2.0, 3.0]), np.array([-3.0, -2.0, -1.0]),
             np.array([0.0, -0.0]), np.array([0.0, -0.0, 1.0]), np.array([1.0, np.nan, 2.0])]
    mode = rng.integers(0, 8)
    if mode < len(pools):
        f = rng.choice(pools[mode], size=N)
    elif mode == 6:
        f = rng.normal(size=N)
    else:
        f = np.round(rng.normal(size=N) * 2) / 2
    r = rng.random()
    if r < 0.05:
        f[0] = np.nan
    elif r < 0.10:
        f[1] = np.nan
    elif r < 0.15:
        f[1] = np.min(f[~np.isnan(f)]) if np.any(~np.isnan(f)) else f[1]     # index 1 ties with the minimum
    return np.ascontiguousarray(f, dtype=np.float64)


def test_sort_permutation_is_simplex_sort(standin):
    """simplex_sort_perm, with the stats gathered as G = 1 ... 32 lanes gather them, against the library's simplexSort on 10^5 arrays of
    N = 2 ... 65 entries: the permutation (hence the multiset of rows, duplicates included) and the resulting f, sentinels included"""
    rng = np.random.default_rng(2024)
    p = lambda a: C.c_void_p(a.ctypes.data)
    seen = dict(regime=0, outside=0, duplicates=0, one_first=0)
    for t in range(100000):
        N = int(rng.integers(2, 66)) if t % 4 else int(rng.integers(2, 10))
        f = _random_fvec(rng, N)
        fa, fb = f.copy(), f.copy()
        pa, pb = np.zeros(N, dtype=np.int32), np.zeros(N, dtype=np.int32)
        standin.standin_simplex_sort_reference(p(fa), N, p(pa))
        G = (1, 4, 8, 16, 32)[t % 5]
        regime = standin.standin_simplex_sort_perm(p(fb), N, G, p(pb))
        assert np.array_equal(pa, pb), (t, f, pa, pb)
        assert np.array_equal(fa.view(np.uint64), fb.view(np.uint64)) or SC.same(fa, fb), (t, f)
        seen["regime" if regime else "outside"] += 1
        seen["duplicates"] += int(len(set(pa.tolist())) < N)
        seen["one_first"] += int(regime and pa[0] == 1 and f[0] == f[1])
    assert min(seen.values()) > 100, seen


_REFUSAL = r"""
import ctypes as C, sys
import numpy as np
lib = C.CDLL(sys.argv[1], mode=C.RTLD_LOCAL)
lib.pnolhost_last_error.restype = C.c_char_p
p = lambda a: C.c_void_p(a.ctypes.data)
X = np.array([[-1.2, 1.0]]); prm = np.array([1.0, 2.0, 0.5, 0.5, 10, 1.0, 1e-7])
lib.pnolhost_set_stream(None, C.c_ulonglong(0), C.c_ulonglong(1), C.c_double(1.0))
f0, fopt = np.zeros(1), np.zeros(1); it, stop = np.zeros(1, dtype=np.int32), np.zeros(1, dtype=np.int32); ev = np.zeros(1, dtype=np.int64)
st = lib.pnolhost_simplex_batch(b"rosenbrock", p(X), C.c_longlong(1), 2, p(prm), 0, p(f0), p(fopt), p(it), p(stop), p(ev), None)
print(st, lib.pnolhost_last_error().decode())
"""


def test_simplex_batch_on_a_c_abi_without_it_is_refused():
    """The host sources reference pnol_simplex_batch weakly: linked against a C-ABI implementation without it (the unmodified stand-in)
    they still build and load, and SimplexSearchBatch fails with PNOL_ERR_NO_FUNCTOR."""
    so = host_standin.base_path()
    if so is None:
        pytest.skip("no g++ on this box")
    r = subprocess.run([sys.executable, "-c", _REFUSAL, so], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    st, msg = r.stdout.strip().split(" ", 1)
    assert int(st) == capi.ERR_NO_FUNCTOR and "pnol_simplex_batch" in msg and "not provided by the C-ABI implementation" in msg, r.stdout


def test_register_functor_simplex_batch_rules():
    from test_user_gradient_cpu import _table
    lib = capi.load_library()
    fn = C.c_void_p(C.cast(lib.pnol_version, C.c_void_p).value)      # any non-NULL code address: registration never calls a launcher
    S, R = capi.F_USER_SCALAR_BASE + 770, capi.F_USER_RESIDUAL_BASE + 770
    keep = [_table(2, True), _table(1, False), _table(2, True), _table(2, True)]
    assert lib.pnol_register_functor(S, C.byref(keep[0])) == capi.PNOL_OK
    assert lib.pnol_register_functor(R, C.byref(keep[1])) == capi.PNOL_OK
    assert lib.pnol_register_functor(S + 1, C.byref(keep[2])) == capi.PNOL_OK
    for kind in (S, S + 1):
        assert lib.pnol_functor_has_simplex_batch(kind) == 0
        assert lib.pnol_register_functor_simplex_batch(kind, fn) == capi.PNOL_OK
        assert lib.pnol_functor_has_simplex_batch(kind) == 1
    # a residual kind, a kind without a table, a built-in kind, a kind outside every range and NULL are refused
    assert lib.pnol_register_functor_simplex_batch(R, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_simplex_batch(S + 2, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_simplex_batch(capi.F_ROSENBROCK, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_simplex_batch(5000, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_simplex_batch(S, None) == capi.ERR_INVALID
    assert lib.pnol_functor_has_simplex_batch(R) == 0 and lib.pnol_functor_has_simplex_batch(S + 2) == 0
    # replacing the table drops the launcher attached to the old one
    assert lib.pnol_register_functor(S, C.byref(keep[3])) == capi.PNOL_OK
    assert lib.pnol_functor_has_simplex_batch(S) == 0 and lib.pnol_functor_registered(S) == 1 and lib.pnol_functor_has_simplex_batch(S + 1) == 1


_SCAN = r"""
import ctypes as C, sys
sys.path.insert(0, sys.argv[1])
from parallelnonlinearoptimizationlibrary_b200 import capi, hostapi
lib = capi.load_library()
hostapi.lib()
for so in sys.argv[2:]:
    C.CDLL(so, mode=C.RTLD_GLOBAL)
print(" ".join(str(k) for k in range(-1, 3101) if lib.pnol_functor_has_simplex_batch(k)))
"""


def _scan(libraries):
    r = subprocess.run([sys.executable, "-c", _SCAN, host_standin.ROOT] + libraries, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return [int(k) for k in r.stdout.split()]


def test_has_simplex_batch_for_every_kind():
    """each scan in a fresh process: the six built-in scalar objectives; with the user libraries of tests/user_functor/ loaded also
    every user scalar kind registered with PNOL_REGISTER_SCALAR_FUNCTOR (with or without derivatives), never a residual model"""
    import user_functor_lib as U
    import user_gradient_lib as UG
    import user_hessian_lib as UH
    import user_jacobian_lib as UJ
    import user_simplex_lib as US
    assert _scan([]) == [1, 2, 3, 4, 5, 6]
    libraries = [m.build_and_load()._name for m in (U, UG, UH, UJ, US)]
    want = sorted([1, 2, 3, 4, 5, 6, U.MY_F_TRID, U.MY_F_STYBLINSKI, UG.MYG_F_TRID, UG.MYG_F_STYBLINSKI, UH.MYH_F_QUADFORM, UH.MYH_F_STYBLINSKI]
                  + list(US.NAMES))
    assert _scan(libraries) == want
