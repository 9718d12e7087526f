"""The case table of tests/test_gpu_functor_kernels_exact.py checked without a GPU: every branch of the generic functor launchers
(include/pnol/device/functor_kernels.cuh, restated in exact_reference.py) is reached by some case, every size limit is run at the
limit, the order witnesses of the population sweep tell the sequential sum from every other order, and the wide residual model's host
jacobian() agrees with a numpy restatement of its operation order (bit for bit)."""
import numpy as np
import pytest

import exact_reference as R
import test_gpu_functor_kernels_exact as T      # its case tables; the module's tests need a GPU
import user_wide_lib as UW

OPTIN = R.SMEM_OPTIN_B200
WAVE_B = 148 * 2048 + 129


def _B(B):
    return WAVE_B if B == "wave" else B


# ---- every branch is reached by some GPU case -----------------------------------------------------------------------------------

def test_eval_batch_cases_reach_every_path_and_boundary():
    paths = {}
    for n, ld, off, B in T.EVAL_CASES:
        for p in R.eval_batch_path(n, ld, off, _B(B), OPTIN):
            paths.setdefault(p, []).append((n, ld, off, _B(B)))
    assert set(paths) == set(R.EVAL_BATCH_PATHS)
    # the boundaries on both sides: B = 63 / 64 of the warp-tile kernel, n = 23 / 24 and 113 / 114 of it, n = 227 / 228 of the tile
    warp = {"warp32_full", "warp32_ragged", "warp_general"}
    assert any(B == 64 and n == 32 for n, ld, off, B in paths["warp32_full"])
    assert any(B == 63 and n == 32 and off % 32 for n, ld, off, B in paths["tile_scalar"] + paths["tile16"])
    assert any(n == 24 for n, *_ in sum((paths[p] for p in warp), []))
    assert any(n == 23 for n, *_ in paths["tile_scalar"])
    assert any(n == 113 for n, *_ in paths["warp_general"])
    assert any(n == 114 for n, *_ in paths["tile_scalar"]) and any(n == 114 for n, *_ in paths["tile16"])
    assert any(n == 227 for n, *_ in paths["tile_scalar"]) and any(n == 226 for n, *_ in paths["tile16"])
    assert any(n == 228 for n, *_ in paths["direct"]) and any(n == 228 for n, *_ in paths["rowwise"])
    # both staging conditions of the tile kernel fail on their own: odd n, ld != n, rows 8 bytes off 16-byte alignment
    assert any(n % 2 and ld == n for n, ld, off, B in paths["tile_scalar"])
    assert any(ld != n for n, ld, off, B in paths["tile_scalar"])
    assert any(n % 2 == 0 and ld == n and off % 16 for n, ld, off, B in paths["tile_scalar"])
    # the warp-tile kernel at n == 32 through misaligned rows and through ld % 4 != 0
    assert any(off % 32 for n, ld, off, B in paths["warp32_full"]) and any(ld % 4 for n, ld, off, B in paths["warp32_full"])
    # batches beyond one wave (2048 threads an SM) on every grid-stride kernel and both row-wise kernels
    big = {p for n, ld, off, B in T.EVAL_CASES if B == "wave" for p in R.eval_batch_path(n, ld, off, WAVE_B, OPTIN)}
    assert big >= {"rowwise16", "rowwise", "warp32_full", "warp32_ragged", "warp_general", "tile16", "tile_scalar"}
    assert set(T.EVAL_B) >= {1, 31, 32, 33, 63, 64, 65}


def test_jacobian_cases_reach_every_tile_size_and_boundary():
    assert R.jacobian_tile_rows(225, OPTIN) == 128 and R.jacobian_tile_rows(226, OPTIN) == 64
    assert R.jacobian_tile_rows(447, OPTIN) == 64 and R.jacobian_tile_rows(448, OPTIN) == 32
    assert R.jacobian_tile_rows(879, OPTIN) == 32 and R.jacobian_tile_rows(880, OPTIN) is None
    ns = {n for n, m in T.AJ_CASES}
    assert {R.jacobian_tile_rows(n, OPTIN) for n in ns} == {128, 64, 32, None}
    assert ns >= {225, 226, 447, 448, 879, 880}
    # a ragged row count at every tile size, several waves at every one, untiled included
    for rows in (128, 64, 32, None):
        assert any(m != "wave" and m % 32 and R.jacobian_tile_rows(n, OPTIN) == rows for n, m in T.AJ_CASES)
    assert {R.jacobian_tile_rows(n, OPTIN) for n, m in T.AJ_CASES if m == "wave"} == {128, 64, 32, None}


def test_fd_jacobian_cases_reach_ragged_passes_both_quotients_and_the_limit():
    ns = set(T.JAC_N)
    assert R.max_n("fd_jacobian", OPTIN) in ns
    assert any(n > 32 and n % 32 for n in ns) and any(n > 32 and n % 32 == 0 for n in ns) and any(n < 32 for n in ns)
    ms = {m for n, m in T.JAC_CASES}
    assert ms >= {1, 127, 128, 129, "wave"}
    rng = np.random.default_rng(0)
    fast = {k: all(R.recip_usable(d) for d in T._dx(k, 5, rng)) for k in T.DX_KINDS}
    slow = {k: not any(R.recip_usable(d) for d in T._dx(k, 5, rng)) for k in T.DX_KINDS}
    assert fast["1e-7"] and fast["1e-5"] and fast["negative"] and slow["1e-70"] and slow["all-ones"]
    assert any(d < 0 for d in T._dx("negative", 5, rng))
    # the 1e-70 step moves some coordinates (nonzero dividends through `/`), not all (zero ones too)
    cols, x, _ = T._wide_problem(40, 300, 1)
    assert np.any(x + 1e-70 != x) and np.any(x + 1e-70 == x)
    J, _ = UW.host_fd_jacobian(cols, x, T._dx("1e-70", 40, rng))
    assert np.count_nonzero(J) >= 4 and np.count_nonzero(J == 0) > 0
    # a dividend below 2^-700 on the rows with t = 2^-760 (the model's forward difference at column a is about dx t)
    assert not R.dividend_in_range(1e-7 * 2.0 ** -760) and R.dividend_in_range(1e-7)


def test_size_limits_are_run_at_the_limit():
    assert R.max_n("fd_points", OPTIN) == 29056 and R.max_n("fd_points", OPTIN) in T.FDG_N
    assert R.max_n("residual", OPTIN) == 29056 and R.max_n("residual", OPTIN) in T.RES_N
    assert R.max_n("fd_jacobian", OPTIN) == 8277
    assert R.max_n("alpha_pool", OPTIN) == 13672
    assert R.max_n("hessian", OPTIN) == 28000 and R.max_n("alpha_slope", OPTIN) == 14528
    # each is the largest n whose shared memory fits, n + 1 does not
    need = {"fd_points": lambda n: 8 * n, "residual": lambda n: 8 * n, "fd_hessian": lambda n: 8 * n, "gradient": lambda n: 8 * n,
            "hessian": lambda n: 8 * (32 * 33 + n), "alpha_pool": lambda n: 17 * n + 16, "alpha_slope": lambda n: 16 * n,
            "fd_jacobian": lambda n: 8 * (3 * n + 128 * 33)}
    for name, bytes_ in need.items():
        n = R.max_n(name, OPTIN)
        assert bytes_(n) <= OPTIN < bytes_(n + 1), name


def test_gpu_cases_cover_the_issue_sizes():
    assert set(T.FDG_N) >= {1, 31, 32, 33, 255, 256, 257}
    assert set(T.FDH_N) == {2, 33, 200, 1000}
    assert {n for n, m in T.JAC_CASES if m == "wave"} >= {1, 33, 100}          # several waves, one pass and several ragged passes


# ---- order witnesses ------------------------------------------------------------------------------------------------------------

def _tree(v):
    if len(v) == 1:
        return float(v[0])
    h = len(v) // 2
    return _tree(v[:h]) + _tree(v[h:])


def _other_orders(v):
    """sums of v in orders a kernel might take instead of the sequential one"""
    n = len(v)
    out = {"reversed": R.seq_sum(v[::-1]), "pairwise": _tree(v), "numpy": float(np.sum(v))}
    if n % 4 == 0:
        s = 0.0
        for k in range(0, n, 4):
            s = s + ((v[k] + v[k + 1]) + (v[k + 2] + v[k + 3]))         # four terms added pairwise, then to the sum
        out["grouped4"] = s
    for st in (2, 4, 8, 16, 32):
        if st < n:
            out["stride%d" % st] = R.seq_sum([R.seq_sum(v[r::st]) for r in range(st)])
    return out


@pytest.mark.parametrize("n", sorted({n for n, *_ in T.EVAL_GEOMS if n >= 3}))
def test_order_witnesses_tell_the_sequential_sum_from_every_other_order(n):
    ws = R.order_witnesses(n)
    seq = [R.seq_sum(w) for w in ws]
    assert seq[0] == 1.0 and seq[2] == (n - 3) * R.U
    others = [_other_orders(w) for w in ws]
    for name in others[0]:
        if name == "numpy" and n < 8:
            continue                                 # numpy adds fewer than 8 terms one by one
        assert any(o[name] != s for o, s in zip(others, seq)), (n, name)


# ---- the wide residual model ----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("n,m", [(1, 5), (2, 40), (3, 40), (7, 300), (33, 300), (1000, 129)])
def test_wide_model_host_jacobian_matches_numpy(n, m):
    rng = np.random.default_rng(n + m)
    cols = UW.columns(m, rng, tiny_rows=np.arange(5, m, T.TINY_DIVIDEND_ROW))
    x = rng.uniform(-2.0, 2.0, n)
    J, F = UW.host_rows(cols, x)
    Jn = UW.np_jacobian(cols, x)
    assert np.array_equal(J.view(np.uint64), Jn.view(np.uint64))
    a, b = UW.cols_ab(m, n)
    t, s, y = cols
    assert np.array_equal(F, y - (x[a] * t + (x[b] * x[b]) * s))
    if n in (7, 33):
        assert np.any(a == b) and np.any(a != b)                 # rows whose two columns coincide, and rows whose do not


def test_wide_model_fd_reference_keeps_the_sign_of_zero_and_reaches_tiny_dividends():
    n, m = 40, 200
    rng = np.random.default_rng(3)
    cols = UW.columns(m, rng, tiny_rows=np.arange(5, m, T.TINY_DIVIDEND_ROW))
    x = rng.uniform(-2.0, 2.0, n)
    dx = -1e-6 * (1.0 + np.arange(n) % 7)
    J, F = UW.host_fd_jacobian(cols, x, dx)
    a, b = UW.cols_ab(m, n)
    untouched = np.ones((m, n), dtype=bool)
    untouched[np.arange(m), a] = untouched[np.arange(m), b] = False
    assert np.all(J[untouched] == 0) and np.all(np.signbit(J[untouched]))        # (r_0 - r_0) / dx with dx < 0 is -0
    Rp = J * dx[None, :]
    tiny = np.arange(5, m, T.TINY_DIVIDEND_ROW)
    assert tiny.size and not any(R.dividend_in_range(v) for v in (J[tiny, a[tiny]] * dx[a[tiny]]))
    assert np.all(np.isfinite(Rp))
