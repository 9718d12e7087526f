"""GA parity (a15 / a16): population, objective values, parent indices and stream position are compared BIT-EXACTLY with
the oracle's restatement of GeneticAlgorithmMPI::findMinBnd driven by the same host-supplied random stream."""
import numpy as np
import pytest

import oracle_lib as O
from parallelnonlinearoptimizationlibrary_b200 import capi

pytestmark = pytest.mark.gpu


def test_pop_sort_stable_with_ties(ctx):
    rng = np.random.default_rng(0)
    for npop, n in ((1, 3), (7, 2), (300, 5), (5000, 32)):
        F = np.round(rng.uniform(0.0, 50.0, npop), 1)          # many ties
        if npop > 3:
            F[3] = -2.5
            F[1] = 1e300
        F = np.abs(F) if npop == 7 else F
        F = np.where(F <= 0, 0.5, F) if False else F
        X = rng.normal(size=(npop, n))
        Fpos = np.abs(F) + 0.1                                  # popSort's 2*FMax sentinel needs FMax > 0
        Xg, Fg = ctx.ga_pop_sort(X, Fpos)
        Xw, Fw = O.ga_pop_sort(X, Fpos)
        assert np.array_equal(Fg, Fw) and np.array_equal(Xg, Xw)
    # negative and mixed-sign keys sort correctly too (the reference's sentinel breaks there; compare with numpy stable)
    F = rng.normal(size=4000)
    X = rng.normal(size=(4000, 3))
    Xg, Fg = ctx.ga_pop_sort(X, F)
    order = np.argsort(F, kind="stable")
    assert np.array_equal(Fg, F[order]) and np.array_equal(Xg, X[order])


def test_check_bounds_stage(ctx):
    rng = np.random.default_rng(1)
    npop, n = 3000, 7
    lb, ub = np.full(n, -1.0), np.linspace(0.5, 2.0, n)
    X = rng.uniform(-1.5, 2.2, size=(npop, n))
    X[10] = 0.0                                                # fully inside
    stream = dict(seed=99, scale=1.0)
    # evaluation flags: repaired rows are set, the others keep what the caller passed
    for ind in (None, rng.integers(0, 2, npop, dtype=np.uint8)):
        Xg, ig, pg = ctx.ga_check_bounds(X, lb, ub, stream, pos=17, ind=ind)
        Xw, iw, pw = O.ga_check_bounds(X, lb, ub, stream, pos=17, ind=ind)
        assert pg == pw and np.array_equal(ig, iw) and np.array_equal(Xg, Xw)
    assert ig[10] == ind[10] and np.any(ig == 0)
    # explicit stream, exhausted -> error
    with pytest.raises(capi.PnolError):
        ctx.ga_check_bounds(X, lb, ub, dict(values=np.linspace(0, 0.9, 5)), pos=0)


def test_check_identical_stage(ctx):
    rng = np.random.default_rng(2)
    npop, n = 2000, 4
    lb, ub = np.full(n, -5.0), np.full(n, 5.0)
    X = rng.normal(size=(npop, n))
    X[5] = X[900]
    X[6] = X[900]
    X[100] = X[101]
    X[1999] = X[0]
    X[300, 0] = 0.0
    X[301] = X[300]
    X[301, 0] = -0.0                                           # -0 == +0 in the reference's comparison
    X[400, 1] = np.nan
    X[401] = X[400]                                            # bit-identical, but NaN != NaN: not duplicates
    stream = dict(seed=5, scale=1.0)
    # evaluation flags: replaced rows are set, the others keep what the caller passed
    for ind in (None, rng.integers(0, 2, npop, dtype=np.uint8)):
        Xg, ig, pg = ctx.ga_check_identical(X, lb, ub, stream, pos=3, ind=ind)
        Xw, iw, pw = O.ga_check_identical(X, lb, ub, stream, pos=3, ind=ind)
        assert pw == 3 + 5 * n
        assert pg == pw and np.array_equal(ig, iw) and np.array_equal(Xg, Xw, equal_nan=True)
        assert np.array_equal(Xg[400:402], X[400:402], equal_nan=True)
    assert np.any(ig == 0)
    # all rows identical (the reference's call on the zero-initialised XpopNew, GeneticAlgorithmMPI.cpp:71)
    Z = np.zeros((500, n))
    Xg, ig, pg = ctx.ga_check_identical(Z, lb, ub, stream, pos=0)
    Xw, iw, pw = O.ga_check_identical(Z, lb, ub, stream, pos=0)
    assert pg == pw == 499 * n and np.array_equal(Xg, Xw) and np.array_equal(ig, iw)


def test_stage_size_limits(ctx):
    """the stand-alone duplicate check counts replaced rows in 24 bits: a larger population is refused, not miscounted"""
    X = np.zeros(((1 << 24) + 1, 1))
    with pytest.raises(capi.PnolError):
        ctx.ga_check_identical(X, [-1.0], [1.0], dict(seed=1, scale=1.0))


GA_CASES = [
    # kind, n, npop, generations, box
    (capi.F_POWER, (2,), 4, 150, 6, 10.0),              # testGAParallel (Source/Examples.cpp:307-337): PowerObject, n = 4, box +-10
    (capi.F_RASTRIGIN, (), 32, 400, 4, 5.12),
    (capi.F_RASTRIGIN, (), 5, 3000, 3, 5.12),
    (capi.F_ROSENBROCK, (), 3, 64, 8, 2.0),
]


@pytest.mark.parametrize("kind,ints,n,npop,gens,box", GA_CASES)
def test_ga_generations_bit_exact(ctx, kind, ints, n, npop, gens, box):
    lb, ub = np.full(n, -box), np.full(n, box)
    x0 = np.full(n, 0.3 * box)
    stream = dict(seed=12345 + n, scale=1.0 - 1.0 / npop)
    f = ctx.functor(kind, (), ints)
    of = O.OFunctor(kind, (), ints)
    ga = ctx.ga_create(f, n, lb, ub, npop, gens, stream)
    f0 = ga.init(x0)
    for g in range(1, gens + 1):
        ga.generation()
        want = O.ga(of, x0, lb, ub, npop, gens, stream, stop_after=g)
        assert want["iters"] == g
        st = ga.status()
        X, F = ga.population()
        cross, mut, elite = ga.indices()
        assert st.generation == g
        assert (st.n_elite, st.n_elite_mut, st.n_cross, st.n_rand) == want["sizes"]
        assert np.array_equal(cross, want["cross_idx"]), "crossover parents, generation %d" % g
        assert np.array_equal(mut, want["mut_idx"]), "mutation parents, generation %d" % g
        assert np.array_equal(elite, want["elite_idx"]), "elite-mutation parents, generation %d" % g
        assert st.stream_pos == want["stream_pos"], "stream position, generation %d" % g
        assert np.array_equal(F, want["F"]) and np.array_equal(X, want["xpop"]), "population, generation %d" % g
    assert f0 == want["f0"]
    ga.close()


def test_ga_static_stop_and_invalid_fractions(ctx):
    n, npop = 3, 50
    lb, ub = np.full(n, -1.0), np.full(n, 1.0)
    f = ctx.functor(capi.F_POWER, (), (2,))
    with pytest.raises(capi.PnolError):                         # the reference prints "666 GA fractions..." and exit(0)s
        ctx.ga_create(f, n, lb, ub, npop, 5, dict(seed=1, scale=0.97), elite_frac=0.5, cross_frac=0.4, elite_mut_frac=0.2)
    stream = dict(seed=3, scale=1.0 - 1.0 / npop)
    ga = ctx.ga_create(f, n, lb, ub, npop, 40, stream, nstatic=2.0)
    ga.run(np.zeros(n), 40)                                     # the optimum is in the start population: F[0] never changes
    want = O.ga(O.OFunctor(capi.F_POWER, (), (2,)), np.zeros(n), lb, ub, npop, 40, stream, nstatic=2.0)
    st = ga.status()
    assert st.stopped == 1 and st.generation == want["iters"] == 2
    X, F = ga.population()
    assert np.array_equal(F, want["F"]) and np.array_equal(X, want["xpop"])


@pytest.mark.parametrize("npop", [70_000, 300_000])
def test_bucket_sort_equals_radix_sort(ctx, npop):
    """popSort at large Npop runs as splitter buckets + per-bucket shared-memory sorts (csrc/ga_pipeline.cu, 6'); PNOL_GA_SORT=radix
    keeps the cooperative radix kernel, which the small-population tests above pin to the oracle. Same generations, same bits:
    objective values, permutation (through the materialised population) and stream position."""
    import os
    n = 8
    f = ctx.functor(capi.F_RASTRIGIN)
    out = []
    for mode in ("radix", None):
        if mode:
            os.environ["PNOL_GA_SORT"] = mode
        else:
            os.environ.pop("PNOL_GA_SORT", None)
        ga = ctx.ga_create(f, n, np.full(n, -5.12), np.full(n, 5.12), npop, 12, dict(seed=99, scale=1.0 - 2.0 ** -20), nstatic=1e9)
        ga.init(np.full(n, 0.7))
        for _ in range(6):
            ga.generation()
        X, F = ga.population()
        out.append((X, F, ga.status().stream_pos))
        ga.close()
    os.environ.pop("PNOL_GA_SORT", None)
    assert np.array_equal(out[0][1], out[1][1]) and np.array_equal(out[0][0], out[1][0]) and out[0][2] == out[1][2]
    assert np.all(np.diff(out[1][1]) >= 0)
