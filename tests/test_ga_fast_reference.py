"""The O(Npop log Npop) GA reference (tests/ga_fast_reference.cpp) against the literal O(Npop^2 n) oracle_ga, bit for bit in every
output, at populations the oracle can run (Npop <= 3000). tests/test_gpu_ga_large.py relies on this equality to check the GPU
generation at 65k - 1M individuals. The last tests show that the comparison notices a wrong tie order and a missed duplicate."""
import numpy as np
import pytest

import ga_fast_reference as R
import oracle_lib as O
from parallelnonlinearoptimizationlibrary_b200 import capi
from test_gpu_ga import GA_CASES

OUTPUTS = ("xpop", "F", "cross_idx", "mut_idx", "elite_idx", "X")
SCALARS = ("iters", "f0", "fOpt", "stream_pos", "sizes")


def _differences(a, b):
    bad = [k for k in OUTPUTS if a[k].tobytes() != b[k].tobytes()]          # bits: -0 and +0 differ
    bad += [k for k in SCALARS if np.asarray(a[k]).tobytes() != np.asarray(b[k]).tobytes()]
    return bad


def _both(*args, **kw):
    fast = R.ga(*args, **kw)
    kw.pop("on_generation", None)
    return fast, R.oracle_ga(*args, **kw)


def _user(kind):
    """(functor, objective pointer) of a test objective of my_ga_objectives.hpp"""
    return O.OFunctor(0), R.objective_fn(kind)


@pytest.fixture(autouse=True)
def _no_faults():
    R.set_faults()
    yield
    R.set_faults()


@pytest.mark.parametrize("kind,ints,n,npop,gens,box", GA_CASES)
def test_ga_cases_of_the_gpu_suite(kind, ints, n, npop, gens, box):
    lb, ub = np.full(n, -box), np.full(n, box)
    stream = dict(seed=12345 + n, scale=1.0 - 1.0 / npop)
    for stop in (1, gens):
        fast, ref = _both(O.OFunctor(kind, (), ints), np.full(n, 0.3 * box), lb, ub, npop, gens, stream, stop_after=stop)
        assert ref["iters"] == stop
        assert _differences(fast, ref) == []


@pytest.mark.parametrize("n,npop,box", [(1, 3000, 1.0), (2, 3000, 0.05), (1, 200, 1e-3)])
def test_small_n_many_duplicates(n, npop, box):
    """n = 1 and 2: crossover children copy whole parents, so most rows of XpopNew repeat an earlier or later one"""
    lb, ub = np.full(n, -box), np.full(n, box)
    stream = dict(seed=31 + n, scale=1.0 - 2.0 ** -20)
    for kind in (capi.F_POWER, capi.F_RASTRIGIN):
        f = O.OFunctor(kind, (), (2,) if kind == capi.F_POWER else ())
        fast, ref = _both(f, np.full(n, 0.5 * box), lb, ub, npop, 5, stream)
        assert ref["iters"] == 5
        assert _differences(fast, ref) == []


@pytest.mark.parametrize("kind", [R.MY_F_QUANTIZED, R.MY_F_SIGNED_ZERO])
@pytest.mark.parametrize("npop", [300, 3000])
def test_user_objectives(kind, npop):
    n = 8
    lb, ub = np.full(n, -5.12), np.full(n, 5.12)
    f, fn = _user(kind)
    fast, ref = _both(f, np.zeros(n), lb, ub, npop, 6, dict(seed=7, scale=1.0 - 2.0 ** -20), fn=fn)
    assert ref["iters"] == 6
    assert _differences(fast, ref) == []
    F = ref["F"]
    if kind == R.MY_F_QUANTIZED:
        assert np.all(np.isin(F, np.arange(33.0))) and F[0] == 0.0
    else:                                                          # both zeros present: their order is the sort's tie order
        assert np.sum((F == 0) & np.signbit(F)) >= 5 and np.sum((F == 0) & ~np.signbit(F)) >= 5


def _counter_run(f, n, npop, gens, box, stop_after, fn=None):
    lb, ub = np.full(n, -box), np.full(n, box)
    return R.ga(f, np.zeros(n), lb, ub, npop, gens, dict(seed=3, scale=1.0 - 2.0 ** -20), stop_after=stop_after, fn=fn)


@pytest.mark.parametrize("objective", ["quantized", "rastrigin"])
def test_explicit_stream_with_zeros_and_exact_ratios(objective):
    """explicit streams holding 0.0, 1.0 and values equal to ratio[k] = fitness[k] / maxFitness of the start population: the
    selection test `selectValue <= ratio` at equality and the index round(0 * Npop) = 0"""
    n, npop, gens, box = 8, 2000, 3, 5.12
    f, fn = _user(R.MY_F_QUANTIZED) if objective == "quantized" else (O.OFunctor(capi.F_RASTRIGIN), None)
    lb, ub = np.full(n, -box), np.full(n, box)
    start = R.ga(f, np.zeros(n), lb, ub, npop, gens, dict(seed=3, scale=1.0 - 2.0 ** -20), stop_after=0, fn=fn)
    F = start["F"]
    ratio = (F[-1] - F) ** 2 / (F[-1] - F[0]) ** 2
    need = _counter_run(f, n, npop, gens, box, gens, fn=fn)["stream_pos"]
    rng = np.random.default_rng(5)
    values = O.stream_array(11, 3 * need, 1.0 - 2.0 ** -20)
    special = np.concatenate([[0.0, 1.0], rng.choice(ratio, 64)])
    hit = rng.random(values.size) < 0.15
    values[hit] = rng.choice(special, hit.sum())
    stream = dict(values=values)
    fast, ref = _both(f, np.zeros(n), lb, ub, npop, gens, stream, fn=fn)
    assert ref["iters"] == gens
    assert _differences(fast, ref) == []
    if objective == "quantized":                                   # ratios (32 - f)^2 / 1024: the edges of the GPU's acceptance table
        assert np.all(np.isin(ratio, np.arange(33.0) ** 2 / 1024))


def test_explicit_stream_that_ends_at_a_generation():
    n, npop, gens, box = 5, 600, 3, 5.12
    f = O.OFunctor(capi.F_RASTRIGIN)
    lb, ub = np.full(n, -box), np.full(n, box)
    end = _counter_run(f, n, npop, gens, box, 2)["stream_pos"]      # generation 2's last draw
    values = O.stream_array(3, end, 1.0 - 2.0 ** -20)
    fast, ref = _both(f, np.zeros(n), lb, ub, npop, gens, dict(values=values), stop_after=2)
    assert ref["iters"] == 2 and ref["stream_pos"] == end
    assert _differences(fast, ref) == []
    fast, ref = _both(f, np.zeros(n), lb, ub, npop, gens, dict(values=values[:-1]), stop_after=2)
    assert ref["iters"] == fast["iters"] == -2


def test_static_stop():
    n, npop = 3, 50
    lb, ub = np.full(n, -1.0), np.full(n, 1.0)
    fast, ref = _both(O.OFunctor(capi.F_POWER, (), (2,)), np.zeros(n), lb, ub, npop, 40, dict(seed=3, scale=1.0 - 1.0 / npop), nstatic=2.0)
    assert ref["iters"] == 2
    assert _differences(fast, ref) == []


def test_generation_callback_sees_every_generation():
    n, npop, gens = 4, 500, 4
    lb, ub = np.full(n, -5.12), np.full(n, 5.12)
    f = O.OFunctor(capi.F_RASTRIGIN)
    seen = {}
    R.ga(f, np.full(n, 1.0), lb, ub, npop, gens, dict(seed=9, scale=0.999), on_generation=lambda g, *out: seen.__setitem__(g, out))
    assert sorted(seen) == list(range(0, gens + 1))
    for g in seen:
        ref = R.oracle_ga(f, np.full(n, 1.0), lb, ub, npop, gens, dict(seed=9, scale=0.999), stop_after=g)
        X, F, cross, mut, elite, pos = seen[g]
        assert np.array_equal(X, ref["xpop"]) and np.array_equal(F, ref["F"]) and pos == ref["stream_pos"]
        assert np.array_equal(cross, ref["cross_idx"]) and np.array_equal(mut, ref["mut_idx"]) and np.array_equal(elite, ref["elite_idx"])


def test_refuses_populations_the_sentinel_sort_does_not_sort():
    """max F <= 0 or a non-finite F: the reference's popSort is not a stable sort there (the GPU library refuses them too)"""
    n, npop = 2, 100
    cube = O.OFunctor(capi.F_POWER, (), (3,))
    neg = R.ga(cube, np.full(n, -1.5), np.full(n, -2.0), np.full(n, -1.0), npop, 3, dict(seed=1, scale=0.99))
    assert neg["iters"] == R.REFUSED
    huge = R.ga(O.OFunctor(capi.F_POWER, (), (2,)), np.full(n, 1e200), np.full(n, -1e200), np.full(n, 1e200), npop, 3,
                dict(seed=1, scale=0.99))
    assert huge["iters"] == R.REFUSED


# ---- sensitivity: a subtly wrong reference must fail the comparison ----
def test_a_flipped_tie_order_is_caught():
    n = 8
    for kind in (R.MY_F_QUANTIZED, R.MY_F_SIGNED_ZERO):
        f, fn = _user(kind)
        args = (f, np.zeros(n), np.full(n, -5.12), np.full(n, 5.12), 3000, 6, dict(seed=7, scale=1.0 - 2.0 ** -20))
        ref = R.oracle_ga(*args, fn=fn)
        R.set_faults(flip_ties=True)
        assert {"F", "xpop"} & set(_differences(R.ga(*args, fn=fn), ref))
        R.set_faults()
        assert _differences(R.ga(*args, fn=fn), ref) == []


def test_one_missed_duplicate_is_caught():
    n, npop = 1, 3000
    f = O.OFunctor(capi.F_POWER, (), (2,))
    args = (f, np.full(n, 0.5), np.full(n, -1.0), np.full(n, 1.0), npop, 3, dict(seed=32, scale=1.0 - 2.0 ** -20))
    ref = R.oracle_ga(*args)
    R.set_faults(miss_duplicate=True)
    bad = _differences(R.ga(*args), ref)
    assert "stream_pos" in bad and "xpop" in bad
