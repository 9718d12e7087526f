"""GA generations at 65k - 1M individuals, bit for bit against the O(Npop log Npop) reference (tests/ga_fast_reference.cpp, itself
equal to oracle_ga bit for bit: tests/test_ga_fast_reference.py). Every generation compares X, F, the crossover / mutation /
elite-mutation parents, the four sizes and the stream position.

Each case exists for a path of csrc/ga_pipeline.cu. Where that path depends on the data, the test restates the host's rule in numpy
and asserts that the path ran:
  * popSort: the bucket sort runs at Npop >= 65536. Its splitters are the previous generation's sorted objective values,
    spl[b] = key(F_old[b N / 4096]) for b >= 1, and a key's bucket is the number of splitters <= key. Buckets of up to 1024 keys
    are sorted by the <128, 8> kernel, those of 1025 - 8192 by <512, 16>, and one bucket above 8192 sends the whole sort to the
    radix kernel. The bucket sizes depend only on the multiset of the new objective values, which is the next sorted F;
  * mutation: the geometry of generation 1 (the host's acceptance-rate estimate starts at 0.25) decides whether the compose
    kernel holds its tables in shared memory and over how many segments it composes them."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import pytest

import ga_fast_reference as R
import oracle_lib as O
import user_functor_lib
from parallelnonlinearoptimizationlibrary_b200 import capi

pytestmark = pytest.mark.gpu

K_BUCKETS, K_CAP, K_CAP_LARGE = 4096, 1024, 8192
SCALE = 1.0 - 2.0 ** -20


@pytest.fixture(scope="module")
def ga_objectives(ctx):
    """tests/user_functor/my_ga_objectives.cu compiled out of tree and loaded: registers the quantized and signed-zero objectives"""
    from parallelnonlinearoptimizationlibrary_b200 import hostapi
    capi.load_library()
    hostapi.lib()
    d = tempfile.mkdtemp(prefix="pnol_ga_objectives_")
    out = os.path.join(d, "libmy_ga_objectives.so")
    cmd = [user_functor_lib.nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-fmad=false", "-Xcompiler",
           "-fPIC,-ffp-contract=off", "-I" + os.path.join(user_functor_lib.ROOT, "include"), "-I" + user_functor_lib.SRC, "-shared",
           "-o", out, os.path.join(user_functor_lib.SRC, "my_ga_objectives.cu"), "-L" + user_functor_lib.LIBDIR, "-lpnol_b200",
           "-Xlinker", "-rpath", "-Xlinker", user_functor_lib.LIBDIR]
    subprocess.run(cmd, check=True, cwd=d, capture_output=True, text=True)
    lib = C.CDLL(out, mode=C.RTLD_GLOBAL)
    assert lib.my_ga_registration_status() == 0
    return lib


def sort_key(F):
    """double_to_key of csrc/ga_common.cuh: order-preserving, -0 and +0 alike"""
    b = np.ascontiguousarray(F, dtype=np.float64).view(np.uint64).copy()
    b[b == np.uint64(1 << 63)] = 0
    return np.where(b >> np.uint64(63) != 0, ~b, b | np.uint64(1 << 63))


def sort_path(F_old, F_new):
    """which kernel sorted a generation under the bucket sort: 'small', 'large' (<512, 16> ran) or 'radix' (fallback)"""
    N = F_old.size
    spl = sort_key(F_old[(np.arange(1, K_BUCKETS, dtype=np.int64) * N) // K_BUCKETS])
    counts = np.bincount(np.searchsorted(spl, sort_key(F_new), side="right"), minlength=K_BUCKETS)
    top = int(counts.max())
    return "radix" if top > K_CAP_LARGE else ("large" if top > K_CAP else "small")


def mut_geometry(n, nrand, sm_count, rate=0.25):
    """the mutation stage's geometry, restated from pipe_enqueue (csrc/ga_pipeline.cu, stage 2) for window_scale = 1"""
    g = 2 if n % 2 == 0 else 1
    stepA, stepR = (n + 2) // g, 2 // g
    sd = stepA
    rate = max(rate, 1e-3)
    cand = nrand * (stepA + stepR * (1.0 / rate - 1.0)) * 1.12 + 8.0 * 1024
    nsub_max = (96 * 1024) // ((1024 // 32) * 4 + sd * 8)
    subs = int(cand / 1024) + 1
    min_subs = (sd + 1023) // 1024
    nsub = max(min_subs, min(nsub_max, (subs + 6 * sm_count - 1) // (6 * sm_count)))
    nctas = (subs + nsub - 1) // nsub
    ctab = nctas * sd
    nseg = (nctas + 31) // 32
    seg_bytes = nseg * sd * 12 + nseg * 12 + 64
    return dict(g=g, nctas=nctas, nseg=nseg, in_smem=ctab * 8 + seg_bytes <= 200 * 1024)


def _digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def reference(kind, n, npop, gens, stream, x0, box, ints=(), nstatic=50.0, stop_after=-1):
    """the fast reference's start population and generations: {g: (X digest, F, cross, mut, elite, pos)}"""
    fn = R.objective_fn(kind)
    f = O.OFunctor(0 if fn is not None else kind, (), ints)
    seen = {}
    R.ga(f, x0, np.full(n, -box), np.full(n, box), npop, gens, stream, nstatic=nstatic, stop_after=stop_after, fn=fn,
         on_generation=lambda g, X, F, cr, mu, el, pos: seen.__setitem__(g, (_digest(X), F, cr, mu, el, pos)))
    return seen


def check_generation(ga, want, g):
    X, F = ga.population()
    cross, mut, elite = ga.indices()
    st = ga.status()
    wx, wF, wc, wm, we, wpos = want
    assert st.generation == g
    assert (st.n_elite, st.n_elite_mut, st.n_cross, st.n_rand) == (ga.npop - wm.size - wc.shape[0] - we.shape[0], we.shape[0],
                                                                 wc.shape[0], wm.size)
    assert st.stream_pos == wpos, "stream position, generation %d" % g
    assert F.tobytes() == wF.tobytes(), "objective values, generation %d: %d differ" % (g, np.sum(F.view(np.uint64) != wF.view(np.uint64)))
    assert _digest(X) == wx, "population, generation %d" % g
    assert np.array_equal(cross[:wc.shape[0]], wc), "crossover parents, generation %d" % g
    assert np.array_equal(mut[:wm.size], wm), "mutation parents, generation %d" % g
    assert np.array_equal(elite[:we.shape[0]], we), "elite-mutation parents, generation %d" % g
    return F


def run_case(ctx, kind, n, npop, gens, x0, box, ints=(), stream=None, max_gens=None, on_generation=None):
    """GPU generations 1..gens against the reference; returns the sorted F of generations 0..gens"""
    stream = stream or dict(seed=1000 + n, scale=SCALE)
    max_gens = max_gens or gens
    want = reference(kind, n, npop, max_gens, stream, x0, box, ints, stop_after=gens)
    f = ctx.functor(kind, (), ints)
    ga = ctx.ga_create(f, n, np.full(n, -box), np.full(n, box), npop, max_gens, stream)
    try:
        ga.init(x0)
        Fs = [check_population(ga, want[0])]
        for g in range(1, gens + 1):
            before = ctx.launches()
            ga.generation()
            if on_generation:
                on_generation(g, ctx.launches() - before)
            Fs.append(check_generation(ga, want[g], g))
    finally:
        ga.close()
    return Fs


def check_population(ga, want):
    """population, objective values and stream position (the start population, or a generation's after a refused one)"""
    X, F = ga.population()
    assert F.tobytes() == want[1].tobytes(), "objective values"
    assert _digest(X) == want[0], "population"
    assert ga.status().stream_pos == want[5]
    return F


# ---- popSort: bucket sort off / on, and its data-dependent kernels ----
@pytest.mark.parametrize("npop", [65535, 65536, 65537])
def test_rastrigin_around_the_bucket_sort_threshold(ctx, npop):
    Fs = run_case(ctx, capi.F_RASTRIGIN, 8, npop, 3, np.full(8, 0.7), 5.12)
    if npop >= 65536:                                              # pipe_create: P->bs_on; below it the radix kernel sorts
        assert [sort_path(Fs[g - 1], Fs[g]) for g in range(1, 4)] == ["small"] * 3


def test_cfg4_bench_size(ctx):
    """1M x 32 Rastrigin, four generations: the whole pipeline at the size bench.py times. Generation 1's children pile up below
    the start population's 10 % mark (radix fallback); generations 2 - 4 have buckets of 1025 - 8192 keys (the <512, 16> kernel)"""
    Fs = run_case(ctx, capi.F_RASTRIGIN, 32, 1 << 20, 4, np.full(32, 0.7), 5.12, max_gens=32)
    assert [sort_path(Fs[g - 1], Fs[g]) for g in range(1, 5)] == ["radix", "large", "large", "large"]


def test_quantized_radix_fallback(ctx, ga_objectives):
    """33 levels over 300k rows: some level always holds more than 8192 rows (tied keys share a bucket), so every generation falls
    back to the radix kernel"""
    Fs = run_case(ctx, R.MY_F_QUANTIZED, 8, 300_000, 4, np.zeros(8), 5.12, max_gens=40)
    assert [sort_path(Fs[g - 1], Fs[g]) for g in range(1, 5)] == ["radix"] * 4


# ---- duplicate table under heavy load ----
@pytest.mark.parametrize("n", [1, 2])
@pytest.mark.parametrize("kind,ints", [(capi.F_POWER, (2,)), (capi.F_RASTRIGIN, ())])
def test_small_n_duplicates_at_200k(ctx, kind, ints, n):
    run_case(ctx, kind, n, 200_000, 3, np.full(n, 0.5), 1.0, ints=ints)


# ---- mutation composition: tables in global memory, several segments ----
@pytest.mark.parametrize("n,in_smem", [(256, False), (33, True)])
def test_mutation_composition_geometry(ctx, n, in_smem):
    npop = 100_000
    nrand = npop - int(np.ceil(0.1 * npop)) - int(np.ceil(0.2 * npop)) - int(np.ceil(0.3 * npop))
    geom = mut_geometry(n, nrand, ctx.sm_count)
    assert geom["in_smem"] == in_smem and geom["nseg"] > 1 and geom["g"] == (2 if n % 2 == 0 else 1), geom
    run_case(ctx, capi.F_RASTRIGIN, n, npop, 1, np.full(n, 0.7), 5.12, max_gens=8)


# ---- selection whose acceptance rate drops between generations ----
def crossover_trials(F, values, pos0, need):
    """trials the crossover of a generation takes (cross_last_trial + 1) and the parents it picks: trial t draws (u[pos0 + 2t], u[pos0 + 2t + 1]), and is
    accepted iff 0 < round(u Npop) < Npop and the second draw <= ratio[index] (Source/GeneticAlgorithmMPI.cpp:134-144); F is the
    generation's sorted parent population"""
    npop = F.size
    ratio = (F[-1] - F) ** 2 / (F[-1] - F[0]) ** 2
    pairs = values[pos0:pos0 + 2 * ((values.size - pos0) // 2)].reshape(-1, 2)
    x = pairs[:, 0] * npop
    idx = np.floor(x)
    idx = (idx + (x - idx >= 0.5)).astype(np.int64)                 # C round(): half away from zero (x >= 0)
    ok = (idx > 0) & (idx < npop)
    acc = ok & (pairs[:, 1] <= ratio[np.where(ok, idx, 0)])
    last = np.searchsorted(np.cumsum(acc), need)                    # the trial that completes `need` genes
    assert last < acc.size
    return int(last) + 1, idx[:last + 1][acc[:last + 1]]


def crossover_round_capacity_bound(need, trials_prev, sm_count):
    """an upper bound on the trials ONE round of ga_cross_kernel evaluates: grid G x W words x 32, with W from the acceptance rate
    the previous generation committed (pipe_enqueue, stage 1); G * W * 32 grows with G, and G <= 4 CTAs per SM"""
    rate = max(need / trials_prev, 1.0 / 512)
    g = 4 * sm_count
    return max(8.0, need / rate * 1.08 / (32.0 * g) + 1.0) * 32.0 * g


def test_acceptance_rate_drop_redoes_the_mutation_window(ctx):
    """generation 1 on ordinary draws; from generation 2 on, each draw is replaced by 1 - 2^-30 with probability 0.86, which
    rejects any trial it touches: the acceptance rate falls about 50-fold. The crossover range of generation 2, sized from
    generation 1's rate, needs more than one round (restated from the trials both generations take), and the mutation window turns
    out short, so the generation is enqueued again with a longer one (the pipeline's launches are counted twice)."""
    n, npop, gens, box = 4, 20_000, 3, 5.12
    x0 = np.full(n, 0.7)
    pos1 = reference(capi.F_RASTRIGIN, n, npop, gens, dict(seed=77, scale=SCALE), x0, box, stop_after=1)[1][5]
    rng = np.random.default_rng(3)
    values = _counter_values(77, 40_000_000)
    tail = values[pos1:]
    tail[rng.random(tail.size) < 0.86] = 1.0 - 2.0 ** -30
    launches = {}
    Fs = run_case(ctx, capi.F_RASTRIGIN, n, npop, 2, x0, box, stream=dict(values=values), max_gens=gens,
                  on_generation=lambda g, count: launches.__setitem__(g, count))
    assert launches[2] >= 2 * launches[1], launches
    need = int(np.ceil(0.3 * npop)) * n
    want = reference(capi.F_RASTRIGIN, n, npop, gens, dict(values=values), x0, box, stop_after=2)
    trials1, parents1 = crossover_trials(Fs[0], values, want[0][5], need)
    trials2, parents2 = crossover_trials(Fs[1], values, want[1][5], need)
    assert np.array_equal(parents1, want[1][2].ravel()) and np.array_equal(parents2, want[2][2].ravel())   # the restatement is right
    assert trials2 > 20 * trials1
    assert trials2 > crossover_round_capacity_bound(need, trials1, ctx.sm_count), (trials1, trials2)


def _counter_values(seed, count):
    """u_k = oracle_stream_uniform(seed, k, SCALE) for k < count, vectorised (the same splitmix64 steps)"""
    k = np.arange(count, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = np.uint64(seed) + (k + np.uint64(1)) * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return ((z >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)) * SCALE


def test_counter_values_are_the_oracle_stream():
    assert np.array_equal(_counter_values(77, 1000), O.stream_array(77, 1000, SCALE))


# ---- explicit stream that ends at generation 2's last draw, or one value earlier ----
@pytest.mark.parametrize("short", [0, 1])
def test_explicit_stream_ends_at_generation_2(ctx, short):
    n, npop, gens, box = 8, 70_000, 4, 5.12
    x0 = np.full(n, 0.7)
    want = reference(capi.F_RASTRIGIN, n, npop, gens, dict(seed=5, scale=SCALE), x0, box, stop_after=2)
    values = _counter_values(5, want[2][5] - short)
    f = ctx.functor(capi.F_RASTRIGIN)
    ga = ctx.ga_create(f, n, np.full(n, -box), np.full(n, box), npop, gens, dict(values=values))
    try:
        ga.init(x0)
        ga.generation()
        check_generation(ga, want[1], 1)
        if short:
            with pytest.raises(capi.PnolError, match="STREAM"):
                ga.generation()
            st = ga.status()                                       # nothing of generation 2 was committed (the index arrays are scratch)
            assert st.generation == 1 and st.stream_pos == want[1][5] and not st.stopped
            check_population(ga, want[1])
        else:
            ga.generation()
            check_generation(ga, want[2], 2)
    finally:
        ga.close()


# ---- -0 and +0 tie in the reference's popSort ----
@pytest.mark.parametrize("npop,box,gens,paths", [
    (3000, 0.5, 4, None),                                        # below 65536: the radix kernel sorts
    (100_000, 0.5, 4, ["radix"] * 4),                            # ~90 % zeros share one key: one bucket, the radix fallback
    (100_000, 2.0, 3, ["small", "large", "large"]),              # zeros spread over buckets of <= 8192 keys: both bucket kernels
])
def test_signed_zero_objective_order(ctx, ga_objectives, npop, box, gens, paths):
    """-0 and +0 in the same generation, sorted by each kernel. The bucket kernels must give every row its own zero"""
    Fs = run_case(ctx, R.MY_F_SIGNED_ZERO, 8, npop, gens, np.zeros(8), box, max_gens=20)
    if paths is not None:
        assert [sort_path(Fs[g - 1], Fs[g]) for g in range(1, gens + 1)] == paths
    for F in Fs[1:]:
        assert np.any((F == 0) & np.signbit(F)) and np.any((F == 0) & ~np.signbit(F))
    F = Fs[-1]
    assert np.sum((F == 0) & np.signbit(F)) > 100 and np.sum((F == 0) & ~np.signbit(F)) > 100


def test_signed_zero_pop_sort(ctx):
    rng = np.random.default_rng(8)
    npop, n = 5000, 3
    F = rng.choice(np.array([0.0, -0.0, 1.0, 2.0]), npop)
    X = rng.normal(size=(npop, n))
    Xg, Fg = ctx.ga_pop_sort(X, F)
    Xw, Fw = O.ga_pop_sort(X, F)
    assert Fg.tobytes() == Fw.tobytes() and np.array_equal(Xg, Xw)
    Xg, Fg = ctx.ga_pop_sort(X[:5], np.array([0.0, -0.0, 1.0, -0.0, 0.0]))
    assert Fg.tobytes() == np.array([0.0, -0.0, -0.0, 0.0, 1.0]).tobytes() and np.array_equal(Xg, X[[0, 1, 3, 4, 2]])


def test_signed_zero_init(ctx, ga_objectives):
    """pnol_ga_init sorts the start population with the radix kernel alone (the bucket sort needs a previous generation's values)"""
    n, npop, box = 8, 3000, 0.5
    want = reference(R.MY_F_SIGNED_ZERO, n, npop, 5, dict(seed=21, scale=SCALE), np.zeros(n), box, stop_after=0)
    f = ctx.functor(R.MY_F_SIGNED_ZERO)
    ga = ctx.ga_create(f, n, np.full(n, -box), np.full(n, box), npop, 5, dict(seed=21, scale=SCALE))
    try:
        ga.init(np.zeros(n))
        F = check_population(ga, want[0])
        assert np.sum((F == 0) & np.signbit(F)) > 10 and np.sum((F == 0) & ~np.signbit(F)) > 10
    finally:
        ga.close()
