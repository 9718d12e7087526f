#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native PNOL hot path (BASELINE.json: "LM iters/sec & Jacobian HBM GB/s at
m=4M,n=256; GA evals/sec; 1/2/4/8 B200").

    python bench.py --gpus 1 --steps K --warmup W            # our arm (1 GPU)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W              # our arm, row-sharded over N GPUs (strong scaling)
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's own CPU code on the host cores
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR  # + what the last timed step computed, as DIR/*.npy

Workload (config.workload = "cfg5"): Levenberg-Marquardt on the tree-summed Lorentzian curve fit of SURVEY.md 8(d),
m = 4 000 000 residuals x n = 256 parameters, FP64. One STEP = one LM iteration of
Source/LevenbergMarquardtMPI.cpp:55-141: FD Jacobian (n+1 model evaluations per row) -> J^T J / J^T r on the FP64 tensor
cores (+ NCCL all-reduce when row-sharded) -> damped Cholesky solve -> trial residual + chi^2 (one C-ABI call, pnol_lm_step, one
synchronisation) -> accept/reject on the host.
Every step recomputes the Jacobian (as the reference does, also after a rejected step) and a fresh findMin starts every
`--restart` steps so that every step does the full work.

  value : LM iterations/s with data, J and all work buffers resident in HBM, timed with CUDA events on the context's
          stream, max over ranks.
  e2e   : the same metric through the reference-facing plugin call LevMarqMPI::findMin (host C++ mirror,
          include/pnol/LevenbergMarquardtMPI.hpp) with HOST buffers: data columns t,y go host->device, F0/FOpt come back,
          every iteration moves x, sigma and chi^2 across PCIe. Wall clock, max over ranks.
  roofline     : the dominant kernel of the step (J^T J SYRK, FP64 DMMA) from CUDA-event scopes inside the timed region.
  cpu_baseline : the verbatim reference (oracle/_ref, compiled from /root/reference/Source) on the host cores, on a bounded
                 row sample of the same problem.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

sys.dont_write_bytecode = True     # the tree may be read-only; the modules imported below must not leave caches in it
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

M_TOTAL = 4_000_000
K_TERMS = 128                      # n = 2 K = 256
LM_PARAMS = dict(lambda0=0.001, factor=10.0, dxgrad=1e-7)
REF_SAMPLE_ROWS = 8192             # rows of the workload one reference step runs on (bounded sample)
METRIC = "lm_iterations_per_second_m4M_n256"
UNIT = "LM iterations/s"


# ----------------------------------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock, power and clock-event reasons of one GPU every 25 ms on a thread (NVML; nvidia-smi fallback)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        self.index, self.samples, self.max_mhz = index, [], None
        self._stop = threading.Event()
        self._thr = None
        self._proc = None
        self._log = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                try:
                    pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                except Exception:
                    pw = 0.0
                self.samples.append((time.perf_counter(), float(mhz), int(rs), pw))
            except Exception:
                pass
            self._stop.wait(0.025)

    def start(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()
        else:
            self._log = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                 "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
            try:
                self._proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                               "-lms", "100"], stdout=self._log, stderr=subprocess.DEVNULL)
            except Exception:
                self._proc = None

    def stop(self):
        self._stop.set()
        if self._thr:
            self._thr.join(timeout=2)
        if self._proc:
            self._proc.terminate()
            try:
                self._proc.wait(timeout=2)
            except Exception:
                pass

    def summary(self, windows):
        """median SM MHz and the union of active reasons over samples that fall into the (t0, t1) windows."""
        if self.nv is not None:
            sel = [s for s in self.samples if any(a <= s[0] <= b for a, b in windows)] or self.samples
            if not sel:
                return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
            bits = 0
            for s in sel:
                bits |= s[2]
            reasons = sorted(name for bit, name in self.REASONS.items() if bits & bit)
            return {"sm_mhz": float(np.median([s[1] for s in sel])), "sm_max_mhz": self.max_mhz, "reasons": reasons,
                    "samples": len(sel), "power_w_max": max(s[3] for s in sel)}
        rows = []
        if self._log:
            self._log.flush()
            self._log.seek(0)
            for line in self._log:
                p = [v.strip() for v in line.split(",")]
                if len(p) >= 7:
                    try:
                        rows.append((float(p[0]), float(p[1]), p[3:7]))
                    except ValueError:
                        pass
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        busy = [r for r in rows if r[0] >= 0.5 * max(x[0] for x in rows)] or rows
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in busy for i in range(4) if r[2][i] == "Active"})
        return {"sm_mhz": float(np.median([r[0] for r in busy])), "sm_max_mhz": busy[0][1], "reasons": reasons, "samples": len(busy)}


# ----------------------------------------------------------------------------------------------------------------------
# reference arm / CPU baseline (the only place bench.py executes oracle/)
# ----------------------------------------------------------------------------------------------------------------------
def _sample_problem(m_total, K, rows):
    from parallelnonlinearoptimizationlibrary_b200 import problems
    pr = problems.lorentz_problem(m_total, K)
    stride = max(1, m_total // rows)
    sl = slice(0, stride * rows, stride)          # every stride-th row: the sample spans the whole abscissa range
    return pr, np.ascontiguousarray(pr["t"][sl][:rows]), np.ascontiguousarray(pr["y"][sl][:rows])


def _run_ref_lm(t, y, w, x0, steps, warmup, nprocs):
    """seconds per LM iteration of the verbatim reference (LevMarqMPI::findMin) on the sample, at `nprocs` mini-MPI ranks."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    r = O.ref_cli("bench_lm", arrays=dict(x=x0, t=t, y=y), obj="lorentz", w=w, steps=steps, warmup=warmup, dxgrad=LM_PARAMS["dxgrad"],
                  lambda0=LM_PARAMS["lambda0"], factor=LM_PARAMS["factor"], nprocs=nprocs, timeout=3600)
    line = [ln for ln in r["_stdout"].splitlines() if ln.startswith("{")][-1]
    return json.loads(line)["s_per_iter"]


def _run_port_lm(t, y, w, x0, steps):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    f = O.OFunctor(103, (w,), (), (t, y), t.size)
    t0 = time.perf_counter()
    O.lm(f, x0, LM_PARAMS["lambda0"], LM_PARAMS["factor"], LM_PARAMS["dxgrad"], steps, 0.0)
    return (time.perf_counter() - t0) / steps


def _time_ref_shape(m, K, P):
    """seconds per LM iteration of the verbatim reference at (m rows, n = 2K) -- a MEASUREMENT at that shape, no scaling"""
    from parallelnonlinearoptimizationlibrary_b200 import problems
    pr = problems.lorentz_problem(m, K)
    return _run_ref_lm(pr["t"], pr["y"], pr["w"], pr["x0"], 1, 0, P)


def cpu_reference(m_total, K, steps, warmup, rows=REF_SAMPLE_ROWS, scaled_shapes=True):
    """Times the reference's CPU implementation of the LM step; returns (iters/s at full m, description).

    The headline figure is the verbatim reference on a row sample of the cfg5 problem scaled by m / rows (every statement of the
    iteration except the n^3 solve is linear in the rows) -- an EXTRAPOLATION, and the line says so. Beside it, measured without any
    scaling (BASELINE.md 4.3): the verbatim reference at m = 4M, n = 16 and at m = 200k, n = 64, the exponent of n those two imply
    for the cost per row, and what that law predicts for cfg5."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    pr, t, y = _sample_problem(m_total, K, rows)
    cores = os.cpu_count() or 1
    scale = m_total / float(rows)
    extra = {}
    if O.have_ref():
        # the reference replicates the dense algebra on every rank and pays n+1 collectives of m doubles per Jacobian, so
        # more ranks are not always faster: calibrate P in {1, min(8, cores)} during warm-up and time the faster one
        cands = sorted({1, min(8, cores)})
        cal = {}
        for P in cands:
            cal[P] = _run_ref_lm(t, y, pr["w"], pr["x0"], 1, max(0, min(warmup, 1)), P)
        P = min(cal, key=cal.get)
        s_iter = _run_ref_lm(t, y, pr["w"], pr["x0"], steps, 0, P)
        kind, used = "reference", P
        note = "verbatim reference LevMarqMPI::findMin (oracle/_ref, mini-MPI ranks=%d; calibration s/iter %s)" % (
            P, {k: round(v, 3) for k, v in cal.items()})
        if scaled_shapes:
            try:
                a = _time_ref_shape(4_000_000, 8, P)           # m = 4M, n = 16
                b = _time_ref_shape(200_000, 32, P)            # m = 200k, n = 64
                pa, pb = a / 4_000_000, b / 200_000            # seconds per row
                expo = float(np.log(pb / pa) / np.log(64.0 / 16.0))
                pred = pb * (2.0 * K / 64.0) ** expo * m_total
                extra = {"measured_shapes": [{"m": 4_000_000, "n": 16, "s_per_iter": a, "ranks": P}, {"m": 200_000, "n": 64, "s_per_iter": b, "ranks": P}],
                         "implied_exponent_of_n_per_row": expo,
                         "cfg5_s_per_iter_predicted_by_that_law": pred,
                         "cfg5_s_per_iter_from_the_row_sample": s_iter * scale}
            except Exception as e:                          # reported, never required
                extra = {"measured_shapes": "failed: %r" % (e,)}
    else:
        s_iter = _run_port_lm(t, y, pr["w"], pr["x0"], steps)
        kind, used = "port", 1
        note = "oracle restatement (oracle/libpnol_oracle.so), scalar"
    value = 1.0 / (s_iter * scale)
    sample = ("EXTRAPOLATED from %d of %d rows (every %d-th), n=%d, %d LM iteration(s): s/iter on the sample %.3f scaled by m/rows=%.1f; %s"
              % (rows, m_total, m_total // rows, 2 * K, steps, s_iter, scale, note))
    d = dict(value=value, unit=UNIT, cores=used, kind=kind, sample=sample, host_cores=cores, s_per_iter_sample=s_iter, extrapolated=True)
    d.update(extra)
    return value, d


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return 0
    t0 = time.perf_counter()
    # every reference step costs about a second on the 8192-row sample: cap the timed steps so that the run ends within a few
    # minutes whatever K the caller asks for (the metric is a rate, the cap only bounds the averaging window)
    timed = max(1, min(args.steps, 40))
    value, cb = cpu_reference(args.m, args.K, timed, args.warmup, rows=args.ref_rows, scaled_shapes=not args.no_scaled_shapes)
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 / value, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": "cfg5: LevenbergMarquardt large least-squares, m=%d residuals x n=%d (tree-summed Lorentzian fit)"
                   % (args.m, 2 * args.K), "m": args.m, "n": 2 * args.K, "sample_rows": args.ref_rows, "steps_timed": timed},
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t0,
    }
    emit(out)
    return 0


# ----------------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------------
class LMDevice:
    """One LM problem resident on one GPU (this rank's row block), stepped through the C-ABI (include/pnol_b200.h)."""

    def __init__(self, ctx, capi, pr, lo, hi):
        self.ctx, self.capi = ctx, capi
        self.m, self.n = hi - lo, pr["n"]
        self.t_dev = ctx.to_device(pr["t"][lo:hi])
        self.y_dev = ctx.to_device(pr["y"][lo:hi])
        self.f = ctx.functor(capi.F_LORENTZ_SUM, (pr["w"],), (), (self.t_dev, self.y_dev), self.m)   # device columns are borrowed
        n, m = self.n, self.m
        self.J = ctx.malloc(m * n * 8)
        self.F, self.Ft = ctx.malloc(m * 8), ctx.malloc(m * 8)
        self.JTJ = ctx.malloc((n * n + n) * 8)          # J^T J followed by -J^T F
        self.dx = ctx.to_device(np.full(n, LM_PARAMS["dxgrad"]))
        self.x0 = pr["x0"].copy()
        self.accepted = self.rejected = 0
        self.start()

    def start(self):
        """findMin prologue (Source/LevenbergMarquardtMPI.cpp:42-51)"""
        self.X = self.x0.copy()
        self.lam = LM_PARAMS["lambda0"]
        _, ss = self.ctx.residual_eval(self.f, self.X, F=self.F, n=self.n)
        self.chi = np.sqrt(ss) ** 2

    def step(self, k=1):
        """k iterations of the while loop (Source/LevenbergMarquardtMPI.cpp:55-141), Jacobian always recomputed: per iteration the
        device work is one pnol_lm_step (one synchronisation) and the accept / reject decision is taken on the host, in C++
        (pnol_lm_iterate) -- no interpreter between two iterations"""
        self.X, self.lam, self.chi, acc, rej, swapped = self.ctx.lm_iterate(self.f, self.X, self.dx, self.n, self.J, self.F, self.Ft, self.JTJ,
                                                                            self.lam, self.chi, LM_PARAMS["factor"], k)
        if swapped:
            self.F, self.Ft = self.Ft, self.F
        self.accepted += acc
        self.rejected += rej


DUMP_SEED = 20240607               # fixed: the sampled rows are the same in every run and every build
DUMP_BUDGET = {"residual": 32 << 20, "jacobian": 16 << 20, "jtj": 8 << 20}     # bytes per array: 56 MiB + the n-vectors in all


def _sample_rows(rows, row_bytes, budget, rng):
    """None if all `rows` rows fit the budget, else a sorted seeded sample of as many rows as fit with their 8-byte indices"""
    if rows * row_bytes <= budget:
        return None
    return np.sort(rng.choice(rows, size=max(1, budget // (row_bytes + 8)), replace=False))


def dump_outputs(out_dir, ctx, prob, lo):
    """Writes what the last timed LM iteration left to its caller, as float64 .npy files: the iterate `x`, `lambda`, `chisq`, and
    the device buffers the caller passed to pnol_lm_iterate: `residual` F at x, `jacobian` J of the last step and `jtj` / `rhs`
    (J^T J and -J^T F). An array over its byte budget is a fixed seeded sample of its rows, with the (global) row indices
    beside it as `<name>_rows`. With the rows sharded over several GPUs, this rank's rows."""
    os.makedirs(out_dir, exist_ok=True)
    m, n = prob.m, prob.n
    rng = np.random.default_rng(DUMP_SEED)
    out = {"x": prob.X, "lambda": np.array([prob.lam]), "chisq": np.array([prob.chi])}
    F = ctx.to_host(prob.F, m)
    rows = _sample_rows(m, 8, DUMP_BUDGET["residual"], rng)
    out["residual"] = F if rows is None else F[rows]
    if rows is not None:
        out["residual_rows"] = (lo + rows).astype(np.float64)
    rows = _sample_rows(m, 8 * n, DUMP_BUDGET["jacobian"], rng)
    rows = np.arange(m) if rows is None else rows
    J = np.empty((rows.size, n))
    for j, i in enumerate(rows):
        ctx.memcpy(J[j], prob.J + int(i) * n * 8, n * 8)
    out["jacobian"], out["jacobian_rows"] = J, (lo + rows).astype(np.float64)
    W = ctx.to_host(prob.JTJ, n * n + n)
    rows = _sample_rows(n, 8 * n, DUMP_BUDGET["jtj"], rng)
    out["jtj"] = W[:n * n].reshape(n, n) if rows is None else W[:n * n].reshape(n, n)[rows]
    if rows is not None:
        out["jtj_rows"] = rows.astype(np.float64)
    out["rhs"] = W[n * n:]
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def run_ours(args):
    import torch
    from parallelnonlinearoptimizationlibrary_b200 import capi, hostapi, launch, problems

    rank, local_rank, world = launch.init_process_group()
    if world != args.gpus and rank == 0:
        print("warning: --gpus %d but WORLD_SIZE %d (launch with torchrun for N > 1)" % (args.gpus, world), file=sys.stderr)
    torch.cuda.set_device(local_rank)
    ctx = capi.Context(local_rank)
    launch.attach_communicator(ctx)
    hostapi.attach(ctx)
    hostapi.set_jacobian_cache(False)      # every iteration recomputes J, as the reference does
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local_rank))

    m_total, K = args.m, args.K
    n = 2 * K
    pr = problems.lorentz_problem(m_total, K)
    lo, hi = launch.row_shard(m_total, world, rank)
    m_loc = hi - lo
    prob = LMDevice(ctx, capi, pr, lo, hi)

    try:
        hbm_peak_early = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0))
    except Exception:
        hbm_peak_early = 6650.0
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()

    def sync_all():
        ctx.sync()
        torch.cuda.synchronize()
        launch.barrier()
        ctx.sync()

    # ---- value: device-resident steps -----------------------------------------------------------------------------
    def run_steps(k, counter0=0):
        i = 0
        while i < k:
            if (counter0 + i) % args.restart == 0:
                prob.start()
            run = min(k - i, args.restart - (counter0 + i) % args.restart)      # up to the next findMin restart
            prob.step(run)
            i += run

    run_steps(args.warmup)
    dmma_peak = ctx.measure_dmma_peak()
    # CUDA-event scopes inside the timed region around the three kernels that carry the step (syrk = the roofline kernel, fd_jacobian,
    # residual); the small scopes are taken in a separate untimed pass below (an event pair costs about 5 us of stream time: seven
    # scopes per iteration were 2 % of an iteration at 8 GPUs)
    ctx.timer_enable(2)
    ctx.timer_reset()
    sync_all()
    l0 = ctx.launches()
    prob.accepted = prob.rejected = 0
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    ev0.record(stream)
    run_steps(args.steps)
    ev1.record(stream)
    sync_all()
    w1 = time.perf_counter()
    launches = ctx.launches() - l0
    ms_total = launch.max_over_ranks(ev0.elapsed_time(ev1))
    timers = {}
    for name in ("fd_jacobian", "syrk", "residual"):
        ms, cnt = ctx.timer_get(name)
        if cnt:
            timers[name] = {"ms_avg": ms / cnt, "count": cnt}
    accepted, rejected = prob.accepted, prob.rejected
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ctx, prob, lo)
    # the small scopes: the same steps once more, untimed, with every scope on
    ctx.timer_enable(1)
    ctx.timer_reset()
    run_steps(min(args.steps, args.restart))
    for name in ("syrk_finish", "allreduce", "spd_solve", "sumsq"):
        ms, cnt = ctx.timer_get(name)
        if cnt:
            timers[name] = {"ms_avg": ms / cnt, "count": cnt, "pass": "untimed repeat of the steps"}
    ctx.timer_enable(False)
    ms_per_step = ms_total / args.steps
    value = 1000.0 / ms_per_step

    # ---- e2e: LevMarqMPI::findMin through the plugin API with host buffers ---------------------------------------
    # The user's objective (LorentzSumObjective holding this rank's rows in host vectors) is built once, as a user of the
    # reference builds his MultiObjective before calling findMin. Every timed call then runs
    # `LevMarqMPI lm; lm.setObjPtr(obj); lm.setParams(...); lm.findMin(X, F0, F)` with a FRESH device twin, so each call pays the
    # host->device upload of the data columns, all device allocations and the F0 / FOpt read-backs into host vectors.
    e2e_prob = hostapi.LMProblem(pr["t"][lo:hi], pr["y"][lo:hi], pr["w"])

    def e2e_call(iters):
        return e2e_prob.run(pr["x0"], LM_PARAMS["lambda0"], LM_PARAMS["factor"], LM_PARAMS["dxgrad"], maxiter=iters, xmindiff=0.0,
                            fresh_device_twin=True)

    e2e_chunk = max(1, min(args.steps, args.restart))
    e2e_call(min(2, e2e_chunk))            # warm-up of the host path (allocator, first-touch of the pageable vectors)
    sync_all()
    e0 = time.perf_counter()
    done, calls = 0, 0
    while done < args.steps:
        k = min(e2e_chunk, args.steps - done)
        rep = e2e_call(k)
        done += rep["iterations"] if rep["iterations"] > 0 else k
        calls += 1
    sync_all()
    e1 = time.perf_counter()
    e2e_s = launch.max_over_ranks(e1 - e0)
    e2e_value = args.steps / e2e_s
    # per call: t,y up and F0,FOpt down; per iteration: x up (Jacobian) + x up (trial), sigma + info + 2 chi^2 down
    h2d = (calls * 2 * m_loc * 8 + args.steps * 2 * n * 8) / args.steps
    d2h = (calls * 2 * m_loc * 8 + args.steps * (n * 8 + 4 + 8) + calls * 8) / args.steps
    e2e_windows = (e0, e1)

    # ---- parity: results of this very run against committed reference-derived fixtures, at every GPU count -----------------
    # LM: 4 iterations from the start point at the FULL cfg5 size against the threaded oracle restatement of
    # Source/LevenbergMarquardtMPI.cpp:12-173 (tests/golden/baseline_lm_golden.npz, case cfg5; the generating script proves that
    # restatement bit-identical to the verbatim reference where the reference finishes). X must also be bit-identical on all ranks.
    import hashlib
    parity = {}
    try:
        GB = np.load(os.path.join(ROOT, "tests", "golden", "baseline_lm_golden.npz"))
        if (m_total, K) == (int(GB["cfg5/m"]), int(GB["cfg5/K"])):
            prob.start()
            prob.step(int(GB["cfg5/maxiter"]))
            want = GB["cfg5/X"]
            rel_x = float(np.linalg.norm(prob.X - want) / np.linalg.norm(want))
            chi_ref = float(GB["cfg5/chisq"])
            xs = launch.gather_over_ranks(prob.X)
            parity["lm"] = {"fixture": "tests/golden/baseline_lm_golden.npz:cfg5 (oracle restatement at m=4M, n=256, 4 iterations)",
                            "rel_err_X": rel_x, "chisq": prob.chi, "chisq_ref": chi_ref, "lambda_equal": bool(prob.lam == float(GB["cfg5/lam"])),
                            "X_bit_identical_on_all_ranks": bool(all(np.array_equal(xs[0], x) for x in xs)),
                            "ok": bool(rel_x <= 1e-9 and prob.lam == float(GB["cfg5/lam"]) and all(np.array_equal(xs[0], x) for x in xs))}
    except Exception as e:
        parity["lm"] = {"ok": False, "error": repr(e)}

    # ---- secondary: FD gradient with the coordinates split by column over the GPUs (cfg3's n = 4096; pnol_fd_gradient,
    #      Source/PNOL_Objective.cpp:88-159), bit for bit against the oracle's gradient (tests/golden/bench_fixture.npz) --------
    fdg = None
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    from make_bench_fixture import GA_SHAPE, fdgrad_inputs, ga_fingerprint      # shapes / inputs only (no oracle import on this path)
    BF = np.load(os.path.join(ROOT, "tests", "golden", "bench_fixture.npz"))
    try:
        xg, dxg = fdgrad_inputs()
        frs = ctx.functor(capi.F_ROSENBROCK)
        g, f0g = ctx.fd_gradient(frs, xg, dxg)
        sync_all()
        reps = 20
        t0g = time.perf_counter()
        for _ in range(reps):
            g, f0g = ctx.fd_gradient(frs, xg, dxg)
        sync_all()
        ms_g = launch.max_over_ranks((time.perf_counter() - t0g) / reps * 1e3)
        ok_g = bool(np.array_equal(g, BF["fdgrad4096/g"]) and f0g == float(BF["fdgrad4096/f0"]))
        gs = launch.gather_over_ranks(g)
        fdg = {"metric": "fd_gradient_n4096_column_split", "ms_per_gradient_host_call": ms_g, "evaluations": 4097, "columns_per_gpu": -(-4096 // world),
               "bit_exact_vs_oracle": ok_g, "bit_identical_on_all_ranks": bool(all(np.array_equal(gs[0], x) for x in gs))}
        parity["fd_gradient"] = {"ok": bool(ok_g and fdg["bit_identical_on_all_ranks"]), "fixture": "tests/golden/bench_fixture.npz:fdgrad4096 (oracle)"}
    except Exception as e:
        parity["fd_gradient"] = {"ok": False, "error": repr(e)}

    # ---- secondary: the dense BFGS / LM pieces at the cfg3 / cfg5 sizes, one GPU each (north_star: they stay on one GPU) -------
    dense = {}
    if not args.no_dense:
        try:
            hbm_pk = hbm_peak_early
            n3 = 4096
            rngd = np.random.default_rng(9)
            D = np.diag(rngd.uniform(0.5, 2.0, n3))
            u3 = rngd.normal(size=(n3, 3)) / np.sqrt(n3)
            D = D + u3 @ u3.T
            g3 = rngd.normal(size=n3)
            s3 = 0.1 * g3 + 0.05 * rngd.normal(size=n3)
            Dd, gd, sd, pd = ctx.to_device(D), ctx.to_device(g3), ctx.to_device(s3), ctx.malloc(n3 * 8)

            def timed_kernel(name, fn, reps, warm=3, groups=3):
                """average kernel time (CUDA-event scope inside the library) of `reps` calls; the best of `groups` such averages, so that
                one disturbed group (another rank's phase on the same host, a clock ramp) does not end in the line; max over ranks"""
                for _ in range(warm):
                    fn()
                ctx.sync()
                best = None
                for _ in range(groups):
                    ctx.timer_enable(True)
                    ctx.timer_reset()
                    for _ in range(reps):
                        fn()
                    ms, cnt = ctx.timer_get(name)
                    ctx.timer_enable(False)
                    avg = ms / max(cnt, 1)
                    best = avg if best is None else min(best, avg)
                return launch.max_over_ranks(best)

            # D (134 MB) exceeds the 126 MB L2; the update rewrites it between matvec calls in the real iteration
            ms = timed_kernel("matvec_neg", lambda: ctx.matvec_neg(Dd, gd, n3, p=pd), 30)
            by = n3 * n3 * 8.0
            dense["matvec_neg"] = {"n": n3, "ms": ms, "bound": "hbm", "algorithmic_bytes": by, "achieved": by / (ms * 1e-3) / 1e9, "unit": "GB/s",
                                   "peak": hbm_pk, "frac": by / (ms * 1e-3) / 1e9 / hbm_pk}
            ms = timed_kernel("hinv_rank2", lambda: ctx.bfgs_update_hinv(Dd, gd, sd, n3, mode=capi.HINV_RANK2), 30)
            by = 3.0 * n3 * n3 * 8.0
            dense["hinv_rank2"] = {"n": n3, "ms": ms, "bound": "hbm", "algorithmic_bytes": by, "achieved": by / (ms * 1e-3) / 1e9, "unit": "GB/s",
                                   "peak": hbm_pk, "frac": by / (ms * 1e-3) / 1e9 / hbm_pk,
                                   "note": "D read twice (u = D g and v = D^T g in one pass, then the update pass) and written once"}
            Dl = ctx.to_device(D)
            ms = timed_kernel("hinv_literal", lambda: ctx.bfgs_update_hinv(Dl, gd, sd, n3, mode=capi.HINV_LITERAL), 3, warm=1, groups=1)
            fl = 4.0 * n3 ** 3
            dense["gemm_nn_literal"] = {"n": n3, "ms": ms, "bound": "tensor", "algorithmic_flops": fl, "achieved": fl / (ms * 1e-3) / 1e12, "unit": "TFLOP/s",
                                        "peak": dmma_peak, "frac": fl / (ms * 1e-3) / 1e12 / dmma_peak,
                                        "note": "updateHessianInv as the reference writes it: two n^3 products (DMMA) + the rank-1 terms"}
            for q in (Dd, gd, sd, pd, Dl):
                ctx.free(q)
            ns = n
            M = rngd.normal(size=(ns, ns))
            A = M @ M.T / ns + np.eye(ns)
            Ad, bd, xd = ctx.to_device(A), ctx.to_device(rngd.normal(size=ns)), ctx.malloc(ns * 8)
            ms = timed_kernel("spd_solve", lambda: ctx.spd_solve(Ad, bd, ns, x=xd), 30)
            dense["spd_solve"] = {"n": ns, "ms": ms, "bound": "latency", "algorithmic_flops": ns ** 3 / 3.0,
                                  "note": "damped Cholesky solve of the LM step (replicated on every GPU): a dependency chain, reported in time only"}
            for q in (Ad, bd, xd):
                ctx.free(q)
        except Exception as e:
            dense["error"] = repr(e)

    # ---- secondary: GA at the cfg4 shape (Rastrigin, Npop = 1M x 32): the fitness sweep alone (this rank's shard) and whole
    #      generations through the GA state machine (rows sharded over the GPUs: every rank creates, repairs and evaluates its own
    #      children; hashes and objective values all-gathered; selection scans and the sort replicated) ----
    ga = None
    if not args.no_ga:
        npop = 1_000_000
        glo, ghi = launch.row_shard(npop, world, rank)
        rng = np.random.default_rng(1234 + rank)
        pts = ctx.to_device(rng.uniform(-5.12, 5.12, size=(ghi - glo, 32)))
        fo = ctx.malloc((ghi - glo) * 8)
        fr = ctx.functor(capi.F_RASTRIGIN)
        for _ in range(3):
            ctx.eval_batch(fr, pts, ghi - glo, 32, f_out=fo)
        # 1M x 32 doubles = 256 MB > L2 (126 MB): every sweep streams from HBM
        sync_all()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 20
        ctx.timer_enable(True)
        ctx.timer_reset()
        for _ in range(reps):
            ctx.eval_batch(fr, pts, ghi - glo, 32, f_out=fo)       # each call returns after a stream sync: time the kernel scope
        tms, tcnt = ctx.timer_get("eval_batch")
        ctx.timer_enable(False)
        sync_all()
        gms = launch.max_over_ranks(tms / max(tcnt, 1))
        ga = {"metric": "ga_fitness_evals_per_second_npop1M_n32", "value": npop / (gms * 1e-3), "unit": "evaluations/s",
              "ms_per_sweep": gms, "hbm_gbs_per_gpu": (ghi - glo) * 33 * 8 / (gms * 1e-3) / 1e9,
              "hbm_frac_of_measured": (ghi - glo) * 33 * 8 / (gms * 1e-3) / 1e9 / hbm_peak_early}
        ctx.free(pts)
        ctx.free(fo)
        gens = GA_SHAPE["gens"]
        gas = ctx.ga_create(fr, 32, np.full(32, -5.12), np.full(32, 5.12), npop, gens + 2, dict(seed=GA_SHAPE["seed"], scale=GA_SHAPE["scale"]), nstatic=1e9)
        gas.init(np.full(32, GA_SHAPE["x0"]))
        gas.generation()
        sync_all()
        g0.record(stream)
        for _ in range(gens):
            gas.generation()
        g1.record(stream)
        sync_all()
        gen_ms = launch.max_over_ranks(g0.elapsed_time(g1)) / gens
        st = gas.status()
        _, Fga = gas.population()
        fp = ga_fingerprint(Fga, st.stream_pos)
        fps = launch.gather_over_ranks(np.frombuffer(bytes.fromhex(fp), dtype=np.uint8).astype(np.float64))
        want_fp = str(BF["ga/sha256"]) if "ga/sha256" in BF else None
        parity["ga"] = {"sha256_F_and_stream_pos": fp, "fixture_sha256_from_the_1_gpu_run": want_fp,
                        "identical_on_all_ranks": bool(all(np.array_equal(fps[0], x) for x in fps)),
                        "ok": bool(want_fp is not None and fp == want_fp and all(np.array_equal(fps[0], x) for x in fps))}
        # per-stage times of two more generations (CUDA-event scopes; they serialise the stages, so they are not part of gen_ms)
        ctx.timer_enable(True)
        ctx.timer_reset()
        gas2 = ctx.ga_create(fr, 32, np.full(32, -5.12), np.full(32, 5.12), npop, gens + 2, dict(seed=GA_SHAPE["seed"], scale=GA_SHAPE["scale"]), nstatic=1e9)
        gas2.init(np.full(32, GA_SHAPE["x0"]))
        ctx.timer_reset()
        for _ in range(3):
            gas2.generation()
        stages = {}
        for name in ("ga_prep", "ga_crossover", "ga_mutation", "ga_elite_mutation", "ga_gather_hash", "ga_check_identical", "ga_check_bounds", "eval_batch",
                     "ga_gather_f", "ga_pop_sort"):
            ms, cnt = ctx.timer_get(name)
            if cnt:
                stages[name] = round(launch.max_over_ranks(ms / cnt), 5)
        ctx.timer_enable(False)
        # algorithmic HBM traffic of a generation: children written once (256 MB), parents read once (256 MB), one more read by
        # the sweep; roofline time at the measured copy bandwidth
        gen_bytes = 3.0 * npop * 32 * 8 / world
        ga.update(ms_per_generation=gen_ms, evals_per_s_whole_generation=(npop - st.n_elite) / (gen_ms * 1e-3), f_best=st.f_best,
                  stream_draws_per_generation=int(st.stream_pos) // (gens + 1), peer_mode=gas.peer_mode(), stage_ms=stages,
                  hbm_frac_whole_generation=gen_bytes / (gen_ms * 1e-3) / 1e9 / hbm_peak_early,
                  note="bound by the counter-based random stream (about 135 M draws of 64-bit integer mixing per generation), not by HBM")
        gas2.close()
        gas.close()
        if world > 1:
            # the other ways of splitting a generation, for the record (include/pnol_b200.h, pnol_ga_set_sharding): the default (auto) at
            # this size is replicas -- the 0.057 ms sweep does not pay for an all-gather of its 8 MB of values (peer_mode 4); "sweep"
            # splits the sweep and all-gathers F as the reference does (3), "rows" shards the population itself (parents over NVLink; 1)
            modes = {"default": {"peer_mode": ga["peer_mode"], "ms_per_generation": gen_ms}}
            for label, shard_mode in (("rows_sharded", 1), ("sweep_sharded", 2)):
                try:
                    ctx.ga_set_sharding(shard_mode)
                    gas3 = ctx.ga_create(fr, 32, np.full(32, -5.12), np.full(32, 5.12), npop, gens + 2, dict(seed=GA_SHAPE["seed"], scale=GA_SHAPE["scale"]), nstatic=1e9)
                    gas3.init(np.full(32, GA_SHAPE["x0"]))
                    gas3.generation()
                    sync_all()
                    g0.record(stream)
                    for _ in range(gens):
                        gas3.generation()
                    g1.record(stream)
                    sync_all()
                    ms3 = launch.max_over_ranks(g0.elapsed_time(g1)) / gens
                    _, F3 = gas3.population()
                    modes[label] = {"peer_mode": gas3.peer_mode(), "ms_per_generation": ms3,
                                    "same_fingerprint": bool(ga_fingerprint(F3, gas3.status().stream_pos) == fp)}
                    gas3.close()
                except Exception as e:
                    modes[label] = {"error": repr(e)}
            ctx.ga_set_sharding(0)
            ga["sharding_modes"] = modes

    if sampler:
        sampler.stop()

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        hbm_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "6650 GB/s (of fallback)"
        traffic = {}
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        except Exception:
            pass

        def tr(kernel):
            t = traffic.get(kernel)
            return t.get("dram_bytes_per_launch") if t and t.get("m") == m_loc and t.get("n") == n else None

        kern = {}
        if "syrk" in timers:
            fl = float(m_loc) * n * (n + 1)                        # lower triangle incl. diagonal, 2 flop per MAC (J^T r is summed by the Jacobian kernel)
            a = fl / (timers["syrk"]["ms_avg"] * 1e-3) / 1e12
            kern["syrk"] = {"bound": "tensor", "achieved": a, "peak": dmma_peak, "unit": "TFLOP/s", "frac": a / dmma_peak,
                            "traffic": tr("syrk"), "ms": timers["syrk"]["ms_avg"], "algorithmic_flops": fl,
                            "peak_source": "FP64 DMMA register-resident microbenchmark of this run (pnol_measure_dmma_peak); "
                                           "MEASURED_PEAKS.json holds no FP64 figure (nominal 148 SM x 128 flop/clk x 1.965 GHz = 37.2)"}
        if "fd_jacobian" in timers:
            by = float(m_loc) * n * 8 + 3.0 * m_loc * 8            # J written once; data columns t, y and the residual F read once
            a = by / (timers["fd_jacobian"]["ms_avg"] * 1e-3) / 1e9
            # the same launch against the FP64-ALU roofline: 221 FP64 warp instructions per row (SASS count of the staged row with the
            # three-operation FD quotient, which the bench's dX = 1e-7 qualifies for: 213 for J, 8 for J^T F; 237 with the five-operation
            # quotient; DESIGN.md section 5.3 / 5.9) x 32 lanes, peak = SMs x 64 lanes x SM clock
            fp64_ops = 221.0 * 32 * m_loc
            fp64_peak = ctx.sm_count * 64 * 1.965e9
            kern["fd_jacobian"] = {"bound": "hbm", "achieved": a, "peak": hbm_peak, "unit": "GB/s", "frac": a / hbm_peak,
                                   "traffic": tr("fd_jacobian"), "ms": timers["fd_jacobian"]["ms_avg"], "algorithmic_bytes": by,
                                   "peak_source": hbm_src,
                                   "fp64_alu_frac": fp64_ops / (timers["fd_jacobian"]["ms_avg"] * 1e-3) / fp64_peak,
                                   "note": "FP64-ALU-bound on B200: 221 FP64 instructions per row (bit-exact FD quotients in three operations + J^T F) put the ceiling at 0.83 of the HBM roofline"}
        if "residual" in timers:
            by = 3.0 * m_loc * 8
            a = by / (timers["residual"]["ms_avg"] * 1e-3) / 1e9
            # row-per-thread kernel: 12 K + (K - 1) + 1 FP64 operations per row (K terms of a / (1 + w (t - c)^2) with IEEE divisions, the tree, y - S)
            res_ops = (13.0 * K) * m_loc
            kern["residual"] = {"bound": "hbm", "achieved": a, "peak": hbm_peak, "unit": "GB/s", "frac": a / hbm_peak, "traffic": tr("residual"),
                                "ms": timers["residual"]["ms_avg"], "algorithmic_bytes": by, "peak_source": hbm_src,
                                "fp64_alu_frac": res_ops / (timers["residual"]["ms_avg"] * 1e-3) / (ctx.sm_count * 64 * 1.965e9),
                                "note": "FP64-ALU-bound: 24 bytes but 13 K = 1664 FP64 operations per row; the HBM fraction says nothing here, the FP64-ALU fraction does"}
        dominant = max(timers, key=lambda k: timers[k]["ms_avg"] * timers[k]["count"]) if timers else None
        roof = kern.get(dominant) or kern.get("syrk") or {}
        roof = dict(roof, kernel=dominant,
                    traffic_source=("profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture at this shape"
                                    if roof.get("traffic") is not None else "not captured at this per-GPU shape (N > 1)"))

        cb = None
        if world == 1 and not args.no_cpu_baseline:
            try:
                _, cb = cpu_reference(m_total, K, 1, 0, rows=args.ref_rows, scaled_shapes=not args.no_scaled_shapes)
            except Exception as e:                               # the baseline is reported, never required
                cb = {"value": None, "unit": UNIT, "cores": 0, "kind": "unavailable", "sample": "failed: %r" % (e,)}

        windows = [(w0, w1), e2e_windows]
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": "cfg5: LevenbergMarquardt large least-squares, m=%d residuals x n=%d (tree-summed Lorentzian fit), "
                                   "Jacobian row-sharded over %d GPU(s), packed J^T J|J^T r all-reduce" % (m_total, n, world),
                       "m": m_total, "n": n, "rows_per_gpu": m_loc, "parallelism": "rows/%d" % world, "restart_every": args.restart,
                       "l2": "inputs exceed L2 (J is %.2f GB per GPU, streamed every step)" % (m_loc * n * 8 / 1e9),
                       "jacobian_cache": False, "accepted_steps": accepted, "rejected_steps": rejected,
                       "lm_exchange": {0: "one rank", 1: "NVLink peer memory inside the step's kernels (csrc/peer.cu)", 2: "NCCL all-reduce"}.get(
                           ctx.lm_exchange_mode(), "undecided")},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "api": "LevMarqMPI::findMin (host C++ mirror of Source/LevenbergMarquardtMPI.hpp) over pageable host vectors",
                    "calls": calls, "iterations_per_call": e2e_chunk},
            "gpu_launches": int(launches),
            "roofline": roof, "kernels": kern, "timers_ms": {k: round(v["ms_avg"], 5) for k, v in timers.items()},
            "jacobian_hbm_gbs": kern.get("fd_jacobian", {}).get("achieved"),
            "cpu_baseline": cb, "secondary": ga, "fd_gradient": fdg, "dense_kernels": dense, "parity": parity,
            "clocks": sampler.summary(windows) if sampler else None,
        }
        emit(out)
    launch.barrier()
    e2e_prob.close()
    hostapi.detach()
    ctx.close()
    try:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass
    return 0


_REAL_STDOUT = None


def _protect_stdout():
    """The contract is ONE JSON line on stdout: route everything libraries print to fd 1 (NCCL's version banner, torchrun
    notices, the reference's own prints) to stderr and keep a private duplicate of stdout for that line."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(obj):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(obj) + "\n")
    out.flush()


def main():
    _protect_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--m", type=int, default=M_TOTAL, help="residual rows (default: the BASELINE.json shape)")
    ap.add_argument("--K", type=int, default=K_TERMS, help="Lorentzian terms, n = 2K")
    ap.add_argument("--restart", type=int, default=10, help="a new findMin starts every this many steps")
    ap.add_argument("--ref-rows", type=int, default=REF_SAMPLE_ROWS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ga", action="store_true")
    ap.add_argument("--no-dense", action="store_true", help="skip the cfg3 dense-kernel lines (matvec, rank-2 / literal update, solve)")
    ap.add_argument("--no-scaled-shapes", action="store_true", help="cpu baseline: skip the measured m=4M,n=16 / m=200k,n=64 reference runs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy (float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
