"""Times pnol_bfgs_batch on the GPU: B random starts of one objective minimised in one call, forward-difference (flags 0) and analytic
(gradient and slope from partial(), flags 3) modes alternated in one process, against the same starts through the BFGS class one at
a time (a sample of 64 starts, timed and extrapolated to B -- labelled as an extrapolation). CUDA events around each call with
device-resident arrays; the first call of every shape and mode is a warm-up; the median of --repeats calls is reported. Prints one JSON
document (and writes it to --out when given) with the card's name, power limit and maximum SM clock read in the same run.

    python tools/time_bfgs_batch.py [--B 65536] [--repeats 3] [--sample 64] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from parallelnonlinearoptimizationlibrary_b200 import capi, hostapi  # noqa: E402

# name, host objective, kind, n, start box half-width
SHAPES = [("rastrigin16", "rastrigin", capi.F_RASTRIGIN, 16, 5.12), ("rosenbrock8", "rosenbrock", capi.F_ROSENBROCK, 8, 2.0),
          ("rosenbrock64", "rosenbrock", capi.F_ROSENBROCK, 64, 2.0), ("goldstein2", "goldstein", capi.F_GOLDSTEIN, 2, 2.0)]
MODES = [("fd", 0), ("analytic", capi.BFGS_ANALYTIC_GRADIENT | capi.BFGS_ANALYTIC_SLOPE)]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().split("\n")[0]
        name, power, clock = [v.strip() for v in q.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:      # the timing itself does not depend on it
        return dict(error=str(e))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=65536)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--sample", type=int, default=64)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    ctx = capi.Context(0)
    hostapi.attach(ctx)
    dev = torch.device("cuda:0")
    res = dict(card=card(), B=a.B, repeats=a.repeats, params="BFGS defaults (c1 1e-4, c2 0.9, dalpha 1e-6, alpha_guess 1, max_iter_ls 1000, "
               "dx_grad 1e-6, max_iter 10000, x_min_diff 1e-5, min_grad_2norm 1e-5, identity D)", shapes=[])
    for name, obj, kind, n, w in SHAPES:
        X0 = np.random.default_rng(n).uniform(-w, w, size=(a.B, n))
        X0d = torch.tensor(X0, device=dev)
        Xd = torch.empty_like(X0d)
        f = ctx.functor(kind)
        out = dict(f0=torch.empty(a.B, dtype=torch.float64, device=dev), fopt=torch.empty(a.B, dtype=torch.float64, device=dev),
                   iters=torch.empty(a.B, dtype=torch.int32, device=dev), stop=torch.empty(a.B, dtype=torch.int32, device=dev))
        times = {m: [] for m, _ in MODES}
        iters = {}
        for rep in range(a.repeats + 1):           # rep 0: warm-up
            for mode, flags in MODES:
                Xd.copy_(X0d)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                ctx.bfgs_batch(f, Xd, flags=flags, n=n, B=a.B, out=out)
                e1.record()
                torch.cuda.synchronize()
                if rep > 0:
                    times[mode].append(e0.elapsed_time(e1) / 1e3)
                iters[mode] = int(out["iters"].sum().item())
        entry = dict(shape=name, n=n, B=a.B)
        for mode, flags in MODES:
            t = float(np.median(times[mode]))
            entry[mode] = dict(seconds=t, fits_per_s=a.B / t, problem_iterations=iters[mode], problem_iterations_per_s=iters[mode] / t,
                               all_seconds=times[mode])
        # the same starts through the BFGS class one at a time (GPU, one host loop per start): a sample, extrapolated
        prm = hostapi.bfgs_params()
        for mode, flags in MODES:
            hostapi.lib().pnolhost_set_analytic_gradient(int(bool(flags & 1)))
            hostapi.lib().pnolhost_set_analytic_slope(int(bool(flags & 2)))
            hostapi.bfgs("bfgs", obj, X0[0], prm)                  # warm-up
            t0 = time.perf_counter()
            for b in range(a.sample):
                hostapi.bfgs("bfgs", obj, X0[b], prm)
            ts = time.perf_counter() - t0
            hostapi.lib().pnolhost_set_analytic_gradient(0)
            hostapi.lib().pnolhost_set_analytic_slope(0)
            entry[mode]["bfgs_class_sample"] = dict(starts=a.sample, seconds=ts)
            entry[mode]["bfgs_class_extrapolated_seconds"] = ts * a.B / a.sample
            entry[mode]["speedup_vs_extrapolated_class_loop"] = ts * a.B / a.sample / entry[mode]["seconds"]
        res["shapes"].append(entry)
        print(json.dumps(dict(shape=name, fd_s=entry["fd"]["seconds"], analytic_s=entry["analytic"]["seconds"],
                              fd_speedup=entry["fd"]["speedup_vs_extrapolated_class_loop"])), file=sys.stderr, flush=True)
    hostapi.detach()
    ctx.close()
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
