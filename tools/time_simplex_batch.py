"""Times pnol_simplex_batch on the GPU: B random starts of one objective minimised in one call, against the same starts through the
SimplexSearch class one at a time (a sample of 64 starts, timed and extrapolated to B -- labelled as an extrapolation). CUDA events
around each call with device-resident arrays and the counter stream; the first call of every shape is a warm-up; the median of
--repeats calls is reported. Prints one JSON document (and writes it to --out when given) with the card's name, power limit and maximum
SM clock read in the same run.

    python tools/time_simplex_batch.py [--B 65536] [--repeats 3] [--sample 64] [--out FILE]
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
SEED = 2024


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
    ap.add_argument("--shapes", default=",".join(s[0] for s in SHAPES))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    ctx = capi.Context(0)
    hostapi.attach(ctx)
    dev = torch.device("cuda:0")
    res = dict(card=card(), B=a.B, repeats=a.repeats, params="SimplexSearch defaults (alpha 1, gamma 2, rho 0.5, sigma 0.5, max_iter 10000, "
               "init_rand_max 1, x_min_diff 1e-7), counter stream seed %d" % SEED, shapes=[])
    stream = capi.StreamDesc(None, 0, SEED, 1.0)
    for name, obj, kind, n, w in SHAPES:
        if name not in a.shapes.split(","):
            continue
        X0 = np.random.default_rng(n).uniform(-w, w, size=(a.B, n))
        X0d = torch.tensor(X0, device=dev)
        Xd = torch.empty_like(X0d)
        f = ctx.functor(kind)
        out = dict(f0=torch.empty(a.B, dtype=torch.float64, device=dev), fopt=torch.empty(a.B, dtype=torch.float64, device=dev),
                   iters=torch.empty(a.B, dtype=torch.int32, device=dev), stop=torch.empty(a.B, dtype=torch.int32, device=dev),
                   evals=torch.empty(a.B, dtype=torch.int64, device=dev))
        times = []
        for rep in range(a.repeats + 1):           # rep 0: warm-up
            Xd.copy_(X0d)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ctx.simplex_batch(f, Xd, stream=stream, n=n, B=a.B, out=out)
            e1.record()
            torch.cuda.synchronize()
            if rep > 0:
                times.append(e0.elapsed_time(e1) / 1e3)
        iters = int(out["iters"].sum().item())
        evals = int(out["evals"].sum().item())
        t = float(np.median(times))
        entry = dict(shape=name, n=n, B=a.B, seconds=t, fits_per_s=a.B / t, problem_iterations=iters, problem_iterations_per_s=iters / t,
                     evaluations=evals, evaluations_per_s=evals / t, stop_max_iter=int((out["stop"] == 0).sum().item()), all_seconds=times)
        # the same starts through the SimplexSearch class one at a time (GPU evaluations, one host loop per start): a sample, each start
        # on its own slice of the stream as in the batch, extrapolated to B
        u = lambda b: np.array([capi.load_library().pnol_stream_uniform(SEED, b * n * n + t, 1.0) for t in range(n * n)])
        hostapi.set_stream(values=u(0))
        hostapi.simplex(obj, X0[0])                 # warm-up
        ts = 0.0
        for b in range(a.sample):
            hostapi.set_stream(values=u(b))
            t0 = time.perf_counter()
            hostapi.simplex(obj, X0[b])
            ts += time.perf_counter() - t0
        entry["class_sample"] = dict(starts=a.sample, seconds=ts)
        entry["class_extrapolated_seconds"] = ts * a.B / a.sample
        entry["speedup_vs_extrapolated_class_loop"] = ts * a.B / a.sample / t
        res["shapes"].append(entry)
        print(json.dumps(dict(shape=name, batch_s=t, class_extrapolated_s=entry["class_extrapolated_seconds"])), file=sys.stderr, flush=True)
    hostapi.detach()
    ctx.close()
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
