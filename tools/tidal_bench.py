#!/usr/bin/env python3
"""Tidal-tensor throughput against the force pass and the field, in one process on one GPU (galaxy scheme, soft 2e8):
  force       b200nb_accel                        (N x N interactions)
  potential   b200nb_potential                    (N x N, self pair excluded)
  tidal_bodies b200nb_tidal_bodies                (N x N, self pair excluded)
  tidal_grid  b200nb_tidal on a 1024 x 1024 grid  (M = 2^20 points)
Kernel time: torch.profiler (CUDA activities) over `--reps` passes of each, the L2 evicted before every pass
(b200nb_flush_l2); G-interactions/s = M * N / kernel time.  End-to-end call time: host clock around the synchronous
call, without the profiler.  The GPU's name and power limit are read in the same run and printed in the JSON line.
    python tools/tidal_bench.py [--n 200000] [--reps 5] [--out FILE]"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "nbody-eurohpc_b200"))
sys.path.insert(0, os.path.join(REPO, "tools"))
import b200nb  # noqa: E402
from field_bench import gpu_info  # noqa: E402

MAIN = ("force_kernel", "field_kernel", "tidal_kernel")
REDUCE = ("field_reduce_kernel", "tidal_reduce_kernel", "integrate_kernel")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=200000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    if not torch.cuda.is_available():
        sys.exit("tidal_bench: no CUDA device (numbers are only taken on the GPU)")

    n = args.n
    d = b200nb.init_bodies("galaxy", n)
    r_sys = float(np.max(np.hypot(np.hypot(d["qx"], d["qy"]), d["qz"])))
    g = np.linspace(-1.5 * r_sys, 1.5 * r_sys, 1024, dtype=np.float32)
    gx, gy = np.meshgrid(g, g)
    grid = [gx.ravel().copy(), gy.ravel().copy(), np.zeros(gx.size, np.float32)]
    cases = {"force": n, "potential": n, "tidal_bodies": n, "tidal_grid": grid[0].size}

    with b200nb.Context(n, b200nb.G_F32, 2e8, 1) as ctx:
        ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
        calls = {"force": lambda: (ctx.accel(), ctx.sync()), "potential": ctx.potential,
                 "tidal_bodies": ctx.tidal_bodies, "tidal_grid": lambda: ctx.tidal(*grid)}
        for f in calls.values():  # warm-up: module load, scratch allocation
            f()
        kernel_ms = {}
        for name, f in calls.items():
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(args.reps):
                    ctx.flush_l2()
                    ctx.sync()
                    f()
            tot = {"main": 0.0, "reduce": 0.0}
            for ev in prof.key_averages():  # kernels appear under their own names, with their device time
                key = "main" if any(k in ev.key for k in MAIN) else "reduce" if any(k in ev.key for k in REDUCE) else None
                if key:
                    tot[key] += getattr(ev, "device_time_total", getattr(ev, "cuda_time_total", 0.0)) / 1000.0  # us -> ms
            kernel_ms[name] = {k: v / args.reps for k, v in tot.items()}
        e2e_ms = {}
        for name, f in calls.items():
            ts = []
            for _ in range(args.reps):
                ctx.sync()
                t0 = time.perf_counter()
                f()
                ts.append((time.perf_counter() - t0) * 1e3)
            e2e_ms[name] = statistics.median(ts)
        # the grid's tidal environment: the share of points with one stretching and two compressive eigenvalues
        lam = np.linalg.eigvalsh(ctx.tidal(*grid).astype(np.float64))
        one_stretch = float(np.mean(np.sum(lam > 0, axis=1) == 1))

    res = {"tool": "tidal_bench", "n": n, "scheme": "galaxy", "soft": 2e8, "reps": args.reps, "l2": "flushed before every pass",
           **gpu_info()}
    for name, m in cases.items():
        k = kernel_ms[name]["main"]
        res[name] = {"targets": m, "kernel_ms": round(k, 4), "reduce_ms": round(kernel_ms[name]["reduce"], 4),
                     "ginter_per_s": round(m * n / (k * 1e-3) / 1e9, 1) if k > 0 else None,
                     "call_ms_host_clock": round(e2e_ms[name], 3)}
    f = res["force"]["ginter_per_s"]
    res["tidal_bodies_vs_force_rate"] = round(res["tidal_bodies"]["ginter_per_s"] / f, 3)
    res["tidal_grid_vs_force_rate"] = round(res["tidal_grid"]["ginter_per_s"] / f, 3)
    res["potential_vs_force_rate"] = round(res["potential"]["ginter_per_s"] / f, 3)
    res["grid_share_one_stretching_axis"] = round(one_stretch, 4)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
