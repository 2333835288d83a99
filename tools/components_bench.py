#!/usr/bin/env python3
"""Field-by-component throughput against the force pass and the field, in one process on one GPU (galaxy scheme, soft 2e8):
  force            b200nb_accel                                   (N x N interactions)
  potential        b200nb_potential                               (N x N, self pair excluded)
  field_grid       b200nb_field on a 1024 x 1024 grid             (M = 2^20 points)
  bodies_c1        b200nb_component_field_bodies, one component holding every body
  bodies_c4        the same, 4 components of consecutive bodies
  bodies_c4_random the same, 4 components of random labels
  bodies_c64       the same, 64 components of consecutive bodies
  grid_c4          b200nb_component_field on the 1024 x 1024 grid, 4 components of consecutive bodies
Kernel time: torch.profiler (CUDA activities) over `--reps` passes of each, the L2 evicted before every pass
(b200nb_flush_l2); the median over the passes of each kernel family's device time per pass; G-interactions/s = M * N /
kernel time (padding sources not counted).  End-to-end call time: median of a host clock around the synchronous call,
without the profiler.  The GPU's name and power limit are read in the same run and printed in the JSON line.
    python tools/components_bench.py [--n 200000] [--reps 7] [--out FILE]"""
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

MAIN = ("force_kernel", "field_kernel")  # component_field_kernel included
OTHER = ("reduce_kernel", "pack_kernel", "integrate_kernel")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=200000)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    if not torch.cuda.is_available():
        sys.exit("components_bench: no CUDA device (numbers are only taken on the GPU)")

    n = args.n
    d = b200nb.init_bodies("galaxy", n)
    r_sys = float(np.max(np.hypot(np.hypot(d["qx"], d["qy"]), d["qz"])))
    g = np.linspace(-1.5 * r_sys, 1.5 * r_sys, 1024, dtype=np.float32)
    gx, gy = np.meshgrid(g, g)
    grid = [gx.ravel().copy(), gy.ravel().copy(), np.zeros(gx.size, np.float32)]
    one = np.zeros(n, np.uint32)
    c4 = (np.arange(n) * 4 // n).astype(np.uint32)
    c4r = np.random.default_rng(0).integers(0, 4, n).astype(np.uint32)
    c64 = (np.arange(n) * 64 // n).astype(np.uint32)
    cases = {"force": n, "potential": n, "field_grid": grid[0].size, "bodies_c1": n, "bodies_c4": n, "bodies_c4_random": n,
             "bodies_c64": n, "grid_c4": grid[0].size}

    with b200nb.Context(n, b200nb.G_F32, 2e8, 1) as ctx:
        ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
        calls = {"force": lambda: (ctx.accel(), ctx.sync()), "potential": ctx.potential,
                 "field_grid": lambda: ctx.field(*grid),
                 "bodies_c1": lambda: ctx.component_field_bodies(one, 1),
                 "bodies_c4": lambda: ctx.component_field_bodies(c4, 4),
                 "bodies_c4_random": lambda: ctx.component_field_bodies(c4r, 4),
                 "bodies_c64": lambda: ctx.component_field_bodies(c64, 64),
                 "grid_c4": lambda: ctx.component_field(c4, 4, *grid)}
        for f in calls.values():  # warm-up: module load, scratch allocation
            f()
        kernel_ms = {}
        for name, f in calls.items():
            per = {"main": [], "other": []}
            for _ in range(args.reps):
                ctx.flush_l2()
                ctx.sync()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    f()
                tot = {"main": 0.0, "other": 0.0}
                for ev in prof.key_averages():  # kernels appear under their own names, with their device time
                    key = "main" if any(k in ev.key for k in MAIN) else "other" if any(k in ev.key for k in OTHER) else None
                    if key:
                        tot[key] += getattr(ev, "device_time_total", getattr(ev, "cuda_time_total", 0.0)) / 1000.0  # us -> ms
                for k in per:
                    per[k].append(tot[k])
            kernel_ms[name] = {k: statistics.median(v) for k, v in per.items()}
        e2e_ms = {}
        for name, f in calls.items():
            ts = []
            for _ in range(args.reps):
                ctx.sync()
                t0 = time.perf_counter()
                f()
                ts.append((time.perf_counter() - t0) * 1e3)
            e2e_ms[name] = statistics.median(ts)
        # the split of the grid's potential between the components, as a check that the grid run computed something
        acc, phi = ctx.component_field(c4, 4, *grid)
        f = ctx.field(*grid)
        sum_rel = float(np.max(np.abs(phi.astype(np.float64).sum(1) - f[3]) / np.abs(f[3].astype(np.float64))))

    res = {"tool": "components_bench", "n": n, "scheme": "galaxy", "soft": 2e8, "reps": args.reps,
           "l2": "flushed before every pass", "statistic": "median over passes", **gpu_info()}
    for name, m in cases.items():
        k = kernel_ms[name]["main"]
        res[name] = {"targets": m, "kernel_ms": round(k, 4), "other_kernels_ms": round(kernel_ms[name]["other"], 4),
                     "ginter_per_s": round(m * n / (k * 1e-3) / 1e9, 1) if k > 0 else None,
                     "call_ms_host_clock": round(e2e_ms[name], 3)}
    for name in ("bodies_c1", "bodies_c4", "bodies_c4_random", "bodies_c64"):
        res[f"{name}_vs_potential_rate"] = round(res[name]["ginter_per_s"] / res["potential"]["ginter_per_s"], 3)
    res["grid_c4_vs_field_grid_rate"] = round(res["grid_c4"]["ginter_per_s"] / res["field_grid"]["ginter_per_s"], 3)
    res["potential_vs_force_rate"] = round(res["potential"]["ginter_per_s"] / res["force"]["ginter_per_s"], 3)
    res["grid_c4_sum_phi_vs_field_max_rel"] = sum_rel
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
