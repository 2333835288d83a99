#!/usr/bin/env python3
"""Nearest-neighbour throughput against the force pass, in one process on one GPU (soft 2e8 for the force pass):
  force          b200nb_accel                               (N x N interactions), galaxy and random schemes
  bodies_k<K>    b200nb_neighbors(k = K)                    (N x N, self pair excluded), K = 1, 6, 8, 32
  grid_k<K>      b200nb_neighbors_at on a 1024 x 1024 grid  (M = 2^20 points, galaxy scheme)
Kernel time: torch.profiler (CUDA activities) over `--reps` passes of each, the L2 evicted before every pass
(b200nb_flush_l2); G-interactions/s = M * N / time of neighbors_kernel (the merge kernel is reported beside it).
End-to-end call time: host clock around the synchronous call, without the profiler.  The GPU's name and power limit are
read in the same run and printed in the JSON line.
    python tools/neighbors_bench.py [--n 200000] [--reps 5] [--out FILE]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "nbody-eurohpc_b200"))
import b200nb  # noqa: E402

KS = (1, 6, 8, 32)


def gpu_info():
    import torch
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return {"gpu": out[0], "power_limit_w": float(out[1]), "sm_clock_max_mhz": float(out[2])}
    except Exception:
        return {"gpu": torch.cuda.get_device_name(0), "power_limit_w": None, "sm_clock_max_mhz": None}


def kernel_ms(ctx, f, reps):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            ctx.flush_l2()
            ctx.sync()
            f()
    tot = {"main": 0.0, "merge": 0.0}
    for ev in prof.key_averages():  # kernels appear under their own names, with their device time
        key = ("main" if ("force_kernel" in ev.key or "neighbors_kernel" in ev.key) else
               "merge" if ("nb_merge_kernel" in ev.key or "integrate_kernel" in ev.key) else None)
        if key:
            tot[key] += getattr(ev, "device_time_total", getattr(ev, "cuda_time_total", 0.0)) / 1000.0  # us -> ms
    return {k: v / reps for k, v in tot.items()}


def host_ms(ctx, f, reps):
    ts = []
    for _ in range(reps):
        ctx.sync()
        t0 = time.perf_counter()
        f()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=200000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("neighbors_bench: no CUDA device (numbers are only taken on the GPU)")

    n = args.n
    res = {"tool": "neighbors_bench", "n": n, "reps": args.reps, "l2": "flushed before every pass", **gpu_info()}
    for scheme in ("galaxy", "random"):
        d = b200nb.init_bodies(scheme, n)
        cases = {"force": (n, None)}
        cases.update({f"bodies_k{k}": (n, k) for k in KS})
        if scheme == "galaxy":
            r_sys = float(np.max(np.hypot(np.hypot(d["qx"], d["qy"]), d["qz"])))
            g = np.linspace(-1.5 * r_sys, 1.5 * r_sys, 1024, dtype=np.float32)
            gx, gy = np.meshgrid(g, g)
            grid = [gx.ravel().copy(), gy.ravel().copy(), np.zeros(gx.size, np.float32)]
            cases.update({f"grid_k{k}": (grid[0].size, k) for k in KS})
        out = {}
        with b200nb.Context(n, b200nb.G_F32, 2e8, 1) as ctx:
            ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
            calls = {}
            for name, (m, k) in cases.items():
                if name == "force":
                    calls[name] = lambda: (ctx.accel(), ctx.sync())
                elif name.startswith("bodies"):
                    calls[name] = (lambda k=k: ctx.neighbors(k))
                else:
                    calls[name] = (lambda k=k: ctx.neighbors_at(*grid, k))
            for f in calls.values():  # warm-up: module load, scratch allocation
                f()
            for name, f in calls.items():
                km = kernel_ms(ctx, f, args.reps)
                m = cases[name][0]
                out[name] = {"targets": m, "kernel_ms": round(km["main"], 4), "merge_ms": round(km["merge"], 4),
                             "ginter_per_s": round(m * n / (km["main"] * 1e-3) / 1e9, 1) if km["main"] > 0 else None,
                             "call_ms_host_clock": round(host_ms(ctx, f, args.reps), 3)}
            for name in cases:
                if name != "force":
                    out[name]["vs_force_rate"] = round(out[name]["ginter_per_s"] / out["force"]["ginter_per_s"], 3)
        res[scheme] = out
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
