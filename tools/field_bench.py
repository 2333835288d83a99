#!/usr/bin/env python3
"""Field and potential throughput against the force pass, in one process on one GPU (galaxy scheme, soft 2e8):
  force   b200nb_accel                       (N x N interactions)
  potential b200nb_potential                 (N x N, self pair excluded)
  grid    b200nb_field on a 1024 x 1024 grid (M = 2^20 points)
  curve   b200nb_field on 100 points of a rotation curve v_c(R) = sqrt(R |a_R|)
Kernel time: torch.profiler (CUDA activities) over `--reps` passes of each, the L2 evicted before every pass
(b200nb_flush_l2); G-interactions/s = M * N / kernel time.  End-to-end call time: host clock around the synchronous
call, without the profiler.  The GPU's name and power limit are read in the same run and printed in the JSON line.
    python tools/field_bench.py [--n 200000] [--reps 5] [--out FILE]"""
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


def gpu_info():
    import torch
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return {"gpu": out[0], "power_limit_w": float(out[1]), "sm_clock_max_mhz": float(out[2])}
    except Exception:
        return {"gpu": torch.cuda.get_device_name(0), "power_limit_w": None, "sm_clock_max_mhz": None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=200000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    if not torch.cuda.is_available():
        sys.exit("field_bench: no CUDA device (numbers are only taken on the GPU)")

    n = args.n
    d = b200nb.init_bodies("galaxy", n)
    r_sys = float(np.max(np.hypot(np.hypot(d["qx"], d["qy"]), d["qz"])))
    g = np.linspace(-1.5 * r_sys, 1.5 * r_sys, 1024, dtype=np.float32)
    gx, gy = np.meshgrid(g, g)
    grid = [gx.ravel().copy(), gy.ravel().copy(), np.zeros(gx.size, np.float32)]
    rc = np.linspace(r_sys / 100, 1.5 * r_sys, 100, dtype=np.float32)
    curve = [rc, np.zeros_like(rc), np.zeros_like(rc)]
    cases = {"force": n, "potential": n, "grid": grid[0].size, "curve": rc.size}

    with b200nb.Context(n, b200nb.G_F32, 2e8, 1) as ctx:
        ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
        calls = {"force": lambda: (ctx.accel(), ctx.sync()), "potential": ctx.potential,
                 "grid": lambda: ctx.field(*grid), "curve": lambda: ctx.field(*curve)}
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
                key = ("main" if ("force_kernel" in ev.key or "field_kernel" in ev.key) else
                       "reduce" if ("field_reduce_kernel" in ev.key or "integrate_kernel" in ev.key) else None)
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
        ax = ctx.field(*curve)[0]
        vc = np.sqrt(rc.astype(np.float64) * np.abs(ax.astype(np.float64)))

    res = {"tool": "field_bench", "n": n, "scheme": "galaxy", "soft": 2e8, "reps": args.reps, "l2": "flushed before every pass",
           **gpu_info()}
    for name, m in cases.items():
        k = kernel_ms[name]["main"]
        res[name] = {"targets": m, "kernel_ms": round(k, 4), "reduce_ms": round(kernel_ms[name]["reduce"], 4),
                     "ginter_per_s": round(m * n / (k * 1e-3) / 1e9, 1) if k > 0 else None,
                     "call_ms_host_clock": round(e2e_ms[name], 3)}
    res["potential_vs_force_rate"] = round(res["potential"]["ginter_per_s"] / res["force"]["ginter_per_s"], 3)
    res["grid_vs_force_rate"] = round(res["grid"]["ginter_per_s"] / res["force"]["ginter_per_s"], 3)
    res["rotation_curve_vc_m_per_s"] = {"R_m": [float(rc[i]) for i in (9, 49, 99)], "vc": [round(float(vc[i]), 2) for i in (9, 49, 99)]}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
