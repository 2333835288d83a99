#!/usr/bin/env python3
"""Friends-of-friends throughput against the force pass, in one process on one GPU (soft 2e8 for the force pass):
  force      b200nb_accel                         (N x N interactions), galaxy and random schemes
  sparse     b200nb_fof, b = half the median first-neighbour distance (mean links per body below 1)
  typical    b200nb_fof, b = the median fourth-neighbour distance (a few links per body)
  one_group  b200nb_fof, b above the system's diameter (every pair linked)
Kernel time: torch.profiler (CUDA activities) over `--reps` passes of each, the L2 evicted before every pass
(b200nb_flush_l2).  G-pairs/s = N (N - 1) / 2 / time of fof_link_kernel, set beside the force pass's N x N
interactions per second; init + merge + finalize kernels are reported beside it.  Mean links per body are counted from
the 32 nearest neighbours (so capped at 32).  End-to-end call time: host clock around the synchronous call, without the
profiler.  The GPU's name and power limit are read in the same run and printed in the JSON line.
    python tools/fof_bench.py [--n 200000] [--reps 5] [--out FILE]"""
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


def kernel_ms(ctx, f, reps):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            ctx.flush_l2()
            ctx.sync()
            f()
    tot = {"main": 0.0, "rest": 0.0}
    for ev in prof.key_averages():  # kernels appear under their own names, with their device time
        key = ("main" if ("force_kernel" in ev.key or "fof_link_kernel" in ev.key) else
               "rest" if any(k in ev.key for k in ("integrate_kernel", "fof_init_kernel", "fof_merge_kernel",
                                                   "fof_finalize_kernel")) else None)
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
        sys.exit("fof_bench: no CUDA device (numbers are only taken on the GPU)")

    n = args.n
    pairs = n * (n - 1) / 2
    res = {"tool": "fof_bench", "n": n, "reps": args.reps, "l2": "flushed before every pass", **gpu_info()}
    for scheme in ("galaxy", "random"):
        d = b200nb.init_bodies(scheme, n)
        out = {}
        with b200nb.Context(n, b200nb.G_F32, 2e8, 1) as ctx:
            ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
            dist = ctx.neighbors(32)[1]
            q = np.stack([d["qx"], d["qy"], d["qz"]]).astype(np.float64)
            bs = {"sparse": 0.5 * float(np.median(dist[:, 0])), "typical": float(np.median(dist[:, 3])),
                  "one_group": 2.01 * float(np.max(np.linalg.norm(q - q.mean(axis=1, keepdims=True), axis=0)))}
            calls = {"force": lambda: (ctx.accel(), ctx.sync())}
            calls.update({name: (lambda b=b: ctx.fof(b)) for name, b in bs.items()})
            for f in calls.values():  # warm-up: module load, scratch allocation
                f()
            for name, f in calls.items():
                km = kernel_ms(ctx, f, args.reps)
                if name == "force":
                    out[name] = {"kernel_ms": round(km["main"], 4),
                                 "ginter_per_s": round(n * n / (km["main"] * 1e-3) / 1e9, 1),
                                 "call_ms_host_clock": round(host_ms(ctx, f, args.reps), 3)}
                    continue
                group = f()
                sizes = np.bincount(group, minlength=n)
                out[name] = {"b": bs[name], "mean_links_capped_32": round(float(np.mean(np.sum(dist <= np.float32(bs[name]), axis=1))), 3),
                             "groups": int(np.count_nonzero(sizes)), "largest_group": int(sizes.max()),
                             "link_kernel_ms": round(km["main"], 4), "merge_finalize_ms": round(km["rest"], 4),
                             "gpairs_per_s": round(pairs / (km["main"] * 1e-3) / 1e9, 1),
                             "call_ms_host_clock": round(host_ms(ctx, f, args.reps), 3)}
                out[name]["vs_force_rate"] = round(out[name]["gpairs_per_s"] / out["force"]["ginter_per_s"], 3)
        res[scheme] = out
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
