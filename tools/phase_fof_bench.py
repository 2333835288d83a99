#!/usr/bin/env python3
"""Phase-space friends-of-friends throughput against the force pass and position friends-of-friends, in one process on
one GPU (soft 2e8 for the force pass):
  force      b200nb_accel                         (N x N interactions), galaxy and random schemes
  fof        b200nb_fof, b = the median fourth-neighbour distance (tools/fof_bench.py's typical setting)
  sparse     b200nb_fof_phase, b_x = half the median first-neighbour distance, b_v = sigma (the 3D velocity dispersion)
  typical    b200nb_fof_phase, b_x = twice the median fourth-neighbour distance, b_v = sigma
  one_group  b200nb_fof_phase, b_x = b_v = inf (every pair linked)
Kernel time: torch.profiler (CUDA activities) over `--reps` passes of each, the L2 evicted before every pass
(b200nb_flush_l2).  G-pairs/s = N (N - 1) / 2 / time of the link kernel, set beside the force pass's N x N interactions
per second; pack + init + merge + finalize kernels are reported beside it, and the time of the peer copies or
all-gather (none on one GPU).  End-to-end call time: host clock around the synchronous call, without the profiler.  The
GPU's name and power limit are read in the same run and printed in the JSON line.
    python tools/phase_fof_bench.py [--n 200000] [--reps 5] [--out FILE]"""
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

MAIN = ("force_kernel", "phase_fof_link_kernel", "fof_link_kernel")
REST = ("integrate_kernel", "phase_fof_pack_kernel", "fof_init_kernel", "fof_merge_kernel", "fof_finalize_kernel")


def gpu_info():
    import torch
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return {"gpu": out[0], "power_limit_w": float(out[1]), "sm_clock_max_mhz": float(out[2])}
    except Exception:
        return {"gpu": torch.cuda.get_device_name(0), "power_limit_w": None, "sm_clock_max_mhz": None}


def _kind(key):
    # substrings, as the force kernel may appear under its mangled name; "fof_link_kernel" is part of the phase one's name
    if any(k in key for k in MAIN):
        return "main"
    return "rest" if any(k in key for k in REST) else "copy" if "Memcpy" in key or "nccl" in key else None


def kernel_ms(ctx, f, reps):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            ctx.flush_l2()
            ctx.sync()
            f()
    tot = {"main": 0.0, "rest": 0.0, "copy": 0.0}
    for ev in prof.key_averages():  # kernels appear under their own names, with their device time
        k = _kind(ev.key)
        if k:
            tot[k] += getattr(ev, "device_time_total", getattr(ev, "cuda_time_total", 0.0)) / 1000.0  # us -> ms
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
        sys.exit("phase_fof_bench: no CUDA device (numbers are only taken on the GPU)")

    n = args.n
    pairs = n * (n - 1) / 2
    res = {"tool": "phase_fof_bench", "n": n, "reps": args.reps, "l2": "flushed before every pass", **gpu_info()}
    for scheme in ("galaxy", "random"):
        d = b200nb.init_bodies(scheme, n)
        out = {}
        with b200nb.Context(n, b200nb.G_F32, 2e8, 1) as ctx:
            ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
            dist = ctx.neighbors(4)[1]
            v = np.stack([d["vx"], d["vy"], d["vz"]]).astype(np.float64)
            sig = float(np.sqrt(np.mean(np.sum((v - v.mean(axis=1, keepdims=True)) ** 2, axis=0))))
            d1, d4 = float(np.median(dist[:, 0])), float(np.median(dist[:, 3]))
            bs = {"sparse": (0.5 * d1, sig), "typical": (2 * d4, sig), "one_group": (float("inf"), float("inf"))}
            calls = {"force": lambda: (ctx.accel(), ctx.sync()), "fof": lambda: ctx.fof(d4)}
            calls.update({name: (lambda b=b: ctx.fof_phase(*b)) for name, b in bs.items()})
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
                b_x, b_v = bs.get(name, (d4, None))
                out[name] = {"b_x": b_x if b_x is None or np.isfinite(b_x) else "inf",
                             "b_v": b_v if b_v is None or np.isfinite(b_v) else "inf",
                             "groups": int(np.count_nonzero(sizes)), "largest_group": int(sizes.max()),
                             "link_kernel_ms": round(km["main"], 4), "other_kernels_ms": round(km["rest"], 4),
                             "copies_ms": round(km["copy"], 4),
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
