#!/usr/bin/env python3
"""Group potential and unbinding against the per-body potential and the force pass, in one process on one GPU
(soft 2e8), galaxy and random schemes:
  force       b200nb_accel                       (N x N interactions)
  potential   b200nb_potential                   (N (N - 1) pairs)
  fof4, fof6  b200nb_group_potential on friends-of-friends labels at the median 4th- / 6th-neighbour distance
  one         b200nb_group_potential with every body in one label
Kernel time: torch.profiler (CUDA activities) over `--reps` passes of each, the L2 evicted before every pass
(b200nb_flush_l2).  G-pairs/s of the group potential = the needed pairs sum n_g (n_g - 1), and the pairs the kernel visits
(each 1024-target tile streams the union of its targets' label ranges), over the time of group_potential_kernel; the
other kernels of the call (sort, pack, reduce, finish) are reported beside it.  `vs_potential` and `vs_force` are
ratios of kernel times in the same run.  End-to-end call time: host clock around the synchronous call, without the
profiler.  b200nb_unbind on the FoF labels: call time, passes, and the bound fraction of the largest group.  The GPU's
name and power limit are read in the same run and printed in the JSON line.
    python tools/groups_bench.py [--n 200000] [--reps 5] [--out FILE]"""
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

TI = 1024  # targets per tile of group_potential_kernel (GP_TI)


def gpu_info():
    import torch
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return {"gpu": out[0], "power_limit_w": float(out[1]), "sm_clock_max_mhz": float(out[2])}
    except Exception:
        return {"gpu": torch.cuda.get_device_name(0), "power_limit_w": None, "sm_clock_max_mhz": None}


MAIN = ("force_kernel", "field_kernel", "group_potential_kernel")


def kernel_ms(ctx, f, reps):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            ctx.flush_l2()
            ctx.sync()
            f()
    tot = {"main": 0.0, "rest": 0.0}
    for ev in prof.key_averages():  # kernels appear under their own names, with their device time
        if "memset" in ev.key.lower() or "memcpy" in ev.key.lower() or "fill" in ev.key.lower():
            continue
        t = getattr(ev, "device_time_total", getattr(ev, "cuda_time_total", 0.0)) / 1000.0  # us -> ms
        tot["main" if any(k in ev.key for k in MAIN) else "rest"] += t
    return {k: v / reps for k, v in tot.items()}


def host_ms(ctx, f, reps):
    ts = []
    for _ in range(reps):
        ctx.sync()
        t0 = time.perf_counter()
        f()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts)


def pair_counts(g):
    """needed pairs sum n_g (n_g - 1) and the pairs group_potential_kernel visits"""
    lab = np.sort(g[g != b200nb.NO_GROUP].astype(np.int64))
    M = len(lab)
    _, start, size = np.unique(lab, return_index=True, return_counts=True)
    needed = float(np.sum(size.astype(np.float64) * (size - 1)))
    lo = np.repeat(start, size)
    hi = lo + np.repeat(size, size)
    visited = 0.0
    for t0 in range(0, M, TI):
        t1 = min(t0 + TI, M)
        visited += float(t1 - t0) * float(hi[t1 - 1] - lo[t0])
    return needed, visited


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=200000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("groups_bench: no CUDA device (numbers are only taken on the GPU)")

    n = args.n
    res = {"tool": "groups_bench", "n": n, "reps": args.reps, "l2": "flushed before every pass", **gpu_info()}
    for scheme in ("galaxy", "random"):
        d = b200nb.init_bodies(scheme, n)
        out = {}
        with b200nb.Context(n, b200nb.G_F32, 2e8, 1) as ctx:
            ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
            dist = ctx.neighbors(6)[1]
            labels = {"fof4": ctx.fof(float(np.median(dist[:, 3]))), "fof6": ctx.fof(float(np.median(dist[:, 5]))),
                      "one": np.zeros(n, np.uint32)}
            calls = {"force": lambda: (ctx.accel(), ctx.sync()), "potential": ctx.potential}
            calls.update({name: (lambda g=g: ctx.group_potential(g)) for name, g in labels.items()})
            for f in calls.values():  # warm-up: module load, scratch allocation
                f()
            for name, f in calls.items():
                km = kernel_ms(ctx, f, args.reps)
                row = {"kernel_ms": round(km["main"], 4), "other_kernels_ms": round(km["rest"], 4),
                       "call_ms_host_clock": round(host_ms(ctx, f, args.reps), 3)}
                if name == "force":
                    row["ginter_per_s"] = round(n * n / (km["main"] * 1e-3) / 1e9, 1)
                elif name == "potential":
                    row["gpairs_per_s"] = round(n * (n - 1) / (km["main"] * 1e-3) / 1e9, 1)
                else:
                    g = labels[name]
                    needed, visited = pair_counts(g)
                    sizes = np.unique(g, return_counts=True)[1]
                    row.update({"groups": int(len(sizes)), "largest_group": int(sizes.max()),
                                "needed_pairs_over_n2": round(needed / n / n, 4), "visited_pairs_over_n2": round(visited / n / n, 4),
                                "gpairs_per_s_needed": round(needed / (km["main"] * 1e-3) / 1e9, 1),
                                "gpairs_per_s_visited": round(visited / (km["main"] * 1e-3) / 1e9, 1)})
                out[name] = row
            for name in labels:
                out[name]["vs_potential_kernel_time"] = round(out["potential"]["kernel_ms"] / out[name]["kernel_ms"], 3)
                out[name]["vs_force_kernel_time"] = round(out["force"]["kernel_ms"] / out[name]["kernel_ms"], 3)
                out[name]["call_vs_potential_call"] = round(out["potential"]["call_ms_host_clock"] / out[name]["call_ms_host_clock"], 3)
                out[name]["rate_vs_potential_rate"] = round(out[name]["gpairs_per_s_visited"] / out["potential"]["gpairs_per_s"], 3)
            for name in ("fof4", "fof6"):
                g = labels[name]
                f = lambda g=g: ctx.unbind(g)  # noqa: E731
                bound, _, it, conv = f()
                big = np.bincount(np.unique(g, return_inverse=True)[1]).argmax()
                root = np.unique(g)[big]
                out[name]["unbind"] = {"call_ms_host_clock": round(host_ms(ctx, f, args.reps), 3), "passes": it, "converged": conv,
                                       "largest_group_bound_fraction": round(float(np.mean(bound[g == root] == root)), 4),
                                       "bound_fraction": round(float(np.mean(bound != b200nb.NO_GROUP)), 4)}
        res[scheme] = out
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
