#!/usr/bin/env python3
"""Cost of the static external potential (b200nb_set_external), in one process on one GPU (galaxy scheme, soft 2e8,
N bodies, a three-term host: Hernquist bulge + Miyamoto-Nagai disk + NFW halo):
  step       b200nb_step of one iteration without terms and with the host, both integrators, on two contexts holding the
             same state; the two arms alternate step by step, device events around each step, the L2 evicted before
             every step (b200nb_flush_l2), median of --steps
  integrate  integrate_kernel alone: mean device time per launch from torch.profiler (CUDA activities), both arms
  tracers    the step with M tracers (a second galaxy realisation), without and with the host, timed as `step`
  field      b200nb_external_field on 2^24 points: wall time of the call (host copies included) and kernel time
The GPU's name and power limit are read in the same run and printed in the JSON line.
    python tools/external_bench.py [--n 200000] [--tracers 2000000] [--steps 9] [--out FILE]"""
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
from tracers_bench import gpu_info  # noqa: E402

DT, SOFT = 3600.0, 2e8
KEYS = ("qx", "qy", "qz", "vx", "vy", "vz")


def host_terms(d):
    gm = float(b200nb.G_F32) * float(np.sum(d["m"], dtype=np.float64))
    r = float(np.max(np.hypot(np.hypot(d["qx"], d["qy"]), d["qz"])))
    return [b200nb.hernquist(2 * gm, 0.25 * r), b200nb.miyamoto_nagai(3 * gm, 0.5 * r, 0.1 * r), b200nb.nfw(5 * gm, 2 * r)]


def one_step_ms(ctx, integrator):
    ctx.flush_l2()
    ctx.sync()
    ctx.event_record(0)
    ctx.step(DT, integrator, 1)
    ctx.event_record(1)
    return ctx.event_elapsed_ms(0, 1)


def alternate(arms, integrator, steps, warmup=2):
    """median step time of each context, the arms timed in turn"""
    for c in arms:
        c.step(DT, integrator, warmup)
    ts = [[] for _ in arms]
    for _ in range(steps):
        for c, t in zip(arms, ts):
            t.append(one_step_ms(c, integrator))
    return [statistics.median(t) for t in ts]


def kernel_ms(ctx, integrator, name, reps):
    """mean device time per launch of the kernels whose name contains `name`, over `reps` steps"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            ctx.flush_l2()
            ctx.sync()
            ctx.step(DT, integrator, 1)
        ctx.sync()
    tot, cnt = 0.0, 0
    for ev in prof.key_averages():
        if name in ev.key:
            tot += getattr(ev, "device_time_total", getattr(ev, "cuda_time_total", 0.0)) / 1000.0
            cnt += ev.count
    return tot / max(cnt, 1), cnt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=200000)
    ap.add_argument("--tracers", type=int, default=2000000)
    ap.add_argument("--steps", type=int, default=9)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("external_bench: no CUDA device (numbers are only taken on the GPU)")

    n = args.n
    d = b200nb.init_bodies("galaxy", n)
    terms = host_terms(d)
    res = {"tool": "external_bench", "n": n, "scheme": "galaxy", "soft": SOFT, "dt": DT, "steps": args.steps,
           "terms": ["hernquist", "miyamoto_nagai", "nfw"], "l2": "flushed before every timed step", **gpu_info()}

    arms = [b200nb.Context(n, b200nb.G_F32, SOFT, 1) for _ in range(2)]
    arms[1].set_external(terms)
    try:
        for integrator, name in ((b200nb.INTEGRATOR_MURB, "murb"), (b200nb.INTEGRATOR_LEAPFROG, "leapfrog")):
            for c in arms:
                c.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
            t0, t1 = alternate(arms, integrator, args.steps)
            k0, c0 = kernel_ms(arms[0], integrator, "integrate_kernel", args.steps)
            k1, c1 = kernel_ms(arms[1], integrator, "integrate_kernel", args.steps)
            res[name] = {"step_ms_0_terms": round(t0, 4), "step_ms_3_terms": round(t1, 4),
                         "step_overhead": round(t1 / t0 - 1, 5),
                         "integrate_kernel_us_0_terms": round(1000 * k0, 2), "integrate_kernel_us_3_terms": round(1000 * k1, 2),
                         "integrate_launches_profiled": [c0, c1]}
        m = args.tracers
        pool = b200nb.init_bodies("galaxy", m, seed=1)
        for integrator, name in ((b200nb.INTEGRATOR_MURB, "murb"), (b200nb.INTEGRATOR_LEAPFROG, "leapfrog")):
            for c in arms:
                c.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
                c.set_tracers(*[pool[k] for k in KEYS])
            t0, t1 = alternate(arms, integrator, max(3, args.steps // 2), warmup=1)
            res[name][f"tracers_{m}"] = {"step_ms_0_terms": round(t0, 3), "step_ms_3_terms": round(t1, 3),
                                          "step_overhead": round(t1 / t0 - 1, 5)}
        for c in arms:
            c.set_tracers(*[np.zeros(0, np.float32)] * 6)

        p = b200nb.init_bodies("galaxy", 1 << 24, seed=2)
        pts = [p["qx"], p["qy"], p["qz"]]
        arms[1].external_field(*pts)  # warm-up: the scratch grows once
        t = time.perf_counter()
        arms[1].external_field(*pts)
        wall = time.perf_counter() - t
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            arms[1].external_field(*pts)
        kt = sum(getattr(ev, "device_time_total", 0.0) for ev in prof.key_averages() if "external_field_kernel" in ev.key) / 1e6
        res["external_field"] = {"points": len(pts[0]), "wall_s": round(wall, 4), "points_per_s": round(len(pts[0]) / wall, 1),
                                 "kernel_s": round(kt, 6), "kernel_points_per_s": round(len(pts[0]) / kt, 1) if kt > 0 else None}
    finally:
        for c in arms:
            c.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
