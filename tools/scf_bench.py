#!/usr/bin/env python3
"""Cost of the basis-function expansion (b200nb_scf_coefficients, b200nb_scf_field), in one process on one GPU:
  coefficients  a flattened Hernquist sample of N = 200k and 1M bodies, (nmax, lmax) = (10, 6) and (24, 12): the wall
                time of the call (it ends in a device join; host tables and copies included), median of --reps, and the
                device time of its two kernels from torch.profiler (CUDA activities), mean per call
  field         b200nb_scf_field at 2^20 points for (10, 6) and (24, 12): wall time and kernel time
  force         b200nb_step of one MUrB iteration on the 200k galaxy scheme (soft 2e8), device events, L2 evicted first,
                median of 5: the scale of the step the expansion sits beside
The fp64 operation counts come from the kernels' structure: the coefficient kernel issues 16 FMAs per register tile and
staged body (tiles: ceil((nmax+1)/4) * ceil((l+1)/2) per l), plus the basis recurrences of each staged body.  The GPU's name
and power limit are read in the same run and printed in the JSON line.
    python tools/scf_bench.py [--reps 7] [--out FILE]"""
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
from tracers_bench import gpu_info, step_ms  # noqa: E402

A = 3e19
SHAPES = ((10, 6), (24, 12))


def sample(n, seed=1):
    rng = np.random.default_rng(seed)
    u = rng.random(n)
    s = np.sqrt(u) / (1 - np.sqrt(u))
    v = rng.normal(size=(n, 3))
    v /= np.linalg.norm(v, axis=1)[:, None]
    P = v * s[:, None] * np.array([1.0, 0.8, 0.5]) * A
    d = {k: P[:, i].astype(np.float32) for i, k in enumerate(("qx", "qy", "qz"))}
    d["m"] = np.full(n, 2e30, np.float32)
    for k in ("vx", "vy", "vz"):
        d[k] = np.zeros(n, np.float32)
    return d


def tiles(nmax, lmax):
    return sum(((nmax + 4) // 4) * ((l + 2) // 2) for l in range(lmax + 1))


def ops(nmax, lmax):
    """fp64 operations per staged body, from scf_coef_kernel: FMAs of the tiles, and the recurrences (radial: 3 per n and
    2 per power of t; angular: 3 per l and 4 per power of w)"""
    K = (nmax + 1) * (lmax + 1) * (lmax + 2) // 2
    fma = 16 * tiles(nmax, lmax)
    rec = sum(4 * nmax + l + 4 for l in range(lmax + 1)) + sum(4 * m + 3 * (lmax - m) for m in range(lmax + 1))
    return {"K": K, "fma_per_body": fma, "fma_per_body_and_coefficient": round(fma / (2 * K), 3),
            "useful_fma_per_body": 2 * K, "recurrence_ops_per_body": rec}


def kernel_ms(fn, names, reps):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
    tot = {k: 0.0 for k in names}
    for e in prof.key_averages():
        for k in names:
            if k in e.key:
                tot[k] += e.device_time_total / 1e3  # us -> ms
    return {k: round(v / reps, 4) for k, v in tot.items()}


def wall(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "needs a CUDA device"
    res = {"tool": "scf_bench", "a": A, "sample": "Hernquist 1 : 0.8 : 0.5, seed 1"}
    res.update(gpu_info())
    coef = {}
    for n in (200000, 1000000):
        d = sample(n)
        with b200nb.Context(n, b200nb.G_F32, 2e8) as ctx:
            ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
            for nm, lm in SHAPES:
                f = lambda: ctx.scf_coefficients(nm, lm, A)  # noqa: E731
                w = wall(f, args.reps)
                k = kernel_ms(f, ["scf_coef_kernel", "scf_reduce_kernel"], args.reps)
                o = ops(nm, lm)
                kt = k["scf_coef_kernel"] + k["scf_reduce_kernel"]
                coef[f"n{n}_{nm}_{lm}"] = {"wall_ms": round(w, 4), "kernel_ms": k,
                                           "fp64_tflops_of_fma": round(2 * o["fma_per_body"] * n / (kt * 1e-3) / 1e12, 3) if kt else None}
    res["coefficients"] = coef
    res["ops"] = {f"{nm}_{lm}": ops(nm, lm) for nm, lm in SHAPES}
    d = sample(200000)
    m = 1 << 20
    rng = np.random.default_rng(2)
    p = [(rng.normal(size=m) * A).astype(np.float32) for _ in range(3)]
    field = {}
    with b200nb.Context(200000, b200nb.G_F32, 2e8) as ctx:
        ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
        for nm, lm in SHAPES:
            S, T = ctx.scf_coefficients(nm, lm, A)
            f = lambda: ctx.scf_field(S, T, A, (0, 0, 0), *p)  # noqa: E731
            w = wall(f, args.reps)
            k = kernel_ms(f, ["scf_field_kernel"], args.reps)["scf_field_kernel"]
            field[f"{nm}_{lm}"] = {"points": m, "wall_ms": round(w, 4), "points_per_s": round(m / (w * 1e-3), 1),
                                   "kernel_ms": k, "kernel_points_per_s": round(m / (k * 1e-3), 1) if k else None}
    res["field"] = field
    g = b200nb.init_bodies("galaxy", 200000)
    with b200nb.Context(200000, b200nb.G_F32, 2e8) as ctx:
        ctx.upload(g["qx"], g["qy"], g["qz"], g["m"], g["vx"], g["vy"], g["vz"])
        res["force_step_ms_200k"] = round(step_ms(ctx, 0, 5), 4)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
