#!/usr/bin/env python3
"""Cost of a frozen basis-function expansion in the external potential (b200nb_set_external_scf), in one process on one
GPU (galaxy scheme, soft 2e8, N bodies).  Four contexts hold the same state: no external potential, the three-term host
of tools/external_bench.py (Hernquist bulge + Miyamoto-Nagai disk + NFW halo), and that host plus an expansion at
(nmax, lmax) = (10, 6) and (24, 12) (coefficients of the galaxy itself, so every S and T entry is a real number):
  step       b200nb_step of one iteration in every arm, both integrators; the arms alternate step by step, device events
             around each step, the L2 evicted before every step (b200nb_flush_l2), median of --steps
  tracers    the step with M tracers (a second galaxy realisation), timed the same way with max(3, steps // 2) samples
  kernel     ext_total_kernel alone: mean device time per launch from torch.profiler (CUDA activities), in a separate run
  field      b200nb_external_field on 2^24 points with each expansion: wall time of the call (host copies included) and
             kernel time
The GPU's name and power limit are read in the same run and printed in the JSON line.
    python tools/external_scf_bench.py [--n 200000] [--tracers 2000000] [--steps 9] [--out FILE]"""
import argparse
import json
import os
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "nbody-eurohpc_b200"))
sys.path.insert(0, os.path.join(REPO, "tools"))
import b200nb  # noqa: E402
from external_bench import DT, KEYS, SOFT, alternate, host_terms, kernel_ms  # noqa: E402
from tracers_bench import gpu_info  # noqa: E402

ARMS = ("none", "3_terms", "3_terms_scf_10_6", "3_terms_scf_24_12")
EXPANSIONS = ((10, 6), (24, 12))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=200000)
    ap.add_argument("--tracers", type=int, default=2000000)
    ap.add_argument("--steps", type=int, default=9)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("external_scf_bench: no CUDA device (numbers are only taken on the GPU)")

    n = args.n
    d = b200nb.init_bodies("galaxy", n)
    terms = host_terms(d)
    a = 0.5 * float(np.max(np.hypot(np.hypot(d["qx"], d["qy"]), d["qz"])))
    res = {"tool": "external_scf_bench", "n": n, "scheme": "galaxy", "soft": SOFT, "dt": DT, "steps": args.steps,
           "terms": ["hernquist", "miyamoto_nagai", "nfw"], "scf_a": a, "l2": "flushed before every timed step", **gpu_info()}

    arms = [b200nb.Context(n, b200nb.G_F32, SOFT, 1) for _ in ARMS]

    def upload_all():
        for c in arms:
            c.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])

    try:
        upload_all()
        for c in arms[1:]:
            c.set_external(terms)
        for c, (nmax, lmax) in zip(arms[2:], EXPANSIONS):
            S, T = arms[0].scf_coefficients(nmax, lmax, a)
            c.set_external_scf(S, T, a)

        def record(integrator, steps, warmup):
            ts = alternate(arms, integrator, steps, warmup=warmup)
            out = {f"step_ms_{k}": round(t, 4) for k, t in zip(ARMS, ts)}
            for k, t in zip(ARMS[2:], ts[2:]):
                out[f"overhead_vs_3_terms_{k}"] = round(t / ts[1] - 1, 5)
            return out

        for integrator, name in ((b200nb.INTEGRATOR_MURB, "murb"), (b200nb.INTEGRATOR_LEAPFROG, "leapfrog")):
            upload_all()
            res[name] = record(integrator, args.steps, 2)
        m = args.tracers
        pool = b200nb.init_bodies("galaxy", m, seed=1)
        for integrator, name in ((b200nb.INTEGRATOR_MURB, "murb"), (b200nb.INTEGRATOR_LEAPFROG, "leapfrog")):
            upload_all()
            for c in arms:
                c.set_tracers(*[pool[k] for k in KEYS])
            res[name][f"tracers_{m}"] = record(integrator, max(3, args.steps // 2), 1)
        for c in arms:
            c.set_tracers(*[np.zeros(0, np.float32)] * 6)

        upload_all()
        for integrator, name in ((b200nb.INTEGRATOR_MURB, "murb"), (b200nb.INTEGRATOR_LEAPFROG, "leapfrog")):
            for c, k in zip(arms[2:], ARMS[2:]):
                c.step(DT, integrator, 2)
                us, cnt = kernel_ms(c, integrator, "ext_total_kernel", args.steps)
                res[name][f"ext_total_kernel_us_{k}"] = round(1000 * us, 2)
                res[name][f"ext_total_launches_profiled_{k}"] = cnt

        p = b200nb.init_bodies("galaxy", 1 << 24, seed=2)
        pts = [p["qx"], p["qy"], p["qz"]]
        from torch.profiler import ProfilerActivity, profile
        for c, k in zip(arms[2:], ARMS[2:]):
            c.external_field(*pts)  # warm-up: the scratch grows once
            t = time.perf_counter()
            c.external_field(*pts)
            wall = time.perf_counter() - t
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                c.external_field(*pts)
            kt = sum(getattr(ev, "device_time_total", 0.0) for ev in prof.key_averages() if "ext_total_kernel" in ev.key) / 1e6
            res[f"external_field_{k}"] = {"points": len(pts[0]), "wall_s": round(wall, 4),
                                          "points_per_s": round(len(pts[0]) / wall, 1), "kernel_s": round(kt, 6),
                                          "kernel_points_per_s": round(len(pts[0]) / kt, 1) if kt > 0 else None}
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
