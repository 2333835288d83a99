#!/usr/bin/env python3
"""Test-particle (tracer) step cost against the field and force passes, in one process on one GPU (galaxy scheme,
soft 2e8, N bodies, both integrators):
  step    b200nb_step of one iteration with M = 0, N and 10 N tracers (positions and velocities of a second galaxy
          realisation): device events around each step, the L2 evicted before every step (b200nb_flush_l2), median;
          tracer G-interactions/s = N * M / (t_M - t_0)
  field   b200nb_field on a 1024 x 1024 grid and the force pass (b200nb_accel): kernel time from torch.profiler (CUDA
          activities) over `--reps` passes, L2 evicted before each; G-interactions/s = targets * N / kernel time
  bodies  the same system as N + M bodies with M of them of zero mass, a few MUrB steps timed the same way
The GPU's name and power limit are read in the same run and printed in the JSON line.
    python tools/tracers_bench.py [--n 200000] [--steps 7] [--reps 5] [--out FILE]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "nbody-eurohpc_b200"))
import b200nb  # noqa: E402

DT, SOFT = 3600.0, 2e8
KEYS = ("qx", "qy", "qz", "vx", "vy", "vz")


def gpu_info():
    import torch
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return {"gpu": out[0], "power_limit_w": float(out[1]), "sm_clock_max_mhz": float(out[2])}
    except Exception:
        return {"gpu": torch.cuda.get_device_name(0), "power_limit_w": None, "sm_clock_max_mhz": None}


def step_ms(ctx, integrator, steps, warmup=2):
    """median device time of one b200nb_step iteration, the L2 evicted before each"""
    ctx.step(DT, integrator, warmup)
    ts = []
    for _ in range(steps):
        ctx.flush_l2()
        ctx.sync()
        ctx.event_record(0)
        ctx.step(DT, integrator, 1)
        ctx.event_record(1)
        ts.append(ctx.event_elapsed_ms(0, 1))
    return statistics.median(ts)


def launches_per_step(ctx, integrator):
    """kernels of one steady-state iteration (step_ms has run the leapfrog's one-off passes already)"""
    before = ctx.launch_count
    ctx.step(DT, integrator, 1)
    return ctx.launch_count - before


def kernel_ms(ctx, f, names, reps):
    from torch.profiler import ProfilerActivity, profile
    f()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            ctx.flush_l2()
            ctx.sync()
            f()
    tot = 0.0
    for ev in prof.key_averages():
        if any(nm in ev.key for nm in names):
            tot += getattr(ev, "device_time_total", getattr(ev, "cuda_time_total", 0.0)) / 1000.0
    return tot / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=200000)
    ap.add_argument("--steps", type=int, default=7)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    if not torch.cuda.is_available():
        sys.exit("tracers_bench: no CUDA device (numbers are only taken on the GPU)")

    n = args.n
    d = b200nb.init_bodies("galaxy", n)
    ms = (n, 10 * n)
    pool = b200nb.init_bodies("galaxy", ms[-1], seed=1)
    res = {"tool": "tracers_bench", "n": n, "scheme": "galaxy", "soft": SOFT, "dt": DT, "steps": args.steps,
           "l2": "flushed before every timed step or pass", **gpu_info()}

    with b200nb.Context(n, b200nb.G_F32, SOFT, 1) as ctx:
        ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
        r_sys = float(np.max(np.hypot(np.hypot(d["qx"], d["qy"]), d["qz"])))
        g = np.linspace(-1.5 * r_sys, 1.5 * r_sys, 1024, dtype=np.float32)
        gx, gy = np.meshgrid(g, g)
        grid = [gx.ravel().copy(), gy.ravel().copy(), np.zeros(gx.size, np.float32)]
        force_k = kernel_ms(ctx, lambda: (ctx.accel(), ctx.sync()), ("force_kernel",), args.reps)
        field_k = kernel_ms(ctx, lambda: ctx.field(*grid), ("field_kernel",), args.reps)
        res["force_pass"] = {"kernel_ms": round(force_k, 4), "ginter_per_s": round(n * n / force_k / 1e6, 1)}
        res["field_grid"] = {"points": grid[0].size, "kernel_ms": round(field_k, 4),
                             "ginter_per_s": round(grid[0].size * n / field_k / 1e6, 1)}
        for integrator, name in ((b200nb.INTEGRATOR_MURB, "murb"), (b200nb.INTEGRATOR_LEAPFROG, "leapfrog")):
            ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
            ctx.set_tracers(*[np.zeros(0, np.float32)] * 6)
            t0 = step_ms(ctx, integrator, args.steps)
            row = {"M0": {"step_ms": round(t0, 3), "launches_per_step": launches_per_step(ctx, integrator)}}
            for m in ms:
                ctx.set_tracers(*[pool[k][:m] for k in KEYS])
                t = step_ms(ctx, integrator, args.steps)
                row[f"M{m}"] = {"step_ms": round(t, 3), "launches_per_step": launches_per_step(ctx, integrator),
                                "tracer_ms": round(t - t0, 3), "tracer_ginter_per_s": round(n * m / (t - t0) / 1e6, 1)}
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    ctx.flush_l2()
                    ctx.sync()
                    ctx.step(DT, integrator, 1)
                    ctx.sync()
                tk = sum(getattr(ev, "device_time_total", 0.0) for ev in prof.key_averages() if "field_kernel" in ev.key) / 1000.0
                row[f"M{m}"]["tracer_field_kernel_ms"] = round(tk, 4)
                row[f"M{m}"]["tracer_kernel_ginter_per_s"] = round(n * m / tk / 1e6, 1) if tk > 0 else None
            res[name] = row
        for name in ("murb", "leapfrog"):
            for m in ms:
                r = res[name][f"M{m}"]
                r["vs_field_rate"] = round(r["tracer_ginter_per_s"] / res["field_grid"]["ginter_per_s"], 3)
                r["vs_force_rate"] = round(r["tracer_ginter_per_s"] / res["force_pass"]["ginter_per_s"], 3)

    res["zero_mass_bodies_murb"] = {}
    for m in ms:
        z = {k: np.concatenate([d[k], pool[k][:m]]) for k in KEYS}
        z["m"] = np.concatenate([d["m"], np.zeros(m, np.float32)])
        with b200nb.Context(n + m, b200nb.G_F32, SOFT, 1) as cz:
            cz.upload(z["qx"], z["qy"], z["qz"], z["m"], z["vx"], z["vy"], z["vz"])
            t = step_ms(cz, b200nb.INTEGRATOR_MURB, 3, warmup=1)
        res["zero_mass_bodies_murb"][f"M{m}"] = {"bodies": n + m, "step_ms": round(t, 3),
                                                 "tracer_step_ms": res["murb"][f"M{m}"]["step_ms"],
                                                 "speedup_of_tracers": round(t / res["murb"][f"M{m}"]["step_ms"], 2)}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
