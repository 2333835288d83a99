#!/usr/bin/env python3
"""bench.py — MUrB all-pairs gravity hot path on B200: billion body-interactions/s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--bodies n] [--scheme galaxy|random]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one computeOneIteration(): the N^2 force pass + the MUrB integrator (+ the position all-gather for N > 1),
i.e. one iteration of `murb -n <bodies> -i <steps> --nv --im gpu+b200 --gf`.
  * --gpus 1 : BASELINE.json configs[1]  (murb -n 200000, galaxy, soft 2e8, dt 3600 — the gpu+tile+full200k shape)
  * --gpus >1: BASELINE.json configs[4]  (n = 4,194,304 strong scaling: targets sharded over the ranks, one in-place
               ncclAllGather of the 16 B/body position blocks per step)
`value` is device-timed (CUDA events on the library's compute stream, state resident in HBM); `e2e` goes through the
public C-ABI with pinned HOST buffers: upload (H2D) + step + download (D2H) inside the timed region, every step.
`--impl reference` times the reference's own CPU path (cpu+omp, compiled from /root/reference into oracle/_ref) on the
host cores: on the configuration itself when it finishes in ~25 s (n = 200 000 does), else on a bounded sample of it.
`--dump-outputs DIR` writes what the last timed step computed, as float32 DIR/<name>.npy: the state a caller receives
(qx qy qz vx vy vz after the step) and the accelerations of its force pass (ax ay az).  The inputs are the seeded
reference generator's, so two builds run with the same arguments can be compared array for array.

Outside the timed region every line also carries: `parity` (a force pass on the final positions checked against the fp64
all-pairs oracle on targets straddling every slice boundary), and on one GPU `roofline_1m` (the N = 1 000 000 force
kernel, BASELINE configs[3]), `prior_art` (the reference's own gpu+tile+full kernels, recompiled for sm_100a, through
the same patched `murb` CLI) and `strong_scaling_base`; on N > 1 GPUs `strong_scaling` (the same 4 M workload re-timed on
one GPU by rank 0 in the same run, and the efficiency that follows).
"""
import argparse
import ctypes
import json
import os
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(REPO, "nbody-eurohpc_b200"))

SOFT, DT = 2e8, 3600.0
STRONG_SCALING_BODIES = 4194304
N_SMS, FP32_LANES = 148, 128
PIPE_SLOTS_PER_INTERACTION = 12  # 3 FADD + 6 FFMA + 3 FMUL (SURVEY §8d); + 1 MUFU.RSQ on its own pipe
METRIC = "billion body-interactions/s (N^2 ordered pairs per force pass, self included)"


def sm_max_mhz():
    try:
        return float(json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))["sm_max_mhz"]), "MEASURED_PEAKS.json sm_max_mhz"
    except Exception:
        return 1965.0, "fallback clocks.max.sm 1965 MHz (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------ clocks (NVML)
class ClockSampler:
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown",
               0x100: "display_clock_setting"}

    def __init__(self, index):
        self.index = index
        self.samples, self.reasons, self.power = [], set(), []
        self._stop = threading.Event()
        self._thread = None
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                bits = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for b, name in self.REASONS.items():
                    if bits & b and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.05)

    def _run_smi(self):
        # fallback without NVML bindings: the recipe's nvidia-smi line (B200_PROFILING.md), polled
        import subprocess
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(int(float(out[0])))
                self.max_mhz = int(float(out[1]))
                self.power.append(float(out[2]))
                for nm, v in zip(names, out[3:]):
                    if "Active" in v and "Not" not in v:
                        self.reasons.add(nm)
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._thread = threading.Thread(target=self._run if self.nv else self._run_smi, daemon=True)
        self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join()
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "power_w_max": (max(self.power) if self.power else None), "samples": len(s)}


# ------------------------------------------------------------------------------------------------ CPU reference
def _cpu_flags():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("flags"):
                return set(line.split(":", 1)[1].split())
    except Exception:
        pass
    return set()


def _cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def load_reference():
    """Best ISA build of the reference CPU path present in oracle/_ref (built from /root/reference by oracle/build_ref.sh)."""
    if os.environ.get("B200NB_BENCH_NO_REF"):  # force the oracle-port fallback (tests)
        return None, None
    flags = _cpu_flags()
    cands = []
    if {"avx512f", "avx512dq", "avx512bw", "avx512vl"} <= flags:
        cands.append(("libmurbref_v4.so", "-O3 -ffast-math -march=x86-64-v4 (AVX-512 MIPP)"))
    if {"avx2", "fma"} <= flags:
        cands.append(("libmurbref_v3.so", "-O3 -ffast-math -march=x86-64-v3 (AVX2 MIPP)"))
    cands.append(("libmurbref.so", "-O3 -ffast-math as shipped (SSE2 MIPP)"))
    FP = ctypes.POINTER(ctypes.c_float)
    for name, desc in cands:
        p = os.path.join(REPO, "oracle", "_ref", name)
        if os.path.exists(p):
            L = ctypes.CDLL(p)
            L.ref_accel.argtypes = [ctypes.c_char_p, ctypes.c_uint64, ctypes.c_char_p, ctypes.c_float, ctypes.c_int] + [FP] * 3
            L.ref_accel.restype = ctypes.c_double
            L.ref_run.argtypes = [ctypes.c_char_p, ctypes.c_uint64, ctypes.c_char_p, ctypes.c_float, ctypes.c_float, ctypes.c_int] + [FP] * 9
            L.ref_run.restype = ctypes.c_double
            return L, desc
    return None, None


def omp_env():
    # the reference's own recipe (README.md:78-89, SimulationNBodyOpenMP.cpp:99-109); must be set before libgomp starts
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    # torchrun exports OMP_NUM_THREADS=1 to every worker unless the user set it; the CPU arm runs on rank 0 alone (the
    # other ranks exit), so it takes every core it is allowed to use.  B200NB_BENCH_OMP_THREADS pins it explicitly.
    pinned = os.environ.get("B200NB_BENCH_OMP_THREADS")
    if pinned:
        os.environ["OMP_NUM_THREADS"] = pinned
    elif "TORCHELASTIC_RUN_ID" in os.environ or "LOCAL_RANK" in os.environ:
        os.environ["OMP_NUM_THREADS"] = str(cores)
    os.environ.setdefault("OMP_NUM_THREADS", str(cores))
    os.environ.setdefault("OMP_DYNAMIC", "FALSE")
    os.environ.setdefault("OMP_PLACES", "cores")
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_SCHEDULE", "static")
    os.environ.setdefault("OMP_WAIT_POLICY", "ACTIVE")
    return int(os.environ["OMP_NUM_THREADS"])


def cpu_reference_rate(scheme, bodies, budget_s, tag="cpu+omp"):
    """G-int/s of the reference CPU implementation: whole iterations of the workload itself when a handful of them fit
    the budget (n = 200 000 does on 16 cores), else of a bounded sample (n = 30 000)."""
    cores = omp_env()
    L, desc = load_reference()
    if L is None:
        return oracle_port_rate(scheme, budget_s)
    none = [None] * 9
    n_small = 30000
    L.ref_run(tag.encode(), n_small, scheme.encode(), SOFT, DT, 1, *none)  # warm-up: thread start, page faults
    ms_small = L.ref_run(tag.encode(), n_small, scheme.encode(), SOFT, DT, 2, *none) / 2
    ms_full = ms_small * (float(bodies) / n_small) ** 2
    n_sample = bodies if 5 * ms_full <= budget_s * 1e3 else n_small     # 1 warm-up + >= 4 timed iterations
    ms1 = ms_full if n_sample == bodies else ms_small
    if n_sample == bodies:
        L.ref_run(tag.encode(), n_sample, scheme.encode(), SOFT, DT, 1, *none)
    iters = int(max(2, min(200, budget_s * 1e3 / max(ms1, 1e-3) - 1)))
    ms = L.ref_run(tag.encode(), n_sample, scheme.encode(), SOFT, DT, iters, *none)
    rate = float(n_sample) ** 2 * iters / (ms * 1e-3) / 1e9
    out = {"value": rate, "unit": "G-int/s", "cores": cores if tag == "cpu+omp" else 1, "kind": "reference",
           "sample": f"reference {tag} ({desc}), {iters} iterations of murb -n {n_sample} -s {scheme} (full force pass + integrator), "
                     f"{ms / iters:.2f} ms/iter" + ("" if n_sample == bodies else f"; bounded sample of the n = {bodies} workload"),
           "ms_per_iter": ms / iters, "iters": iters, "n_sample": n_sample, "same_config": n_sample == bodies,
           "cpu_model": _cpu_model()}
    if tag == "cpu+omp":
        # the other reference CPU paths the north star asks for, single thread, same ICs (bounded: a few seconds each)
        others = {}
        for t, it in (("cpu+simd", 3), ("cpu+naive", 1)):
            n_t = n_small if t == "cpu+simd" else 8000   # cpu+naive at 30000 is ~8 s/iteration; 8000 is the Report's own size
            L.ref_run(t.encode(), n_t, scheme.encode(), SOFT, DT, 1 if t == "cpu+simd" else 0, *none)
            ms_t = L.ref_run(t.encode(), n_t, scheme.encode(), SOFT, DT, it, *none)
            others[t] = {"value": float(n_t) ** 2 * it / (ms_t * 1e-3) / 1e9, "unit": "G-int/s", "cores": 1, "n_sample": n_t,
                         "iters": it, "ms_per_iter": ms_t / it}
        # the same cpu+omp exactly as the reference ships it (no -march: SSE2 MIPP, CMakeLists.txt:128-131)
        shipped = os.path.join(REPO, "oracle", "_ref", "libmurbref.so")
        if os.path.exists(shipped) and "as shipped" not in desc:
            FP = ctypes.POINTER(ctypes.c_float)
            S = ctypes.CDLL(shipped)
            S.ref_run.argtypes = [ctypes.c_char_p, ctypes.c_uint64, ctypes.c_char_p, ctypes.c_float, ctypes.c_float, ctypes.c_int] + [FP] * 9
            S.ref_run.restype = ctypes.c_double
            S.ref_run(b"cpu+omp", n_small, scheme.encode(), SOFT, DT, 1, *none)
            ms_s = S.ref_run(b"cpu+omp", n_small, scheme.encode(), SOFT, DT, 10, *none)
            others["cpu+omp as shipped (-O3 -ffast-math, SSE2 MIPP)"] = {
                "value": float(n_small) ** 2 * 10 / (ms_s * 1e-3) / 1e9, "unit": "G-int/s", "cores": cores, "n_sample": n_small,
                "iters": 10, "ms_per_iter": ms_s / 10}
        out["other_reference_paths"] = others
    return out


def oracle_port_rate(scheme, budget_s):
    """Fallback when oracle/_ref was not built: the scalar C restatement (oracle/liboracle.so), one core."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("pyoracle", os.path.join(REPO, "oracle", "pyoracle.py"))
    pyoracle = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(pyoracle)
    o = pyoracle.load()  # builds oracle/liboracle.so if needed
    n = 8000
    d = o.init_bodies(scheme, n)
    t0 = time.perf_counter()
    it = 0
    while time.perf_counter() - t0 < max(2.0, budget_s / 2):
        o.accel_naive(d)
        it += 1
    dt = time.perf_counter() - t0
    return {"value": float(n) ** 2 * it / dt / 1e9, "unit": "G-int/s", "cores": 1, "kind": "port",
            "sample": f"oracle port of cpu+naive (oracle/nbody_oracle.c), {it} force passes at n={n}", "n_sample": n}


# ------------------------------------------------------------------------------------------------ arms
def workload_config(args, world):
    """The `config` object, identical for both arms (the driver compares them)."""
    return {"workload": f"murb -n {args.bodies} -i {args.steps} --nv --gf ({args.scheme}, soft {SOFT:g}, dt {DT:g})"
            + ("" if world == 1 else f"; strong scaling over {world} GPUs (BASELINE configs[4])"),
            "bodies": args.bodies, "scheme": args.scheme, "integrator": "murb-explicit", "soft": SOFT, "dt": DT,
            "n_gpus": world}


REF_ARM_BUDGET_S = 25.0   # CPU seconds the reference arm may spend on its warm-up + timed steps


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    cores = omp_env()
    L, desc = load_reference()
    total_steps = args.steps + max(args.warmup, 1)
    if L is None:
        r = oracle_port_rate(args.scheme, 10)
        ms_per_step, value, n_run = None, r["value"], r["n_sample"]
        base = r
    else:
        none = [None] * 9
        tag = b"cpu+omp"
        # probe the rate on a small system (also starts the OpenMP team), then run the configuration itself if all its
        # steps fit the budget; otherwise the largest system that does (a bounded sample of the same workload)
        L.ref_run(tag, 30000, args.scheme.encode(), SOFT, DT, 1, *none)
        probe_ms = L.ref_run(tag, 30000, args.scheme.encode(), SOFT, DT, 2, *none) / 2
        rate = 30000.0 ** 2 / (probe_ms * 1e-3)   # interactions / s
        n_fit = int((REF_ARM_BUDGET_S * rate / total_steps) ** 0.5)
        n_run = args.bodies if args.bodies <= n_fit else max(30000, n_fit // 10000 * 10000)
        L.ref_run(tag, n_run, args.scheme.encode(), SOFT, DT, max(args.warmup, 1), *none)
        ms = L.ref_run(tag, n_run, args.scheme.encode(), SOFT, DT, args.steps, *none)
        ms_per_step = ms / args.steps
        value = float(n_run) ** 2 * args.steps / (ms * 1e-3) / 1e9
        what = "the configuration itself" if n_run == args.bodies else f"a bounded sample of the workload (n = {n_run} of {args.bodies})"
        base = {"value": value, "unit": "G-int/s", "cores": cores, "kind": "reference",
                "sample": f"reference cpu+omp ({desc}), {cores} OpenMP threads, {args.steps} timed iterations after "
                          f"{max(args.warmup, 1)} warm-up of murb -n {n_run} -s {args.scheme}: {what}",
                "n_sample": n_run, "same_config": n_run == args.bodies, "cpu_model": _cpu_model()}
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "G-int/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic (reference Bodies generator, srand(0))",
        "config": workload_config(args, world), "impl_tag": "cpu+omp", "sample_bodies": n_run,
        "cpu_baseline": base,
        "e2e": {"value": value, "unit": "G-int/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


class StdoutToStderr:
    """NCCL (and anything else native) may print to fd 1; the contract is ONE JSON line on stdout.  Everything written
    to fd 1 while this is active goes to stderr; emit() writes the line to the real stdout."""

    def __init__(self):
        sys.stdout.flush()
        self._saved = os.dup(1)
        os.dup2(2, 1)

    def emit(self, line):
        sys.stdout.flush()
        os.dup2(self._saved, 1)
        print(line, flush=True)
        os.dup2(2, 1)


# ------------------------------------------------------------------------------------------------ checks and side legs
def load_pyoracle():
    """oracle/pyoracle.py — the CHECKER (and, in cpu_baseline, the thing timed); never on the product path."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("pyoracle", os.path.join(REPO, "oracle", "pyoracle.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def boundary_targets(n, L, world, extra=40, seed=11):
    """Targets on both sides of every slice boundary, the two ends of the system and a few random ones."""
    idx = [0, n - 1]
    for k in range(1, world):
        idx += [k * L - 2, k * L - 1, k * L, k * L + 1]
    idx += list(np.random.default_rng(seed).integers(0, n, extra))
    return np.unique(np.clip(np.array(idx, dtype=np.int64), 0, n - 1)).astype(np.uint64)


def parity_check(b200nb, ctx, bodies, n, world, rank, scheme):
    """After the timed region: one more force pass on the positions the last exchange published, state + accelerations
    back to the host (collective), and on rank 0 the fp64 all-pairs oracle on the sampled targets (O(targets x N))."""
    ctx.accel()
    state = ctx.download_state()
    acc = ctx.download_accel()
    if rank != 0:
        return None
    pyoracle = load_pyoracle()
    idx = boundary_targets(n, b200nb.slice_length(n, world), world)
    moved = dict(bodies)
    moved.update({k: state[k] for k in ("qx", "qy", "qz")})
    t0 = time.perf_counter()
    a64 = np.stack(pyoracle.load().accel_f64(moved, idx))
    ii = idx.astype(np.int64)
    got = np.stack([a[ii] for a in acc]).astype(np.float64)
    err_each = np.linalg.norm(got - a64, axis=0) / np.linalg.norm(a64, axis=0)
    finite = all(bool(np.all(np.isfinite(state[k]))) for k in ("qx", "qy", "qz", "vx", "vy", "vz"))
    # Body 0 of the galaxy scheme is the 2e24 kg central mass (Bodies.cpp:158-214): its acceleration is the residual of N
    # nearly cancelling pulls (|a_0| ~ 1e-3 of everyone else's, condition number sum|t_j| / |sum t_j| ~ 1e3), so its
    # relative error is ~1e3 x the per-term rounding (measured 5e-7 at the initial positions, 5e-6..9e-6 once it has left
    # the origin; every other target stays below 2e-7, tools/parity_probe.py).  It is reported on its own, against a
    # bound that scales with that conditioning, so that the 1e-5 bound on everyone else stays meaningful.
    central = scheme == "galaxy"
    regular = (ii != 0) if central else np.ones(len(ii), bool)
    err = float(err_each[regular].max())
    out = {"max_rel_err": err, "tol": 1e-5, "targets": int(regular.sum()), "ok": bool(err <= 1e-5 and finite), "state_finite": finite,
           "median_rel_err": float(np.median(err_each[regular])),
           "what": "max |a - a_fp64| / |a_fp64| of a force pass on the final positions of this run, fp64 all-pairs oracle "
                   "(oracle/nbody_oracle.c: oracle_accel_f64) on targets straddling every slice boundary + both ends + random",
           "oracle_s": time.perf_counter() - t0}
    if central:
        e0 = float(err_each[ii == 0][0])
        out["central_body"] = {"rel_err": e0, "tol": 1e-4, "abs_a": float(np.linalg.norm(a64[:, ii == 0])),
                               "typical_abs_a": float(np.median(np.linalg.norm(a64[:, regular], axis=0))),
                               "why": "body 0 = the 2e24 kg central mass: |a_0| is the residual of N cancelling pulls, ~1e-3 of a typical "
                                      "|a| (condition number ~1e3), so it gets its own bound"}
        out["ok"] = bool(out["ok"] and e0 <= 1e-4)
    return out


DUMP_NAMES = ("qx", "qy", "qz", "vx", "vy", "vz", "ax", "ay", "az")
DUMP_MAX_BODIES = 1 << 20   # 9 float32 arrays of 2^20 bodies: 36 MiB, under the 64 MiB a dump may take


def dump_sample(n):
    """Bodies --dump-outputs writes: all of them up to DUMP_MAX_BODIES, else a fixed seeded sample (sorted, the same in
    every run with the same n)."""
    if n <= DUMP_MAX_BODIES:
        return None
    return np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_BODIES, replace=False))


def outputs_of_last_step(ctx, n):
    """The state after the last step and the accelerations of that step's force pass (downloads are collective)."""
    state = ctx.download_state()
    out = {k: state[k] for k in ("qx", "qy", "qz", "vx", "vy", "vz")}
    out.update(zip(("ax", "ay", "az"), ctx.download_accel()))
    idx = dump_sample(n)
    return {k: out[k] if idx is None else out[k][idx] for k in DUMP_NAMES}


def write_outputs(path, arrays):
    os.makedirs(path, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), np.ascontiguousarray(v, dtype=np.float32))


def timed_steps_single_gpu(b200nb, scheme, n, steps, warmup):
    """`steps` flushed, event-timed computeOneIteration() of an n-body system on the current device (one GPU)."""
    names = ("qx", "qy", "qz", "m", "vx", "vy", "vz")
    big = b200nb.init_bodies(scheme, n)
    with b200nb.Context(n, b200nb.G_F32, SOFT, 1) as c2:
        c2.upload(*[big[k] for k in names])
        for _ in range(warmup):
            c2.step(DT, 0, 1)
        c2.sync()
        ms = 0.0
        for _ in range(steps):
            c2.flush_l2()
            c2.event_record(0)
            c2.step(DT, 0, 1)
            c2.event_record(1)
            ms += c2.event_elapsed_ms(0, 1)
        kernel = c2.kernel_name
    return {"bodies": n, "n_gpus": 1, "value": float(n) ** 2 * steps / (ms * 1e-3) / 1e9, "unit": "G-int/s",
            "ms_per_step": ms / steps, "steps": steps, "warmup": warmup, "l2_flush_between_steps": True, "kernel": kernel}


def roofline_at(b200nb, scheme, n, reps, max_mhz):
    """Force kernel alone (b200nb_accel) at n bodies on one GPU: `reps` event-timed launches, L2 flushed between them."""
    names = ("qx", "qy", "qz", "m", "vx", "vy", "vz")
    d = b200nb.init_bodies(scheme, n)
    with b200nb.Context(n, b200nb.G_F32, SOFT, 1) as c:
        c.upload(*[d[k] for k in names])
        c.accel()
        c.sync()
        c.profile_enable(True)
        for _ in range(reps):
            c.flush_l2()
            c.accel()
        ms, launches = c.profile_get()
        c.profile_enable(False)
        kernel = c.kernel_name
    avg = ms / max(launches, 1)
    rate = float(n) ** 2 / (avg * 1e-3)
    return {"bodies": n, "kernel": kernel, "launches": int(launches), "avg_launch_ms": avg, "kernel_gint_per_s": rate / 1e9,
            "achieved": 2 * PIPE_SLOTS_PER_INTERACTION * rate / 1e12, "peak": N_SMS * FP32_LANES * 2 * max_mhz * 1e6 / 1e12,
            "unit": "TFLOP/s", "frac": PIPE_SLOTS_PER_INTERACTION * rate / (N_SMS * FP32_LANES * max_mhz * 1e6),
            "interactions_per_clk_per_sm": rate / (max_mhz * 1e6) / N_SMS,
            "note": "BASELINE configs[3] / north-star target (>= 0.70 at N = 1M): same definition as `roofline`, CUDA events around "
                    "every force launch, 256 MiB L2 flush between launches"}


def prior_art_leg(scheme, cases):
    """The reference's own GPU kernels (gpu+tile+full, gpu+tile+full200k: SimulationNBodyCUDATileFullDevice.cu:53-153,
    ...200k.cu:102-175) compiled unchanged for sm_100a into oracle/_ref/murb_b200, and gpu+b200, through the SAME patched
    CLI (`murb -n N -i I --nv --im TAG --gf`, main.cpp:348-371 times every iteration incl. its device sync)."""
    import re
    import subprocess
    exe = os.path.join(REPO, "oracle", "_ref", "murb_b200")
    if not os.path.exists(exe):
        return {"unavailable": "oracle/_ref/murb_b200 not built (needs the reference sources at build time)"}
    out = {"how": "oracle/_ref/murb_b200 -n N -i I --nv -s " + scheme + " --im TAG --gf; G-int/s = N^2 * I / 'Entire simulation took' ms",
           "cases": []}
    env = dict(os.environ)
    env.pop("MURB_B200_NGPUS", None)
    for n, iters in cases:
        case = {"bodies": n, "iterations": iters, "gint_per_s": {}}
        for tag in ("gpu+tile+full", "gpu+tile+full200k", "gpu+b200"):
            try:
                r = subprocess.run([exe, "-n", str(n), "-i", str(iters), "--nv", "-s", scheme, "--im", tag, "--gf"],
                                   capture_output=True, text=True, timeout=600, env=env)
                m = re.search(r"Entire simulation took ([0-9.eE+-]+) ms", r.stdout)
                if r.returncode != 0 or not m:
                    case["gint_per_s"][tag] = None
                    case.setdefault("errors", {})[tag] = (r.stdout + r.stderr)[-300:]
                    continue
                case["gint_per_s"][tag] = float(n) ** 2 * iters / (float(m.group(1)) * 1e-3) / 1e9
            except Exception as e:  # a comparator that fails must not take the bench line down
                case["gint_per_s"][tag] = None
                case.setdefault("errors", {})[tag] = repr(e)[-300:]
        g = case["gint_per_s"]
        best = max([v for k, v in g.items() if k != "gpu+b200" and v], default=None)
        case["b200_over_best_prior_art"] = (g.get("gpu+b200") / best) if best and g.get("gpu+b200") else None
        out["cases"].append(case)
    return out


def run_b200_arm(args, rank, world, local_rank):
    out_guard = StdoutToStderr()
    import torch
    import b200nb

    from b200nb import dist as bdist

    dist = bdist.init_process_group()     # None for a single rank
    nccl_id = None
    if dist is not None:
        nccl_id = bdist.broadcast_bytes(dist, b200nb.Context.unique_id() if rank == 0 else None)
    torch.cuda.set_device(local_rank)
    torch.cuda.init()
    n = args.bodies
    bodies = b200nb.init_bodies(args.scheme, n)
    if world > 1:
        ctx = b200nb.Context(n, b200nb.G_F32, SOFT, rank=rank, n_ranks=world, device=local_rank, nccl_id=nccl_id)
    else:
        ctx = b200nb.Context(n, b200nb.G_F32, SOFT, 1)
    names = ("qx", "qy", "qz", "m", "vx", "vy", "vz")
    pinned = b200nb.PinnedArrays(list(names), n)
    for k in names:
        pinned[k][:] = bodies[k]
    up = [pinned[k] for k in names]
    down = {k: pinned[k] for k in ("qx", "qy", "qz", "vx", "vy", "vz")}
    ctx.upload_raw(up)
    own_first, own_count = ctx.slice_bounds(0)

    def barrier():
        ctx.sync()
        if dist is not None:
            dist.barrier()
        ctx.sync()

    def reduce_max(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident arm: K x computeOneIteration, per-step CUDA events, L2 evicted between steps
    for _ in range(args.warmup):
        ctx.step(DT, 0, 1)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ctx.profile_enable(True)
    launches0 = ctx.launch_count
    barrier()
    t_wall0 = time.perf_counter()
    dev_ms = 0.0
    for i in range(args.steps):
        ctx.flush_l2()
        ctx.event_record(0)
        ctx.step(DT, 0, 1)
        ctx.event_record(1)
        dev_ms += ctx.event_elapsed_ms(0, 1)
    barrier()
    bracket_ms = (time.perf_counter() - t_wall0) * 1e3
    clocks = sampler.stop()
    launches = ctx.launch_count - launches0
    force_ms, force_launches = ctx.profile_get()
    ctx.profile_enable(False)
    if args.dump_outputs:
        last = outputs_of_last_step(ctx, n)
        if rank == 0:
            write_outputs(args.dump_outputs, last)
    dev_ms = reduce_max(dev_ms)
    force_ms = reduce_max(force_ms)
    interactions_per_step = float(n) * float(n)
    value = interactions_per_step * args.steps / (dev_ms * 1e-3) / 1e9

    # ---- end-to-end arm: pinned host state in, host state out, every step, through the public C ABI.
    # Every rank's host holds the state; a rank moves its own targets across its own host link (H2D 28 B, D2H 24 B per
    # body) and the step's exchange replicates positions on the GPUs, so the job moves 52 B per body per step in total.
    # same number of steps, but bounded to ~30 s of wall time for long-step workloads (at least 3 steps)
    e2e_steps = int(max(min(args.steps, 3), min(args.steps, 30e3 / max(dev_ms / args.steps, 1e-3))))
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        ctx.upload_raw(up)               # H2D: qx qy qz m vx vy vz of the rank's own bodies (+ the exchange)
        ctx.step(DT, 0, 1)
        ctx.download_slice(down)         # D2H: qx qy qz vx vy vz of the rank's own bodies (joins the device)
    barrier()
    e2e_s = reduce_max(time.perf_counter() - t0)
    e2e_value = interactions_per_step * e2e_steps / e2e_s / 1e9

    # ---- parity of this very run (all ranks: the downloads are collective)
    parity = parity_check(b200nb, ctx, bodies, n, world, rank, args.scheme)

    if rank != 0:
        ctx.close()
        if dist is not None:
            dist.barrier()       # rank 0 re-times the workload on one GPU (strong_scaling) before everyone leaves
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (the force pass): FP32 pipe, not HBM, not tensor
    max_mhz, peak_src = sm_max_mhz()
    peak_tflops = N_SMS * FP32_LANES * 2 * max_mhz * 1e6 / 1e12
    per_gpu_int_per_launch = interactions_per_step / world * args.steps / max(force_launches, 1)
    avg_launch_ms = force_ms / max(force_launches, 1)
    kernel_int_per_s = per_gpu_int_per_launch / (avg_launch_ms * 1e-3)
    achieved_tflops = 2 * PIPE_SLOTS_PER_INTERACTION * kernel_int_per_s / 1e12
    meas_mhz = clocks.get("sm_mhz") or max_mhz
    traffic, traffic_src = None, None
    try:  # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture
        t = json.load(open(os.path.join(REPO, "profiles", "ncu_traffic.json")))
        if t["workload_bodies"] == n and world == 1 and ctx.kernel_name.startswith(t.get("kernel_name", "")):
            traffic = t["dram_bytes_per_launch"]
            traffic_src = "constant from the committed ncu --set full capture of this workload (" + t["source"] + "), not measured by this run"
    except Exception:
        pass
    roofline = {
        "bound": "fp32_pipe", "achieved": achieved_tflops, "peak": peak_tflops, "unit": "TFLOP/s",
        "frac": achieved_tflops / peak_tflops,
        "traffic": traffic, "traffic_source": traffic_src,
        "note": "compute-bound kernel: neither 'hbm' nor 'tensor' applies (SURVEY §8d). achieved = 12 FP32-pipe slots per "
                "interaction counted as FMA (2 flop) x interactions per launch / CUDA-event launch duration; peak = "
                f"148 SMs x 128 lanes x 2 x {max_mhz:.0f} MHz ({peak_src}; MEASURED_PEAKS.json has no FP32 entry), so "
                "frac == 12*int/s / (148*128*f). The pipe peak is reachable: a pure FFMA2 loop measures 1.987 of 2.0 "
                "warp-instr/clk/SM and FFMA 3.9 of 4.0 on this part (profiles/r01_microbench_pipes.txt).",
        "kernel": ctx.kernel_name, "avg_launch_ms": avg_launch_ms, "launches": force_launches,
        "kernel_share_of_step": force_ms / dev_ms,
        "kernel_gint_per_s_per_gpu": kernel_int_per_s / 1e9,
        "interactions_per_clk_per_sm": kernel_int_per_s / (meas_mhz * 1e6) / N_SMS,
        "frac_at_measured_clock": 2 * PIPE_SLOTS_PER_INTERACTION * kernel_int_per_s / (N_SMS * FP32_LANES * 2 * meas_mhz * 1e6),
        "murb_gflops_20flop_2p30": 20.0 * value * 1e9 / 2 ** 30,
        "hbm_algorithmic_bytes_per_launch": 28.0 * n / world, "hbm_gbs_algorithmic": 28.0 * n / world / (avg_launch_ms * 1e-3) / 1e9,
    }
    exchange = ctx.exchange_name
    ctx.close()
    cpu = cpu_reference_rate(args.scheme, n, 12.0) if world == 1 and not args.no_cpu else None
    extra = {}
    if world == 1 and not args.no_side_legs:
        # BASELINE configs[3]: the north-star roofline target is stated at N = 1M
        if n != 1000000:
            extra["roofline_1m"] = roofline_at(b200nb, args.scheme, 1000000, 3, max_mhz)
        # the on-box prior-art bar (SURVEY §8 f1): the reference's GPU kernels through the same CLI, this line's N, and 1M
        extra["prior_art"] = prior_art_leg(args.scheme, [(n, max(args.steps, 50) if n <= 300000 else 5), (1000000, 5)]
                                           if n != 1000000 else [(n, 5)])
    # The --gpus N>1 lines run the strong-scaling workload (n = 4,194,304).  Every line is self-contained: the 1-GPU line
    # carries the 1-GPU rate of that workload, and every N>1 line re-times it on ONE GPU (rank 0, the other ranks idle at
    # a barrier) and states the efficiency that follows.
    if not args.no_scaling_base:
        if world == 1 and n != STRONG_SCALING_BODIES:
            base = timed_steps_single_gpu(b200nb, args.scheme, STRONG_SCALING_BODIES, 3, 1)
            base["note"] = ("same workload as the --gpus N>1 lines (BASELINE configs[4]), 3 flushed event-timed steps after 1 "
                            "warm-up; efficiency(N) = value(N) / (N * this)")
            extra["strong_scaling_base"] = base
        elif world > 1:
            base = timed_steps_single_gpu(b200nb, args.scheme, n, 3, 1)
            extra["strong_scaling"] = {"base": base, "efficiency": value / (world * base["value"]),
                                       "definition": "value / (n_gpus * base.value); base = the same workload on ONE GPU (rank 0, "
                                                     "other ranks idle), 3 flushed event-timed steps after 1 warm-up, in this run"}
    cfg = workload_config(args, world)
    out = {
        "metric": METRIC, "value": value, "unit": "G-int/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
        # the 1..8 GPU series is the strong-scaling one of BASELINE configs[4]; the --gpus 1 line's own `value` is
        # configs[1] (n = 200 000), its `strong_scaling_base` is the 1-GPU point of the series
        "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic (reference Bodies generator restated, srand(0))",
        "config": cfg, "impl_tag": "gpu+b200",
        "exchange": exchange if world > 1 else "none",
        "l2": "256 MiB memset between timed steps (outside the per-step event pair); inputs are 16 B/body and L2-resident by design",
        "timing": "sum over steps of CUDA-event pairs on the library's compute stream, max over ranks",
        "gpu_launches": int(launches), "bracket_wall_ms": bracket_ms,
        "clocks": {"sm_mhz": clocks["sm_mhz"], "sm_max_mhz": clocks["sm_max_mhz"], "reasons": clocks["reasons"],
                   "power_w_max": clocks["power_w_max"], "samples": clocks["samples"]},
        "e2e": {"value": e2e_value, "unit": "G-int/s", "h2d_bytes_per_step": 7 * 4 * n, "d2h_bytes_per_step": 6 * 4 * n,
                "ms_per_step": e2e_s * 1e3 / e2e_steps, "steps": e2e_steps,
                "path": "b200nb_upload (pinned host SoA; each rank copies its own targets) + b200nb_step + b200nb_download_slice "
                        "(each rank reads its own targets back), host wall clock; bytes are the job's total over all ranks",
                "rank0_own_bodies": own_count},
        "roofline": roofline,
        "parity": parity,
    }
    if cpu is not None:
        out["cpu_baseline"] = cpu
    out.update(extra)
    out_guard.emit(json.dumps(out))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--bodies", type=int, default=None)
    ap.add_argument("--scheme", default="galaxy", choices=["galaxy", "random"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-scaling-base", action="store_true", help="skip the 1-GPU run of the strong-scaling workload")
    ap.add_argument("--no-side-legs", action="store_true", help="skip roofline_1m and prior_art (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the state and accelerations of the last timed step as float32 DIR/<name>.npy "
                         f"(a fixed seeded sample of {DUMP_MAX_BODIES} bodies above that size)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the GPU path computed: use it with --impl b200")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != max(args.gpus, 1) and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if args.gpus > 1 and world == 1:
        raise SystemExit("for --gpus N > 1 launch with: python -m torch.distributed.run --nnodes=1 --nproc-per-node N "
                         "--master-addr 127.0.0.1 --master-port P bench.py --gpus N ...")
    if args.bodies is None:
        args.bodies = 200000 if args.gpus <= 1 else STRONG_SCALING_BODIES
    if args.steps is None:
        args.steps = 200 if args.gpus <= 1 else 5
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
    else:
        run_b200_arm(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
