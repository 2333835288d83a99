"""bench.py keeps the driver's contract: exactly ONE JSON line on stdout with the required keys, for both arms."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import REPO

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "e2e"}


def _run(args, timeout):
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), *args], capture_output=True, text=True, timeout=timeout, cwd=REPO)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.split("\n") if l.strip()]
    assert len(lines) == 1, f"stdout must be one JSON line, got {len(lines)}: {r.stdout[:500]}"
    return json.loads(lines[0])


@pytest.mark.skipif(not os.path.exists(os.path.join(REPO, "oracle", "_ref", "libmurbref.so")), reason="oracle/_ref not built")
def test_reference_arm_line():
    d = _run(["--impl", "reference", "--steps", "2", "--warmup", "1"], 600)
    assert BASE_KEYS <= set(d)
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["dtype"] == "f32"
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["value"] > 0
    # the arm runs the configuration itself when it fits its CPU budget (2+1 iterations at n = 200 000 do)
    assert d["config"]["bodies"] == 200000 and d["sample_bodies"] == 200000 and d["cpu_baseline"]["same_config"] is True


@pytest.mark.skipif(not os.path.exists(os.path.join(REPO, "oracle", "_ref", "libmurbref.so")), reason="oracle/_ref not built")
def test_reference_arm_takes_all_cores_under_torchrun(monkeypatch):
    """torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU arm (rank 0 alone) must still use every allowed core."""
    monkeypatch.setenv("OMP_NUM_THREADS", "1")
    monkeypatch.setenv("LOCAL_RANK", "0")
    monkeypatch.setenv("RANK", "0")
    monkeypatch.setenv("WORLD_SIZE", "2")
    d = _run(["--impl", "reference", "--gpus", "2", "--steps", "2", "--warmup", "1"], 600)
    assert d["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0)) and d["n_gpus"] == 2
    monkeypatch.setenv("RANK", "1")  # the other ranks exit 0 without work and print nothing
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=REPO)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_reference_arm_falls_back_to_the_oracle_port(monkeypatch):
    """Without oracle/_ref (the reference could not be compiled) the arm times the oracle's C restatement instead."""
    monkeypatch.setenv("B200NB_BENCH_NO_REF", "1")
    d = _run(["--impl", "reference", "--steps", "2", "--warmup", "1"], 600)
    assert d["impl"] == "reference" and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 1
    assert d["value"] > 0 and BASE_KEYS - {"ms_per_step"} <= set(d)


def test_dump_sample_is_fixed_and_bounded():
    import bench
    assert bench.dump_sample(200000) is None and bench.dump_sample(bench.DUMP_MAX_BODIES) is None
    idx = bench.dump_sample(4194304)
    assert len(idx) == bench.DUMP_MAX_BODIES and np.all(np.diff(idx) > 0) and idx[-1] < 4194304
    assert np.array_equal(idx, bench.dump_sample(4194304))
    assert 4 * len(bench.DUMP_NAMES) * len(idx) <= 64 << 20


def test_dump_outputs_needs_the_gpu_arm(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=60, cwd=REPO)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and r.stdout == ""


@pytest.mark.gpu
def test_dump_outputs_sample_above_the_limit(b200, tmp_path):
    """Above DUMP_MAX_BODIES the dump holds the bodies dump_sample() names, in that order, bit for bit."""
    import bench
    n = bench.DUMP_MAX_BODIES + 4096
    _run(["--bodies", str(n), "--steps", "1", "--warmup", "3", "--no-cpu", "--no-scaling-base", "--no-side-legs",
          "--dump-outputs", str(tmp_path)], 900)
    idx = bench.dump_sample(n)
    init = b200.init_bodies("galaxy", n)
    with b200.Context(n, b200.G_F32, 2e8, 1) as ctx:
        ctx.upload(*[init[k] for k in ("qx", "qy", "qz", "m", "vx", "vy", "vz")])
        for _ in range(3 + 1):
            ctx.step(3600.0, 0, 1)
        want = ctx.download_state()
        want.update(zip(("ax", "ay", "az"), ctx.download_accel()))
    for k in bench.DUMP_NAMES:
        got = np.load(tmp_path / f"{k}.npy")
        assert got.dtype == np.float32 and np.array_equal(got.view(np.uint32), want[k][idx].view(np.uint32)), k


@pytest.mark.gpu
def test_b200_arm_line(b200, tmp_path):
    dump = tmp_path / "dump"
    d = _run(["--steps", "5", "--warmup", "3", "--no-cpu", "--no-scaling-base", "--no-side-legs", "--dump-outputs", str(dump)], 900)
    assert BASE_KEYS | {"gpu_launches", "clocks", "roofline", "parity"} <= set(d)
    assert d["parity"]["ok"] is True and d["parity"]["max_rel_err"] <= 1e-5 and d["parity"]["targets"] >= 40
    assert d["n_gpus"] == 1 and d["steps"] == 5 and d["warmup"] == 3 and d["dtype"] == "f32" and d["vs_baseline"] is None
    assert d["gpu_launches"] == 10                        # one force + one integrator launch per step
    assert d["e2e"]["h2d_bytes_per_step"] == 7 * 4 * 200000 and d["e2e"]["d2h_bytes_per_step"] == 6 * 4 * 200000
    assert 0 < d["e2e"]["value"] < d["value"] * 1.02
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r)
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and 0.5 < r["frac"] < 1.0
    assert r["kernel_share_of_step"] > 0.99
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    assert "workload" in d["config"] and "200000" in d["config"]["workload"]
    # the dump is the state after warm-up + timed steps and the accelerations of the last step's force pass
    got = {p.stem: np.load(p) for p in dump.glob("*.npy")}
    assert sorted(got) == sorted(("qx", "qy", "qz", "vx", "vy", "vz", "ax", "ay", "az"))
    init = b200.init_bodies("galaxy", 200000)
    with b200.Context(200000, b200.G_F32, 2e8, 1) as ctx:
        ctx.upload(*[init[k] for k in ("qx", "qy", "qz", "m", "vx", "vy", "vz")])
        for _ in range(3 + 5):
            ctx.step(3600.0, 0, 1)
        want = ctx.download_state()
        want.update(zip(("ax", "ay", "az"), ctx.download_accel()))
    for k, v in got.items():
        assert v.dtype == np.float32 and np.array_equal(v.view(np.uint32), want[k].view(np.uint32)), k
    # both arms describe the workload with the identical `config` object (the driver compares them)
    if os.path.exists(os.path.join(REPO, "oracle", "_ref", "libmurbref.so")):
        ref = _run(["--impl", "reference", "--steps", "5", "--warmup", "3"], 900)
        assert ref["config"] == d["config"] and ref["metric"] == d["metric"] and ref["unit"] == d["unit"]
        assert ref["cpu_baseline"]["same_config"] is True
