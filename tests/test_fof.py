"""b200nb_fof on the GPU: exact agreement with the CPU restatement of the definition (tests/fof_oracle.c), invariance
over shards, ranks and asynchronous steps, ties, padding, non-finite positions, untouched simulation state, bounded
scratch and the error contract.  Labels are integers: every comparison is exact."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import DT, G_F32, REPO, SOFT
from fof_oracle import FofOracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def foracle():
    return FofOracle()


def _ctx(b200, d, **kw):
    ctx = b200.Context(len(d["qx"]), G_F32, SOFT, **kw)
    ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
    return ctx


def _bodies(q, m=None):
    n = q.shape[1]
    d = {c: np.ascontiguousarray(q[i], np.float32) for i, c in enumerate(("qx", "qy", "qz"))}
    for c in ("vx", "vy", "vz"):
        d[c] = np.zeros(n, np.float32)
    d["m"] = np.full(n, 1e20, np.float32) if m is None else np.asarray(m, np.float32)
    return d


def _linking_lengths(ctx, d):
    """From the data: the median distance to the first neighbour (mostly small groups), to the sixth (large groups),
    and a length above the system's diameter (one group)."""
    dist = ctx.neighbors(6)[1]
    bs = []
    for col in (0, 5):
        v = dist[:, col][np.isfinite(dist[:, col])]
        bs.append(float(np.median(v)) if len(v) else 1e9)
    q = np.stack([d["qx"], d["qy"], d["qz"]]).astype(np.float64)
    bs.append(2.01 * float(np.max(np.linalg.norm(q - q.mean(axis=1, keepdims=True), axis=0))) + 1.0)
    return bs


# ------------------------------------------------------------------------------------------------ exact agreement
@pytest.mark.parametrize("scheme", ["galaxy", "random"])
@pytest.mark.parametrize("n", [1, 2, 129, 2049, 20000, 200000])
def test_exact_vs_restatement(b200, oracle, foracle, scheme, n):
    d = oracle.init_bodies(scheme, n)
    with _ctx(b200, d) as ctx:
        bs = _linking_lengths(ctx, d)
        if n >= 200000:  # one group at 200k would take 2e10 unions in the restatement
            bs = bs[:2]
        sizes = []
        for b in bs:
            got = ctx.fof(b)
            assert np.array_equal(got, foracle.groups(d, b)), b
            sizes.append(len(np.unique(got)))
        if n > 2:
            assert sizes[0] >= sizes[1] and sizes[0] > 1
        if len(bs) == 3:
            assert sizes[2] == 1


@pytest.mark.parametrize("integrator", [0, 1])
def test_exact_after_steps(b200, oracle, foracle, integrator):
    d = oracle.init_bodies("galaxy", 2049)
    with _ctx(b200, d) as ctx:
        ctx.step(DT, integrator, 5)
        st = ctx.download_state()
        assert not np.array_equal(st["qx"], d["qx"])
        for b in _linking_lengths(ctx, st):
            assert np.array_equal(ctx.fof(b), foracle.groups(st, b))


# ------------------------------------------------------------------------------------------------ invariance
def test_virtual_shards_and_reruns(b200, oracle):
    for scheme in ("galaxy", "random"):
        d = oracle.init_bodies(scheme, 20011)
        res = []
        for k in (1, 2, 3):
            with _ctx(b200, d, devices=[0] * k) as ctx:
                if k == 1:
                    bs = _linking_lengths(ctx, d)
                res.append([ctx.fof(b) for b in bs])
                assert all(np.array_equal(a, ctx.fof(b)) for a, b in zip(res[-1], bs))  # rerun
        for r in res[1:]:
            assert all(np.array_equal(a, b) for a, b in zip(res[0], r))


def test_ordered_after_async_step(b200, oracle):
    d = oracle.init_bodies("random", 20011)
    with _ctx(b200, d) as ctx:
        bs = _linking_lengths(ctx, d)[:2]
    for devs in ([0], [0, 0, 0]):
        res = []
        for join in (False, True):
            with _ctx(b200, d, devices=devs) as ctx:
                ctx.step(DT, 0, 3)
                if join:
                    ctx.sync()
                res.append([ctx.fof(b) for b in bs])
        assert all(np.array_equal(a, b) for a, b in zip(*res))


def _n_devices():
    import torch
    return torch.cuda.device_count()


def test_two_gpus(b200, oracle):
    if _n_devices() < 2:
        pytest.skip("needs 2 GPUs")
    d = oracle.init_bodies("galaxy", 20011)
    res = []
    for devs in ([0], [0, 1]):
        with _ctx(b200, d, devices=devs) as ctx:
            ctx.step(DT, 0, 2)
            if devs == [0]:
                bs = _linking_lengths(ctx, ctx.download_state())
            res.append([ctx.fof(b) for b in bs])
    assert all(np.array_equal(a, b) for a, b in zip(*res))


def test_torchrun_ranks():
    if _n_devices() < 2:
        pytest.skip("needs 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29583", os.path.join(REPO, "tests", "mp_fof_parity.py")],
                       capture_output=True, text=True, timeout=600)
    print(r.stdout[-2000:])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert r.stdout.count("ok=True") == 2


# ------------------------------------------------------------------------------------------------ edge cases
def test_lattice_ties(b200, foracle):
    """Spacing 1.0 over several AoSoA blocks: d2 = 1 exactly between lattice neighbours."""
    g = np.arange(16, dtype=np.float64)
    X, Y, Z = np.meshgrid(np.arange(17.0), g, g, indexing="ij")
    d = _bodies(np.stack([X.ravel(), Y.ravel(), Z.ravel()]))
    n = len(d["qx"])
    below = np.nextafter(np.float32(1), np.float32(0))
    with _ctx(b200, d) as ctx:
        assert np.all(ctx.fof(1.0) == 0)
        assert np.array_equal(ctx.fof(below), np.arange(n))
        assert np.array_equal(ctx.fof(np.sqrt(np.float32(2))), foracle.groups(d, np.sqrt(np.float32(2))))


def test_b_zero_links_coincident_bodies(b200, oracle, foracle):
    d = oracle.init_bodies("random", 3000)
    for c in ("qx", "qy", "qz"):  # body 2k + 1 sits on body 2k, and body 2999 on body 5
        d[c][1::2] = d[c][0::2][:1500]
        d[c][2999] = d[c][5]
    with _ctx(b200, d) as ctx:
        got = ctx.fof(0.0)
    assert np.array_equal(got, foracle.groups(d, 0.0))
    want = np.arange(3000) & ~1
    want[2998:] = [2998, 4]
    assert np.array_equal(got, want)


@pytest.mark.parametrize("n", [129, 257])
def test_padding_never_linked(b200, oracle, n):
    """One real body in the last AoSoA block: its 127 padding bodies sit exactly on it."""
    d = oracle.init_bodies("random", n)
    with _ctx(b200, d) as ctx:
        assert np.array_equal(ctx.fof(0.0), np.arange(n))


def test_non_finite_positions_stay_alone(b200, oracle, foracle):
    d = oracle.init_bodies("galaxy", 2049)
    for c in ("qx", "qy", "qz"):
        d[c] = d[c].copy()
    bad = [3, 500, 1000, 1500]
    d["qx"][3], d["qy"][500], d["qz"][1000], d["qx"][1500] = np.nan, np.inf, -np.inf, np.nan
    with _ctx(b200, d) as ctx:
        for b in (1e7, 1e18):
            got = ctx.fof(b)
            assert np.array_equal(got, foracle.groups(d, b))
            assert np.array_equal(got[bad], bad)
        assert np.all(np.delete(ctx.fof(1e18), bad) == 0)


def test_zero_mass_bodies_link(b200, oracle, foracle):
    d = oracle.init_bodies("random", 1000)
    with _ctx(b200, d) as ctx:
        b = _linking_lengths(ctx, d)[1]
        want = ctx.fof(b)
    d["m"] = d["m"].copy()
    d["m"][::3] = 0
    with _ctx(b200, d) as ctx:
        got = ctx.fof(b)
    assert np.array_equal(got, want) and np.array_equal(got, foracle.groups(d, b))
    assert np.any(np.bincount(got, minlength=1000)[got[::3]] > 1)


# ------------------------------------------------------------------------------------------------ contract
@pytest.mark.parametrize("integrator", [0, 1])
@pytest.mark.parametrize("steps", [1, 32])  # 32: the cached step-graph path
def test_state_untouched(b200, oracle, integrator, steps):
    d = oracle.init_bodies("galaxy", 5000)
    out = []
    for probe in (False, True):
        with _ctx(b200, d) as ctx:
            ctx.step(DT, integrator, steps)
            if probe:
                ctx.fof(1e9)
                ctx.fof(1e18)
            ctx.step(DT, integrator, steps)
            st = ctx.download_state()
            out.append([st[k] for k in ctx._STATE] + list(ctx.download_accel()))
    for a, b in zip(out[0], out[1]):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.mark.parametrize("shards", [1, 3])
def test_scratch_is_bounded(b200, oracle, shards):
    n = 10000
    d = oracle.init_bodies("galaxy", n)
    with _ctx(b200, d, devices=[0] * shards) as ctx:
        n_pad = shards * b200.slice_length(n, shards)
        before, launches = ctx.allocated_bytes, ctx.launch_count
        ctx.fof(1e9)
        grown = ctx.allocated_bytes
        # a forest of 4 N_pad bytes per shard; the first one holds all P of them
        assert grown - before == 4 * n_pad * (shards + shards - 1), grown - before
        assert ctx.launch_count - launches == 2 * shards + (2 if shards > 1 else 1)
        for b in (0.0, 1e11, 1e18):
            ctx.fof(b)
        assert ctx.allocated_bytes == grown


def test_errors(b200, oracle):
    L = b200.lib()
    d = oracle.init_bodies("galaxy", 1000)
    g = np.empty(1000, np.uint32)
    gp = g.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32))
    with b200.Context(1000, G_F32, SOFT) as ctx:
        assert L.b200nb_fof(ctx._ctx, 1.0, gp) == b200.ESTATE
        ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
        assert L.b200nb_fof(ctx._ctx, 1.0, None) == b200.EINVAL
        for bad in (-1.0, float("nan"), float("inf"), -float("inf"), 2e19, 3.4e38):
            assert L.b200nb_fof(ctx._ctx, bad, gp) == b200.EINVAL, bad
        for ok in (0.0, -0.0, 1.8e19):
            assert L.b200nb_fof(ctx._ctx, ok, gp) == b200.OK, ok
        assert np.all(g == 0)  # 1.8e19 spans the system
        for bad in (-1.0, float("nan"), 2e19, True):
            with pytest.raises(ValueError):
                ctx.fof(bad)
