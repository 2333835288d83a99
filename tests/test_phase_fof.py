"""b200nb_fof_phase on the GPU: exact agreement with the CPU restatement of the definition (tests/phase_fof_oracle.c),
b200nb_fof's labels for a power-of-two b_x and b_v = inf, the two overlapping systems, invariance over shards, ranks and
asynchronous steps, padding, non-finite inputs, untouched simulation state, bounded scratch and the error contract.
Labels are integers: every comparison is exact."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import DT, G_F32, REPO, SOFT
from phase_fof_oracle import PhaseFofOracle
from test_phase_fof_cpu import KEYS, two_systems

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def poracle():
    return PhaseFofOracle()


def _ctx(b200, d, **kw):
    ctx = b200.Context(len(d["qx"]), G_F32, SOFT, **kw)
    ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
    return ctx


def _settings(ctx, d):
    """(b_x, b_v) from the data, from sparse to one group and from b_v = inf down to every body alone: b_x at the median
    first- and sixth-neighbour distance and above the diameter, b_v at the velocity dispersion and far below it."""
    dist = ctx.neighbors(6)[1]
    bx = []
    for col in (0, 5):
        v = dist[:, col][np.isfinite(dist[:, col])]
        bx.append(float(np.median(v)) if len(v) else 1e9)
    q = np.stack([d["qx"], d["qy"], d["qz"]]).astype(np.float64)
    v = np.stack([d["vx"], d["vy"], d["vz"]]).astype(np.float64)
    diam = 2.01 * float(np.max(np.linalg.norm(q - q.mean(axis=1, keepdims=True), axis=0))) + 1.0
    sig = float(np.sqrt(np.mean(np.sum((v - v.mean(axis=1, keepdims=True)) ** 2, axis=0)))) or 1.0
    return [(bx[0], np.inf), (bx[1], np.inf), (bx[1], sig), (bx[1], 0.1 * sig), (diam, np.inf), (diam, sig),
            (np.inf, np.inf), (bx[1], 1e-6 * sig)]


# ------------------------------------------------------------------------------------------------ exact agreement
@pytest.mark.parametrize("scheme", ["galaxy", "random"])
@pytest.mark.parametrize("n", [1, 2, 127, 128, 129, 1023, 1024, 1025, 4097, 20000])
def test_exact_vs_restatement(b200, oracle, poracle, scheme, n):
    d = oracle.init_bodies(scheme, n)
    with _ctx(b200, d) as ctx:
        sizes = []
        for b_x, b_v in _settings(ctx, d):
            got = ctx.fof_phase(b_x, b_v)
            assert np.array_equal(got, poracle.groups(d, b_x, b_v)), (b_x, b_v)
            sizes.append(len(np.unique(got)))
    assert sizes[4] == 1 and sizes[6] == 1  # one group
    if n > 2:
        assert sizes[0] > sizes[1] and sizes[3] >= sizes[2] >= sizes[1]
        assert sizes[7] == n  # every body alone


@pytest.mark.parametrize("integrator", [0, 1])
def test_exact_after_steps(b200, oracle, poracle, integrator):
    d = oracle.init_bodies("galaxy", 2049)
    with _ctx(b200, d) as ctx:
        ctx.step(DT, integrator, 5)
        st = ctx.download_state()
        assert not np.array_equal(st["qx"], d["qx"]) and not np.array_equal(st["vx"], d["vx"])
        for b_x, b_v in _settings(ctx, st):
            assert np.array_equal(ctx.fof_phase(b_x, b_v), poracle.groups(st, b_x, b_v)), (b_x, b_v)


@pytest.mark.parametrize("scheme", ["galaxy", "random"])
def test_power_of_two_bx_is_fof_200k(b200, oracle, scheme):
    d = oracle.init_bodies(scheme, 200000)
    with _ctx(b200, d) as ctx:
        for k in (22, 24):
            got, want = ctx.fof_phase(2.0 ** k, np.inf), ctx.fof(2.0 ** k)
            assert np.array_equal(got, want), k
            assert 1 < len(np.unique(got)) < 200000


def test_two_overlapping_systems(b200, oracle, poracle):
    d = two_systems(b200.init_bodies)
    n = len(d["qx"]) // 2
    truth = np.repeat([0, 1], n)
    with _ctx(b200, d) as ctx:
        b = float(np.median(ctx.neighbors(4)[1][:, 3]))
        pos = ctx.fof(b)
        big = np.bincount(pos).argmax()
        assert np.all(np.bincount(truth[pos == big], minlength=2) > 1000)  # position FoF mixes the systems
        for b_v in (2000.0, 3000.0):
            g = ctx.fof_phase(2 * b, b_v)
            assert np.array_equal(g, poracle.groups(d, 2 * b, b_v))
            sizes = np.bincount(g, minlength=2 * n)
            roots = np.flatnonzero(sizes >= 20)
            assert len(roots) == 2, sizes[roots]
            for r in roots:
                assert len(np.unique(truth[g == r])) == 1 and sizes[r] > 9000
            cat = b200.fof_groups(g, d["m"], ctx.download_state(), 20)  # the labels feed the catalogue unchanged
            assert list(cat["root"]) == sorted(roots, key=lambda r: (-sizes[r], r))


# ------------------------------------------------------------------------------------------------ invariance
def test_virtual_shards_and_reruns(b200, oracle):
    for scheme in ("galaxy", "random"):
        d = oracle.init_bodies(scheme, 20011)
        res = []
        for k in (1, 2, 3, 8):
            with _ctx(b200, d, devices=[0] * k) as ctx:
                if k == 1:
                    bs = _settings(ctx, d)[:6]
                res.append([ctx.fof_phase(*b) for b in bs])
                assert all(np.array_equal(a, ctx.fof_phase(*b)) for a, b in zip(res[-1], bs))  # rerun
        for r in res[1:]:
            assert all(np.array_equal(a, b) for a, b in zip(res[0], r))


def test_ordered_after_async_step(b200, oracle):
    d = oracle.init_bodies("random", 20011)
    with _ctx(b200, d) as ctx:
        bs = _settings(ctx, d)[1:4]
    for devs in ([0], [0, 0, 0]):
        res = []
        for join in (False, True):
            with _ctx(b200, d, devices=devs) as ctx:
                ctx.step(DT, 0, 3)
                if join:
                    ctx.sync()
                res.append([ctx.fof_phase(*b) for b in bs])
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
                bs = _settings(ctx, ctx.download_state())[:6]
            res.append([ctx.fof_phase(*b) for b in bs])
    assert all(np.array_equal(a, b) for a, b in zip(*res))


def test_torchrun_ranks():
    if _n_devices() < 2:
        pytest.skip("needs 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29587", os.path.join(REPO, "tests", "mp_phase_fof_parity.py")],
                       capture_output=True, text=True, timeout=600)
    print(r.stdout[-2000:])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert r.stdout.count("ok=True") == 2


# ------------------------------------------------------------------------------------------------ edge cases
@pytest.mark.parametrize("n", [129, 257])
def test_padding_never_linked(b200, n):
    """Bodies 0 and n - 1 (alone in the last AoSoA block) sit at scaled x = +0.9 and -0.9: too far apart to link, but
    each within reach of the padding lanes at the origin.  Every other body is far away."""
    d = {c: np.zeros(n, np.float32) for c in KEYS}
    d["qx"][:] = 1e3 * np.arange(n, dtype=np.float32) + 1e4
    d["qx"][0], d["qx"][n - 1] = 0.9, -0.9
    d["m"] = np.full(n, 1e20, np.float32)
    with _ctx(b200, d) as ctx:
        assert np.array_equal(ctx.fof_phase(1.0, np.inf), np.arange(n))
        assert np.array_equal(ctx.fof_phase(1.0, 1.0), np.arange(n))


def test_non_finite_inputs_stay_alone(b200, oracle, poracle):
    d = oracle.init_bodies("galaxy", 2049)
    d = {c: d[c].copy() for c in KEYS + ("m",)}
    bad = [3, 500, 1000, 1500]
    with _ctx(b200, d) as ctx:
        b_x, b_v = _settings(ctx, d)[2]
    d["qx"][3], d["vy"][500], d["vz"][1000], d["vx"][1500] = np.nan, np.inf, -np.inf, np.nan
    with _ctx(b200, d) as ctx:
        for bs in ((b_x, b_v), (np.inf, np.inf), (1e30, 1e30)):
            got = ctx.fof_phase(*bs)
            assert np.array_equal(got, poracle.groups(d, *bs))
            assert np.array_equal(got[bad], bad)
        assert np.all(np.delete(ctx.fof_phase(np.inf, np.inf), bad) == 0)
        # a tiny b overflows the scaled coordinates: every body alone
        assert np.array_equal(ctx.fof_phase(1e-38, np.inf), np.arange(2049))


def test_zero_mass_bodies_link(b200, oracle, poracle):
    d = oracle.init_bodies("random", 1000)
    with _ctx(b200, d) as ctx:
        b = _settings(ctx, d)[2]
        want = ctx.fof_phase(*b)
    d["m"] = d["m"].copy()
    d["m"][::3] = 0
    with _ctx(b200, d) as ctx:
        got = ctx.fof_phase(*b)
    assert np.array_equal(got, want) and np.array_equal(got, poracle.groups(d, *b))


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
                ctx.fof_phase(1e9, 1e3)
                ctx.fof_phase(np.inf, np.inf)
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
        ctx.fof_phase(1e9, 1e3)
        grown = ctx.allocated_bytes
        # the scaled array of all bodies on every shard, then a forest of 4 N_pad bytes per shard; the first holds all P
        assert grown - before == 24 * n_pad * shards + 4 * n_pad * (shards + shards - 1), grown - before
        # pack, init and link per shard, merge (P > 1) and finalize
        assert ctx.launch_count - launches == 3 * shards + (2 if shards > 1 else 1)
        for bs in ((1e7, 1.0), (1e11, np.inf), (np.inf, np.inf)):
            ctx.fof_phase(*bs)
        assert ctx.allocated_bytes == grown
        ctx.fof(1e9)  # position FoF fits in the same scratch
        assert ctx.allocated_bytes == grown


def test_errors(b200, oracle):
    L = b200.lib()
    d = oracle.init_bodies("galaxy", 1000)
    g = np.empty(1000, np.uint32)
    gp = g.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32))
    inf, nan = float("inf"), float("nan")
    with b200.Context(1000, G_F32, SOFT) as ctx:
        assert L.b200nb_fof_phase(ctx._ctx, 1.0, 1.0, gp) == b200.ESTATE
        ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
        assert L.b200nb_fof_phase(ctx._ctx, 1.0, 1.0, None) == b200.EINVAL
        for bad in (0.0, -0.0, -1.0, nan, -inf):
            assert L.b200nb_fof_phase(ctx._ctx, bad, 1.0, gp) == b200.EINVAL, bad
            assert L.b200nb_fof_phase(ctx._ctx, 1.0, bad, gp) == b200.EINVAL, bad
        for ok in ((1.0, inf), (inf, 1.0), (1e-45, 3.4e38)):
            assert L.b200nb_fof_phase(ctx._ctx, *ok, gp) == b200.OK, ok
        assert L.b200nb_fof_phase(ctx._ctx, inf, inf, gp) == b200.OK
        assert np.all(g == 0)  # both parts switched off: one group
        for bad in (0.0, -1.0, nan, -inf, True):
            with pytest.raises(ValueError):
                ctx.fof_phase(bad, 1.0)
            with pytest.raises(ValueError):
                ctx.fof_phase(1.0, bad)
