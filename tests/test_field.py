"""b200nb_field / b200nb_potential on the GPU: against the fp64 field reference (tests/field_oracle.c), against the
library's own energy and force pass, bitwise invariance of every result (reruns, batching, shards, ranks), untouched
simulation state, ordering after an asynchronous step, and the error contract."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import DT, G_F32, REPO, SOFT, max_rel_err
from field_oracle import FieldOracle

pytestmark = pytest.mark.gpu

BATCH = 128 * 512  # FIELD_BATCH in csrc/field_sm100.cuh: targets per launch


@pytest.fixture(scope="module")
def foracle():
    return FieldOracle()


def _ctx(b200, d, soft=SOFT, **kw):
    ctx = b200.Context(len(d["qx"]), G_F32, soft, **kw)
    ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
    return ctx


def _points(d, M, rng):
    """M points mixing five kinds: inside the system, just outside it, 10^3 system radii away, exactly on a body, and
    on body 0 (the galaxy's central body)."""
    q = np.stack([d["qx"], d["qy"], d["qz"]]).astype(np.float64)
    R = max(float(np.max(np.linalg.norm(q, axis=0))), 1e8)
    kind = rng.integers(0, 5, M)
    kind[: min(M, 5)] = np.arange(min(M, 5))[::-1]  # the first point is on the central body, every kind occurs
    u = rng.normal(size=(3, M))
    u /= np.linalg.norm(u, axis=0)
    radius = np.select([kind == 0, kind == 1, kind == 2], [R * rng.random(M) ** (1 / 3), R * (1.5 + rng.random(M)), 1e3 * R], 0.0)
    p = u * radius
    on = rng.integers(0, q.shape[1], M)
    p[:, kind == 3] = q[:, on[kind == 3]]
    p[:, kind == 4] = q[:, [0]]
    return [p[k].astype(np.float32) for k in range(3)]


def _check_field(got, ref):
    ax, ay, az, phi, amag = ref
    da = np.linalg.norm(np.stack(got[:3]).astype(np.float64) - np.stack([ax, ay, az]), axis=0)
    amod = np.linalg.norm(np.stack([ax, ay, az]), axis=0)
    assert np.all(da <= 1e-6 * amag), float(np.max(da / np.maximum(amag, 1e-300)))
    big = amod >= 0.05 * amag
    assert np.all(da[big] <= 1e-5 * amod[big]), float(np.max(da[big] / amod[big]))
    dphi = np.abs(got[3].astype(np.float64) - phi)
    assert np.all(dphi <= 1e-6 * np.abs(phi)), float(np.max(dphi / np.abs(phi)))


# ------------------------------------------------------------------------------------------------ accuracy
@pytest.mark.parametrize("scheme,n", [("galaxy", 1), ("random", 129), ("galaxy", 2049), ("galaxy", 200000)])
def test_field_vs_fp64(b200, oracle, foracle, scheme, n):
    d = oracle.init_bodies(scheme, n)
    rng = np.random.default_rng(n)
    with _ctx(b200, d) as ctx:
        for M in (1, 127, 128, 129, 4097):
            p = _points(d, M, rng)
            got = ctx.field(*p)
            _check_field(got, foracle.field(d, *p))


@pytest.mark.parametrize("soft", [2e8, 1e4])
@pytest.mark.parametrize("n", [2049, 200000])
def test_potential_vs_fp64(b200, oracle, foracle, n, soft):
    """soft = 1e4: the self term G m_i / soft is ~3000x the rest, so an implementation that subtracts it fails."""
    d = oracle.init_bodies("galaxy", n)
    with _ctx(b200, d, soft) as ctx:
        phi = ctx.potential()
    idx = None if n <= 4096 else np.unique(np.concatenate([[0, 1, 127, 128, n - 1], np.random.default_rng(1).integers(0, n, 400)]))
    ref = foracle.potential(d, idx, soft=soft)
    got = phi if idx is None else phi[idx.astype(np.int64)]
    err = np.abs(got.astype(np.float64) - ref) / np.abs(ref)
    assert np.max(err) <= 1e-6, float(np.max(err))


def test_potential_coincident_bodies(b200, oracle, foracle):
    """Exclusion is by index: two bodies at the same position each see the other (and a third one, far off)."""
    n = 3
    d = {k: np.zeros(n, np.float32) for k in ("qx", "qy", "qz", "vx", "vy", "vz")}
    d["qx"][:] = [1e8, 1e8, -3e8]
    d["m"] = np.array([2e24, 5e20, 1e22], np.float32)
    for soft in (2e8, 1e4):
        with _ctx(b200, d, soft) as ctx:
            phi = ctx.potential()
        ref = foracle.potential(d, soft=soft)
        assert np.all(np.abs(phi - ref) <= 1e-6 * np.abs(ref)), (phi, ref)
        assert phi[1] < -0.5 * float(G_F32) * 2e24 / soft  # body 1 sees body 0 at zero distance


# ------------------------------------------------------------------------------------------------ consistency
def test_consistent_with_energy_and_force_pass(b200, oracle):
    n = 20000
    d = oracle.init_bodies("galaxy", n)
    with _ctx(b200, d) as ctx:
        ctx.step(DT, 0, 2)
        st = ctx.download_state()
        e = ctx.energy()
        phi = ctx.potential()
        ctx.accel()
        acc = ctx.download_accel()
        f = ctx.field(st["qx"], st["qy"], st["qz"])
    m = d["m"].astype(np.float64)
    kin = 0.5 * np.sum(m * sum(st[k].astype(np.float64) ** 2 for k in ("vx", "vy", "vz")))
    pot = 0.5 * np.sum(m * phi.astype(np.float64))
    assert abs((e - kin) - pot) <= 1e-6 * abs(pot), ((e - kin), pot)
    # the field at a body includes its (zero) self force: the same sum as the force pass; body 0 is the central body
    assert max_rel_err([a[1:] for a in acc], [a[1:] for a in f[:3]]) <= 2e-6


# ------------------------------------------------------------------------------------------------ bitwise invariance
def _same(a, b):
    for x, y in zip(a, b):
        assert np.array_equal(x.view(np.uint32), y.view(np.uint32))


def test_bitwise_reruns_batches_and_alone(b200, oracle):
    n = 30000
    d = oracle.init_bodies("galaxy", n)
    rng = np.random.default_rng(3)
    big = _points(d, 100000, rng)
    sel = np.array([0, 1, 511, 512, 4096, BATCH - 1, BATCH, BATCH + 1, 99999])
    with _ctx(b200, d) as ctx:
        r1 = ctx.field(*big)
        _same(r1, ctx.field(*big))  # rerun
        alone = [ctx.field(*[p[i:i + 1] for p in big]) for i in sel]
        for j, i in enumerate(sel):
            _same([a[i:i + 1] for a in r1], alone[j])
        # just above one internal batch, and a shifted window: the same point at another position of the call
        part = ctx.field(*[p[:BATCH + 37] for p in big])
        _same([a[:BATCH + 37] for a in r1], part)
        shifted = ctx.field(*[p[5:BATCH + 300] for p in big])
        _same([a[5:BATCH + 300] for a in r1], shifted)
        phi = ctx.potential()
        _same([phi], [ctx.potential()])


def test_bitwise_virtual_shards(b200, oracle):
    n = 20011
    d = oracle.init_bodies("random", n)
    p = _points(d, 3001, np.random.default_rng(4))
    res = []
    for k in (1, 2, 3):
        with _ctx(b200, d, devices=[0] * k) as ctx:
            res.append((ctx.field(*p), ctx.potential()))
    for r in res[1:]:
        _same(res[0][0], r[0])
        _same([res[0][1]], [r[1]])


def _n_devices():
    import torch
    return torch.cuda.device_count()


def test_bitwise_two_gpus(b200, oracle):
    if _n_devices() < 2:
        pytest.skip("needs 2 GPUs")
    n = 20011
    d = oracle.init_bodies("galaxy", n)
    p = _points(d, 3001, np.random.default_rng(5))
    res = []
    for devs in ([0], [0, 1]):
        with _ctx(b200, d, devices=devs) as ctx:
            ctx.step(DT, 0, 2)
            res.append((ctx.field(*p), ctx.potential()))
    _same(res[0][0], res[1][0])
    _same([res[0][1]], [res[1][1]])


def test_bitwise_torchrun_ranks():
    if _n_devices() < 2:
        pytest.skip("needs 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29579", os.path.join(REPO, "tests", "mp_field_parity.py")],
                       capture_output=True, text=True, timeout=600)
    print(r.stdout[-2000:])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert r.stdout.count("ok=True") == 2


# ------------------------------------------------------------------------------------------------ state and ordering
@pytest.mark.parametrize("integrator", [0, 1])
@pytest.mark.parametrize("steps", [1, 32])  # 32: the cached step-graph path
def test_state_untouched(b200, oracle, integrator, steps):
    n = 5000
    d = oracle.init_bodies("galaxy", n)
    p = _points(d, 1000, np.random.default_rng(6))
    out = []
    for probe in (False, True):
        with _ctx(b200, d) as ctx:
            ctx.step(DT, integrator, steps)
            if probe:
                ctx.field(*p)
                ctx.potential()
            ctx.step(DT, integrator, steps)
            st = ctx.download_state()
            out.append([st[k] for k in ctx._STATE] + list(ctx.download_accel()))
    _same(out[0], out[1])


def test_ordered_after_async_step(b200, oracle):
    n = 20011
    d = oracle.init_bodies("random", n)
    p = _points(d, 2000, np.random.default_rng(7))
    res = []
    for join in (False, True):
        with _ctx(b200, d, devices=[0, 0, 0]) as ctx:
            ctx.step(DT, 0, 3)
            if join:
                ctx.sync()
            res.append((ctx.field(*p), ctx.potential()))
    _same(res[0][0], res[1][0])
    _same([res[0][1]], [res[1][1]])


def test_scratch_is_bounded(b200, oracle):
    d = oracle.init_bodies("galaxy", 10000)
    rng = np.random.default_rng(8)
    with _ctx(b200, d) as ctx:
        before = ctx.allocated_bytes
        ctx.field(*_points(d, 3 * BATCH, rng))
        grown = ctx.allocated_bytes
        assert grown > before
        ctx.field(*_points(d, 7 * BATCH + 5, rng))
        ctx.potential()
        assert ctx.allocated_bytes == grown


# ------------------------------------------------------------------------------------------------ errors
def test_errors(b200, oracle):
    L = b200.lib()
    d = oracle.init_bodies("galaxy", 1000)
    x = np.zeros(4, np.float32)
    xp = x.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
    with b200.Context(1000, G_F32, SOFT) as ctx:
        assert L.b200nb_field(ctx._ctx, 4, xp, xp, xp, None, None, None, None) == b200.ESTATE
        assert L.b200nb_potential(ctx._ctx, xp) == b200.ESTATE
        ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
        assert L.b200nb_field(ctx._ctx, 4, None, xp, xp, xp, xp, xp, xp) == b200.EINVAL
        assert L.b200nb_field(ctx._ctx, 4, xp, xp, None, xp, xp, xp, xp) == b200.EINVAL
        assert L.b200nb_potential(ctx._ctx, None) == b200.EINVAL
        assert L.b200nb_field(ctx._ctx, 0, None, None, None, None, None, None, None) == b200.OK
        a = ctx.field(x, x, x)
        assert all(v.shape == (4,) for v in a)
        # only phi requested
        phi = np.empty(4, np.float32)
        assert L.b200nb_field(ctx._ctx, 4, xp, xp, xp, None, None, None, phi.ctypes.data_as(ctypes.POINTER(ctypes.c_float))) == b200.OK
        assert np.array_equal(phi, a[3])
        with pytest.raises(ValueError):
            ctx.field(x, x, x[:3])
