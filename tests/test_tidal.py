"""b200nb_tidal / b200nb_tidal_bodies on the GPU: against the fp64 reference (tests/tidal_oracle.c) under the header's
per-entry bound, the physics (point mass, trace identity, derivative of b200nb_field, points vs bodies mode), bitwise
invariance (reruns, batching, shards, ranks), untouched simulation state, ordering after an asynchronous step, bounded
scratch and the error contract."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import DT, G_F32, REPO, SOFT
from field_oracle import FieldOracle
from test_field import _points
from tidal_oracle import TidalOracle, six

pytestmark = pytest.mark.gpu

BATCH = 32768  # TIDAL_BATCH in csrc/tidal_sm100.cuh: targets per launch
BOUND = 5e-6   # |T_ab - T_ab^fp64| <= BOUND * A_ab (include/b200nb.h)
G = float(G_F32)


@pytest.fixture(scope="module")
def toracle():
    return TidalOracle()


def _ctx(b200, d, soft=SOFT, **kw):
    ctx = b200.Context(len(d["qx"]), G_F32, soft, **kw)
    ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
    return ctx


def _check(got, ref, what=""):
    """got: float32 [m][3][3] from the library; ref: (t, amag, s5) of the oracle"""
    t, amag, _ = ref
    g6 = six(got).astype(np.float64)
    err = np.abs(g6 - t)
    ok = err <= BOUND * amag
    worst = float(np.max(np.where(amag > 0, err / np.where(amag > 0, amag, 1.0), 0.0)))
    assert np.all(ok), (what, worst, np.argwhere(~ok)[:5])
    return worst


# ------------------------------------------------------------------------------------------------ accuracy
@pytest.mark.parametrize("soft", [2e8, 1e4])
@pytest.mark.parametrize("scheme,n", [("galaxy", 1), ("random", 129), ("galaxy", 2049), ("galaxy", 200000)])
def test_tidal_vs_fp64(b200, oracle, toracle, scheme, n, soft):
    """the five kinds of points of test_field: inside, just outside, 10^3 system radii away, on a body, on body 0"""
    d = oracle.init_bodies(scheme, n)
    rng = np.random.default_rng(n)
    worst = 0.0
    with _ctx(b200, d, soft) as ctx:
        for M in (1, 127, 128, 129, 4097):
            p = _points(d, M, rng)
            got = ctx.tidal(*p)
            assert got.shape == (M, 3, 3) and got.dtype == np.float32
            assert np.array_equal(got, np.transpose(got, (0, 2, 1)))
            worst = max(worst, _check(got, toracle.tidal(d, *p, soft=soft), (M,)))
    print(f"{scheme} n={n} soft={soft}: max |T - T64| / A = {worst:.2e}")


@pytest.mark.parametrize("soft", [2e8, 1e4])
@pytest.mark.parametrize("n", [2049, 200000])
def test_tidal_bodies_vs_fp64(b200, oracle, toracle, n, soft):
    """soft = 1e4: the self term G m_i / soft^3 would dwarf everything, so it must be excluded, never subtracted"""
    d = oracle.init_bodies("galaxy", n)
    with _ctx(b200, d, soft) as ctx:
        t = ctx.tidal_bodies()
    assert t.shape == (n, 3, 3) and t.dtype == np.float32
    idx = None if n <= 4096 else np.unique(np.concatenate([[0, 1, 127, 128, n - 1], np.random.default_rng(1).integers(0, n, 400)]))
    got = t if idx is None else t[idx.astype(np.int64)]
    worst = _check(got, toracle.tidal_bodies(d, idx, soft=soft))
    print(f"bodies n={n} soft={soft}: max |T - T64| / A = {worst:.2e}")


def test_tidal_bodies_coincident(b200, toracle):
    """Exclusion is by index: two bodies at the same position each see the other (and a third one, far off)."""
    n = 3
    d = {k: np.zeros(n, np.float32) for k in ("qx", "qy", "qz", "vx", "vy", "vz")}
    d["qx"][:] = [1e8, 1e8, -3e8]
    d["m"] = np.array([2e24, 5e20, 1e22], np.float32)
    for soft in (2e8, 1e4):
        with _ctx(b200, d, soft) as ctx:
            t = ctx.tidal_bodies()
        _check(t, toracle.tidal_bodies(d, soft=soft), soft)
        # body 1 sees body 0 at zero distance: -G m_0 / soft^3 on the diagonal
        assert np.allclose(np.diag(t[1]), -G * 2e24 / float(np.float32(soft)) ** 3, rtol=1e-3)


# ------------------------------------------------------------------------------------------------ physics
def test_point_mass(b200):
    """one body, soft = 1 m (a context needs soft > 0; s^2 = r^2 + 1 differs from r^2 by <= 1e-12 here):
    T = G m / r^3 (3 u u^T - 1), stretching along the line to the body"""
    d = {k: np.zeros(1, np.float32) for k in ("qx", "qy", "qz", "vx", "vy", "vz")}
    d["m"] = np.array([2e24], np.float32)
    rng = np.random.default_rng(2)
    u = rng.normal(size=(3, 200))
    u /= np.linalg.norm(u, axis=0)
    r = 10 ** rng.uniform(6, 12, 200)
    p = [(u[k] * r).astype(np.float32) for k in range(3)]
    p[0][0], p[1][0], p[2][0] = 3e8, 0, 0
    with _ctx(b200, d, 1.0) as ctx:
        t = ctx.tidal(*p).astype(np.float64)
    pd = np.stack(p).astype(np.float64)
    rr = np.linalg.norm(pd, axis=0)
    uu = pd / rr
    gm = G * 2e24
    want = gm / rr[:, None, None] ** 3 * (3 * np.einsum("im,jm->mij", uu, uu) - np.eye(3))
    scale = gm / rr**3
    assert np.all(np.abs(t - want) <= 4 * BOUND * scale[:, None, None])
    assert np.allclose(np.diag(t[0]), gm / 3e8**3 * np.array([2, -1, -1]), rtol=BOUND, atol=0)
    assert np.all(np.linalg.eigvalsh(t)[:, -1] > 0)


@pytest.mark.parametrize("soft", [2e8, 1e4])
def test_trace_identity(b200, oracle, toracle, soft):
    """tr T = -3 soft^2 sum_j G m_j / s^5 (Poisson's equation for the Plummer-softened kernel)"""
    d = oracle.init_bodies("galaxy", 20000)
    p = _points(d, 3000, np.random.default_rng(3))
    with _ctx(b200, d, soft) as ctx:
        t = ctx.tidal(*p).astype(np.float64)
        tb = ctx.tidal_bodies().astype(np.float64)
    for got, (_, amag, s5) in ((t, toracle.tidal(d, *p, soft=soft)), (tb, toracle.tidal_bodies(d, soft=soft))):
        tr = np.trace(got, axis1=1, axis2=2)
        want = -3.0 * float(np.float32(soft)) ** 2 * s5
        assert np.all(np.abs(tr - want) <= BOUND * amag[:, :3].sum(axis=1))


def test_derivative_of_the_field(b200, oracle, toracle):
    """T_ab = d a_a / d p_b: central differences of b200nb_field at p +- h e_b, p and p +- h exact in fp32.
    Tolerance, per entry: the fp64 truncation error of the same difference (from the references) + the field's own
    error bound 1e-6 * amag at p +- h over 2h + the tidal bound.  That is below 1e-3 of A_ab on the diagonal and about
    1e-3 of it off the diagonal, whose A_ab can be much smaller than the field's scale."""
    d = oracle.init_bodies("galaxy", 20000)
    rng = np.random.default_rng(4)
    M, h = 500, 2.0**20
    p = np.round(rng.normal(size=(3, M)) * 1e8 / 64.0) * 64.0  # |p| < 2^28: multiples of 64 are exact, and so is p +- h
    assert np.array_equal(p.astype(np.float32).astype(np.float64), p)
    fo = FieldOracle()
    t64, amag, _ = toracle.tidal(d, *p.astype(np.float32))
    with _ctx(b200, d) as ctx:
        t = six(ctx.tidal(*p.astype(np.float32))).astype(np.float64)
        jg, j64, rnd = np.empty((M, 3, 3)), np.empty((M, 3, 3)), np.zeros((M, 3))
        for b in range(3):
            e = np.zeros((3, 1))
            e[b] = h
            pp, pm = (p + e).astype(np.float32), (p - e).astype(np.float32)
            assert np.array_equal(pp.astype(np.float64), p + e) and np.array_equal(pm.astype(np.float64), p - e)
            gp, gm_ = ctx.field(*pp), ctx.field(*pm)
            rp, rm = fo.field(d, *pp), fo.field(d, *pm)
            jg[:, :, b] = (np.stack(gp[:3], 1).astype(np.float64) - np.stack(gm_[:3], 1)) / (2 * h)
            j64[:, :, b] = (np.stack(rp[:3], 1) - np.stack(rm[:3], 1)) / (2 * h)
            rnd[:, b] = 1e-6 * (rp[4] + rm[4]) / (2 * h)
    trunc = np.abs(six(j64) - t64)
    tol = trunc + rnd[:, [0, 1, 2, 1, 2, 2]] + BOUND * amag
    assert np.all(tol[:, :3] <= 1e-3 * amag[:, :3]) and np.median(tol / amag) <= 1e-3  # a meaningful comparison
    assert np.all(np.abs(six(jg) - t) <= tol), float(np.max(np.abs(six(jg) - t) / amag))


def test_bodies_equal_points_minus_self(b200, oracle):
    """At a body's position the points-mode tensor carries the self term -G m_i / soft^3 * I that bodies mode leaves out.
    Light bodies keep the self term small, so the comparison is well conditioned."""
    n, soft = 4099, 2e8
    d = oracle.init_bodies("galaxy", n)
    light = np.array([1, 2, 129, 2048, n - 1])
    d["m"] = d["m"].copy()
    d["m"][light] = np.float32(1e12)
    with _ctx(b200, d, soft) as ctx:
        tb = ctx.tidal_bodies()[light].astype(np.float64)
        tp = ctx.tidal(d["qx"][light], d["qy"][light], d["qz"][light]).astype(np.float64)
    _, amag, _ = TidalOracle().tidal_bodies(d, light, soft=soft)
    self_term = -G * float(np.float32(1e12)) / float(np.float32(soft)) ** 3
    diff = six(tp - tb) - self_term * np.array([1, 1, 1, 0, 0, 0])
    assert np.all(np.abs(diff) <= 2 * BOUND * amag)


# ------------------------------------------------------------------------------------------------ bitwise invariance
def _same(a, b):
    assert np.array_equal(np.asarray(a).view(np.uint32), np.asarray(b).view(np.uint32))


def test_bitwise_reruns_batches_and_alone(b200, oracle):
    n = 30000
    d = oracle.init_bodies("galaxy", n)
    big = _points(d, 100000, np.random.default_rng(5))
    sel = np.array([0, 1, 511, 512, 4096, BATCH - 1, BATCH, BATCH + 1, 3 * BATCH + 5, 99999])
    with _ctx(b200, d) as ctx:
        r1 = ctx.tidal(*big)
        _same(r1, ctx.tidal(*big))  # rerun
        for i in sel:
            _same(r1[i:i + 1], ctx.tidal(*[p[i:i + 1] for p in big]))
        _same(r1[:BATCH + 37], ctx.tidal(*[p[:BATCH + 37] for p in big]))
        _same(r1[5:2 * BATCH + 300], ctx.tidal(*[p[5:2 * BATCH + 300] for p in big]))
        tb = ctx.tidal_bodies()
        _same(tb, ctx.tidal_bodies())


def test_bitwise_virtual_shards(b200, oracle):
    n = 20011
    d = oracle.init_bodies("random", n)
    p = _points(d, 3001, np.random.default_rng(6))
    res = []
    for k in (1, 2, 3):
        with _ctx(b200, d, devices=[0] * k) as ctx:
            res.append((ctx.tidal(*p), ctx.tidal_bodies()))
    for r in res[1:]:
        _same(res[0][0], r[0])
        _same(res[0][1], r[1])


def _n_devices():
    import torch
    return torch.cuda.device_count()


def test_bitwise_two_gpus(b200, oracle):
    if _n_devices() < 2:
        pytest.skip("needs 2 GPUs")
    n = 20011
    d = oracle.init_bodies("galaxy", n)
    p = _points(d, 3001, np.random.default_rng(7))
    res = []
    for devs in ([0], [0, 1]):
        with _ctx(b200, d, devices=devs) as ctx:
            ctx.step(DT, 0, 2)
            res.append((ctx.tidal(*p), ctx.tidal_bodies()))
    _same(res[0][0], res[1][0])
    _same(res[0][1], res[1][1])


def test_bitwise_torchrun_ranks():
    if _n_devices() < 2:
        pytest.skip("needs 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29583", os.path.join(REPO, "tests", "mp_tidal_parity.py")],
                       capture_output=True, text=True, timeout=600)
    print(r.stdout[-2000:])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert r.stdout.count("ok=True") == 2


# ------------------------------------------------------------------------------------------------ state and ordering
@pytest.mark.parametrize("tracers", [False, True])
@pytest.mark.parametrize("integrator", [0, 1])
@pytest.mark.parametrize("steps", [1, 32])  # 32: the cached step-graph path
def test_state_untouched(b200, oracle, integrator, steps, tracers):
    n = 5000
    d = oracle.init_bodies("galaxy", n)
    rng = np.random.default_rng(8)
    p = _points(d, 1000, rng)
    tr = [(rng.normal(size=700) * 2e8).astype(np.float32) for _ in range(3)] + [np.zeros(700, np.float32)] * 3
    out = []
    for probe in (False, True):
        with _ctx(b200, d) as ctx:
            if tracers:
                ctx.set_tracers(*tr)
            ctx.step(DT, integrator, steps)
            if probe:
                ctx.tidal(*p)
                ctx.tidal_bodies()
            ctx.step(DT, integrator, steps)
            st = ctx.download_state()
            res = [st[k] for k in ctx._STATE] + list(ctx.download_accel())
            if tracers:
                res += list(ctx.download_tracers().values())
            out.append(res)
    for a, b in zip(*out):
        _same(a, b)


def test_ordered_after_async_step(b200, oracle):
    n = 20011
    d = oracle.init_bodies("random", n)
    p = _points(d, 2000, np.random.default_rng(9))
    res = []
    for join in (False, True):
        with _ctx(b200, d, devices=[0, 0, 0]) as ctx:
            ctx.step(DT, 0, 3)
            if join:
                ctx.sync()
            res.append((ctx.tidal(*p), ctx.tidal_bodies()))
    _same(res[0][0], res[1][0])
    _same(res[0][1], res[1][1])


def test_scratch_and_launches(b200, oracle):
    """Growth of allocated_bytes is the header's 28 S B + 36 B; two launches per batch; steps launch and allocate the
    same before and after tidal calls as in a context that never made one."""
    n = 10000
    d = oracle.init_bodies("galaxy", n)
    nblk = (n + 127) // 128
    S = min(64, max(1, (nblk + 31) // 32))
    rng = np.random.default_rng(10)

    def steps(c):
        before, b0 = c.launch_count, c.allocated_bytes
        c.step(DT, 0, 1)
        c.step(DT, 1, 1)
        return c.launch_count - before, c.allocated_bytes - b0

    with _ctx(b200, d) as ctx, _ctx(b200, d) as ref:
        assert ctx.allocated_bytes == ref.allocated_bytes
        assert steps(ctx) == steps(ref)
        assert ctx.allocated_bytes == ref.allocated_bytes
        before, L0 = ctx.allocated_bytes, ctx.launch_count
        ctx.tidal(*_points(d, 3 * BATCH, rng))
        assert ctx.launch_count - L0 == 2 * 3
        grown = ctx.allocated_bytes
        assert grown - before == 28 * S * BATCH + 36 * BATCH
        L0 = ctx.launch_count
        ctx.tidal(*_points(d, 7 * BATCH + 5, rng))
        assert ctx.launch_count - L0 == 2 * 8
        L0 = ctx.launch_count
        ctx.tidal_bodies()
        assert ctx.launch_count - L0 == 2
        assert ctx.allocated_bytes == grown
        assert steps(ctx) == steps(ref)


# ------------------------------------------------------------------------------------------------ errors
def test_errors(b200, oracle):
    L = b200.lib()
    d = oracle.init_bodies("galaxy", 1000)
    x = np.zeros(4, np.float32)
    xp = x.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
    t = np.zeros((4, 6), np.float32)
    tp = t.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
    with b200.Context(1000, G_F32, SOFT) as ctx:
        assert L.b200nb_tidal(ctx._ctx, 4, xp, xp, xp, tp) == b200.ESTATE
        assert L.b200nb_tidal_bodies(ctx._ctx, tp) == b200.ESTATE
        ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
        assert L.b200nb_tidal(ctx._ctx, 4, None, xp, xp, tp) == b200.EINVAL
        assert L.b200nb_tidal(ctx._ctx, 4, xp, None, xp, tp) == b200.EINVAL
        assert L.b200nb_tidal(ctx._ctx, 4, xp, xp, None, tp) == b200.EINVAL
        assert L.b200nb_tidal(ctx._ctx, 4, xp, xp, xp, None) == b200.EINVAL
        assert L.b200nb_tidal_bodies(ctx._ctx, None) == b200.EINVAL
        assert L.b200nb_tidal(ctx._ctx, 0, None, None, None, None) == b200.OK
        a = ctx.tidal(x, x, x)
        assert a.shape == (4, 3, 3)
        assert ctx.tidal(x[:0], x[:0], x[:0]).shape == (0, 3, 3)
        with pytest.raises(ValueError):
            ctx.tidal(x, x, x[:3])
        with pytest.raises(ValueError):
            ctx.tidal(x.reshape(2, 2), x.reshape(2, 2), x.reshape(2, 2))
