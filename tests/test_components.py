"""b200nb_component_field / b200nb_component_field_bodies on the GPU: against the fp64 reference (tests/components_oracle.c)
under the header's per-component bound, bit-identity with b200nb_field / b200nb_potential for one all-body component,
locality (relabelling, n_comp, renumbering, reruns, batching, shards, ranks), the physics of the budget built on the
output, untouched simulation state, ordering after an asynchronous step, bounded scratch and the error contract."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from components_oracle import ComponentsOracle
from conftest import DT, G_F32, REPO, SOFT
from test_field import _points

pytestmark = pytest.mark.gpu

NONE = 0xFFFFFFFF
G = float(G_F32)


@pytest.fixture(scope="module")
def co():
    return ComponentsOracle()


def _ctx(b200, d, soft=SOFT, **kw):
    ctx = b200.Context(len(d["qx"]), G_F32, soft, **kw)
    ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
    return ctx


def _same(a, b):
    assert np.array_equal(np.asarray(a).view(np.uint32), np.asarray(b).view(np.uint32))


def _check(got, ref, what=""):
    """got: (acc [m][C][3], phi [m][C]) from the library; ref: the oracle's (acc, phi, amag)"""
    acc, phi = got
    racc, rphi, amag = ref
    da = np.linalg.norm(acc.astype(np.float64) - racc, axis=2)
    assert np.all(da <= 1e-6 * amag), (what, float(np.max(np.where(amag > 0, da / np.where(amag > 0, amag, 1), da))))
    dphi = np.abs(phi.astype(np.float64) - rphi)
    assert np.all(dphi <= 1e-6 * np.abs(rphi)), (what, float(np.max(np.where(rphi != 0, dphi / np.abs(np.where(rphi != 0, rphi, 1)), dphi))))
    return float(np.max(np.where(amag > 0, da / np.where(amag > 0, amag, 1), 0), initial=0))


def _labels(kind, n, C, rng):
    if kind == "contiguous":
        return (np.arange(n) * C // max(n, 1)).astype(np.uint32)
    if kind == "interleaved":
        return (np.arange(n) % C).astype(np.uint32)
    if kind == "random":
        g = rng.integers(0, C, n).astype(np.uint32)
        g[rng.random(n) < 0.05] = NONE
        return g
    if kind == "none":
        return np.full(n, NONE, np.uint32)
    if kind == "sizes":  # components of 127, 128, 129 and 1 members, one empty, the rest in the last one
        g = np.full(n, C - 1, np.uint32)
        cuts = np.cumsum([0, 127, 128, 129, 1])
        for h in range(min(4, C - 2)):
            g[cuts[h]:cuts[h + 1]] = h
        return rng.permutation(g)
    raise ValueError(kind)


# ------------------------------------------------------------------------------------------------ accuracy
CASES = [("galaxy", 1, 1, "contiguous"), ("random", 129, 2, "interleaved"), ("galaxy", 129, 3, "random"),
         ("galaxy", 2049, 3, "contiguous"), ("random", 2049, 64, "random"), ("galaxy", 2049, 64, "interleaved"),
         ("galaxy", 2049, 2, "none"), ("random", 2049, 8, "sizes"), ("galaxy", 200000, 3, "contiguous"),
         ("galaxy", 200000, 64, "random")]


@pytest.mark.parametrize("soft", [2e8, 1e4])
@pytest.mark.parametrize("scheme,n,C,kind", CASES)
def test_components_vs_fp64(b200, oracle, co, scheme, n, C, kind, soft):
    d = oracle.init_bodies(scheme, n)
    rng = np.random.default_rng(n + C)
    comp = _labels(kind, n, C, rng)
    M = 129 if n > 10000 else 600
    p = _points(d, M, rng)
    idx = None if n <= 4096 else np.unique(np.concatenate([[0, 1, 127, 128, n - 1], rng.integers(0, n, 300)]))
    with _ctx(b200, d, soft) as ctx:
        got = ctx.component_field(comp, C, *p)
        assert got[0].shape == (M, C, 3) and got[1].shape == (M, C) and got[0].dtype == np.float32
        w1 = _check(got, co.field(d, comp, C, *p, soft=soft), "points")
        acc, phi = ctx.component_field_bodies(comp, C)
        assert acc.shape == (n, C, 3) and phi.shape == (n, C)
    if idx is not None:
        acc, phi = acc[idx], phi[idx]
    w2 = _check((acc, phi), co.bodies(d, comp, C, idx, soft=soft), "bodies")
    print(f"{scheme} n={n} C={C} {kind} soft={soft}: max |da| / sum|a_ij| = {w1:.2e} (points), {w2:.2e} (bodies)")


# ------------------------------------------------------------------------------------------------ bit-identity
@pytest.mark.parametrize("n", [1, 129, 2049, 200000])
def test_one_component_is_the_field_bitwise(b200, oracle, n):
    d = oracle.init_bodies("galaxy", n)
    p = _points(d, 4097, np.random.default_rng(3))
    comp = np.zeros(n, np.uint32)
    with _ctx(b200, d) as ctx:
        ax, ay, az, phi = ctx.field(*p)
        acc, cphi = ctx.component_field(comp, 1, *p)
        _same(acc[:, 0, 0], ax)
        _same(acc[:, 0, 1], ay)
        _same(acc[:, 0, 2], az)
        _same(cphi[:, 0], phi)
        _, bphi = ctx.component_field_bodies(comp, 1)
        _same(bphi[:, 0], ctx.potential())


# ------------------------------------------------------------------------------------------------ locality
def test_locality_relabelling(b200, oracle):
    """component h's values depend only on h's members: other bodies relabelled, merged, split, set to NO_GROUP, a
    growing n_comp and a renumbered h leave them bitwise unchanged"""
    n = 30011
    d = oracle.init_bodies("galaxy", n)
    rng = np.random.default_rng(4)
    p = _points(d, 3000, rng)
    base = rng.integers(0, 4, n).astype(np.uint32)
    h_members = base == 1
    with _ctx(b200, d) as ctx:
        ref = ctx.component_field(base, 4, *p), ctx.component_field_bodies(base, 4)

        def check(comp, C, h):
            a, f = ctx.component_field(comp, C, *p)
            _same(a[:, h], ref[0][0][:, 1])
            _same(f[:, h], ref[0][1][:, 1])
            a, f = ctx.component_field_bodies(comp, C)
            _same(a[:, h], ref[1][0][:, 1])
            _same(f[:, h], ref[1][1][:, 1])

        others = np.where(h_members, 1, rng.integers(2, 9, n)).astype(np.uint32)  # the others split and renumbered
        check(others, 9, 1)
        merged = np.where(h_members, 1, 0).astype(np.uint32)
        check(merged, 2, 1)
        check(np.where(h_members, 1, NONE).astype(np.uint32), 2, 1)
        check(np.where(h_members, 1, base).astype(np.uint32), 64, 1)  # growing n_comp
        check(np.where(h_members, 63, np.where(base == 3, 1, base)).astype(np.uint32), 64, 63)  # h renumbered


def test_bitwise_reruns_batches_and_alone(b200, oracle):
    """C = 64 on 30k bodies: one chunk per component, 64 in all, so a batch holds 65536 points; 130000 points take two"""
    n, C = 30000, 64
    d = oracle.init_bodies("galaxy", n)
    rng = np.random.default_rng(5)
    comp = rng.integers(0, C, n).astype(np.uint32)
    big = _points(d, 130000, rng)
    with _ctx(b200, d) as ctx:
        a1, f1 = ctx.component_field(comp, C, *big)
        a2, f2 = ctx.component_field(comp, C, *big)
        _same(a1, a2)
        _same(f1, f2)
        for i in (0, 1, 511, 512, 65535, 65536, 129999):
            a, f = ctx.component_field(comp, C, *[q[i:i + 1] for q in big])
            _same(a, a1[i:i + 1])
            _same(f, f1[i:i + 1])
        a, f = ctx.component_field(comp, C, *[q[7:70000] for q in big])
        _same(a, a1[7:70000])
        _same(f, f1[7:70000])
        b1 = ctx.component_field_bodies(comp, C)
        b2 = ctx.component_field_bodies(comp, C)
        _same(b1[0], b2[0])
        _same(b1[1], b2[1])


def test_bitwise_virtual_shards(b200, oracle):
    n, C = 20011, 3
    d = oracle.init_bodies("random", n)
    rng = np.random.default_rng(6)
    comp = rng.integers(0, C, n).astype(np.uint32)
    comp[::7] = NONE
    p = _points(d, 3001, rng)
    res = []
    for k in (1, 2, 3, 8):
        with _ctx(b200, d, devices=[0] * k) as ctx:
            res.append(ctx.component_field(comp, C, *p) + ctx.component_field_bodies(comp, C))
    for r in res[1:]:
        for a, b in zip(res[0], r):
            _same(a, b)


def _n_devices():
    import torch
    return torch.cuda.device_count()


def test_bitwise_two_gpus(b200, oracle):
    if _n_devices() < 2:
        pytest.skip("needs 2 GPUs")
    n, C = 20011, 3
    d = oracle.init_bodies("galaxy", n)
    rng = np.random.default_rng(7)
    comp = rng.integers(0, C, n).astype(np.uint32)
    p = _points(d, 3001, rng)
    res = []
    for devs in ([0], [0, 1]):
        with _ctx(b200, d, devices=devs) as ctx:
            ctx.step(DT, 0, 2)
            res.append(ctx.component_field(comp, C, *p) + ctx.component_field_bodies(comp, C))
    for a, b in zip(*res):
        _same(a, b)


def test_bitwise_torchrun_ranks():
    if _n_devices() < 2:
        pytest.skip("needs 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29587", os.path.join(REPO, "tests", "mp_components_parity.py")],
                       capture_output=True, text=True, timeout=600)
    print(r.stdout[-2000:])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert r.stdout.count("ok=True") == 2


# ------------------------------------------------------------------------------------------------ physics
def test_sum_over_components_and_own_group(b200, oracle):
    """sum_h a^h = b200nb_field's a, sum_h phi^h = b200nb_potential, phi^(comp[i]) = b200nb_group_potential, to 1e-6"""
    n, C = 50000, 5
    d = oracle.init_bodies("galaxy", n)
    rng = np.random.default_rng(8)
    comp = rng.integers(0, C, n).astype(np.uint32)
    p = _points(d, 2000, rng)
    with _ctx(b200, d) as ctx:
        acc, phi = ctx.component_field(comp, C, *p)
        f = ctx.field(*p)
        bacc, bphi = ctx.component_field_bodies(comp, C)
        pot, gpot = ctx.potential(), ctx.group_potential(comp)
    _, _, amag = ComponentsOracle().field(d, comp, C, *p)
    a = np.stack(f[:3], 1).astype(np.float64)
    assert np.all(np.linalg.norm(acc.astype(np.float64).sum(1) - a, axis=1) <= 2e-6 * amag.sum(1))
    assert np.all(np.abs(phi.astype(np.float64).sum(1) - f[3]) <= 2e-6 * np.abs(f[3]))
    assert np.all(np.abs(bphi.astype(np.float64).sum(1) - pot) <= 2e-6 * np.abs(pot))
    own = bphi[np.arange(n), comp].astype(np.float64)
    assert np.all(np.abs(own - gpot) <= 2e-6 * np.abs(gpot))


def test_budget_on_gpu_output(b200, oracle):
    """Newton's third law and the energy on the library's rows: |F_gh + F_hg| <= 1e-6 sum |m a|, and
    sum K + W / 2 = b200nb_energy to 1e-6 of the cancellation-free scale sum K + |sum W| / 2"""
    n, C = 40000, 4
    d = oracle.init_bodies("galaxy", n)
    comp = (np.arange(n) * C // n).astype(np.uint32)
    with _ctx(b200, d) as ctx:
        ctx.step(DT, 0, 3)
        st = ctx.download_state()
        acc, phi = ctx.component_field_bodies(comp, C)
        e = ctx.energy()
    m = d["m"]
    b = b200.component_budget(comp, C, m, st, acc, phi)
    ma = np.sum(m.astype(np.float64)[:, None] * np.linalg.norm(acc.astype(np.float64), axis=2))
    assert np.all(np.abs(b["force"] + np.transpose(b["force"], (1, 0, 2))) <= 1e-6 * ma)
    got = b["kinetic"].sum() + 0.5 * b["W"].sum()
    assert abs(got - e) <= 1e-6 * (b["kinetic"].sum() + 0.5 * abs(b["W"].sum())), (got, e)


def test_two_galaxies_attract(b200):
    """two well-separated Plummer-like clouds: F_01 = G M0 M1 / d^2 up to the tidal (quadrupole) term, F_10 = -F_01"""
    rng = np.random.default_rng(9)
    n0, n1, R, D = 3000, 2000, 1e9, 4e10
    q = np.concatenate([rng.normal(size=(n0, 3)) * R, rng.normal(size=(n1, 3)) * 0.5 * R + [D, 0, 0]]).astype(np.float32)
    m = np.concatenate([np.full(n0, 2e24), np.full(n1, 1e24)]).astype(np.float32)
    z = np.zeros(n0 + n1, np.float32)
    comp = np.concatenate([np.zeros(n0), np.ones(n1)]).astype(np.uint32)
    with b200.Context(n0 + n1, G_F32, 1e7) as ctx:
        ctx.upload(q[:, 0], q[:, 1], q[:, 2], m, z, z, z)
        acc, phi = ctx.component_field_bodies(comp, 2)
    st = {"qx": q[:, 0], "qy": q[:, 1], "qz": q[:, 2], "vx": z, "vy": z, "vz": z}
    b = b200.component_budget(comp, 2, m, st, acc, phi)
    M0, M1 = b["mass"]
    c0, c1 = b["com"]
    dvec = c1 - c0
    dist = np.linalg.norm(dvec)
    want = G * M0 * M1 / dist**2 * dvec / dist
    rms = np.sqrt(np.mean(np.sum((q[:n0] - c0) ** 2, 1))) + np.sqrt(np.mean(np.sum((q[n0:] - c1) ** 2, 1)))
    tol = 3 * (rms / dist) ** 2 * np.linalg.norm(want) + 1e-5 * np.linalg.norm(want)
    assert np.linalg.norm(b["force"][0, 1] - want) <= tol
    assert np.linalg.norm(b["force"][1, 0] + want) <= tol
    assert b["W"][0, 1] < 0 and np.isclose(b["W"][0, 1], b["W"][1, 0], rtol=1e-6)


# ------------------------------------------------------------------------------------------------ state and ordering
@pytest.mark.parametrize("tracers", [False, True])
@pytest.mark.parametrize("integrator", [0, 1])
@pytest.mark.parametrize("steps", [1, 32])  # 32: the cached step-graph path
def test_state_untouched(b200, oracle, integrator, steps, tracers):
    n, C = 5000, 3
    d = oracle.init_bodies("galaxy", n)
    rng = np.random.default_rng(10)
    comp = rng.integers(0, C, n).astype(np.uint32)
    p = _points(d, 1000, rng)
    tr = [(rng.normal(size=700) * 2e8).astype(np.float32) for _ in range(3)] + [np.zeros(700, np.float32)] * 3
    out = []
    for probe in (False, True):
        with _ctx(b200, d) as ctx:
            if tracers:
                ctx.set_tracers(*tr)
            ctx.step(DT, integrator, steps)
            if probe:
                ctx.component_field(comp, C, *p)
                ctx.component_field_bodies(comp, C)
            ctx.step(DT, integrator, steps)
            st = ctx.download_state()
            res = [st[k] for k in ctx._STATE] + list(ctx.download_accel())
            if tracers:
                res += list(ctx.download_tracers().values())
            out.append(res)
    for a, b in zip(*out):
        _same(a, b)


def test_ordered_after_async_step(b200, oracle):
    n, C = 20011, 3
    d = oracle.init_bodies("random", n)
    rng = np.random.default_rng(11)
    comp = rng.integers(0, C, n).astype(np.uint32)
    p = _points(d, 2000, rng)
    res = []
    for join in (False, True):
        with _ctx(b200, d, devices=[0, 0, 0]) as ctx:
            ctx.step(DT, 0, 3)
            if join:
                ctx.sync()
            res.append(ctx.component_field(comp, C, *p) + ctx.component_field_bodies(comp, C))
    for a, b in zip(*res):
        _same(a, b)


def _r(x):
    return (x + 255) // 256 * 256


def test_scratch_and_launches(b200, oracle):
    """growth of allocated_bytes is the header's formula; launches: one pack per call, then two per batch"""
    n, C = 10000, 3
    d = oracle.init_bodies("galaxy", n)
    rng = np.random.default_rng(12)
    comp = rng.integers(0, C, n).astype(np.uint32)
    cnt = np.bincount(comp, minlength=C)
    T = int(np.sum((cnt + 127) // 128 * 128))
    S = int(sum(min(64, max(1, -(-(-(-c // 128)) // 32))) for c in cnt if c))
    B = min(65536, max(1, 2**22 // (512 * S)) * 512)

    def need(bodies, Bc):
        return (_r(16 * S * Bc) + _r(16 * T) + _r(4 * T) + (_r(4 * n) if bodies else 0) + _r(8 * S) + _r(4 * (C + 1))
                + 12 * Bc + 16 * C * Bc)

    with _ctx(b200, d) as ctx, _ctx(b200, d) as ref:
        before, L0 = ctx.allocated_bytes, ctx.launch_count
        ctx.component_field(comp, C, *_points(d, 3 * B, rng))
        assert ctx.launch_count - L0 == 1 + 2 * 3
        assert ctx.allocated_bytes - before == need(False, B)
        L0 = ctx.launch_count
        ctx.component_field(comp, C, *_points(d, 7 * B + 5, rng))
        assert ctx.launch_count - L0 == 1 + 2 * 8
        L0 = ctx.launch_count
        ctx.component_field_bodies(comp, C)
        assert ctx.launch_count - L0 == 1 + 2
        assert ctx.allocated_bytes - before == max(need(False, B), need(True, (b200.slice_length(n, 1) + 511) // 512 * 512))
        L0 = ctx.launch_count
        ctx.component_field(np.full(n, 0xFFFFFFFF, np.uint32), C, *_points(d, 100, rng))
        assert ctx.launch_count - L0 == 1  # no member: the reduction alone
        b0 = ref.launch_count
        ref.step(DT, 0, 1)
        L0 = ctx.launch_count
        ctx.step(DT, 0, 1)
        assert ctx.launch_count - L0 == ref.launch_count - b0


# ------------------------------------------------------------------------------------------------ errors
def test_errors(b200, oracle):
    L = b200.lib()
    n = 1000
    d = oracle.init_bodies("galaxy", n)
    x = np.zeros(4, np.float32)
    xp = x.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
    acc = np.zeros((n, 2, 3), np.float32)
    ap = acc.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
    comp = np.zeros(n, np.uint32)
    up = lambda g: g.ctypes.data_as(ctypes.POINTER(ctypes.c_uint))  # noqa: E731
    with b200.Context(n, G_F32, SOFT) as ctx:
        assert L.b200nb_component_field(ctx._ctx, up(comp), 1, 4, xp, xp, xp, ap, ap) == b200.ESTATE
        assert L.b200nb_component_field_bodies(ctx._ctx, up(comp), 1, ap, ap) == b200.ESTATE
        ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
        assert L.b200nb_component_field(ctx._ctx, None, 1, 4, xp, xp, xp, ap, ap) == b200.EINVAL
        assert L.b200nb_component_field_bodies(ctx._ctx, None, 1, ap, ap) == b200.EINVAL
        for C in (0, 65):
            assert L.b200nb_component_field(ctx._ctx, up(comp), C, 4, xp, xp, xp, ap, ap) == b200.EINVAL
            assert L.b200nb_component_field_bodies(ctx._ctx, up(comp), C, ap, ap) == b200.EINVAL
        bad = comp.copy()
        bad[n - 1] = 2
        assert L.b200nb_component_field(ctx._ctx, up(bad), 2, 4, xp, xp, xp, ap, ap) == b200.EINVAL
        assert L.b200nb_component_field_bodies(ctx._ctx, up(bad), 2, ap, ap) == b200.EINVAL
        bad[n - 1] = 0xFFFFFFFE
        assert L.b200nb_component_field_bodies(ctx._ctx, up(bad), 64, ap, ap) == b200.EINVAL
        for k in range(3):
            pts = [xp, xp, xp]
            pts[k] = None
            assert L.b200nb_component_field(ctx._ctx, up(comp), 1, 4, *pts, ap, ap) == b200.EINVAL
        assert L.b200nb_component_field(ctx._ctx, up(comp), 1, 0, None, None, None, None, None) == b200.OK
        assert L.b200nb_component_field(ctx._ctx, up(comp), 1, 4, xp, xp, xp, None, None) == b200.OK
        assert L.b200nb_component_field_bodies(ctx._ctx, up(comp), 1, None, ap) == b200.OK
        a, f = ctx.component_field(comp, 1, x[:0], x[:0], x[:0])
        assert a.shape == (0, 1, 3) and f.shape == (0, 1)
        for bad_c in (0, 65, 1.0, True):
            with pytest.raises(ValueError):
                ctx.component_field_bodies(comp, bad_c)
        with pytest.raises(ValueError):
            ctx.component_field_bodies(np.full(n, 3, np.uint32), 3)
        with pytest.raises(ValueError):
            ctx.component_field_bodies(comp[:-1], 1)
        with pytest.raises(ValueError):
            ctx.component_field(comp, 1, x, x, x[:3])
