"""b200nb_scf_coefficients and b200nb_scf_field on the GPU: agreement with the long-double restatement (tests/scf_oracle.c)
within the header's bound, bit-identity over reruns, shards, ranks, asynchronous and graph-replayed steps, relabelling
and truncation, locality of the evaluator, the physics of Hernquist and flattened samples against b200nb_field, the
gradient, the centre and the z axis, symmetries and linearity, edge cases, untouched state, scratch, launches and
errors."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import DT, G_F32, REPO
from scf_oracle import ScfOracle
from test_scf_cpu import A_SCALE, hernquist_sample

pytestmark = pytest.mark.gpu
SOFT = 1e-6 * A_SCALE
KEYS = ("qx", "qy", "qz", "vx", "vy", "vz")


@pytest.fixture(scope="module")
def so():
    return ScfOracle()


def _system(n, seed, flatten=(1.0, 0.8, 0.5), offset=(0.15, -0.1, 0.05), zero_v=False):
    q = hernquist_sample(n, A_SCALE, seed, flatten=flatten, offset=offset)
    rng = np.random.default_rng(seed + 11)
    d = {"qx": q[0], "qy": q[1], "qz": q[2], "m": (rng.random(n) * 2e29 + 1e29).astype(np.float32)}
    for c in ("vx", "vy", "vz"):
        d[c] = np.zeros(n, np.float32) if zero_v else (rng.normal(size=n) * 1e5).astype(np.float32)
    return d


def _ctx(b200, d, G=G_F32, **kw):
    ctx = b200.Context(len(d["qx"]), G, SOFT, **kw)
    ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
    return ctx


def _gm(d, G=G_F32):
    return (np.float32(G) * d["m"].astype(np.float32)).astype(np.float32)


def _bits(*arrs):
    return [np.ascontiguousarray(a).view(np.uint64).copy() for a in arrs]


def _same(x, y):
    return all(np.array_equal(a, b) for a, b in zip(_bits(*x), _bits(*y)))


CENTRE = (0.1 * A_SCALE, -0.05 * A_SCALE, 0.02 * A_SCALE)


# ------------------------------------------------------------------------------------------------ accuracy
@pytest.mark.parametrize("n,nmax,lmax", [(1, 0, 0), (127, 6, 4), (129, 31, 15), (1000, 10, 6), (2500, 31, 15), (20000, 10, 6)])
def test_coefficients_vs_oracle(b200, so, n, nmax, lmax):
    d = _system(n, n)
    with _ctx(b200, d) as ctx:
        S, T = ctx.scf_coefficients(nmax, lmax, A_SCALE, CENTRE)
    S0, T0, Ss, Ts = so.coefficients([d["qx"], d["qy"], d["qz"]], _gm(d), nmax, lmax, A_SCALE, CENTRE)
    assert np.all(np.abs(S - S0) <= 1e-12 * Ss), np.max(np.abs(S - S0) / np.maximum(Ss, 1e-300))
    assert np.all(np.abs(T - T0) <= 1e-12 * Ts), np.max(np.abs(T - T0) / np.maximum(Ts, 1e-300))
    iu = np.triu_indices(lmax + 1, 1)
    assert np.all(S[:, iu[0], iu[1]] == 0) and np.all(T[:, :, 0] == 0)


def _points(m, seed, lo=0.05, hi=8.0, centre=CENTRE):
    rng = np.random.default_rng(seed)
    x = rng.normal(size=(m, 3))
    x *= (rng.uniform(lo, hi, m) / np.linalg.norm(x, axis=1))[:, None] * A_SCALE
    x += np.asarray(centre)
    return [x[:, k].astype(np.float32) for k in range(3)]


@pytest.mark.parametrize("nmax,lmax", [(0, 0), (8, 6), (31, 15)])
def test_field_vs_oracle(b200, so, nmax, lmax):
    d = _system(3000, 5)
    p = _points(777, 6)
    with _ctx(b200, d) as ctx:
        S, T = ctx.scf_coefficients(nmax, lmax, A_SCALE, CENTRE)
        ax, ay, az, phi = ctx.scf_field(S, T, A_SCALE, CENTRE, *p)
    ox, oy, oz, ophi, sa, sphi = so.field(S, T, A_SCALE, CENTRE, *p)
    assert np.all(np.abs(phi - ophi) <= 1e-12 * sphi)
    for k, (g, o) in enumerate(((ax, ox), (ay, oy), (az, oz))):
        assert np.all(np.abs(g - o) <= 1e-12 * sa[k]), k


# ------------------------------------------------------------------------------------------------ bit-identity
def test_truncation_is_a_sub_block(b200):
    d = _system(20000, 3)
    with _ctx(b200, d) as ctx:
        S, T = ctx.scf_coefficients(31, 15, A_SCALE, CENTRE)
        for nm, lm in ((0, 0), (10, 6), (24, 12), (31, 0), (0, 15), (5, 15), (31, 14)):
            s, t = ctx.scf_coefficients(nm, lm, A_SCALE, CENTRE)
            assert _same((s, t), (S[:nm + 1, :lm + 1, :lm + 1], T[:nm + 1, :lm + 1, :lm + 1])), (nm, lm)


def test_shards_reruns_and_labels(b200):
    d = _system(20011, 4)
    n = len(d["qx"])
    rng = np.random.default_rng(0)
    grp = rng.integers(0, 3, n).astype(np.uint32)
    res = []
    for devs in ([0], [0, 0], [0, 0, 0], [0] * 8):
        with _ctx(b200, d, devices=devs) as ctx:
            r = [ctx.scf_coefficients(8, 6, A_SCALE, CENTRE), ctx.scf_coefficients(8, 6, A_SCALE, CENTRE),
                 ctx.scf_coefficients(8, 6, A_SCALE, CENTRE, group=np.full(n, 7, np.uint32), label=7),
                 ctx.scf_coefficients(8, 6, A_SCALE, CENTRE, group=grp, label=1)]
            other = np.where(grp == 1, 1, rng.integers(2, 2 ** 32 - 1, n)).astype(np.uint32)  # non-members relabelled
            r.append(ctx.scf_coefficients(8, 6, A_SCALE, CENTRE, group=other, label=1))
            res.append(r)
    for r in res:
        assert _same(r[0], r[1]) and _same(r[0], r[2]) and _same(r[3], r[4])
        assert _same(r[0], res[0][0]) and _same(r[3], res[0][3])


@pytest.mark.parametrize("integrator", [0, 1])
def test_after_async_steps_and_graphs(b200, integrator):
    """Right after an asynchronous step (and 64 graph-replayed ones), the coefficients are those of the positions the
    steps leave, bit for bit, and the call changes nothing: the run continues exactly as a twin that never called it."""
    d = _system(20000, 8)
    for devs in ([0], [0, 0, 0]):
        with _ctx(b200, d, devices=devs) as a, _ctx(b200, d, devices=devs) as b:
            for steps in (1, 64):
                a.step(DT, integrator, steps)
                got = a.scf_coefficients(6, 4, A_SCALE, CENTRE)
                a.step(DT, integrator, 1)
                b.step(DT, integrator, steps)
                st = b.download_state()
                b.step(DT, integrator, 1)
                with _ctx(b200, {**st, "m": d["m"]}) as c:
                    assert _same(c.scf_coefficients(6, 4, A_SCALE, CENTRE), got)
            sa, sb = a.download_state(), b.download_state()
            assert all(np.array_equal(sa[k], sb[k]) for k in KEYS)
            assert all(np.array_equal(x, y) for x, y in zip(a.download_accel(), b.download_accel()))


def test_field_locality(b200):
    d = _system(5000, 9)
    p = _points(3000, 10)
    with _ctx(b200, d) as ctx:
        S, T = ctx.scf_coefficients(12, 8, A_SCALE, CENTRE)
        full = ctx.scf_field(S, T, A_SCALE, CENTRE, *p)
        perm = np.random.default_rng(1).permutation(3000)
        shuf = ctx.scf_field(S, T, A_SCALE, CENTRE, *[x[perm] for x in p])
        part = ctx.scf_field(S, T, A_SCALE, CENTRE, *[x[1000:1300] for x in p])
        one = ctx.scf_field(S, T, A_SCALE, CENTRE, *[x[5:6] for x in p])
    assert _same([f[perm] for f in full], shuf)
    assert _same([f[1000:1300] for f in full], part) and _same([f[5:6] for f in full], one)


def test_field_batches(b200):
    """2^20 points per launch: 2^20 + 300 points go through two launches and agree with one-point calls."""
    S = np.zeros((3, 3, 3))
    S[0, 0, 0], S[1, 2, 1], S[2, 1, 1] = 1e12, 3e10, -2e10
    T = np.zeros_like(S)
    T[1, 2, 2] = 1e10
    m = (1 << 20) + 300
    p = _points(m, 11)
    with b200.Context(1, G_F32, SOFT) as ctx:  # allowed before an upload
        l0 = ctx.launch_count
        full = ctx.scf_field(S, T, A_SCALE, CENTRE, *p)
        assert ctx.launch_count - l0 == 2
        for i in (0, (1 << 20) - 1, 1 << 20, m - 1):
            assert _same([f[i:i + 1] for f in full], ctx.scf_field(S, T, A_SCALE, CENTRE, *[x[i:i + 1] for x in p]))


# ------------------------------------------------------------------------------------------------ physics
def test_hernquist_sphere(b200):
    n, GM = 200000, 4e20
    q = hernquist_sample(n, A_SCALE, 1, rmax=np.inf)
    d = {"qx": q[0], "qy": q[1], "qz": q[2], "m": np.full(n, GM / n, np.float32)}
    for c in ("vx", "vy", "vz"):
        d[c] = np.zeros(n, np.float32)
    with _ctx(b200, d, G=1.0) as ctx:
        S, T = ctx.scf_coefficients(2, 2, A_SCALE)
    M = float(np.sum(d["m"].astype(np.float64)))
    assert abs(S[0, 0, 0] / (M / A_SCALE) - 1) < 5e-3
    assert np.abs(S).ravel()[1:].max() < 2e-2 * M / A_SCALE and np.abs(T).max() < 2e-2 * M / A_SCALE


def test_flattened_sample_vs_direct_summation(b200):
    d = _system(20000, 1, zero_v=True)
    q = np.stack([d["qx"], d["qy"], d["qz"]], axis=1).astype(np.float64)
    keep = np.linalg.norm(q - np.array([0.15, -0.1, 0.05]) * A_SCALE, axis=1) < 50 * A_SCALE
    d = {k: v[keep] for k, v in d.items()}
    p = _points(200, 12, lo=0.3, hi=5.0, centre=(0, 0, 0))
    with _ctx(b200, d) as ctx:
        S, T = ctx.scf_coefficients(16, 8, A_SCALE)
        phi = ctx.scf_field(S, T, A_SCALE, (0, 0, 0), *p)[3]
        direct = ctx.field(*p)[3].astype(np.float64)
        S0, T0 = ctx.scf_coefficients(16, 0, A_SCALE)
        phi0 = ctx.scf_field(S0, T0, A_SCALE, (0, 0, 0), *p)[3]
    rel = np.abs(phi / direct - 1)
    assert np.median(rel) < 2e-3 and rel.max() < 1e-2, (np.median(rel), rel.max())
    assert np.abs(phi0 / direct - 1).max() > 5e-2  # the monopole alone misses: l, m > 0 carry the shape


def test_gradient_vs_finite_differences(b200):
    d = _system(5000, 13)
    p = _points(300, 14, lo=0.3, hi=5.0)
    h = 2.0 ** np.floor(np.log2(A_SCALE * 1e-4))  # the divisor is the fp64 difference of the two fp32 points
    with _ctx(b200, d) as ctx:
        S, T = ctx.scf_coefficients(12, 8, A_SCALE, CENTRE)
        a3 = ctx.scf_field(S, T, A_SCALE, CENTRE, *p)[:3]
        scale = np.abs(ctx.scf_field(S, T, A_SCALE, CENTRE, *p)[3]) / A_SCALE
        for k in range(3):
            pp, pm = list(p), list(p)
            pp[k] = (p[k].astype(np.float64) + h).astype(np.float32)
            pm[k] = (p[k].astype(np.float64) - h).astype(np.float32)
            dx = pp[k].astype(np.float64) - pm[k].astype(np.float64)
            fd = -(ctx.scf_field(S, T, A_SCALE, CENTRE, *pp)[3] - ctx.scf_field(S, T, A_SCALE, CENTRE, *pm)[3]) / dx
            assert np.all(np.abs(fd - a3[k]) <= 1e-5 * scale + 1e-4 * np.abs(a3[k])), k


def test_centre_and_z_axis(b200):
    d = _system(5000, 15)
    c = (0.0, 0.0, 0.0)
    z = np.array([0.0, 0.01, 0.3, 1.0, 4.0, -0.5, -2.0]) * A_SCALE
    with _ctx(b200, d) as ctx:
        S, T = ctx.scf_coefficients(12, 8, A_SCALE, c)
        zero = np.zeros(len(z), np.float32)
        on = ctx.scf_field(S, T, A_SCALE, c, zero, zero, z.astype(np.float32))
        off = ctx.scf_field(S, T, A_SCALE, c, (1e-6 * np.abs(z)).astype(np.float32), zero, z.astype(np.float32))
        ctr = ctx.scf_field(S, T, A_SCALE, c, np.zeros(1, np.float32), np.zeros(1, np.float32), np.zeros(1, np.float32))
        near = ctx.scf_field(S, T, A_SCALE, c, *[np.full(1, 1e-6 * A_SCALE, np.float32)] * 3)
    assert all(np.all(np.isfinite(f)) for f in on + ctr)
    assert ctr[0][0] == 0 and ctr[1][0] == 0 and ctr[2][0] == 0
    assert abs(ctr[3][0] / near[3][0] - 1) < 1e-5
    amag = np.sqrt(sum(f[1:] ** 2 for f in on[:3]))
    for k in range(3):
        assert np.all(np.abs(on[k][1:] - off[k][1:]) <= 1e-4 * amag), k
    assert np.all(np.abs(on[3] / off[3] - 1) < 1e-5)


# ------------------------------------------------------------------------------------------------ symmetries, linearity
def test_rotation_reflection_and_linearity(b200, so):
    d = _system(4000, 16, offset=(0.2, 0.1, -0.1))
    c = (0.0, 0.0, 0.0)
    nmax, lmax = 10, 8
    q = [d["qx"], d["qy"], d["qz"]]
    _, _, Ss, Ts = so.coefficients(q, _gm(d), nmax, lmax, A_SCALE, c)
    tol = 3e-12 * (Ss + Ts) + 1e-300
    m = np.arange(lmax + 1)[None, None, :]
    l = np.arange(lmax + 1)[None, :, None]
    with _ctx(b200, d) as ctx:
        S, T = ctx.scf_coefficients(nmax, lmax, A_SCALE, c)
    rot = dict(d, qx=-d["qy"], qy=d["qx"].copy())
    with _ctx(b200, rot) as ctx:
        Sr, Tr = ctx.scf_coefficients(nmax, lmax, A_SCALE, c)
    ca, sa = np.round(np.cos(m * np.pi / 2)), np.round(np.sin(m * np.pi / 2))
    assert np.all(np.abs(Sr - (S * ca - T * sa)) <= tol) and np.all(np.abs(Tr - (S * sa + T * ca)) <= tol)
    ref = dict(d, qz=-d["qz"])
    with _ctx(b200, ref) as ctx:
        Sz, Tz = ctx.scf_coefficients(nmax, lmax, A_SCALE, c)
    sign = (-1.0) ** (l + m)
    assert np.all(np.abs(Sz - sign * S) <= tol) and np.all(np.abs(Tz - sign * T) <= tol)
    g = np.random.default_rng(2).integers(0, 3, len(d["qx"])).astype(np.uint32)
    with _ctx(b200, d) as ctx:
        parts = [ctx.scf_coefficients(nmax, lmax, A_SCALE, c, group=g, label=k) for k in (0, 1)]
        both = ctx.scf_coefficients(nmax, lmax, A_SCALE, c, group=np.where(g < 2, 0, 2).astype(np.uint32), label=0)
    for k in range(2):
        assert np.all(np.abs(parts[0][k] + parts[1][k] - both[k]) <= tol)


# ------------------------------------------------------------------------------------------------ edge cases
def test_zero_mass_and_non_finite(b200):
    n = 3000
    d = _system(n, 17)
    z = dict(d, m=np.zeros(n, np.float32))
    with _ctx(b200, z) as ctx:
        S, T = ctx.scf_coefficients(31, 15, A_SCALE, CENTRE)
    assert np.all(S == 0) and np.all(T == 0)
    bad = {k: v.copy() for k, v in d.items()}
    bad["qy"][100], bad["qz"][2000] = np.nan, np.inf
    grp = np.zeros(n, np.uint32)
    grp[[100, 2000]] = 1
    lm = np.tril(np.ones((9, 9), bool))
    with _ctx(b200, bad) as ctx, _ctx(b200, d) as good:
        S, T = ctx.scf_coefficients(6, 8, A_SCALE, CENTRE)
        assert np.all(np.isnan(S[:, lm])) and np.all(np.isnan(T[:, lm & (np.arange(9)[None, :] > 0)]))
        assert np.all(T[:, :, 0] == 0)
        others = ctx.scf_coefficients(6, 8, A_SCALE, CENTRE, group=grp, label=0)
        g2 = good.scf_coefficients(6, 8, A_SCALE, CENTRE, group=grp, label=0)
        assert _same(others, g2)  # non-members at non-finite positions take no part
        nanp = ctx.scf_field(np.ones_like(S), np.zeros_like(T), A_SCALE, CENTRE, np.array([np.nan, 3 * A_SCALE], np.float32),
                             np.zeros(2, np.float32), np.zeros(2, np.float32))
        assert np.all(np.isnan([f[0] for f in nanp])) and np.all(np.isfinite([f[1] for f in nanp]))


def test_body_at_the_centre(b200, so):
    d = _system(257, 18)
    for k in ("qx", "qy", "qz"):
        d[k][[0, 128, 256]] = 0.0
    with _ctx(b200, d) as ctx:
        S, T = ctx.scf_coefficients(8, 6, A_SCALE)
    assert np.all(np.isfinite(S)) and np.all(np.isfinite(T))
    S0, T0, Ss, Ts = so.coefficients([d["qx"], d["qy"], d["qz"]], _gm(d), 8, 6, A_SCALE)
    assert np.all(np.abs(S - S0) <= 1e-12 * Ss) and np.all(np.abs(T - T0) <= 1e-12 * Ts)


def test_state_scratch_launches_and_errors(b200):
    n = 20000
    d = _system(n, 19)
    with b200.Context(n, G_F32, SOFT) as ctx:
        with pytest.raises(b200.B200Error) as e:
            ctx.scf_coefficients(2, 2, A_SCALE)
        assert e.value.code == b200.ESTATE
        ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
        ctx.step(DT, 1, 2)
        before = ctx.download_state(), ctx.download_accel()
        b0, l0 = ctx.allocated_bytes, ctx.launch_count
        ctx.scf_coefficients(31, 15, A_SCALE)
        assert ctx.launch_count - l0 == 2
        grown = ctx.allocated_bytes - b0
        K, C = 32 * 136, min(512, -(-n // 64))
        r = lambda x: -(-x // 256) * 256  # noqa: E731
        assert 0 <= grown <= r(12952) + r(8 * K) + r(16 * K) + r(16 * K * C) + r(4 * n)
        b1 = ctx.allocated_bytes
        ctx.scf_coefficients(31, 15, A_SCALE, group=np.zeros(n, np.uint32))
        ctx.scf_coefficients(10, 6, A_SCALE)
        assert ctx.allocated_bytes - b1 <= r(4 * n)
        after = ctx.download_state(), ctx.download_accel()
        assert all(np.array_equal(before[0][k], after[0][k]) for k in KEYS)
        assert all(np.array_equal(x, y) for x, y in zip(before[1], after[1]))
        L = b200.lib()
        cen = (ctypes.c_double * 3)(0, 0, 0)
        bad_c = (ctypes.c_double * 3)(0, float("nan"), 0)
        S = (ctypes.c_double * 4352)()
        f = np.zeros(1, np.float32).ctypes.data_as(ctypes.POINTER(ctypes.c_float))
        for args in ((32, 0, A_SCALE, cen, S, S), (0, 16, A_SCALE, cen, S, S), (0, 0, 0.0, cen, S, S), (0, 0, -1.0, cen, S, S),
                     (0, 0, float("inf"), cen, S, S), (0, 0, float("nan"), cen, S, S), (0, 0, A_SCALE, None, S, S),
                     (0, 0, A_SCALE, bad_c, S, S), (0, 0, A_SCALE, cen, None, S), (0, 0, A_SCALE, cen, S, None)):
            nm, lm, a, c, s_, t_ = args
            assert L.b200nb_scf_coefficients(ctx._ctx, nm, lm, a, c, None, 0, s_, t_) == b200.EINVAL, args
            assert L.b200nb_scf_field(ctx._ctx, nm, lm, a, c, s_, t_, 1, f, f, f, None, None, None, None) == b200.EINVAL, args
        assert L.b200nb_scf_field(ctx._ctx, 0, 0, A_SCALE, cen, S, S, 1, None, f, f, None, None, None, None) == b200.EINVAL
        assert L.b200nb_scf_field(ctx._ctx, 0, 0, A_SCALE, cen, S, S, 0, None, None, None, None, None, None, None) == b200.OK


def _n_devices():
    import torch
    return torch.cuda.device_count()


def test_two_gpus(b200):
    if _n_devices() < 2:
        pytest.skip("needs 2 GPUs")
    d = _system(20011, 20)
    res = []
    for devs in ([0], [0, 1], [1, 0]):
        with _ctx(b200, d, devices=devs) as ctx:
            res.append(ctx.scf_coefficients(10, 6, A_SCALE, CENTRE))
    assert _same(res[0], res[1]) and _same(res[0], res[2])


def test_torchrun_ranks():
    if _n_devices() < 2:
        pytest.skip("needs 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29591", os.path.join(REPO, "tests", "mp_scf_parity.py")],
                       capture_output=True, text=True, timeout=600)
    print(r.stdout[-2000:])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert r.stdout.count("ok=True") == 4
