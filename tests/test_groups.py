"""b200nb_group_potential and b200nb_unbind on the GPU: agreement with the fp64 reference (tests/groups_oracle.c), the
analytic two-body case, pass-by-pass unbinding, bitwise invariance over reruns, shards, asynchronous steps and
order-keeping relabellings, edge cases, untouched simulation state, bounded scratch and the error contract."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import DT, G_F32, REPO, SOFT
from groups_oracle import GroupsOracle

pytestmark = pytest.mark.gpu
NO = 0xFFFFFFFF


@pytest.fixture(scope="module")
def goracle():
    return GroupsOracle()


def _ctx(b200, d, **kw):
    ctx = b200.Context(len(d["qx"]), G_F32, SOFT, **kw)
    ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
    return ctx


def _fof_lengths(ctx, d):
    """median first- and sixth-neighbour distances and one above the diameter (the FoF tests' choice)"""
    if len(d["qx"]) < 2:
        return [1.0]
    dist = ctx.neighbors(min(6, len(d["qx"]) - 1))[1]
    bs = [float(np.median(dist[:, 0])), float(np.median(dist[:, -1]))]
    q = np.stack([d["qx"], d["qy"], d["qz"]]).astype(np.float64)
    bs.append(2.01 * float(np.max(np.linalg.norm(q - q.mean(axis=1, keepdims=True), axis=0))) + 1.0)
    return bs


def _label_sets(ctx, d, rng):
    n = len(d["qx"])
    sets = {f"fof{k}": ctx.fof(b) for k, b in enumerate(_fof_lengths(ctx, d))}
    sets["random7"] = rng.integers(0, 7, n).astype(np.uint32)
    sets["one"] = np.full(n, 12345, np.uint32)
    sets["distinct"] = np.arange(n, dtype=np.uint32)
    sets["none"] = np.full(n, NO, np.uint32)
    mix = rng.integers(0, 3, n).astype(np.uint32)
    mix[rng.random(n) < 0.3] = NO
    sets["mix_none"] = mix
    return sets


def _sample(n, rng, k=48):
    return np.unique(np.concatenate([[0, n - 1], rng.integers(0, n, k)])).astype(np.int64)


def _check_phi(got, want, what):
    zero = want == 0
    assert np.all(got[zero] == 0) and not np.any(np.signbit(got[zero])), what  # +0 exactly
    err = np.abs(got[~zero].astype(np.float64) - want[~zero])
    assert np.all(err <= 1e-6 * np.abs(want[~zero])), (what, float(np.max(err / np.abs(want[~zero]))))


# ------------------------------------------------------------------------------------------------ group potential
@pytest.mark.parametrize("scheme", ["galaxy", "random"])
@pytest.mark.parametrize("n", [1, 127, 128, 129, 4097, 30000, 200000])
def test_potential_vs_oracle(b200, oracle, goracle, scheme, n):
    d = oracle.init_bodies(scheme, n)
    rng = np.random.default_rng(n)
    with _ctx(b200, d) as ctx:
        sets = _label_sets(ctx, d, rng)
        for name, g in sets.items():
            got = ctx.group_potential(g)
            idx = _sample(n, rng)
            _check_phi(got[idx], goracle.potential(d, g, idx), name)
            if name in ("distinct", "none"):
                assert np.all(got == 0) and not np.any(np.signbit(got)), name
            if name == "one" and n > 1:
                full = ctx.potential()
                assert np.all(np.abs(got.astype(np.float64) - full) <= 1e-6 * np.abs(full.astype(np.float64)))
            if name == "mix_none":
                assert np.all(got[g == NO] == 0)


@pytest.mark.parametrize("integrator", [0, 1])
def test_potential_after_steps(b200, oracle, goracle, integrator):
    d = oracle.init_bodies("galaxy", 4097)
    with _ctx(b200, d) as ctx:
        ctx.step(DT, integrator, 5)
        st = dict(ctx.download_state(), m=d["m"])
        assert not np.array_equal(st["qx"], d["qx"])
        for b in _fof_lengths(ctx, st)[:2]:
            g = ctx.fof(b)
            _check_phi(ctx.group_potential(g), goracle.potential(st, g), b)


# ------------------------------------------------------------------------------------------------ unbinding
def _moving(b200, oracle, scheme, n, seed):
    """bodies with random velocities of a fifth of the typical escape speed added, so that passes remove some members"""
    d = oracle.init_bodies(scheme, n)
    with _ctx(b200, d) as ctx:
        scale = float(np.sqrt(np.median(np.abs(ctx.potential()))))
    rng = np.random.default_rng(seed)
    for c in ("vx", "vy", "vz"):
        d[c] = (d[c] + rng.normal(size=n) * scale * 0.2).astype(np.float32)
    return d


@pytest.mark.parametrize("scheme,n", [("galaxy", 4097), ("random", 4097), ("galaxy", 30000)])
def test_unbind_pass_by_pass(b200, oracle, goracle, scheme, n):
    d = _moving(b200, oracle, scheme, n, 7)
    with _ctx(b200, d) as ctx:
        g0 = ctx.fof(_fof_lengths(ctx, d)[1])
        cur, k = g0, 0
        for k in range(1, 30):
            bound, phi, it, conv = ctx.unbind(cur, 1)
            assert it == 1
            want_phi, E = goracle.unbind_pass(d, cur)
            mem = cur != NO
            _check_phi(phi[mem], want_phi[mem], f"pass {k}")
            assert np.all(phi[~mem] == 0)
            left = mem & (bound == NO)
            want_left = mem & ~(E < 0)
            close = np.abs(E) <= 1e-5 * np.abs(want_phi)
            assert np.array_equal(left & ~close, want_left & ~close), k
            assert np.array_equal(bound[mem & ~left], cur[mem & ~left])
            if conv:
                assert not np.any(left)
                break
            cur = bound
            if np.all(cur == NO):  # everybody left: the next pass starts from an empty set
                b_e, phi_e, it_e, conv_e = ctx.unbind(cur, 1)
                assert it_e == 0 and conv_e and np.all(b_e == NO) and np.all(phi_e == 0)
                bound, phi, k = b_e, phi_e, k + 1
                conv = True
                break
        assert conv and k > 1
        # the chained passes equal one call of k passes, bit for bit; a converged result is a fixed point
        b_all, phi_all, it_all, conv_all = ctx.unbind(g0, k)
        assert it_all == k and conv_all
        assert np.array_equal(b_all, bound) and np.array_equal(phi_all.view(np.uint32), phi.view(np.uint32))
        b2, phi2, it2, conv2 = ctx.unbind(b_all, 1)
        assert it2 == (1 if np.any(b_all != NO) else 0) and conv2 and np.array_equal(b2, b_all) and np.array_equal(phi2.view(np.uint32), phi_all.view(np.uint32))
        # unbind(unbind(g, 1).bound, 1) == unbind(g, 2)
        one = ctx.unbind(g0, 1)
        two = ctx.unbind(g0, 2)
        chain = ctx.unbind(one[0], 1)
        assert np.array_equal(chain[0], two[0]) and np.array_equal(chain[1].view(np.uint32), two[1].view(np.uint32))
        assert two[2] == 2 and not two[3]


def test_unbind_full_loop_vs_oracle(b200, oracle, goracle):
    d = _moving(b200, oracle, "galaxy", 2049, 3)
    with _ctx(b200, d) as ctx:
        g = ctx.fof(_fof_lengths(ctx, d)[1])
        bound, phi, it, conv = ctx.unbind(g)
    wb, wphi, wit, wconv = goracle.unbind(d, g)
    assert conv and wconv
    assert np.mean(bound == wb) > 0.999 and abs(it - wit) <= 1


def _two_body(m1, m2, u, d=1e9, third=False):
    n = 3 if third else 2
    q = np.zeros((3, n), np.float32)
    q[0, 1] = d
    if third:
        q[1, 2] = 5e12
    v = np.zeros((3, n), np.float32)
    v[1, 1] = u
    dd = {c: q[i] for i, c in enumerate(("qx", "qy", "qz"))}
    dd.update({c: v[i] for i, c in enumerate(("vx", "vy", "vz"))})
    dd["m"] = np.array([m1, m2] + ([1e24] if third else []), np.float32)
    return dd


def test_two_body_threshold(b200):
    m, dist = 1e24, 1e9
    ucrit = np.sqrt(8 * float(G_F32) * m / np.sqrt(dist * dist + SOFT * SOFT))
    for f, stays in ((0.99, True), (1.01, False)):
        d = _two_body(m, m, ucrit * f, dist, third=True)
        with _ctx(b200, d) as ctx:
            bound, phi, it, conv = ctx.unbind(np.array([4, 4, 9], np.uint32))
        assert conv
        if stays:
            assert list(bound) == [4, 4, NO] and it == 2  # the lone body leaves in pass 1
        else:
            assert list(bound) == [NO, NO, NO] and it == 2
    # unequal masses: the light body leaves first, then the heavy one is alone and leaves
    m2 = 1e24
    m1 = 4 * m2
    r = np.sqrt(dist * dist + SOFT * SOFT)
    u = np.sqrt(25 * float(G_F32) * m2 / r)
    d = _two_body(m1, m2, u, dist)
    with _ctx(b200, d) as ctx:
        g = np.array([1, 1], np.uint32)
        b1, _, it1, conv1 = ctx.unbind(g, 1)
        assert list(b1) == [1, NO] and it1 == 1 and not conv1
        b, phi, it, conv = ctx.unbind(g)
        assert list(b) == [NO, NO] and it == 3 and conv and np.all(phi == 0)


# ------------------------------------------------------------------------------------------------ invariance
def test_invariance_bitwise(b200, oracle):
    d = _moving(b200, oracle, "galaxy", 20011, 5)
    res = []
    for k in (1, 2, 3):
        with _ctx(b200, d, devices=[0] * k) as ctx:
            if k == 1:
                g = ctx.fof(_fof_lengths(ctx, d)[1])
                mix = g.copy()
                mix[::5] = NO
            r = (ctx.group_potential(g), ctx.group_potential(mix), ctx.unbind(g, 3), ctx.unbind(mix))
            r2 = (ctx.group_potential(g), ctx.group_potential(mix), ctx.unbind(g, 3), ctx.unbind(mix))
            res.append(r)
            _same(r, r2)
            if k == 1:  # a relabelling that keeps the sorted order
                rel = np.where(g == NO, NO, g.astype(np.uint64) * 3 + 11).astype(np.uint32)
                assert np.array_equal(ctx.group_potential(rel).view(np.uint32), r[0].view(np.uint32))
                b, phi, it, conv = ctx.unbind(rel, 3)
                assert np.array_equal(b, np.where(r[2][0] == NO, NO, r[2][0].astype(np.uint64) * 3 + 11).astype(np.uint32))
                assert np.array_equal(phi.view(np.uint32), r[2][1].view(np.uint32)) and it == r[2][2]
    for r in res[1:]:
        _same(res[0], r)


def _same(a, b):
    assert np.array_equal(a[0].view(np.uint32), b[0].view(np.uint32))
    assert np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32))
    for x, y in ((a[2], b[2]), (a[3], b[3])):
        assert np.array_equal(x[0], y[0]) and np.array_equal(x[1].view(np.uint32), y[1].view(np.uint32)) and x[2:] == y[2:]


def test_ordered_after_async_step(b200, oracle):
    d = _moving(b200, oracle, "random", 20011, 2)
    for devs in ([0], [0, 0, 0]):
        res = []
        for join in (False, True):
            with _ctx(b200, d, devices=devs) as ctx:
                ctx.step(DT, 0, 3)
                if join:
                    ctx.sync()
                g = ctx.fof(_fof_lengths(ctx, d)[1]) if not res else res[0][2]
                res.append((ctx.group_potential(g), ctx.unbind(g), g))
        assert np.array_equal(res[0][0].view(np.uint32), res[1][0].view(np.uint32))
        assert np.array_equal(res[0][1][0], res[1][1][0]) and np.array_equal(res[0][1][1].view(np.uint32), res[1][1][1].view(np.uint32))


def _n_devices():
    import torch
    return torch.cuda.device_count()


def test_two_gpus(b200, oracle):
    if _n_devices() < 2:
        pytest.skip("needs 2 GPUs")
    d = _moving(b200, oracle, "galaxy", 20011, 4)
    res = []
    for devs in ([0], [0, 1]):
        with _ctx(b200, d, devices=devs) as ctx:
            ctx.step(DT, 0, 2)
            if devs == [0]:
                g = ctx.fof(_fof_lengths(ctx, ctx.download_state())[1])
            res.append((ctx.group_potential(g), ctx.unbind(g)))
    assert np.array_equal(res[0][0].view(np.uint32), res[1][0].view(np.uint32))
    assert np.array_equal(res[0][1][0], res[1][1][0]) and np.array_equal(res[0][1][1].view(np.uint32), res[1][1][1].view(np.uint32))


def test_torchrun_ranks():
    if _n_devices() < 2:
        pytest.skip("needs 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29587", os.path.join(REPO, "tests", "mp_groups_parity.py")],
                       capture_output=True, text=True, timeout=600)
    print(r.stdout[-2000:])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert r.stdout.count("ok=True") == 2


# ------------------------------------------------------------------------------------------------ edge cases
def test_zero_mass_members(b200, oracle, goracle):
    d = oracle.init_bodies("random", 3000)
    d["m"] = d["m"].copy()
    d["m"][::3] = 0
    g = np.random.default_rng(1).integers(0, 4, 3000).astype(np.uint32)
    with _ctx(b200, d) as ctx:
        got = ctx.group_potential(g)
    want = goracle.potential(d, g)
    _check_phi(got, want, "zero mass")
    assert np.all(got[::3] < 0)  # they feel the potential


def test_padding_never_contributes(b200, oracle, goracle):
    for n in (129, 257):  # one real body in the last AoSoA block; the padding sits on it
        d = oracle.init_bodies("random", n)
        g = np.zeros(n, np.uint32)
        g[-1] = 5
        with _ctx(b200, d) as ctx:
            got = ctx.group_potential(g)
        assert got[-1] == 0 and not np.signbit(got[-1])
        _check_phi(got, goracle.potential(d, g), n)


def test_non_finite_body(b200, oracle, goracle):
    d = oracle.init_bodies("galaxy", 2049)
    d["qx"] = d["qx"].copy()
    d["qx"][700] = np.nan
    g = (np.arange(2049) % 3).astype(np.uint32)  # body 700 has label 1
    with _ctx(b200, d) as ctx:
        phi = ctx.group_potential(g)
        assert np.all(np.isnan(phi[g == 1])) and np.all(np.isfinite(phi[g != 1]))
        bound = ctx.unbind(g)[0]
        assert np.all(bound[g == 1] == NO)
        # through friends-of-friends labels the body is alone: it leaves, nobody else is affected
        f = ctx.fof(_fof_lengths(ctx, d)[1])
        assert f[700] == 700 and np.sum(f == 700) == 1
        phi_f = ctx.group_potential(f)
        assert phi_f[700] == 0 and np.all(np.isfinite(phi_f))
        bf = ctx.unbind(f)[0]
        assert bf[700] == NO
    _check_phi(phi_f, goracle.potential(d, f), "fof labels")  # the other groups are untouched


# ------------------------------------------------------------------------------------------------ contract
@pytest.mark.parametrize("integrator", [0, 1])
@pytest.mark.parametrize("steps", [1, 32])  # 32: the cached step-graph path
def test_state_untouched(b200, oracle, integrator, steps):
    d = oracle.init_bodies("galaxy", 5000)
    g = (np.arange(5000) % 4).astype(np.uint32)
    out = []
    for probe in (False, True):
        with _ctx(b200, d) as ctx:
            ctx.step(DT, integrator, steps)
            if probe:
                ctx.group_potential(g)
                ctx.unbind(g)
            ctx.step(DT, integrator, steps)
            st = ctx.download_state()
            out.append([st[k] for k in ctx._STATE] + list(ctx.download_accel()))
    for a, b in zip(out[0], out[1]):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.mark.parametrize("shards", [1, 3])
def test_scratch_and_launches(b200, oracle, shards):
    n = 10000
    d = oracle.init_bodies("galaxy", n)
    g = (np.arange(n) % 5).astype(np.uint32)
    with _ctx(b200, d, devices=[0] * shards) as ctx:
        n_pad = shards * b200.slice_length(n, shards)
        before, launches = ctx.allocated_bytes, ctx.launch_count
        ctx.group_potential(g)
        grown = ctx.allocated_bytes
        cap = -(-n // 1024) * 1024
        assert 0 < grown - before <= shards * (102 * n + 16 * n_pad + 20 * 256 + 4 * 64 * cap + (16 << 20)), grown - before
        first = ctx.launch_count - launches
        if shards == 1:  # iota, sort, members, pack; potential + reduce; finish
            assert first == 7, first
        ctx.unbind(g)
        ctx.group_potential(np.full(n, NO, np.uint32))
        ctx.unbind(np.arange(n, dtype=np.uint32), 5)
        assert ctx.allocated_bytes == grown
        l0 = ctx.launch_count
        ctx.group_potential(g)
        assert ctx.launch_count - l0 == first


def test_errors(b200, oracle):
    L = b200.lib()
    n = 1000
    d = oracle.init_bodies("galaxy", n)
    g = np.zeros(n, np.uint32)
    phi = np.empty(n, np.float32)
    bound = np.empty(n, np.uint32)
    UP, FP = ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(ctypes.c_float)
    gp, pp, bp = g.ctypes.data_as(UP), phi.ctypes.data_as(FP), bound.ctypes.data_as(UP)
    it, conv = ctypes.c_uint(), ctypes.c_int()
    with b200.Context(n, G_F32, SOFT) as ctx:
        assert L.b200nb_group_potential(ctx._ctx, gp, pp) == b200.ESTATE
        assert L.b200nb_unbind(ctx._ctx, gp, 1, bp, pp, ctypes.byref(it), ctypes.byref(conv)) == b200.ESTATE
        ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
        assert L.b200nb_group_potential(ctx._ctx, None, pp) == b200.EINVAL
        assert L.b200nb_group_potential(ctx._ctx, gp, None) == b200.EINVAL
        assert L.b200nb_unbind(ctx._ctx, None, 1, bp, pp, None, None) == b200.EINVAL
        assert L.b200nb_unbind(ctx._ctx, gp, 1, None, pp, None, None) == b200.EINVAL
        assert L.b200nb_unbind(ctx._ctx, gp, 0, bp, pp, None, None) == b200.EINVAL
        assert L.b200nb_unbind(ctx._ctx, gp, 2, bp, None, None, None) == b200.OK
        assert L.b200nb_unbind(ctx._ctx, gp, 2, bp, pp, ctypes.byref(it), ctypes.byref(conv)) == b200.OK
        assert 1 <= it.value <= 2
        for bad in (np.zeros(n - 1, np.uint32), np.zeros((n, 1), np.uint32), np.zeros(n, np.float32), np.full(n, -1),
                    np.full(n, 2**32, np.int64), np.zeros(n, bool)):
            with pytest.raises(ValueError):
                ctx.group_potential(bad)
            with pytest.raises(ValueError):
                ctx.unbind(bad)
        for bad in (0, -1, 2**32, 1.0, True):
            with pytest.raises(ValueError):
                ctx.unbind(g, bad)
    assert L.b200nb_group_potential(None, gp, pp) == b200.EINVAL
    assert L.b200nb_unbind(None, gp, 1, bp, pp, None, None) == b200.EINVAL
