"""b200nb_neighbors / b200nb_neighbors_at on the GPU: bit-exact agreement with the CPU restatement of the definition
(tests/neighbors_oracle.c), bitwise invariance (reruns, k, batching, shards, ranks), edge cases, untouched simulation
state, ordering after an asynchronous step, bounded scratch and the error contract."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import DT, G_F32, REPO, SOFT
from neighbors_oracle import NONE, NeighborsOracle

pytestmark = pytest.mark.gpu

BATCH_K32 = 65536  # targets per launch at k in (16, 32]: nb_batch(32) in csrc/neighbors_sm100.cuh


@pytest.fixture(scope="module")
def noracle():
    return NeighborsOracle()


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


def _points(d, M, rng):
    """M points: inside the system, far outside it (10^3 system radii), exactly on a body, and on body 0 (the galaxy's
    central body)."""
    q = np.stack([d["qx"], d["qy"], d["qz"]]).astype(np.float64)
    R = max(float(np.max(np.linalg.norm(q, axis=0))), 1e8)
    kind = rng.integers(0, 4, M)
    kind[: min(M, 4)] = np.arange(min(M, 4))[::-1]
    u = rng.normal(size=(3, M))
    u /= np.linalg.norm(u, axis=0)
    p = u * np.where(kind == 0, R * rng.random(M) ** (1 / 3), 1e3 * R)
    on = rng.integers(0, q.shape[1], M)
    p[:, kind == 2] = q[:, on[kind == 2]]
    p[:, kind == 3] = q[:, [0]]
    return [p[k].astype(np.float32) for k in range(3)]


def _same(a, b):
    assert a[0].shape == b[0].shape
    assert np.array_equal(a[0], b[0])
    assert np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32))


def _check_bodies(ctx, noracle, d, k, rng, sample=2000):
    n = len(d["qx"])
    got = ctx.neighbors(k)
    if n <= 4096:
        _same(got, noracle.bodies(d, k))
        return got
    sel = np.unique(np.concatenate([[0, 1, 127, 128, n - 129, n - 1], rng.integers(0, n, sample)])).astype(np.uint64)
    _same((got[0][sel.astype(np.int64)], got[1][sel.astype(np.int64)]), noracle.bodies(d, k, sel))
    return got


# ------------------------------------------------------------------------------------------------ exact agreement
@pytest.mark.parametrize("scheme", ["galaxy", "random"])
@pytest.mark.parametrize("n", [1, 2, 129, 2049, 200000])
def test_bit_exact_vs_restatement(b200, oracle, noracle, scheme, n):
    d = oracle.init_bodies(scheme, n)
    rng = np.random.default_rng(n)
    M = 2000 if n > 4096 else 700
    p = _points(d, M, rng)
    with _ctx(b200, d) as ctx:
        for k in (1, 6, 8, 16, 32):
            _check_bodies(ctx, noracle, d, k, rng)
            _same(ctx.neighbors_at(*p, k), noracle.points(d, *p, k))


@pytest.mark.parametrize("integrator", [0, 1])
def test_bit_exact_after_steps(b200, oracle, noracle, integrator):
    n = 2049
    d = oracle.init_bodies("galaxy", n)
    with _ctx(b200, d) as ctx:
        ctx.step(DT, integrator, 5)
        st = ctx.download_state()
        moved = {c: st[c] for c in ("qx", "qy", "qz")}
        assert not np.array_equal(moved["qx"], d["qx"])
        p = _points(moved, 500, np.random.default_rng(9))
        for k in (1, 8, 32):
            _same(ctx.neighbors(k), noracle.bodies(moved, k))
            _same(ctx.neighbors_at(*p, k), noracle.points(moved, *p, k))


# ------------------------------------------------------------------------------------------------ invariance
def test_bitwise_reruns_k_prefix_and_batches(b200, oracle):
    n = 20000
    d = oracle.init_bodies("galaxy", n)
    p = _points(d, BATCH_K32 + 4000, np.random.default_rng(3))
    with _ctx(b200, d) as ctx:
        full = ctx.neighbors(32)
        _same(full, ctx.neighbors(32))  # rerun
        for k in (1, 3, 6, 8, 12, 16, 20):
            _same(ctx.neighbors(k), (full[0][:, :k].copy(), full[1][:, :k].copy()))
        big = ctx.neighbors_at(*p, 32)  # crosses the batch boundary at k = 32
        sel = np.array([0, 1, 127, 128, BATCH_K32 - 1, BATCH_K32, BATCH_K32 + 1, len(p[0]) - 1])
        for i in sel:
            _same(ctx.neighbors_at(*[a[i:i + 1] for a in p], 32), (big[0][i:i + 1], big[1][i:i + 1]))
        shifted = ctx.neighbors_at(*[a[7:BATCH_K32 + 300] for a in p], 32)
        _same(shifted, (big[0][7:BATCH_K32 + 300], big[1][7:BATCH_K32 + 300]))
        small = ctx.neighbors_at(*p, 3)  # another bucket: other batch size, tile and chunk count
        _same(small, (big[0][:, :3].copy(), big[1][:, :3].copy()))


def test_bitwise_virtual_shards(b200, oracle):
    n = 20011
    d = oracle.init_bodies("random", n)
    p = _points(d, 3001, np.random.default_rng(4))
    res = []
    for k in (1, 2, 3):
        with _ctx(b200, d, devices=[0] * k) as ctx:
            res.append((ctx.neighbors(8), ctx.neighbors_at(*p, 8)))
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
    p = _points(d, 3001, np.random.default_rng(5))
    res = []
    for devs in ([0], [0, 1]):
        with _ctx(b200, d, devices=devs) as ctx:
            ctx.step(DT, 0, 2)
            res.append((ctx.neighbors(8), ctx.neighbors_at(*p, 8)))
    _same(res[0][0], res[1][0])
    _same(res[0][1], res[1][1])


def test_bitwise_torchrun_ranks():
    if _n_devices() < 2:
        pytest.skip("needs 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29581", os.path.join(REPO, "tests", "mp_neighbors_parity.py")],
                       capture_output=True, text=True, timeout=600)
    print(r.stdout[-2000:])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert r.stdout.count("ok=True") == 2


# ------------------------------------------------------------------------------------------------ edge cases
def test_single_body_gives_empty_slots(b200, oracle):
    d = oracle.init_bodies("galaxy", 1)
    with _ctx(b200, d) as ctx:
        idx, dist = ctx.neighbors(5)
        assert np.all(idx == NONE) and np.all(np.isinf(dist))
        idx, dist = ctx.neighbors_at([1.0], [2.0], [3.0], 3)
        assert idx[0, 0] == 0 and np.all(idx[0, 1:] == NONE) and np.all(np.isinf(dist[0, 1:]))


def test_k_above_n_pads_with_empty_slots(b200, oracle, noracle):
    d = oracle.init_bodies("random", 9)
    with _ctx(b200, d) as ctx:
        idx, dist = ctx.neighbors(20)
        _same((idx, dist), noracle.bodies(d, 20))
        assert np.all(idx[:, 8:] == NONE) and np.all(np.isinf(dist[:, 8:])) and np.all(idx[:, :8] < 9)
        pidx, _ = ctx.neighbors_at(*[np.zeros(2, np.float32)] * 3, 12)
        assert np.all(pidx[:, 9:] == NONE) and np.all(pidx[:, :9] < 9)


def test_coincident_bodies_by_index(b200, noracle):
    q = np.zeros((3, 7))
    q[0] = [1e9, -2e9, 1e9, 1e9, 5e9, 1e9, -2e9]
    d = _bodies(q)
    with _ctx(b200, d) as ctx:
        idx, dist = ctx.neighbors(4)
        _same((idx, dist), noracle.bodies(d, 4))
        assert list(idx[0]) == [2, 3, 5, 1] and list(dist[0][:3]) == [0, 0, 0]
        assert list(idx[3][:3]) == [0, 2, 5]
        pidx, pdist = ctx.neighbors_at([1e9], [0.0], [0.0], 4)
        assert list(pidx[0]) == [0, 2, 3, 5] and np.all(pdist == 0)


def test_lattice_ties_in_index_order(b200, noracle):
    g = np.arange(5, dtype=np.float64) * 1e8
    X, Y, Z = np.meshgrid(g, g, g, indexing="ij")
    d = _bodies(np.stack([X.ravel(), Y.ravel(), Z.ravel()]))
    with _ctx(b200, d) as ctx:
        idx, dist = ctx.neighbors(6)
        _same((idx, dist), noracle.bodies(d, 6))
        c = 2 * 25 + 2 * 5 + 2  # the centre: six face neighbours at exactly 1e8 m, in index order
        assert list(idx[c]) == sorted([c - 25, c - 5, c - 1, c + 1, c + 5, c + 25]) and np.all(dist[c] == np.float32(1e8))


@pytest.mark.parametrize("n", [129, 257])
def test_padding_never_returned(b200, oracle, noracle, n):
    """One real body in the last AoSoA block: its 127 padding neighbours sit exactly on it (G m = 0)."""
    d = oracle.init_bodies("random", n)
    with _ctx(b200, d) as ctx:
        idx, dist = ctx.neighbors(32)
        assert np.all(idx < n)
        _same((idx, dist), noracle.bodies(d, 32))
        last = [np.full(4, d[c][n - 1]) for c in ("qx", "qy", "qz")]
        pidx, pdist = ctx.neighbors_at(*last, 32)
        assert np.all(pidx < n) and np.all(pidx[:, 0] == n - 1) and np.all(pdist[:, 0] == 0)


def test_zero_mass_bodies_found(b200, oracle, noracle):
    d = oracle.init_bodies("random", 1000)
    d["m"] = d["m"].copy()
    d["m"][::3] = 0
    with _ctx(b200, d) as ctx:
        idx, dist = ctx.neighbors(8)
        _same((idx, dist), noracle.bodies(d, 8))
        assert np.any(idx % 3 == 0)


# ------------------------------------------------------------------------------------------------ contract
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
                ctx.neighbors(8)
                ctx.neighbors_at(*p, 32)
            ctx.step(DT, integrator, steps)
            st = ctx.download_state()
            out.append([st[k] for k in ctx._STATE] + list(ctx.download_accel()))
    for a, b in zip(out[0], out[1]):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


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
            res.append((ctx.neighbors(6), ctx.neighbors_at(*p, 6)))
    _same(res[0][0], res[1][0])
    _same(res[0][1], res[1][1])


def test_scratch_is_bounded(b200, oracle):
    d = oracle.init_bodies("galaxy", 10000)
    rng = np.random.default_rng(8)
    with _ctx(b200, d) as ctx:
        before = ctx.allocated_bytes
        ctx.neighbors_at(*_points(d, 3 * BATCH_K32, rng), 32)
        ctx.neighbors(1)
        ctx.neighbors_at(*_points(d, 1100000, rng), 1)  # more than one batch at k = 1
        grown = ctx.allocated_bytes
        assert 0 < grown - before <= 100 << 20, grown - before
        ctx.neighbors_at(*_points(d, 5 * BATCH_K32 + 3, rng), 32)
        for k in (1, 8, 16, 32):
            ctx.neighbors(k)
        ctx.neighbors_at(*_points(d, 300000, rng), 8)
        assert ctx.allocated_bytes == grown


def test_errors(b200, oracle):
    L = b200.lib()
    d = oracle.init_bodies("galaxy", 1000)
    x = np.zeros(4, np.float32)
    xp = x.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
    with b200.Context(1000, G_F32, SOFT) as ctx:
        assert L.b200nb_neighbors(ctx._ctx, 4, None, None) == b200.ESTATE
        assert L.b200nb_neighbors_at(ctx._ctx, 4, xp, xp, xp, 4, None, None) == b200.ESTATE
        ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
        for k in (0, 33):
            assert L.b200nb_neighbors(ctx._ctx, k, None, None) == b200.EINVAL
            assert L.b200nb_neighbors_at(ctx._ctx, 4, xp, xp, xp, k, None, None) == b200.EINVAL
        assert L.b200nb_neighbors_at(ctx._ctx, 4, None, xp, xp, 4, None, None) == b200.EINVAL
        assert L.b200nb_neighbors_at(ctx._ctx, 4, xp, xp, None, 4, None, None) == b200.EINVAL
        assert L.b200nb_neighbors_at(ctx._ctx, 0, None, None, None, 4, None, None) == b200.OK
        # either output may be NULL
        idx, dist = ctx.neighbors(4)
        only = np.empty((1000, 4), np.float32)
        assert L.b200nb_neighbors(ctx._ctx, 4, None, only.ctypes.data_as(ctypes.POINTER(ctypes.c_float))) == b200.OK
        assert np.array_equal(only.view(np.uint32), dist.view(np.uint32))
        for bad in (0, 33, 2.0, True):
            with pytest.raises(ValueError):
                ctx.neighbors(bad)
        with pytest.raises(ValueError):
            ctx.neighbors_at(x, x, x[:3], 4)
