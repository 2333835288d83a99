"""Massless test particles (b200nb_set_tracers) on the GPU: bit for bit against a twin context whose tracers are advanced
on the host from b200nb_field and the integrator's exact operation sequence (tests/tracers_oracle.c), physics checks
that do not go through the field call (zero-mass bodies, Kepler orbits against an fp64 host integration), bitwise
invariance (subsets, shards, reruns, asynchronous steps), the lifecycle rules of include/b200nb.h and the error codes."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import DT, G_F32, REPO, SOFT
from field_oracle import FieldOracle
from tracers_oracle import KEYS, TracersOracle

pytestmark = pytest.mark.gpu

FIELD_TI = 512
BATCH = 128 * FIELD_TI  # FIELD_BATCH in csrc/field_sm100.cuh: tracers per field launch
DT32 = np.float32(DT)


@pytest.fixture(scope="module")
def to():
    return TracersOracle()


def _upload(ctx, d):
    ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])


def _ctx(b200, d, soft=SOFT, **kw):
    ctx = b200.Context(len(d["qx"]), G_F32, soft, **kw)
    _upload(ctx, d)
    return ctx


def _tracers(d, M, rng):
    """M tracers: inside the system, just outside it, far away, exactly on a body and on body 0; velocities of the
    bodies' scale in random directions."""
    q = np.stack([d["qx"], d["qy"], d["qz"]]).astype(np.float64)
    R = max(float(np.max(np.linalg.norm(q, axis=0))), 1e8)
    kind = rng.integers(0, 5, M)
    kind[: min(M, 5)] = np.arange(min(M, 5))[::-1]
    u = rng.normal(size=(3, M))
    u /= np.linalg.norm(u, axis=0)
    radius = np.select([kind == 0, kind == 1, kind == 2], [R * rng.random(M) ** (1 / 3), R * (1.5 + rng.random(M)), 1e3 * R], 0.0)
    p = u * radius
    on = rng.integers(0, q.shape[1], M)
    p[:, kind == 3] = q[:, on[kind == 3]]
    p[:, kind == 4] = q[:, [0]]
    vs = max(float(np.std(np.concatenate([d["vx"], d["vy"]]))), 1e3)
    v = rng.normal(size=(3, M)) * vs
    return {k: np.ascontiguousarray(x, np.float32) for k, x in zip(KEYS, list(p) + list(v))}


def _set(ctx, t):
    ctx.set_tracers(*[t[k] for k in KEYS])


def _same(a, b, what=""):
    for k in KEYS:
        assert np.array_equal(np.asarray(a[k]).view(np.uint32), np.asarray(b[k]).view(np.uint32)), (what, k)


class Twin:
    """A context without tracers, and tracers advanced on the host from its b200nb_field and the integrator's operation
    sequence, one step at a time."""

    def __init__(self, ctx, t, to):
        self.ctx, self.to = ctx, to
        self.t = {k: v.copy() for k, v in t.items()}
        self.a = None  # stored a(p_n; q_n) of the leapfrog

    def field(self):
        return [x.copy() for x in self.ctx.field(self.t["qx"], self.t["qy"], self.t["qz"])[:3]]

    def step(self, integrator, dt=DT32):
        if integrator == 0:
            a = self.field()
            self.ctx.step(dt, 0, 1)
            self.to.murb(self.t, a, dt)
            self.a = None
        else:
            if self.a is None:
                self.a = self.field()
            self.to.kick_drift(self.t, self.a, dt)
            self.ctx.step(dt, 1, 1)
            self.a = self.field()
            self.to.kick(self.t, self.a, dt)


def _check_twin(A, twin, what):
    _same(A.download_tracers(), twin.t, what + " tracers")
    _same(A.download_state(), twin.ctx.download_state(), what + " bodies")


# ------------------------------------------------------------------------------------------------ exact semantics
@pytest.mark.parametrize("steps", [3, 40])  # 40: one context on one shard replays the captured step graph
@pytest.mark.parametrize("integrator", [0, 1])
@pytest.mark.parametrize("shards", [1, 2, 3])
@pytest.mark.parametrize("n", [1, 129, 2049, 20000])
def test_twin(b200, oracle, to, n, shards, integrator, steps):
    d = oracle.init_bodies("galaxy", n)
    rng = np.random.default_rng(n + 7 * shards + integrator)
    devs = [0] * shards
    with _ctx(b200, d, devices=devs) as A, _ctx(b200, d, devices=devs) as B:
        for M in (1, 511, 512, 513, BATCH + 1):
            _upload(A, d)
            _upload(B, d)
            t = _tracers(d, M, rng)
            _set(A, t)
            assert A.n_tracers == M
            twin = Twin(B, t, to)
            if steps == 3:
                for i in range(3):
                    A.step(DT32, integrator, 1)
                    twin.step(integrator)
                    _check_twin(A, twin, f"M={M} step {i + 1}")
            else:
                A.step(DT32, integrator, steps)
                for _ in range(steps):
                    twin.step(integrator)
                _check_twin(A, twin, f"M={M} after {steps} steps")


# ------------------------------------------------------------------------------------------------ physics
def test_zero_mass_bodies(b200, oracle):
    """The same points as zero-mass bodies: after one MUrB step the velocities agree within the field tests'
    acceleration bound (1e-6 of sum_j |a_ij|) times dt, for the tracer and for the zero-mass body."""
    n, M = 2049, 3000
    d = oracle.init_bodies("galaxy", n)
    t = _tracers(d, M, np.random.default_rng(11))
    z = {k: np.concatenate([d[k], t[k]]) for k in KEYS}
    z["m"] = np.concatenate([d["m"], np.zeros(M, np.float32)])
    with _ctx(b200, z) as cz:
        cz.step(DT32, 0, 1)
        vz = cz.download_state()
    with _ctx(b200, d) as ct:
        _set(ct, t)
        ct.step(DT32, 0, 1)
        w = ct.download_tracers()
    amag = FieldOracle().field(d, t["qx"], t["qy"], t["qz"])[4]
    for k in ("vx", "vy", "vz"):
        a, b = w[k].astype(np.float64), vz[k][n:].astype(np.float64)
        ulp = np.spacing(np.maximum(np.abs(w[k]), np.abs(vz[k][n:]))).astype(np.float64)
        assert np.all(np.abs(a - b) <= 2e-6 * amag * DT + 2 * ulp), float(np.max(np.abs(a - b) / (amag * DT)))


def test_kepler_orbits(b200):
    """One point mass, small softening, tracers on circular orbits at three radii and four phases, tilted: 1000 leapfrog
    steps (about 1.2 orbits at the smallest radius) agree with an fp64 host KDK of the same point-mass problem to 1e-4
    of the orbit's radius and speed."""
    mc, soft, dt = np.float32(2e30), 1.0, np.float32(2e4)
    gm = float(np.float32(G_F32 * mc))  # the G*m the library folds into the body array
    r = np.repeat([1e11, 2e11, 5e11], 4)
    ph = np.tile(np.arange(4) * np.pi / 2 + 0.3, 3)
    tilt = 0.4
    p = np.stack([r * np.cos(ph), r * np.sin(ph) * np.cos(tilt), r * np.sin(ph) * np.sin(tilt)])
    v = np.sqrt(gm / r) * np.stack([-np.sin(ph), np.cos(ph) * np.cos(tilt), np.cos(ph) * np.sin(tilt)])
    t = {k: x.astype(np.float32) for k, x in zip(KEYS, list(p) + list(v))}
    body = {k: np.zeros(1, np.float32) for k in KEYS}
    body["m"] = np.array([mc], np.float32)
    hp = np.stack([t[k] for k in KEYS[:3]]).astype(np.float64)
    hv = np.stack([t[k] for k in KEYS[3:]]).astype(np.float64)

    def acc(x):
        d2 = np.sum(x * x, axis=0) + soft * soft
        return -gm * x / (d2 * np.sqrt(d2))

    a = acc(hp)
    with _ctx(b200, body, soft) as ctx:
        _set(ctx, t)
        for _ in range(10):
            ctx.step(dt, 1, 100)
            for _ in range(100):
                hv += a * (dt / 2)
                hp += hv * dt
                a = acc(hp)
                hv += a * (dt / 2)
            g = ctx.download_tracers()
            gp = np.stack([g[k] for k in KEYS[:3]]).astype(np.float64)
            gv = np.stack([g[k] for k in KEYS[3:]]).astype(np.float64)
            assert np.all(np.linalg.norm(gp - hp, axis=0) <= 1e-4 * r)
            assert np.all(np.linalg.norm(gv - hv, axis=0) <= 1e-4 * np.sqrt(gm / r))
        assert np.all(ctx.download_state()["qx"] == 0)  # the central body feels no self force


# ------------------------------------------------------------------------------------------------ invariance
def _run(b200, d, t, integrator, steps, devices=None, step_calls=1):
    with _ctx(b200, d, devices=devices or [0]) as ctx:
        _set(ctx, t)
        for _ in range(step_calls):
            ctx.step(DT32, integrator, steps)
        return ctx.download_tracers()


@pytest.mark.parametrize("integrator", [0, 1])
def test_subset_alone(b200, oracle, integrator):
    d = oracle.init_bodies("galaxy", 5000)
    t = _tracers(d, 3000, np.random.default_rng(12))
    full = _run(b200, d, t, integrator, 5)
    sel = np.array([0, 1, 511, 512, 1999, 2999])
    sub = _run(b200, d, {k: v[sel].copy() for k, v in t.items()}, integrator, 5)
    _same({k: v[sel] for k, v in full.items()}, sub)
    alone = _run(b200, d, {k: v[[1999]].copy() for k, v in t.items()}, integrator, 5)
    _same({k: v[[1999]] for k, v in full.items()}, alone)


@pytest.mark.parametrize("integrator", [0, 1])
@pytest.mark.parametrize("M", [5, 3000])  # 5: fewer tracers than shards; 3000 on 8 shards: the last two own none
def test_shard_counts(b200, oracle, integrator, M):
    d = oracle.init_bodies("random", 20011)
    t = _tracers(d, M, np.random.default_rng(M))
    ref = _run(b200, d, t, integrator, 4)
    for k in (2, 3, 8):
        _same(ref, _run(b200, d, t, integrator, 4, devices=[0] * k), f"{k} shards")


@pytest.mark.parametrize("integrator", [0, 1])
def test_reruns_and_async_download(b200, oracle, integrator):
    d = oracle.init_bodies("galaxy", 20000)
    t = _tracers(d, 70000, np.random.default_rng(13))
    r1 = _run(b200, d, t, integrator, 40)
    _same(r1, _run(b200, d, t, integrator, 40))
    for devs in ([0], [0, 0, 0]):
        out = []
        for join in (False, True):
            with _ctx(b200, d, devices=devs) as ctx:
                _set(ctx, t)
                ctx.step(DT32, integrator, 3)
                if join:
                    ctx.sync()
                out.append(ctx.download_tracers())  # straight after the asynchronous step: the post-step state
        _same(out[0], out[1])
        _same(out[0], _run(b200, d, t, integrator, 3, devices=devs))


# ------------------------------------------------------------------------------------------------ lifecycle
def _cdiv(a, b):
    return (a + b - 1) // b


def _expected_bytes(n, M, P, local):
    """include/b200nb.h: 36 T + 16 S min(T, 65536) on every local shard"""
    T = _cdiv(_cdiv(M, P), FIELD_TI) * FIELD_TI
    S = min(64, max(1, _cdiv(_cdiv(n, 128), 32)))
    return local * (36 * T + 16 * S * min(T, BATCH))


def test_no_tracers_is_unchanged(b200, oracle, monkeypatch):
    """set_tracers(M) then set_tracers(0): the same launches per step, graphs and allocated bytes as a context that
    never had tracers, and the same state."""
    n = 3000
    d = oracle.init_bodies("galaxy", n)
    t = _tracers(d, 1000, np.random.default_rng(14))
    # several shards merge the force pass into one launch when the exchange has already landed at enqueue time, which
    # depends on timing: always split, so that launch counts compare
    monkeypatch.setenv("B200NB_SPLIT_LAUNCHES", "1")
    for devs in ([0], [0, 0]):
        res = []
        for had in (False, True):
            with _ctx(b200, d, devices=devs) as ctx:
                if had:
                    _set(ctx, t)
                    ctx.step(DT32, 1, 40)
                    _upload(ctx, d)
                    ctx.set_tracers(*[np.zeros(0, np.float32)] * 6)
                    assert ctx.n_tracers == 0
                counts = []
                for integrator, steps in ((0, 1), (1, 1), (1, 1), (0, 40), (1, 40), (1, 40)):
                    before = ctx.launch_count
                    ctx.step(DT32, integrator, steps)
                    counts.append(ctx.launch_count - before)
                st = ctx.download_state()
                res.append((counts, ctx.allocated_bytes, st))
        assert res[0][0] == res[1][0]
        assert res[0][1] == res[1][1]
        _same(res[0][2], res[1][2])


@pytest.mark.parametrize("devs", [[0], [0, 0, 0]])
def test_allocated_bytes_formula(b200, oracle, devs):
    for n in (129, 200000):
        d = oracle.init_bodies("galaxy", n)
        with _ctx(b200, d, devices=devs) as ctx:
            base = ctx.allocated_bytes
            for M in (1, 1025, 3 * BATCH + 7):
                _set(ctx, _tracers(d, M, np.random.default_rng(M)))
                assert ctx.allocated_bytes - base == _expected_bytes(n, M, len(devs), len(devs)), (n, M)
            ctx.set_tracers(*[np.zeros(0, np.float32)] * 6)
            assert ctx.allocated_bytes == base


def test_set_before_upload(b200, oracle, to):
    d = oracle.init_bodies("galaxy", 2049)
    t = _tracers(d, 700, np.random.default_rng(15))
    with b200.Context(2049, G_F32, SOFT) as A, _ctx(b200, d) as B:
        _set(A, t)
        _same(A.download_tracers(), t)
        with pytest.raises(b200.B200Error) as e:
            A.step(DT32, 1, 1)
        assert e.value.code == b200.ESTATE
        _upload(A, d)
        twin = Twin(B, t, to)
        for integrator in (1, 1, 0):
            A.step(DT32, integrator, 1)
            twin.step(integrator)
            _check_twin(A, twin, f"integrator {integrator}")


@pytest.mark.parametrize("devs", [[0], [0, 0]])
def test_stored_acceleration_invalidated(b200, oracle, to, devs):
    """A body re-upload, and b200nb_integrate_host_accel, leave the tracers but invalidate their stored a(p): the next
    leapfrog step matches a twin that takes a(p) anew."""
    n = 2049
    d = oracle.init_bodies("galaxy", n)
    d2 = oracle.init_bodies("random", n, seed=3)
    t = _tracers(d, 1500, np.random.default_rng(16))
    with _ctx(b200, d, devices=devs) as A, _ctx(b200, d, devices=devs) as B:
        _set(A, t)
        twin = Twin(B, t, to)
        for _ in range(2):
            A.step(DT32, 1, 1)
            twin.step(1)
        _upload(A, d2)
        _upload(B, d2)
        twin.a = None
        A.step(DT32, 1, 1)
        twin.step(1)
        _check_twin(A, twin, "after re-upload")
        acc = [np.full(n, 1e-3, np.float32), np.zeros(n, np.float32), np.full(n, -2e-3, np.float32)]
        before = A.download_tracers()
        A.integrate_host_accel(*acc, DT32)
        B.integrate_host_accel(*acc, DT32)
        _same(A.download_tracers(), before, "integrate_host_accel moved no tracer")
        twin.a = None
        for steps in (1, 40):
            A.step(DT32, 1, steps)
            for _ in range(steps):
                twin.step(1)
            _check_twin(A, twin, f"after integrate_host_accel, {steps} steps")


def test_replace_between_graph_runs(b200, oracle):
    n = 4000
    d = oracle.init_bodies("galaxy", n)
    rng = np.random.default_rng(17)
    t1, t2 = _tracers(d, 900, rng), _tracers(d, 2100, rng)
    for integrator in (0, 1):
        with _ctx(b200, d) as ctx:
            _set(ctx, t1)
            ctx.step(DT32, integrator, 40)
            st = ctx.download_state()
            _set(ctx, t2)
            ctx.step(DT32, integrator, 40)
            got = ctx.download_tracers()
        with _ctx(b200, {**d, **{k: st[k] for k in KEYS}}) as fresh:
            _set(fresh, t2)
            fresh.step(DT32, integrator, 40)
            _same(got, fresh.download_tracers())


@pytest.mark.parametrize("integrator", [0, 1])
def test_queries_change_nothing(b200, oracle, integrator):
    n = 5000
    d = oracle.init_bodies("galaxy", n)
    t = _tracers(d, 1200, np.random.default_rng(18))
    p = [t[k][:300].copy() for k in ("qx", "qy", "qz")]
    out = []
    for probe in (False, True):
        with _ctx(b200, d, devices=[0, 0]) as ctx:
            _set(ctx, t)
            ctx.step(DT32, integrator, 2)
            if probe:
                ctx.field(*p)
                ctx.potential()
                ctx.neighbors(4)
                ctx.fof(1e9)
                ctx.energy()
                ctx.metrics()
                ctx.accel()
                ctx.download_accel()
            ctx.step(DT32, integrator, 2)
            out.append((ctx.download_tracers(), ctx.download_state()))
    _same(out[0][0], out[1][0])
    _same(out[0][1], out[1][1])


def test_errors(b200, oracle):
    L = b200.lib()
    x = np.zeros(4, np.float32)
    xp = x.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
    d = oracle.init_bodies("galaxy", 1000)
    with _ctx(b200, d) as ctx:
        assert L.b200nb_set_tracers(ctx._ctx, 4, xp, xp, xp, None, xp, xp) == b200.EINVAL
        assert L.b200nb_set_tracers(ctx._ctx, 4, *[None] * 6) == b200.EINVAL
        assert L.b200nb_set_tracers(ctx._ctx, 0, *[None] * 6) == b200.OK
        # per-shard slices of 2^31 and more (the arrays are never read: the call fails first)
        assert L.b200nb_set_tracers(ctx._ctx, 2 ** 31, *[xp] * 6) == b200.EINVAL
        assert L.b200nb_set_tracers(ctx._ctx, 2 ** 31 - 511, *[xp] * 6) == b200.EINVAL  # 2^31 after rounding to tiles
        assert L.b200nb_download_tracers(ctx._ctx, *[None] * 6) == b200.OK
        with pytest.raises(ValueError):
            ctx.set_tracers(x, x, x, x, x, x[:3])
        _set(ctx, {k: x.copy() for k in KEYS})
        assert ctx.n_tracers == 4
        assert L.b200nb_download_tracers(ctx._ctx, *[None] * 6) == b200.OK
    # more than the device holds (three shards on one device, ~77 GB each): refused before anything is allocated, and
    # the context is left with no tracers
    M = 3 * (2 ** 31 - 512)
    with _ctx(b200, d, devices=[0, 0, 0]) as ctx:
        _set(ctx, _tracers(d, 100, np.random.default_rng(19)))
        base = ctx.allocated_bytes
        assert L.b200nb_set_tracers(ctx._ctx, M, *[xp] * 6) == b200.ECUDA
        assert "bytes on device" in L.b200nb_last_error(ctx._ctx).decode()
        assert ctx.n_tracers == 0
        assert ctx.allocated_bytes < base
        ctx.step(DT32, 1, 2)
        assert ctx.download_tracers()["qx"].shape == (0,)


# ------------------------------------------------------------------------------------------------ two GPUs, two ranks
def _n_devices():
    import torch
    return torch.cuda.device_count()


def test_two_gpus(b200, oracle):
    if _n_devices() < 2:
        pytest.skip("needs 2 GPUs")
    d = oracle.init_bodies("galaxy", 20011)
    t = _tracers(d, BATCH + 1001, np.random.default_rng(20))
    for integrator in (0, 1):
        _same(_run(b200, d, t, integrator, 3), _run(b200, d, t, integrator, 3, devices=[0, 1]))


def test_torchrun_ranks():
    if _n_devices() < 2:
        pytest.skip("needs 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29583", os.path.join(REPO, "tests", "mp_tracers_parity.py")],
                       capture_output=True, text=True, timeout=600)
    print(r.stdout[-2000:])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert r.stdout.count("ok=True") == 4
