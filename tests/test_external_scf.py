"""A frozen basis-function expansion as part of the external potential (b200nb_set_external_scf) on the GPU:
b200nb_external_field against fl(analytic terms + b200nb_scf_field) bit for bit, zero-mass bodies and tracers bit for
bit against a host twin, the stored accelerations, invariance over shards, graphs, tracers and asynchronous steps, the
energy, the physics against the analytic Hernquist term, conservation in axisymmetric and barred hosts, a frozen host
against the live one, and the lifecycle rules, launches, device memory and errors of include/b200nb.h."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import DT, G_F32, REPO, SOFT
from test_external import BATCH, GM, RSYS, Twin, _ctx, _same_state, _upload, _zero_mass, host, points
from test_scf_cpu import hernquist_sample
from tracers_oracle import KEYS, TracersOracle

pytestmark = pytest.mark.gpu

A_H = 0.5 * RSYS  # scale radius of the expansions' host samples
CENTRE = (1e6, -2e6, 5e5)
FIELD_TI = 512  # tracer slots per shard come in whole field tiles (csrc/field_sm100.cuh)
_EXP = {}


@pytest.fixture(scope="module")
def to():
    return TracersOracle()


def _bits(x):
    x = np.asarray(x)
    return x.view(np.uint64 if x.dtype == np.float64 else np.uint32)


def _eq(a, b, what=""):
    assert np.array_equal(_bits(a), _bits(b)), what


def expansion(b200, nmax, lmax, n=20000, seed=1, flatten=(1.0, 0.8, 0.5), offset=(0.15, -0.1, 0.05), centre=CENTRE, gm=3 * GM,
              a=A_H):
    """(S, T) of a flattened, offset Hernquist sample of total G M = gm and scale a, about `centre`"""
    key = (nmax, lmax, n, seed, flatten, offset, centre, gm, a)
    if key not in _EXP:
        q = hernquist_sample(n, a, seed, flatten=flatten, offset=offset)
        m = np.full(n, gm / float(G_F32) / n, np.float32)
        z = np.zeros(n, np.float32)
        with b200.Context(n, G_F32, SOFT) as ctx:
            ctx.upload(q[0], q[1], q[2], m, z, z, z)
            _EXP[key] = ctx.scf_coefficients(nmax, lmax, a, centre)
    return _EXP[key]


def _set(ctx, S, T, centre=CENTRE):
    ctx.set_external_scf(S, T, A_H, centre)


# ------------------------------------------------------------------------------------------------ consistency
@pytest.mark.parametrize("nmax,lmax", [(0, 0), (4, 3), (10, 6), (24, 12), (31, 15)])
@pytest.mark.parametrize("n_terms", [0, 3])
def test_external_field_is_terms_plus_expansion(b200, nmax, lmax, n_terms):
    S, T = expansion(b200, nmax, lmax)
    terms = host(b200, centre=(3e6, 1e6, -2e6))[:n_terms]
    p = points(20000)
    with b200.Context(1, G_F32, SOFT) as a, b200.Context(1, G_F32, SOFT) as b:
        if terms:
            a.set_external(terms)
            b.set_external(terms)
        _set(a, S, T)
        got = a.external_field(*p)
        e0 = b.external_field(*p)
        s = b.scf_field(S, T, A_H, CENTRE, *p)
    for q in range(4):
        _eq(got[q], e0[q] + s[q], (nmax, lmax, n_terms, q))


def test_external_field_batches(b200):
    """across the 2^20 batch boundary, and any batching of the points gives the same bits"""
    S, T = expansion(b200, 10, 6)
    with b200.Context(1, G_F32, SOFT) as a, b200.Context(1, G_F32, SOFT) as b:
        for c in (a, b):
            c.set_external(host(b200))
        _set(a, S, T)
        for n in (BATCH - 1, BATCH + 1):
            p = points(n, seed=n)
            got = a.external_field(*p)
            e0 = b.external_field(*p)
            s = b.scf_field(S, T, A_H, CENTRE, *p)
            for q in range(4):
                _eq(got[q], e0[q] + s[q], (n, q))
            tail = a.external_field(*[x[-5:] for x in p])
            for g, t in zip(got, tail):
                _eq(g[-5:], t, n)


# ------------------------------------------------------------------------------------------------ zero-mass twin
@pytest.mark.parametrize("integrator", [0, 1])
@pytest.mark.parametrize("shards", [1, 3])
@pytest.mark.parametrize("graph", [False, True])
def test_zero_mass_bodies_and_tracers_match_host_twin(b200, to, integrator, shards, graph):
    d = _zero_mass(b200)
    t = {k: d[k].copy() for k in KEYS}
    S, T = expansion(b200, 10, 6)
    with _ctx(b200, d, host(b200, centre=(1e6, -2e6, 5e5)), devices=[0] * shards) as ctx:
        _set(ctx, S, T)
        ctx.set_tracers(*[t[k] for k in KEYS])
        twin = Twin(ctx, t, to)
        calls = [1] * 60 + [40] if graph else [1] * 100
        done = 0
        for c in calls:
            ctx.step(DT, integrator, c)
            for _ in range(c):
                twin.step(integrator)
            done += c
            if c > 1 or done % 25 == 0:
                st, tr = ctx.download_state(), ctx.download_tracers()
                _same_state(st, twin.t, ("bodies", done))
                _same_state(tr, twin.t, ("tracers", done))  # a zero-mass body and a tracer move together
        ax = ctx.download_accel()
        if integrator == 1:
            for q in range(3):
                _eq(ax[q], twin.a[q], q)


# ------------------------------------------------------------------------------------------------ massive bodies
def test_accel_includes_expansion(b200):
    d = b200.init_bodies("galaxy", 4097)
    S, T = expansion(b200, 16, 8)
    with _ctx(b200, d) as a0, _ctx(b200, d, host(b200)) as a1:
        _set(a1, S, T)
        a0.accel()
        a1.accel()
        s = a0.download_accel()
        w = a1.download_accel()
        e = a1.external_field(d["qx"], d["qy"], d["qz"])
    for q in range(3):
        want = (s[q].astype(np.float64) + e[q]).astype(np.float32)
        tol = np.spacing(np.abs(s[q])) + np.spacing(np.abs(want))
        assert np.all(np.abs(w[q].astype(np.float64) - want) <= tol), q


def _run(b200, d, integrator, devices=(0,), calls=(1,) * 40, tracers=None, sync=False, exp=True):
    with _ctx(b200, d, host(b200), devices=devices) as ctx:
        if exp:
            _set(ctx, *expansion(b200, 10, 6))
        if tracers is not None:
            ctx.set_tracers(*[tracers[k] for k in KEYS])
        for c in calls:
            ctx.step(DT, integrator, c)
            if sync:
                ctx.sync()
        return ctx.download_state()


@pytest.mark.parametrize("integrator", [0, 1])
def test_trajectories_bit_identical(b200, integrator):
    """reruns, graph and single steps, with and without tracers, asynchronous and joined steps, on each shard count"""
    d = b200.init_bodies("galaxy", 2049)
    rng = np.random.default_rng(3)
    t = {k: (rng.normal(size=777) * (RSYS if k[0] == "q" else 1e3)).astype(np.float32) for k in KEYS}
    refs = []
    for devs in ([0], [0, 0], [0, 0, 0]):
        ref = _run(b200, d, integrator, devices=devs)
        _same_state(ref, _run(b200, d, integrator, devices=devs), (devs, "rerun"))
        _same_state(ref, _run(b200, d, integrator, devices=devs, calls=(40,)), (devs, "one call"))
        _same_state(ref, _run(b200, d, integrator, devices=devs, calls=(40,), sync=True), (devs, "one call, joined"))
        _same_state(ref, _run(b200, d, integrator, devices=devs, sync=True), (devs, "synchronous"))
        _same_state(ref, _run(b200, d, integrator, devices=devs, tracers=t), (devs, "tracers"))
        _same_state(ref, _run(b200, d, integrator, devices=devs, tracers=t, calls=(40,)), (devs, "tracers, one call"))
        refs.append(ref)
    for r in refs[1:]:
        for c in ("qx", "qy", "qz"):
            assert np.all(np.abs(r[c].astype(np.float64) - refs[0][c]) <= 2e-6 * 2e8), c
    assert not np.array_equal(_run(b200, d, integrator, exp=False)["qx"], refs[0]["qx"])


def test_energy_includes_expansion(b200):
    d = b200.init_bodies("galaxy", 4096)
    S, T = expansion(b200, 16, 8)
    with _ctx(b200, d) as c0, _ctx(b200, d, host(b200, centre=(2e6, 0.0, 1e6))) as c1:
        _set(c1, S, T)
        c0.step(DT, 1, 3)
        c1.step(DT, 1, 3)
        st = c1.download_state()
        e1, m1 = c1.energy(), c1.metrics()
        c0.upload(st["qx"], st["qy"], st["qz"], d["m"], st["vx"], st["vy"], st["vz"])
        e0, m0 = c0.energy(), c0.metrics()
        phi = c1.external_field(st["qx"], st["qy"], st["qz"])[3]
    w = d["m"].astype(np.float64) * phi
    assert abs((e1 - e0) - w.sum()) <= 1e-12 * np.abs(w).sum()
    assert m1["energy"] == e1
    for k in m0:
        if k != "energy":
            assert m0[k] == m1[k], k


# ------------------------------------------------------------------------------------------------ physics
def _monopole(gm, a):
    S = np.full((1, 1, 1), gm / a)
    return S, np.zeros_like(S)


def test_monopole_is_the_hernquist_term(b200):
    """S_000 = GM/a alone is the Hernquist potential -GM/(r + a), from 1e-3 a to 1e3 a and at the centre"""
    a = A_H
    rng = np.random.default_rng(4)
    r = a * 10.0 ** rng.uniform(-3, 3, 5000)
    u = rng.normal(size=(3, 5000))
    u /= np.linalg.norm(u, axis=0)
    p = [np.append((u[k] * r).astype(np.float32), np.float32(0.0)) for k in range(3)]
    with b200.Context(1, G_F32, SOFT) as ce, b200.Context(1, G_F32, SOFT) as ch:
        ce.set_external_scf(*_monopole(3 * GM, a), a)
        ch.set_external([b200.hernquist(3 * GM, a)])
        e, h = ce.external_field(*p), ch.external_field(*p)
    assert np.all(np.abs(e[3] / h[3] - 1) <= 1e-14)
    ae, ah = np.sqrt(e[0] ** 2 + e[1] ** 2 + e[2] ** 2), np.sqrt(h[0] ** 2 + h[1] ** 2 + h[2] ** 2)
    assert np.all(np.abs(ae[:-1] / ah[:-1] - 1) <= 1e-14)
    assert ae[-1] == 0.0 and ah[-1] == 0.0


def test_circular_orbit(b200):
    a = A_H
    with b200.Context(1, G_F32, SOFT) as ctx:
        ctx.set_external_scf(*_monopole(GM, a), a)
        R = np.float32(RSYS)
        acc = ctx.external_field(np.array([R]), np.zeros(1), np.zeros(1))[0][0]
        v = np.sqrt(-acc * float(R))
        dt = 2 * np.pi * float(R) / v / 1000
        z = np.zeros(1, np.float32)
        ctx.upload(np.array([R]), z, z, z, z, np.array([v], np.float32), z)
        rmax = rmin = float(R)
        for _ in range(100):
            ctx.step(dt, 1, 100)
            s = ctx.download_state()
            rr = float(np.hypot(s["qx"][0], s["qy"][0]))
            rmax, rmin = max(rmax, rr), min(rmin, rr)
    dev = max(rmax - float(R), float(R) - rmin) / float(R)
    print(f"circular orbit in the S_000 expansion, 10 periods at 1000 leapfrog steps: |dr|/r {dev:.3e}")
    assert dev <= 1e-4


def _keep_m(S, T, ms):
    S, T = S.copy(), T.copy()
    drop = [m for m in range(S.shape[2]) if m not in ms]
    S[:, :, drop] = 0.0
    T[:, :, drop] = 0.0
    return S, T


# the conservation hosts: 8 GM at scale 4 RSYS, stepped at DT / 16.  Measured on a B200 at DT / 4, an analytic Hernquist
# host of 8 GM at scale 2 RSYS already drifts by 1.4e-4 in E (the galaxy's orbits through the cusp are under-resolved),
# and the (1, 0.4, 0.3) bar's m = 2 terms swing L_z by 64 % at DT / 4: the expansion behaves as the analytic term does
A_C = 4 * RSYS


def _conserve(b200, S, T):
    d = b200.init_bodies("galaxy", 2048)
    with _ctx(b200, d) as ctx:
        ctx.set_external_scf(S, T, A_C, (0.0, 0.0, 0.0))
        m0, e0 = ctx.metrics(), ctx.energy()
        dl, de = 0.0, 0.0
        for _ in range(10):
            ctx.step(DT / 16, 1, 100)
            m, e = ctx.metrics(), ctx.energy()
            dl = max(dl, abs(m["ang_z"] - m0["ang_z"]) / abs(m0["ang_z"]))
            de = max(de, abs(e - e0) / abs(e0))
    return dl, de


def _host_200k(b200, seed, flatten):
    return expansion(b200, 10, 6, n=200000, seed=seed, flatten=flatten, offset=(0.0, 0.0, 0.0), centre=(0.0, 0.0, 0.0),
                     gm=8 * GM, a=A_C)


def test_galaxy_in_axisymmetric_expansion_conserves(b200):
    """every m > 0 coefficient of a centred, flattened 200k sample zeroed: an axisymmetric host"""
    dl, de = _conserve(b200, *_keep_m(*_host_200k(b200, 5, (1.0, 1.0, 0.5)), (0,)))
    print(f"galaxy N=2048 in a centred axisymmetric expansion, 1000 leapfrog steps: |dLz|/|Lz| {dl:.3e}, |dE|/|E| {de:.3e}")
    assert dl <= 1e-6 and de <= 1e-4


def test_galaxy_in_barred_expansion(b200):
    """the m = 0 and m = 2 coefficients of an x-elongated sample: energy is kept, L_z is not (the bar exerts a torque)"""
    dl, de = _conserve(b200, *_keep_m(*_host_200k(b200, 6, (1.0, 0.7, 0.5)), (0, 2)))
    print(f"galaxy N=2048 in a barred (m = 0, 2) expansion, 1000 leapfrog steps: |dLz|/|Lz| {dl:.3e}, |dE|/|E| {de:.3e}")
    assert de <= 1e-4 and dl > 1e-5


def test_frozen_host_matches_live_host(b200):
    """a (16, 8) expansion of a 100k-body Hernquist host against that host's own field at a satellite's bodies"""
    a = 2 * RSYS
    nh, ns = 100000, 2048
    q = hernquist_sample(nh, a, 7)
    sat = b200.init_bodies("galaxy", ns)
    off = np.float32(3 * a)
    d = {"qx": np.concatenate([q[0], sat["qx"] + off]), "qy": np.concatenate([q[1], sat["qy"]]),
         "qz": np.concatenate([q[2], sat["qz"]]),
         "m": np.concatenate([np.full(nh, 10 * 2.51e24 / nh, np.float32), sat["m"]])}
    for c in ("vx", "vy", "vz"):
        d[c] = np.zeros(nh + ns, np.float32)
    labels = np.concatenate([np.zeros(nh, np.uint32), np.ones(ns, np.uint32)])
    with b200.Context(nh + ns, G_F32, 1e-6 * a) as A:
        _upload(A, d)
        S, T = A.scf_coefficients(16, 8, a, (0.0, 0.0, 0.0), group=labels, label=0)
        acc, phi = A.component_field_bodies(labels, 2)
    ps = [d[k][nh:] for k in ("qx", "qy", "qz")]
    with b200.Context(ns, G_F32, 1e-6 * a) as B:
        B.set_external_scf(S, T, a)
        e = B.external_field(*ps)
    r = np.sqrt(sum(x.astype(np.float64) ** 2 for x in ps))
    keep = (r > 0.3 * a) & (r < 5 * a)
    assert keep.sum() > ns // 2
    live_a = acc[nh:, 0, :].astype(np.float64)[keep]
    frozen_a = np.stack(e[:3], axis=1)[keep]
    rel_phi = np.abs(e[3][keep] / phi[nh:, 0].astype(np.float64)[keep] - 1)
    rel_a = np.linalg.norm(frozen_a - live_a, axis=1) / np.linalg.norm(live_a, axis=1)
    print(f"frozen vs live host at {keep.sum()} satellite bodies: Phi median {np.median(rel_phi):.2e} max {rel_phi.max():.2e}; "
          f"|a| median {np.median(rel_a):.2e} max {rel_a.max():.2e}")
    assert np.median(rel_phi) < 2e-3 and rel_phi.max() < 1e-2
    # the live a also carries the discreteness of 100k host bodies, a few of which pass close to any satellite body
    # (measured on a B200: median 1.4e-2); the expansion is the smooth part of it
    assert np.median(rel_a) < 3e-2


# ------------------------------------------------------------------------------------------------ lifecycle
def test_set_before_upload_and_get(b200):
    d = b200.init_bodies("galaxy", 1500)
    S, T = expansion(b200, 10, 6)
    with b200.Context(1500, G_F32, SOFT) as a, b200.Context(1500, G_F32, SOFT) as b:
        assert a.external_scf is None
        _set(a, S, T)
        _upload(a, d)
        _upload(b, d)
        _set(b, S, T)
        for c in (a, b):
            c.step(DT, 1, 5)
        _same_state(a.download_state(), b.download_state())
        S2, T2, a2, c2 = a.external_scf
        assert np.array_equal(S2, S) and np.array_equal(T2, T) and a2 == A_H and c2 == CENTRE


@pytest.mark.parametrize("integrator", [0, 1])
def test_change_between_steps_is_fresh_context(b200, integrator):
    d = b200.init_bodies("galaxy", 1500)
    rng = np.random.default_rng(5)
    t = {k: (rng.normal(size=300) * (RSYS if k[0] == "q" else 1e3)).astype(np.float32) for k in KEYS}
    S1, T1 = expansion(b200, 4, 3)
    S2, T2 = expansion(b200, 24, 12, seed=2)
    with _ctx(b200, d, host(b200)) as ctx:
        _set(ctx, S1, T1)
        ctx.set_tracers(*[t[k] for k in KEYS])
        ctx.step(DT, integrator, 4)
        _set(ctx, S2, T2)
        st, tr = ctx.download_state(), ctx.download_tracers()
        ctx.step(DT, integrator, 4)
        got, got_t = ctx.download_state(), ctx.download_tracers()
    with b200.Context(1500, G_F32, SOFT) as fresh:
        fresh.set_external(host(b200))
        _set(fresh, S2, T2)
        fresh.upload(st["qx"], st["qy"], st["qz"], d["m"], st["vx"], st["vy"], st["vz"])
        fresh.set_tracers(*[tr[k] for k in KEYS])
        fresh.step(DT, integrator, 4)
        _same_state(got, fresh.download_state())
        _same_state(got_t, fresh.download_tracers())


@pytest.mark.parametrize("integrator", [0, 1])
def test_set_and_clear_is_never_set(b200, integrator):
    d = b200.init_bodies("galaxy", 2000)
    t = {k: d[k][:100].copy() for k in KEYS}
    S, T = expansion(b200, 24, 12)
    out = []
    for cleared in (False, True):
        with b200.Context(2000, G_F32, SOFT) as ctx:
            ctx.set_external(host(b200))
            if cleared:
                _set(ctx, S, T)
                ctx.set_external_scf(None)
                assert ctx.external_scf is None
            _upload(ctx, d)
            ctx.set_tracers(*[t[k] for k in KEYS])
            if cleared:  # also after a step with the expansion and tracers
                _set(ctx, S, T)
                ctx.step(DT, integrator, 2)
                ctx.set_external_scf(None)
                _upload(ctx, d)
                ctx.set_tracers(*[t[k] for k in KEYS])
            l0 = ctx.launch_count
            ctx.step(DT, integrator, 3)
            ctx.step(DT, integrator, 40)
            out.append((ctx.download_state(), ctx.download_tracers(), ctx.energy(), ctx.launch_count - l0,
                        ctx.allocated_bytes))
    _same_state(out[0][0], out[1][0])
    _same_state(out[0][1], out[1][1])
    assert out[0][2:] == out[1][2:]


def test_terms_and_expansion_are_independent(b200):
    S, T = expansion(b200, 4, 3)
    terms = host(b200)
    with b200.Context(1000, G_F32, SOFT) as ctx:
        _set(ctx, S, T)
        ctx.set_external(terms)
        assert ctx.external_scf[2] == A_H and np.array_equal(ctx.external_scf[0], S)
        ctx.set_external([])
        assert ctx.external_scf is not None
        ctx.set_external(terms)
        ctx.set_external_scf(None)
        assert [bytes(x) for x in ctx.external] == [bytes(x) for x in terms]


@pytest.mark.parametrize("shards,tracers", [(1, True), (3, False)])
def test_one_extra_launch_per_evaluation(b200, monkeypatch, shards, tracers):
    """counted over the call sequence of test_external.py::test_terms_add_no_launches"""
    # several shards merge their two force launches into one when the exchange has landed at enqueue time, which
    # depends on timing: count with the split form, which is always taken then
    monkeypatch.setenv("B200NB_SPLIT_LAUNCHES", "1")
    d = b200.init_bodies("galaxy", 2000)
    S, T = expansion(b200, 10, 6)
    counts = []
    for exp in (False, True):
        with _ctx(b200, d, host(b200), devices=[0] * shards) as ctx:
            if exp:
                _set(ctx, S, T)
            if tracers:
                ctx.set_tracers(*[d[k][:50].copy() for k in KEYS])
            l0 = ctx.launch_count
            for integrator in (0, 1):
                ctx.step(DT, integrator, 2)
                ctx.step(DT, integrator, 40)
            counts.append(ctx.launch_count - l0)
    per_shard = 42 + 1 + 42  # MUrB: one force pass per step; leapfrog: a(x_0) once, then one per step
    want = shards * per_shard + (per_shard if tracers else 0)  # the tracer pass evaluates e once per evaluation too
    assert counts[1] - counts[0] == want, counts


def _r256(x):
    return (x + 255) // 256 * 256


@pytest.mark.parametrize("shards", [1, 3])
def test_allocated_bytes_formula(b200, shards):
    n, M = 2000, 1000
    d = b200.init_bodies("galaxy", n)
    L = b200.slice_length(n, shards)
    Tslots = -(-(-(-M // shards)) // FIELD_TI) * FIELD_TI

    def block(nmax, lmax):
        return _r256(12952) + _r256(16 * (nmax + 1) * (lmax + 1) * (lmax + 2) // 2)

    t = {k: d[k][:M].copy() for k in KEYS}
    S1, T1 = expansion(b200, 24, 12)
    S2, T2 = expansion(b200, 10, 6)
    none = [np.zeros(0, np.float32)] * 6
    with _ctx(b200, d, devices=[0] * shards) as ctx:
        base = ctx.allocated_bytes
        ctx.set_tracers(*[t[k] for k in KEYS])
        tr_own = ctx.allocated_bytes - base  # the tracer set's own buffers
        ctx.set_tracers(*none)
        _set(ctx, S1, T1)
        assert ctx.allocated_bytes - base == shards * (block(24, 12) + 32 * L)
        _set(ctx, S2, T2)  # grow-only
        assert ctx.allocated_bytes - base == shards * (block(24, 12) + 32 * L)
        ctx.set_tracers(*[t[k] for k in KEYS])  # the expansion first, then tracers
        assert ctx.allocated_bytes - base == tr_own + shards * (block(24, 12) + 32 * L + 32 * Tslots)
        ctx.set_tracers(*none)
        assert ctx.allocated_bytes - base == shards * (block(24, 12) + 32 * L)
        ctx.set_external_scf(None)
        assert ctx.allocated_bytes == base
        ctx.set_tracers(*[t[k] for k in KEYS])  # tracers first, then the expansion
        _set(ctx, S2, T2)
        assert ctx.allocated_bytes - base == tr_own + shards * (block(10, 6) + 32 * L + 32 * Tslots)
        ctx.step(DT, 1, 3)  # tracers set before the expansion move in it
        tr = ctx.download_tracers()
        ctx.set_external_scf(None)
        assert ctx.allocated_bytes - base == tr_own
    with _ctx(b200, d, devices=[0] * shards) as ref:
        _set(ref, S2, T2)
        ref.set_tracers(*[t[k] for k in KEYS])
        ref.step(DT, 1, 3)
        _same_state(tr, ref.download_tracers())


def test_host_accel_ignores_expansion(b200):
    d = b200.init_bodies("galaxy", 1500)
    rng = np.random.default_rng(2)
    a = [(rng.normal(size=1500) * 1e-3).astype(np.float32) for _ in range(3)]
    out = []
    for exp in (False, True):
        with _ctx(b200, d) as ctx:
            if exp:
                _set(ctx, *expansion(b200, 10, 6))
            ctx.integrate_host_accel(*a, DT)
            ctx.integrate_host_accel(*a, DT)
            out.append(ctx.download_state())
    _same_state(out[0], out[1])


def test_field_calls_unchanged(b200):
    d = b200.init_bodies("galaxy", 3000)
    p = points(500)
    lab = (np.arange(3000) % 2).astype(np.uint32)
    out = []
    for exp in (False, True):
        with _ctx(b200, d) as ctx:
            if exp:
                _set(ctx, *expansion(b200, 10, 6))
            out.append((ctx.field(*p), ctx.potential(), ctx.tidal(*p), ctx.tidal_bodies(), ctx.component_field_bodies(lab, 2),
                        ctx.scf_coefficients(6, 4, A_H)))
    for x, y in zip(out[0], out[1]):
        for u, v in zip(x if isinstance(x, tuple) else (x,), y if isinstance(y, tuple) else (y,)):
            _eq(u, v)


def test_errors_leave_expansion(b200):
    L = b200.lib()
    S, T = expansion(b200, 4, 3)
    Sp, Tp = b200._scf_pack(S).ravel(), b200._scf_pack(T).ravel()
    DP = ctypes.POINTER(ctypes.c_double)

    def dp(x):
        return None if x is None else np.ascontiguousarray(x, np.float64).ctypes.data_as(DP)

    c0 = np.zeros(3)
    with b200.Context(1000, G_F32, SOFT) as ctx:
        _set(ctx, S, T)
        Tbad = Tp.copy()
        Tbad[2 * 10 + 1] = 1.0  # n = 2, l = 1, m = 0
        Snan = Sp.copy()
        Snan[5] = np.nan
        Tinf = Tp.copy()
        Tinf[7] = np.inf
        bad = [(4, 3, 1.0, c0, Sp, None), (4, 3, 1.0, c0, None, Tp), (32, 3, 1.0, c0, Sp, Tp), (4, 16, 1.0, c0, Sp, Tp),
               (4, 3, 0.0, c0, Sp, Tp), (4, 3, -1.0, c0, Sp, Tp), (4, 3, np.inf, c0, Sp, Tp), (4, 3, np.nan, c0, Sp, Tp),
               (4, 3, 1.0, None, Sp, Tp), (4, 3, 1.0, np.array([0, np.nan, 0]), Sp, Tp), (4, 3, 1.0, c0, Snan, Tp),
               (4, 3, 1.0, c0, Sp, Tinf), (4, 3, 1.0, c0, Sp, Tbad)]
        for i, (nm, lm, a, c, s, t) in enumerate(bad):
            assert L.b200nb_set_external_scf(ctx._ctx, nm, lm, a, dp(c), dp(s), dp(t)) == b200.EINVAL, i
        S2, T2, a2, c2 = ctx.external_scf
        assert np.array_equal(S2, S) and np.array_equal(T2, T) and a2 == A_H and c2 == CENTRE
        u = ctypes.c_uint()
        assert L.b200nb_get_external_scf(ctx._ctx, None, None, None, None, None, None, None) == b200.EINVAL
        assert L.b200nb_get_external_scf(ctx._ctx, ctypes.byref(u), None, None, None, None, None, None) == b200.OK
        assert u.value == 1
        with pytest.raises(ValueError):
            ctx.set_external_scf(S, None, A_H)


# ------------------------------------------------------------------------------------------------ ranks
def test_torchrun_ranks():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29591", os.path.join(REPO, "tests", "mp_external_scf_parity.py")],
                       capture_output=True, text=True, timeout=600)
    print(r.stdout[-2000:])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert r.stdout.count("ok=True") == 2
