"""Static external potential (b200nb_set_external) on the GPU: b200nb_external_field against the host restatement
(tests/external_oracle.c), zero-mass bodies and tracers bit for bit against a host twin, massive bodies against the
fp64 oracle and across shards, graphs, tracers and asynchronous steps, the physics of orbits and conservation laws, the
lifecycle rules of include/b200nb.h and the error codes."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import DT, G_F32, REPO, SOFT
from external_oracle import ExternalOracle
from tracers_oracle import KEYS, TracersOracle

pytestmark = pytest.mark.gpu

DT32 = np.float32(DT)
BATCH = 1 << 20  # EXTERNAL_BATCH in csrc/context.cu
GM = float(G_F32) * 2.51e24  # G times the mass of the galaxy initial conditions
RSYS = 2e8  # their size [m]


@pytest.fixture(scope="module")
def eo(b200):
    return ExternalOracle(b200.ExternalTerm)


@pytest.fixture(scope="module")
def to():
    return TracersOracle()


def host(b200, centre=(0.0, 0.0, 0.0)):
    """bulge + disk + halo, several times the galaxy's own mass"""
    return [b200.hernquist(2 * GM, 0.25 * RSYS, centre), b200.miyamoto_nagai(3 * GM, 0.5 * RSYS, 0.1 * RSYS, centre),
            b200.nfw(5 * GM, 2 * RSYS, centre)]


def kinds(b200, c=(1e7, -2e7, 3e6)):
    return {"plummer": b200.plummer(GM, 0.3 * RSYS, c), "hernquist": b200.hernquist(GM, 0.3 * RSYS, c),
            "nfw": b200.nfw(GM, 0.3 * RSYS, c), "miyamoto_nagai": b200.miyamoto_nagai(GM, 0.3 * RSYS, 0.05 * RSYS, c),
            "logarithmic": b200.logarithmic(1e6, 0.3 * RSYS, 0.7, c)}


def eight(b200):
    rng = np.random.default_rng(8)
    ks = list(kinds(b200).values())
    out = []
    for i in range(8):
        c = tuple(rng.normal(size=3) * 0.3 * RSYS)
        t = ks[i % 5]
        out.append(type(t)(t.kind, 0, t.gm * (1 + i), t.a * (1 + 0.1 * i), t.b, (ctypes.c_double * 3)(*c)))
    return out


def points(n, seed=0):
    rng = np.random.default_rng(seed)
    r = RSYS * 10.0 ** rng.uniform(-6, 3, n)
    u = rng.normal(size=(3, n))
    u /= np.linalg.norm(u, axis=0)
    p = (u * r).astype(np.float32)
    p[:, :3] = 0.0
    p[2, 3:6] = 0.0  # in the plane
    p[:2, 6:9] = 0.0  # on the z axis
    return p[0].copy(), p[1].copy(), p[2].copy()


def _bits(x):
    x = np.asarray(x)
    return x.view(np.uint64 if x.dtype == np.float64 else np.uint32)


def _eq(a, b, what=""):
    assert np.array_equal(_bits(a), _bits(b)), what


def _upload(ctx, d):
    ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])


def _ctx(b200, d, terms=(), devices=(0,), **kw):
    ctx = b200.Context(len(d["qx"]), G_F32, SOFT, devices=list(devices), **kw)
    if terms:
        ctx.set_external(terms)
    _upload(ctx, d)
    return ctx


def _same_state(a, b, what=""):
    for k in KEYS:
        _eq(a[k], b[k], (what, k))


def _scale(eo, terms, p):
    """sum over terms of |a_term| and |phi_term|: the cancellation-free size of the sums"""
    sa, sp = 0.0, 0.0
    for t in terms:
        a = eo.eval([t], *p)
        sa = sa + np.sqrt(a[0] ** 2 + a[1] ** 2 + a[2] ** 2)
        sp = sp + np.abs(a[3])
    return sa, sp


# ------------------------------------------------------------------------------------------------ external_field
@pytest.mark.parametrize("case", ["plummer", "hernquist", "nfw", "miyamoto_nagai", "logarithmic", "three", "eight"])
def test_external_field_matches_oracle(b200, eo, case):
    terms = {"three": host(b200), "eight": eight(b200)}.get(case) or [kinds(b200)[case]]
    p = points(20000)
    with b200.Context(1, G_F32, SOFT) as ctx:  # allowed before an upload
        ctx.set_external(terms)
        got = ctx.external_field(*p)
    ref = eo.eval(terms, *p)
    logs = {t.kind for t in terms} & {b200.EXT_NFW, b200.EXT_LOGARITHMIC}
    if not logs:
        for g, r in zip(got, ref):
            _eq(g, r, case)
        return
    if logs == {b200.EXT_LOGARITHMIC}:  # the logarithmic a_ext involves no log
        for q in range(3):
            _eq(got[q], ref[q], (case, q))
    sa, sp = _scale(eo, terms, p)
    for q in range(3):
        assert np.all(np.abs(got[q] - ref[q]) <= 1e-14 * sa), (case, q)
    assert np.all(np.abs(got[3] - ref[3]) <= 1e-14 * sp), case


def test_external_field_batches(b200, eo):
    """a batch boundary (+-1 point) and results bitwise independent of the other points of the call"""
    terms = [kinds(b200)["plummer"], kinds(b200)["miyamoto_nagai"], kinds(b200)["hernquist"]]
    with b200.Context(1, G_F32, SOFT) as ctx:
        ctx.set_external(terms)
        for n in (BATCH - 1, BATCH, BATCH + 1):
            p = points(n, seed=n)
            got = ctx.external_field(*p)
            ref = eo.eval(terms, *p)
            for g, r in zip(got, ref):
                _eq(g, r, n)
            tail = ctx.external_field(*[x[-5:] for x in p])
            for g, t in zip(got, tail):
                _eq(g[-5:], t, n)
        assert ctx.external_field(np.zeros(0), np.zeros(0), np.zeros(0))[0].shape == (0,)


# ------------------------------------------------------------------------------------------------ zero-mass twin
class Twin:
    """bodies (or tracers) without self-gravity advanced on the host: a = fp32(external_field) and the integrator's
    operation sequence (tests/tracers_oracle.c)"""

    def __init__(self, ctx, t, to):
        self.ctx, self.to = ctx, to
        self.t = {k: v.copy() for k, v in t.items()}
        self.a = None

    def acc(self):
        e = self.ctx.external_field(self.t["qx"], self.t["qy"], self.t["qz"])
        return [x.astype(np.float32) for x in e[:3]]

    def step(self, integrator):
        if integrator == 0:
            self.to.murb(self.t, self.acc(), DT32)
            return
        if self.a is None:
            self.a = self.acc()
        self.to.kick_drift(self.t, self.a, DT32)
        self.a = self.acc()
        self.to.kick(self.t, self.a, DT32)


def _zero_mass(b200, n=300):
    d = b200.init_bodies("galaxy", n)
    d["m"][:] = 0
    return d


@pytest.mark.parametrize("integrator", [0, 1])
@pytest.mark.parametrize("shards", [1, 3])
@pytest.mark.parametrize("graph", [False, True])
def test_zero_mass_bodies_and_tracers_match_host_twin(b200, to, integrator, shards, graph):
    d = _zero_mass(b200)
    t = {k: d[k].copy() for k in KEYS}
    terms = host(b200, centre=(1e6, -2e6, 5e5))
    with _ctx(b200, d, terms, devices=[0] * shards) as ctx:
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
def test_accel_includes_terms(b200):
    d = b200.init_bodies("galaxy", 4097)
    terms = host(b200, centre=(3e6, 1e6, -2e6))
    with _ctx(b200, d) as a0, _ctx(b200, d, terms) as a1:
        a0.accel()
        a1.accel()
        s = a0.download_accel()
        w = a1.download_accel()
        e = a1.external_field(d["qx"], d["qy"], d["qz"])
    for q in range(3):
        want = (s[q].astype(np.float64) + e[q]).astype(np.float32)
        tol = np.spacing(np.abs(s[q])) + np.spacing(np.abs(want))
        assert np.all(np.abs(w[q].astype(np.float64) - want) <= tol), q


def _run(b200, d, terms, integrator, devices=(0,), calls=(1,) * 40, tracers=None, sync=False):
    with _ctx(b200, d, terms, devices=devices) as ctx:
        if tracers is not None:
            ctx.set_tracers(*[tracers[k] for k in KEYS])
        for c in calls:
            ctx.step(DT, integrator, c)
            if sync:
                ctx.sync()
        return ctx.download_state()


@pytest.mark.parametrize("integrator", [0, 1])
def test_trajectories_bit_identical(b200, integrator):
    """Bit-identical across reruns, graph and single steps, with and without tracers, asynchronous and joined steps, on
    each shard count.  The force pass chunks the sources by shard count, so massive bodies on different shard counts
    agree to the force pass's accuracy rather than bitwise; the terms themselves are shard-independent bit for bit
    (test_zero_mass_bodies_and_tracers_match_host_twin)."""
    d = b200.init_bodies("galaxy", 2049)
    terms = host(b200)
    rng = np.random.default_rng(3)
    t = {k: (rng.normal(size=777) * (RSYS if k[0] == "q" else 1e3)).astype(np.float32) for k in KEYS}
    refs = []
    for devs in ([0], [0, 0], [0, 0, 0]):
        ref = _run(b200, d, terms, integrator, devices=devs)
        _same_state(ref, _run(b200, d, terms, integrator, devices=devs), (devs, "rerun"))
        _same_state(ref, _run(b200, d, terms, integrator, devices=devs, calls=(40,)), (devs, "one call"))
        _same_state(ref, _run(b200, d, terms, integrator, devices=devs, calls=(40,), sync=True), (devs, "one call, joined"))
        _same_state(ref, _run(b200, d, terms, integrator, devices=devs, sync=True), (devs, "synchronous"))
        _same_state(ref, _run(b200, d, terms, integrator, devices=devs, tracers=t), (devs, "tracers"))
        _same_state(ref, _run(b200, d, terms, integrator, devices=devs, tracers=t, calls=(40,)), (devs, "tracers, one call"))
        refs.append(ref)
    for r in refs[1:]:
        for c in ("qx", "qy", "qz"):
            assert np.all(np.abs(r[c].astype(np.float64) - refs[0][c]) <= 2e-6 * 2e8), c
    without = _run(b200, d, (), integrator)
    assert not np.array_equal(without["qx"], refs[0]["qx"])


@pytest.mark.parametrize("integrator", [0, 1])
def test_matches_fp64_oracle(b200, oracle, eo, to, integrator):
    """20 steps against an fp64 self-force plus the oracle's terms, at test_gpu_parity.py's tolerance without terms"""
    d = oracle.init_bodies("galaxy", 2048)
    terms = host(b200, centre=(1e6, 2e6, -1e6))
    with _ctx(b200, d, terms) as ctx:
        ctx.step(DT, integrator, 20)
        out = ctx.download_state()

    def acc(s):
        a = oracle.accel_f64(s)
        e = eo.eval(terms, s["qx"], s["qy"], s["qz"])
        return [(x + y).astype(np.float32) for x, y in zip(a, e[:3])]

    s = {k: d[k].copy() for k in list(KEYS) + ["m"]}
    a = acc(s)
    for _ in range(20):
        if integrator == 0:
            to.murb(s, acc(s), DT32)
        else:
            to.kick_drift(s, a, DT32)
            a = acc(s)
            to.kick(s, a, DT32)
    for c in ("qx", "qy", "qz"):
        assert np.all(np.abs(out[c].astype(np.float64) - s[c]) <= 2e-6 * 2e8), c
    for c in ("vx", "vy", "vz"):
        assert np.all(np.abs(out[c].astype(np.float64) - s[c]) <= 1e-5 * np.abs(s[c]).max()), c


# ------------------------------------------------------------------------------------------------ physics
def test_energy_includes_external_potential(b200):
    d = b200.init_bodies("galaxy", 4096)
    terms = host(b200, centre=(2e6, 0.0, 1e6))
    with _ctx(b200, d) as c0, _ctx(b200, d, terms) as c1:
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


def _circular_orbit(b200, term, plane_radius):
    """one zero-mass body on a circular orbit in the plane z = 0 of a term centred at the origin: the relative radius
    excursion over 10 orbits of 1000 leapfrog steps each"""
    with b200.Context(1, G_F32, SOFT) as ctx:
        ctx.set_external([term])
        R = np.float32(plane_radius)
        a = ctx.external_field(np.array([R]), np.zeros(1), np.zeros(1))[0][0]
        v = np.sqrt(-a * float(R))
        period = 2 * np.pi * float(R) / v
        dt = period / 1000
        z = np.zeros(1, np.float32)
        ctx.upload(np.array([R]), z, z, z, z, np.array([v], np.float32), z)
        rmax = rmin = float(R)
        for _ in range(100):
            ctx.step(dt, 1, 100)
            s = ctx.download_state()
            r = float(np.hypot(s["qx"][0], s["qy"][0]))
            rmax, rmin = max(rmax, r), min(rmin, r)
        return max(rmax - float(R), float(R) - rmin) / float(R)


def test_circular_orbits(b200):
    dev_h = _circular_orbit(b200, b200.hernquist(GM, 0.25 * RSYS), RSYS)
    dev_mn = _circular_orbit(b200, b200.miyamoto_nagai(GM, 0.5 * RSYS, 0.1 * RSYS), RSYS)
    print(f"circular orbits, 10 periods at 1000 leapfrog steps: |dr|/r Hernquist {dev_h:.3e}, Miyamoto-Nagai {dev_mn:.3e}")
    assert dev_h <= 1e-4 and dev_mn <= 1e-4  # measured on a B200: 1.8e-5 and 2.2e-5


def test_galaxy_in_axisymmetric_host_conserves(b200):
    d = b200.init_bodies("galaxy", 2048)
    terms = [b200.miyamoto_nagai(3 * GM, 0.5 * RSYS, 0.1 * RSYS), b200.nfw(5 * GM, 2 * RSYS)]
    with _ctx(b200, d, terms) as ctx:
        m0, e0 = ctx.metrics(), ctx.energy()
        dl, de = 0.0, 0.0
        for _ in range(10):
            ctx.step(DT / 4, 1, 100)
            m, e = ctx.metrics(), ctx.energy()
            dl = max(dl, abs(m["ang_z"] - m0["ang_z"]) / abs(m0["ang_z"]))
            de = max(de, abs(e - e0) / abs(e0))
    print(f"galaxy N=2048 in a centred axisymmetric host, 1000 leapfrog steps: |dLz|/|Lz| {dl:.3e}, |dE|/|E| {de:.3e}")
    assert dl <= 1e-6 and de <= 1e-4  # measured on a B200: 5.9e-8 and 1.9e-5


# ------------------------------------------------------------------------------------------------ lifecycle
def test_set_before_upload(b200):
    d = b200.init_bodies("galaxy", 1500)
    terms = host(b200)
    with b200.Context(1500, G_F32, SOFT) as a, b200.Context(1500, G_F32, SOFT) as b:
        a.set_external(terms)
        _upload(a, d)
        _upload(b, d)
        b.set_external(terms)
        for c in (a, b):
            c.step(DT, 1, 5)
        _same_state(a.download_state(), b.download_state())
        assert [bytes(t) for t in a.external] == [bytes(t) for t in terms]


@pytest.mark.parametrize("integrator", [0, 1])
def test_change_between_steps_is_fresh_context(b200, integrator):
    d = b200.init_bodies("galaxy", 1500)
    rng = np.random.default_rng(5)
    t = {k: (rng.normal(size=300) * (RSYS if k[0] == "q" else 1e3)).astype(np.float32) for k in KEYS}
    with _ctx(b200, d, host(b200)) as ctx:
        ctx.set_tracers(*[t[k] for k in KEYS])
        ctx.step(DT, integrator, 4)
        ctx.set_external(eight(b200))
        st, tr = ctx.download_state(), ctx.download_tracers()
        ctx.step(DT, integrator, 4)
        got, got_t = ctx.download_state(), ctx.download_tracers()
    with b200.Context(1500, G_F32, SOFT) as fresh:
        fresh.set_external(eight(b200))
        fresh.upload(st["qx"], st["qy"], st["qz"], d["m"], st["vx"], st["vy"], st["vz"])
        fresh.set_tracers(*[tr[k] for k in KEYS])
        fresh.step(DT, integrator, 4)
        _same_state(got, fresh.download_state())
        _same_state(got_t, fresh.download_tracers())


@pytest.mark.parametrize("integrator", [0, 1])
def test_set_and_clear_is_no_terms(b200, integrator):
    d = b200.init_bodies("galaxy", 2000)
    t = {k: d[k][:100].copy() for k in KEYS}
    out = []
    for cleared in (False, True):
        with b200.Context(2000, G_F32, SOFT) as ctx:
            if cleared:
                ctx.set_external(host(b200))
                ctx.set_external([])
                assert ctx.external == []
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


def test_terms_add_no_launches(b200):
    d = b200.init_bodies("galaxy", 2000)
    counts = []
    for terms in ((), host(b200)):
        with _ctx(b200, d, terms) as ctx:
            ctx.set_tracers(*[d[k][:50].copy() for k in KEYS])
            l0 = ctx.launch_count
            for integrator in (0, 1):
                ctx.step(DT, integrator, 2)
                ctx.step(DT, integrator, 40)
            counts.append((ctx.launch_count - l0, ctx.allocated_bytes))
    assert counts[0] == counts[1]


def test_change_between_graph_runs(b200):
    d = b200.init_bodies("galaxy", 1500)
    res = []
    for calls in ((40,), (1,) * 40):
        with _ctx(b200, d, host(b200)) as ctx:
            for c in calls:
                ctx.step(DT, 1, c)
            ctx.set_external(eight(b200))
            for c in calls:
                ctx.step(DT, 1, c)
            res.append(ctx.download_state())
    _same_state(res[0], res[1])


def test_host_accel_ignores_terms(b200):
    d = b200.init_bodies("galaxy", 1500)
    rng = np.random.default_rng(2)
    a = [(rng.normal(size=1500) * 1e-3).astype(np.float32) for _ in range(3)]
    out = []
    for terms in ((), host(b200)):
        with _ctx(b200, d, terms) as ctx:
            ctx.integrate_host_accel(*a, DT)
            ctx.integrate_host_accel(*a, DT)
            out.append(ctx.download_state())
    _same_state(out[0], out[1])


def test_field_calls_unchanged(b200):
    d = b200.init_bodies("galaxy", 3000)
    p = points(500)
    out = []
    for terms in ((), host(b200)):
        with _ctx(b200, d, terms) as ctx:
            out.append((ctx.field(*p), ctx.potential(), ctx.tidal(*p), ctx.tidal_bodies()))
    for x, y in zip(out[0], out[1]):
        for u, v in zip(x if isinstance(x, tuple) else (x,), y if isinstance(y, tuple) else (y,)):
            _eq(u, v)


def test_errors_leave_terms(b200):
    L = b200.lib()
    good = host(b200)
    with b200.Context(1000, G_F32, SOFT) as ctx:
        ctx.set_external(good)
        T = b200.ExternalTerm

        def arr(ts):
            return (T * len(ts))(*ts)

        def mod(t, **kw):
            u = T.from_buffer_copy(bytes(t))
            for k, v in kw.items():
                setattr(u, k, v)
            return u

        p, h, n, mn, lg = kinds(b200).values()
        bad = [mod(p, kind=5), mod(p, kind=-1), mod(p, reserved=1), mod(p, gm=-1.0), mod(p, gm=np.nan), mod(p, a=-1.0),
               mod(p, b=1.0), mod(h, a=0.0), mod(h, b=1.0), mod(n, a=0.0), mod(n, a=np.inf), mod(mn, b=0.0),
               mod(mn, a=-1.0), mod(lg, a=0.0), mod(lg, b=0.0), mod(lg, b=-1.0)]
        c = mod(p)
        c.centre[2] = np.inf
        bad.append(c)
        for i, t in enumerate(bad):
            assert L.b200nb_set_external(ctx._ctx, 2, arr([good[0], t])) == b200.EINVAL, i
        assert L.b200nb_set_external(ctx._ctx, 9, arr([good[0]] * 9)) == b200.EINVAL
        assert L.b200nb_set_external(ctx._ctx, 1, None) == b200.EINVAL
        z = np.zeros(4, np.float32)
        fp = z.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
        assert L.b200nb_external_field(ctx._ctx, 4, None, fp, fp, *[None] * 4) == b200.EINVAL
        assert L.b200nb_external_field(ctx._ctx, 0, None, None, None, *[None] * 4) == b200.OK
        assert [bytes(t) for t in ctx.external] == [bytes(t) for t in good]
        with pytest.raises(ValueError):
            ctx.set_external([good[0]] * 9)


# ------------------------------------------------------------------------------------------------ ranks
def _n_devices():
    import torch
    return torch.cuda.device_count()


def test_torchrun_ranks():
    if _n_devices() < 2:
        pytest.skip("needs 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29587", os.path.join(REPO, "tests", "mp_external_parity.py")],
                       capture_output=True, text=True, timeout=600)
    print(r.stdout[-2000:])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert r.stdout.count("ok=True") == 2
