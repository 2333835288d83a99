"""CPU checks of the external potential: the host restatement of the evaluator (tests/external_oracle.c) against an
independent numpy longdouble restatement of the formulas, a_ext = -grad Phi_ext, the NFW series, Miyamoto-Nagai against
Plummer, the ctypes mirror of the term struct, the constructors' validation, the C ABI's argument checks and the
registers of the new kernel instantiations."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import REPO
from external_oracle import ExternalOracle

L0 = 1e19  # scale length of the test terms [m]
GM = 1.3e30


@pytest.fixture(scope="module")
def eo(b200):
    return ExternalOracle(b200.ExternalTerm)


def _kinds(b200, centre=(0.0, 0.0, 0.0)):
    return {
        "plummer": b200.plummer(GM, L0, centre),
        "hernquist": b200.hernquist(GM, L0, centre),
        "nfw": b200.nfw(GM, L0, centre),
        "miyamoto_nagai": b200.miyamoto_nagai(GM, L0, 0.3 * L0, centre),
        "logarithmic": b200.logarithmic(4.8e10, L0, 0.8, centre),
    }


def _mu_ld(x):
    """ln(1+x) - x/(1+x) in longdouble; a 40-term positive series below 1e-2, where the difference cancels"""
    x = np.asarray(x, np.longdouble)
    y = x / (1 + x)
    s = np.zeros_like(x)
    for j in range(40, 1, -1):
        s = np.longdouble(1) / j + y * s
    return np.where(x < 1e-2, y * y * s, np.log1p(x) - x / (1 + x))


def _ref(t, px, py, pz):
    """(ax, ay, az, phi) of one term in longdouble, straight from the formulas of include/b200nb.h"""
    ld = np.longdouble
    d = [np.asarray(p, np.float32).astype(ld) - ld(c) for p, c in zip((px, py, pz), t.centre)]
    gm, a, b = ld(t.gm), ld(t.a), ld(t.b)
    R2 = d[0] ** 2 + d[1] ** 2
    r2 = R2 + d[2] ** 2
    r = np.sqrt(r2)
    with np.errstate(divide="ignore", invalid="ignore"):
        if t.kind == 0:
            s2 = r2 + a * a
            phi = -gm / np.sqrt(s2)
            k = gm / s2 ** 1.5
            kz = k
        elif t.kind == 1:
            phi = -gm / (r + a)
            k = np.where(r > 0, gm / (r * (r + a) ** 2), 0)
            kz = k
        elif t.kind == 2:
            x = r / a
            phi = np.where(r > 0, -gm * np.log1p(x) / r, -gm / a)
            k = np.where(r > 0, gm * _mu_ld(x) / r ** 3, 0)
            kz = k
        elif t.kind == 3:
            zeta = np.sqrt(d[2] ** 2 + b * b)
            D2 = R2 + (a + zeta) ** 2
            phi = -gm / np.sqrt(D2)
            k = gm / D2 ** 1.5
            kz = k * (a + zeta) / zeta
        else:
            S = R2 + d[2] ** 2 / (b * b) + a * a
            phi = gm / 2 * np.log(S)
            k = gm / S
            kz = k / (b * b)
    return -k * d[0], -k * d[1], -kz * d[2], phi


def _points(scale):
    """fp32 points at r = 1e-9 .. 1e6 scale lengths on the axes, in the plane, off the plane, plus the centre"""
    radii = scale * 10.0 ** np.arange(-9, 6.5, 0.5)
    dirs = np.array([[1, 0, 0], [0, 1, 0], [0, 0, 1], [-1, 0, 0], [0, 0, -1], [0.6, 0.8, 0], [0.48, 0.64, 0.6],
                     [-0.3, 0.2, -0.932737905308882]])
    p = (radii[:, None, None] * dirs[None, :, :]).reshape(-1, 3)
    p = np.vstack([np.zeros((1, 3)), p]).astype(np.float32)
    return p[:, 0].copy(), p[:, 1].copy(), p[:, 2].copy()


@pytest.mark.parametrize("kind", ["plummer", "hernquist", "nfw", "miyamoto_nagai", "logarithmic"])
def test_oracle_matches_longdouble(b200, eo, kind):
    t = _kinds(b200)[kind]
    p = _points(L0)
    got = eo.eval([t], *p)
    ref = [np.asarray(x, np.longdouble) for x in _ref(t, *p)]
    amag = np.sqrt(ref[0] ** 2 + ref[1] ** 2 + ref[2] ** 2)
    for q in range(3):
        err = np.abs(got[q].astype(np.longdouble) - ref[q])
        assert np.all(err <= 1e-13 * amag), (kind, q, float(np.max(err / np.where(amag > 0, amag, 1))))
    assert np.all(np.abs(got[3] - ref[3]) <= 1e-13 * np.abs(ref[3])), kind
    if kind in ("hernquist", "nfw"):  # exactly 0 at the centre
        assert got[0][0] == 0 and got[1][0] == 0 and got[2][0] == 0


def test_terms_sum_in_order(b200, eo):
    terms = list(_kinds(b200, centre=(1e18, -2e18, 5e17)).values())
    p = _points(L0)
    acc = [np.zeros(len(p[0])) for _ in range(4)]
    for t in terms:
        one = eo.eval([t], *p)
        acc = [a + o for a, o in zip(acc, one)]
    got = eo.eval(terms, *p)
    for a, g in zip(acc, got):
        assert np.array_equal(a, g)


@pytest.mark.parametrize("kind", ["plummer", "hernquist", "nfw", "miyamoto_nagai", "logarithmic"])
def test_acceleration_is_minus_gradient(b200, eo, kind):
    t = _kinds(b200, centre=(2e18, -1e18, 3e18))[kind]
    rng = np.random.default_rng(1)
    n = 200
    r = L0 * 10.0 ** rng.uniform(-2, 2, n)
    u = rng.normal(size=(3, n))
    u /= np.linalg.norm(u, axis=0)
    p = (u * r + np.asarray(t.centre)[:, None]).astype(np.float32)
    a = eo.eval([t], *p)
    amag = np.sqrt(a[0] ** 2 + a[1] ** 2 + a[2] ** 2)
    for q in range(3):
        h = (1e-3 * np.minimum(r, 0.3 * L0)).astype(np.float32)  # below every scale length of the terms
        hi, lo = p.copy(), p.copy()
        hi[q] = (p[q] + h).astype(np.float32)
        lo[q] = (p[q] - h).astype(np.float32)
        step = hi[q].astype(np.float64) - lo[q].astype(np.float64)
        g = (eo.eval([t], *hi)[3] - eo.eval([t], *lo)[3]) / step
        assert np.all(np.abs(a[q] + g) <= 1e-5 * amag), (kind, q)


def test_nfw_series(b200, eo):
    t = b200.nfw(GM, L0)
    x = np.logspace(-12, 3, 3001)
    px = (x * L0).astype(np.float32)
    z = np.zeros_like(px)
    ax, _, _, phi = eo.eval([t], px, z, z)
    xe = px.astype(np.longdouble) / np.longdouble(L0)  # the fp32 point's own x
    r = xe * np.longdouble(L0)
    phi_ref = -np.longdouble(GM) * np.log1p(xe) / r
    a_ref = np.longdouble(GM) * _mu_ld(xe) / r ** 2
    assert np.all(np.abs(phi - phi_ref) <= 1e-12 * np.abs(phi_ref))
    assert np.all(np.abs(-ax - a_ref) <= 1e-12 * a_ref)
    # continuous across the cutoff x = 0.1: the last point of the series and the first of the log1p form
    below = np.float32(np.nextafter(np.float32(0.1 * L0), np.float32(0)))
    while below / L0 >= 0.1:
        below = np.nextafter(below, np.float32(0))
    above = np.nextafter(below, np.float32(np.inf))
    while above / L0 < 0.1:
        above = np.nextafter(above, np.float32(np.inf))
    a2 = eo.eval([t], np.array([below, above], np.float32), np.zeros(2, np.float32), np.zeros(2, np.float32))[0]
    mu2 = _mu_ld(np.array([below, above], np.longdouble) / np.longdouble(L0))
    ratio = (a2[1] / a2[0]) / float((mu2[1] / float(above) ** 2) / (mu2[0] / float(below) ** 2))
    assert abs(ratio - 1) <= 1e-13


def test_miyamoto_nagai_a0_is_plummer(b200, eo):
    b = 0.3 * L0
    p = _points(L0)
    mn = eo.eval([b200.miyamoto_nagai(GM, 0.0, b)], *p)
    pl = eo.eval([b200.plummer(GM, b)], *p)
    amag = np.sqrt(pl[0] ** 2 + pl[1] ** 2 + pl[2] ** 2)
    for q in range(3):
        assert np.all(np.abs(mn[q] - pl[q]) <= 1e-14 * amag)
    assert np.all(np.abs(mn[3] - pl[3]) <= 1e-14 * np.abs(pl[3]))


def test_struct_layout(b200):
    T = b200.ExternalTerm
    assert ctypes.sizeof(T) == 56
    assert [(f, getattr(T, f).offset) for f, _ in T._fields_] == [("kind", 0), ("reserved", 4), ("gm", 8), ("a", 16),
                                                                  ("b", 24), ("centre", 32)]
    assert b200.EXTERNAL_MAX == 8
    h = open(os.path.join(REPO, "include", "b200nb.h")).read()
    assert "#define B200NB_EXTERNAL_MAX 8" in h
    for name, v in (("PLUMMER", 0), ("HERNQUIST", 1), ("NFW", 2), ("MIYAMOTO_NAGAI", 3), ("LOGARITHMIC", 4)):
        assert re.search(rf"B200NB_EXT_{name} = {v}\b", h) and getattr(b200, f"EXT_{name}") == v


def test_constructors(b200):
    t = b200.miyamoto_nagai(1.0, 2.0, 3.0, centre=(4, 5, 6))
    assert (t.kind, t.reserved, t.gm, t.a, t.b, tuple(t.centre)) == (3, 0, 1.0, 2.0, 3.0, (4.0, 5.0, 6.0))
    assert b200.logarithmic(1.0, 2.0, 0.9).b == 0.9 and b200.nfw(1.0, 2.0).kind == b200.EXT_NFW
    assert b200.plummer(1.0, 0.0).a == 0.0  # a point mass
    assert b200.miyamoto_nagai(1.0, 0.0, 1.0).a == 0.0
    bad = [lambda: b200.plummer(-1.0, 1.0), lambda: b200.plummer(1.0, -1.0), lambda: b200.hernquist(1.0, 0.0),
           lambda: b200.nfw(1.0, 0.0), lambda: b200.nfw(np.inf, 1.0), lambda: b200.miyamoto_nagai(1.0, -1.0, 1.0),
           lambda: b200.miyamoto_nagai(1.0, 1.0, 0.0), lambda: b200.logarithmic(1.0, 0.0, 1.0),
           lambda: b200.logarithmic(1.0, 1.0, 0.0), lambda: b200.hernquist(1.0, 1.0, centre=(0, np.nan, 0)),
           lambda: b200.hernquist(1.0, 1.0, centre=(0, 0))]
    for f in bad:
        with pytest.raises(ValueError):
            f()


def test_null_context(b200):
    L = b200.lib()
    t = (b200.ExternalTerm * 1)(b200.plummer(1.0, 1.0))
    n = ctypes.c_uint()
    assert L.b200nb_set_external(None, 0, None) == b200.EINVAL
    assert L.b200nb_set_external(None, 1, t) == b200.EINVAL
    assert L.b200nb_get_external(None, t, ctypes.byref(n)) == b200.EINVAL
    assert L.b200nb_external_field(None, 0, *[None] * 7) == b200.EINVAL
    assert L.b200nb_external_field(None, 4, *[None] * 7) == b200.EINVAL


def test_new_kernels_do_not_spill(tmp_path):
    """The instantiations with terms stay in registers at their launch bounds."""
    src = os.path.join(REPO, "nbody-eurohpc_b200", "csrc", "context.cu")
    r = subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-c",
                        "-o", str(tmp_path / "ctx.o"), src], capture_output=True, text=True, cwd=REPO)
    assert r.returncode == 0, r.stderr[-2000:]
    props = dict(re.findall(r"Function properties for (\S+)\n\s*(\d+ bytes stack frame, \d+ bytes spill stores)", r.stderr))
    for name in ("integrate_kernelILb1E", "tracer_update_kernelILb1E", "energy_kernelILb1E"):
        hits = [v for k, v in props.items() if name in k]
        assert hits and all(v.startswith("0 bytes stack frame, 0 bytes spill") for v in hits), (name, hits)
