"""CPU checks of the tidal-tensor feature: the fp64 reference (tests/tidal_oracle.c) against the analytic point mass,
its own symmetry and trace identity, and central differences of the fp64 field reference; the C ABI's argument checks
and the Python expansion of the six columns."""
import numpy as np

from conftest import G_F32
from field_oracle import FieldOracle
from tidal_oracle import TidalOracle, matrix, six

G = float(G_F32)


def _one_body(mass, pos=(0.0, 0.0, 0.0)):
    d = {k: np.zeros(1, np.float32) for k in ("qx", "qy", "qz", "vx", "vy", "vz")}
    d["qx"][0], d["qy"][0], d["qz"][0] = pos
    d["m"] = np.array([mass], np.float32)
    return d


def test_analytic_point_mass():
    mass, r = 2e24, 3e8
    d = _one_body(mass)
    p = [np.array([v], np.float32) for v in (r, 0.0, 0.0)]
    to = TidalOracle()
    t, amag, _ = to.tidal(d, *p, soft=0.0)
    gm = G * float(np.float32(mass))
    # stretching along the line to the body, compression across it
    assert np.allclose(t[0], gm / r**3 * np.array([2.0, -1.0, -1.0, 0.0, 0.0, 0.0]), rtol=1e-13, atol=0)
    assert np.allclose(amag[0], gm / r**3 * np.array([4.0, 1.0, 1.0, 0.0, 0.0, 0.0]), rtol=1e-13, atol=0)
    # softened: T_xx = G m (3 r^2 / s^5 - 1 / s^3), T_yy = T_zz = -G m / s^3
    eps = 1e8
    t, _, _ = to.tidal(d, *p, soft=eps)
    s = np.sqrt(r * r + float(np.float32(eps)) ** 2)
    want = [gm * (3 * r * r / s**5 - 1 / s**3), -gm / s**3, -gm / s**3, 0.0, 0.0, 0.0]
    assert np.allclose(t[0], want, rtol=1e-13, atol=0)
    # the same body seen along another direction: T = G m / r^3 (3 u u^T - 1)
    u = np.array([2.0, -3.0, 6.0]) / 7.0
    p = [np.array([v], np.float32) for v in (r * u)]
    t, _, _ = to.tidal(d, *p, soft=0.0)
    pd = np.array([float(a[0]) for a in p])
    rr = np.linalg.norm(pd)
    uu = pd / rr
    want = gm / rr**3 * (3 * np.outer(uu, uu) - np.eye(3))
    assert np.allclose(matrix(t)[0], want, rtol=0, atol=1e-12 * gm / rr**3)


def test_amag_bounds_every_entry(oracle):
    d = oracle.init_bodies("galaxy", 800)
    rng = np.random.default_rng(0)
    p = [(rng.normal(size=50) * 1e9).astype(np.float32) for _ in range(3)]
    t, amag, _ = TidalOracle().tidal(d, *p)
    assert np.all(np.abs(t) <= amag * (1 + 1e-12))
    assert np.all(amag[:, :3] > 0)


def test_symmetric_under_axis_permutation(oracle):
    """Swapping the x and y axes of bodies and points swaps rows and columns of T: T'_xy = T_yx, T'_xz = T_yz, ..."""
    d = oracle.init_bodies("random", 500)
    rng = np.random.default_rng(1)
    p = [(rng.normal(size=40) * 5e8).astype(np.float32) for _ in range(3)]
    to = TidalOracle()
    t = matrix(to.tidal(d, *p)[0])
    dp = dict(d, qx=d["qy"], qy=d["qx"])
    tp = matrix(to.tidal(dp, p[1], p[0], p[2])[0])
    perm = [1, 0, 2]
    assert np.array_equal(tp, t[:, perm][:, :, perm])
    assert np.array_equal(t, np.transpose(t, (0, 2, 1)))


def test_trace_identity(oracle):
    d = oracle.init_bodies("galaxy", 1000)
    rng = np.random.default_rng(2)
    p = [(rng.normal(size=60) * 3e8).astype(np.float32) for _ in range(3)]
    to = TidalOracle()
    for soft in (2e8, 1e4, 0.0):
        t, amag, s5 = to.tidal(d, *p, soft=soft)
        tr = t[:, 0] + t[:, 1] + t[:, 2]
        want = -3.0 * float(np.float32(soft)) ** 2 * s5
        assert np.all(np.abs(tr - want) <= 1e-12 * amag[:, :3].sum(axis=1)), soft
        tb, ab, s5b = to.tidal_bodies(d, soft=soft)
        trb = tb[:, 0] + tb[:, 1] + tb[:, 2]
        assert np.all(np.abs(trb + 3.0 * float(np.float32(soft)) ** 2 * s5b) <= 1e-12 * ab[:, :3].sum(axis=1)), soft


def test_central_differences_of_the_field(oracle):
    """T_ab = d a_a / d p_b: central differences of the fp64 field at p +- h e_b, with p and h exact in fp32 and h << soft."""
    d = oracle.init_bodies("galaxy", 600)
    rng = np.random.default_rng(3)
    M, h = 40, 16384.0
    p = np.round(rng.normal(size=(3, M)) * 2e8 / 64.0) * 64.0  # multiples of 64: p +- h is exact in fp32
    assert np.array_equal(p.astype(np.float32).astype(np.float64), p)
    fo, to = FieldOracle(), TidalOracle()
    t, amag, _ = to.tidal(d, *p.astype(np.float32))
    jac = np.empty((M, 3, 3))
    for b in range(3):
        e = np.zeros((3, 1))
        e[b] = h
        ap = np.stack(fo.field(d, *(p + e).astype(np.float32))[:3], axis=1)
        am = np.stack(fo.field(d, *(p - e).astype(np.float32))[:3], axis=1)
        jac[:, :, b] = (ap - am) / (2 * h)
    assert np.all(np.abs(six(jac) - t) <= 1e-6 * amag), float(np.max(np.abs(six(jac) - t) / amag))


def test_bodies_mode_excludes_self_by_index(oracle):
    d = oracle.init_bodies("galaxy", 300)
    to = TidalOracle()
    idx = np.array([0, 7, 299], np.uint64)
    tb = to.tidal_bodies(d)[0]
    assert np.array_equal(to.tidal_bodies(d, idx)[0], tb[idx.astype(np.int64)])
    # with softening the points-mode value at a body is the bodies-mode value plus the self term -G m_i / soft^3 * I
    soft = 2e8
    i = idx.astype(np.int64)
    tp = to.tidal(d, d["qx"][i], d["qy"][i], d["qz"][i], soft=soft)[0]
    self_term = -G * d["m"][i].astype(np.float64) / float(np.float32(soft)) ** 3
    want = tb[i] + np.outer(self_term, [1, 1, 1, 0, 0, 0])
    assert np.allclose(tp, want, rtol=1e-12, atol=1e-12 * np.max(np.abs(tp)))
    # two coincident bodies see each other
    c = {k: np.zeros(2, np.float32) for k in ("qx", "qy", "qz", "vx", "vy", "vz")}
    c["m"] = np.array([1e24, 1e24], np.float32)
    tc = to.tidal_bodies(c, soft=1e4)[0]
    assert np.allclose(tc[:, :3], -G * 1e24 / float(np.float32(1e4)) ** 3, rtol=1e-6)


def test_python_expands_six_columns(b200):
    t6 = np.arange(12, dtype=np.float32).reshape(2, 6)
    t = b200.Context._tidal_matrix(t6)
    assert t.shape == (2, 3, 3) and t.dtype == np.float32
    assert np.array_equal(t, np.transpose(t, (0, 2, 1)))
    assert np.array_equal(t[1], [[6, 9, 10], [9, 7, 11], [10, 11, 8]])
    assert np.array_equal(six(t), t6)


def test_null_context(b200):
    L = b200.lib()
    assert L.b200nb_tidal(None, 1, None, None, None, None) == b200.EINVAL
    assert L.b200nb_tidal_bodies(None, None) == b200.EINVAL
