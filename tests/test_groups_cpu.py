"""CPU checks of the group potential and unbinding feature: the fp64 reference (tests/groups_oracle.c) against brute-force
numpy, the b200nb.bound_groups catalogue against a plain loop, and the argument checks that need no context."""
import numpy as np
import pytest

from groups_oracle import GroupsOracle

G = float(np.float32(6.67384e-11))
SOFT = 2e8
NO = 0xFFFFFFFF


@pytest.fixture(scope="module")
def goracle():
    return GroupsOracle()


def _system(n, seed):
    rng = np.random.default_rng(seed)
    centres = rng.normal(size=(3, 3)) * 1e10
    q = centres[rng.integers(0, 3, n)] + rng.normal(size=(n, 3)) * 1e9
    d = {c: q[:, i].astype(np.float32) for i, c in enumerate(("qx", "qy", "qz"))}
    d.update({c: (rng.normal(size=n) * 2e3).astype(np.float32) for c in ("vx", "vy", "vz")})
    d["m"] = (rng.random(n) * 1e24).astype(np.float32)
    d["m"][::11] = 0
    return d


def _labels(n, seed):
    rng = np.random.default_rng(seed)
    g = rng.integers(0, 6, n).astype(np.uint32)
    g[rng.random(n) < 0.2] = NO
    g[5] = 1000  # alone
    return g


def _numpy_pass(d, g):
    q = np.stack([d[c] for c in ("qx", "qy", "qz")], axis=1).astype(np.float64)
    v = np.stack([d[c] for c in ("vx", "vy", "vz")], axis=1).astype(np.float64)
    m = d["m"].astype(np.float64)
    n = len(m)
    phi, E = np.zeros(n), np.zeros(n)
    for lab in np.unique(g[g != NO]):
        idx = np.flatnonzero(g == lab)
        r = np.sqrt(np.sum((q[idx, None, :] - q[None, idx, :]) ** 2, axis=2) + SOFT * SOFT)
        t = G * m[idx][None, :] / r
        np.fill_diagonal(t, 0)
        phi[idx] = -t.sum(axis=1)
        M = m[idx].sum()
        V = (m[idx][:, None] * v[idx]).sum(axis=0) / M if M != 0 else np.zeros(3)
        E[idx] = 0.5 * np.sum((v[idx] - V) ** 2, axis=1) + phi[idx]
    return phi, E


def test_oracle_vs_numpy(goracle):
    d = _system(600, 1)
    g = _labels(600, 2)
    phi, E = goracle.unbind_pass(d, g, soft=SOFT)
    wphi, wE = _numpy_pass(d, g)
    assert np.allclose(phi, wphi, rtol=1e-12, atol=0) and np.allclose(E, wE, rtol=1e-9, atol=1e-9 * np.abs(wphi).max())
    assert phi[5] == 0 and np.all(phi[g == NO] == 0)
    idx = np.array([0, 5, 17, 599], np.uint64)
    assert np.allclose(goracle.potential(d, g, idx, soft=SOFT), wphi[idx.astype(np.int64)], rtol=1e-12, atol=0)


def test_oracle_loop(goracle):
    d = _system(400, 3)
    g = _labels(400, 4)
    bound, phi, it, conv = goracle.unbind(d, g, soft=SOFT)
    assert conv and it >= 2
    cur = g.copy()
    for _ in range(it):  # the loop restated with numpy passes
        p, E = _numpy_pass(d, cur)
        left = (cur != NO) & ~(E < 0)
        last_phi = p
        cur = np.where(left, NO, cur).astype(np.uint32)
    assert np.array_equal(bound, cur) and np.allclose(phi, last_phi, rtol=1e-12, atol=0)
    assert bound[5] == NO
    b1, _, it1, conv1 = goracle.unbind(d, g, 1, soft=SOFT)
    assert it1 == 1 and not conv1
    empty = goracle.unbind(d, np.full(400, NO, np.uint32), soft=SOFT)
    assert empty[2] == 0 and empty[3] and np.all(empty[0] == NO)


def _catalogue_loop(bound, m, st, phi, min_size):
    rows = []
    for lab in sorted(set(bound.tolist()) - {NO}):
        mem = [i for i in range(len(bound)) if bound[i] == lab]
        if len(mem) < min_size:
            continue
        M = sum(float(m[i]) for i in mem)
        com = [sum(float(m[i]) * float(st[c][i]) for i in mem) / M for c in ("qx", "qy", "qz")]
        vel = [sum(float(m[i]) * float(st[c][i]) for i in mem) / M for c in ("vx", "vy", "vz")]
        kin = sum(0.5 * float(m[i]) * sum((float(st[c][i]) - vel[k]) ** 2 for k, c in enumerate(("vx", "vy", "vz"))) for i in mem)
        pot = sum(0.5 * float(m[i]) * float(phi[i]) for i in mem)
        rows.append((-len(mem), lab, M, com, vel, kin, pot))
    rows.sort(key=lambda t: (t[0], t[1]))
    return rows


@pytest.mark.parametrize("min_size", [1, 5, 20])
def test_bound_groups_vs_loop(b200, min_size):
    rng = np.random.default_rng(min_size)
    n = 500
    bound = rng.integers(0, 12, n).astype(np.uint32) * 1000003
    bound[rng.random(n) < 0.3] = NO
    st = {c: rng.normal(size=n).astype(np.float32) * 1e3 for c in ("qx", "qy", "qz", "vx", "vy", "vz")}
    m = (rng.random(n) * 1e22).astype(np.float32)
    phi = -(rng.random(n) * 1e6).astype(np.float32)
    cat = b200.bound_groups(bound, m, st, phi, min_size)
    ref = _catalogue_loop(bound, m, st, phi, min_size)
    assert len(ref) > 1 and len(cat["label"]) == len(ref)
    assert cat["label"].dtype == np.uint32 and cat["com"].shape == (len(ref), 3)
    for g, (neg, lab, M, com, vel, kin, pot) in enumerate(ref):
        assert cat["label"][g] == lab and cat["size"][g] == -neg
        assert np.isclose(cat["mass"][g], M, rtol=1e-12, atol=0)
        assert np.allclose(cat["com"][g], com, rtol=1e-12, atol=0) and np.allclose(cat["vel"][g], vel, rtol=1e-12, atol=0)
        assert np.isclose(cat["kinetic"][g], kin, rtol=1e-10, atol=0) and np.isclose(cat["potential"][g], pot, rtol=1e-12, atol=0)


def test_bound_groups_arguments(b200):
    st = {c: np.zeros(3, np.float32) for c in ("qx", "qy", "qz", "vx", "vy", "vz")}
    b = np.array([7, 7, NO], np.uint32)
    cat = b200.bound_groups(b, np.array([0, 0, 1], np.float32), st, np.zeros(3), 1)
    assert list(cat["label"]) == [7] and list(cat["size"]) == [2] and np.all(np.isnan(cat["com"][0]))
    assert len(b200.bound_groups(np.full(3, NO, np.uint32), np.ones(3), st, np.zeros(3), 1)["label"]) == 0
    for bad in (0, -1, 2.0, True):
        with pytest.raises(ValueError):
            b200.bound_groups(b, np.ones(3), st, np.zeros(3), bad)
    for bad_b in (np.array([0, -1, 2]), np.array([0, 2**32, 1]), np.zeros(3, np.float32), np.zeros((3, 1), np.uint32)):
        with pytest.raises(ValueError):
            b200.bound_groups(bad_b, np.ones(3), st, np.zeros(3), 1)
    with pytest.raises(ValueError):
        b200.bound_groups(b, np.ones(4), st, np.zeros(3), 1)
    with pytest.raises(ValueError):
        b200.bound_groups(b, np.ones(3), st, np.zeros(2), 1)
    assert b200.NO_GROUP == NO


def test_null_context(b200):
    L = b200.lib()
    assert L.b200nb_group_potential(None, None, None) == b200.EINVAL
    assert L.b200nb_unbind(None, None, 1, None, None, None, None) == b200.EINVAL
