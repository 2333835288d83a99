"""CPU checks of the friends-of-friends feature: the fp32 restatement (tests/fof_oracle.c) against connected components
of an independent fp64 link graph, the b200nb.fof_groups catalogue against a plain loop, and the argument checks of the
Python and C entry points that need no context."""
import numpy as np
import pytest
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components
from scipy.spatial.distance import pdist, squareform

from fof_oracle import FofOracle


@pytest.fixture(scope="module")
def foracle():
    return FofOracle()


def _min_labels(labels):
    """component labels -> the smallest member index of each body's component"""
    first = np.full(labels.max() + 1, len(labels), np.int64)
    np.minimum.at(first, labels, np.arange(len(labels)))
    return first[labels].astype(np.uint32)


def _fp64_groups(d, b):
    q = np.stack([d["qx"], d["qy"], d["qz"]], axis=1).astype(np.float64)
    adj = squareform(pdist(q)) <= b
    return _min_labels(connected_components(coo_matrix(adj), directed=False)[1])


def _clear_b(d, links_per_body):
    """A linking length at about `links_per_body` mean links, moved up to a gap in the fp64 pair distances so that no
    distance lies within a relative 1e-5 of it (there fp32 and fp64 must decide every pair alike)."""
    q = np.stack([d["qx"], d["qy"], d["qz"]], axis=1).astype(np.float64)
    r = np.sort(pdist(q))
    k = min(int(links_per_body * len(q) / 2), len(r) - 2)
    while not r[k + 1] > r[k] * (1 + 3e-5):
        k += 1
    b = np.float32(np.sqrt(r[k] * r[k + 1]))
    assert np.all(np.abs(r - b) > 1e-5 * b)
    return b


def _clumps(n, seed):
    rng = np.random.default_rng(seed)
    centres = rng.normal(size=(5, 3)) * 1e10
    q = centres[rng.integers(0, 5, n)] + rng.normal(size=(n, 3)) * 1e9 * rng.random((n, 1))
    return {c: q[:, i].astype(np.float32) for i, c in enumerate(("qx", "qy", "qz"))}


def _systems(oracle):
    return [("galaxy", oracle.init_bodies("galaxy", 300)), ("random", oracle.init_bodies("random", 257)),
            ("clumps", _clumps(700, 1))]


@pytest.mark.parametrize("links", [0.3, 2.0, 6.0, 40.0])
def test_restatement_vs_fp64_components(oracle, foracle, links):
    for name, d in _systems(oracle):
        b = _clear_b(d, links)
        got = foracle.groups(d, b)
        assert np.array_equal(got, _fp64_groups(d, float(b))), name
        assert np.all(got <= np.arange(len(got)))


def test_restatement_extremes(oracle, foracle):
    d = _clumps(500, 2)
    n = len(d["qx"])
    assert np.array_equal(foracle.groups(d, 0.0), np.arange(n))  # no two bodies coincide
    assert np.all(foracle.groups(d, 1e15) == 0)  # b above the diameter: one group
    # coincident bodies link at b = 0; non-finite positions never link
    e = {c: d[c].copy() for c in ("qx", "qy", "qz")}
    e["qx"][7], e["qy"][7], e["qz"][7] = e["qx"][3], e["qy"][3], e["qz"][3]
    e["qx"][11], e["qy"][12], e["qz"][13] = np.nan, np.inf, -np.inf
    g0 = foracle.groups(e, 0.0)
    assert g0[7] == 3 and np.array_equal(np.delete(g0, 7), np.delete(np.arange(n), 7))
    g = foracle.groups(e, 1e15)
    assert list(g[11:14]) == [11, 12, 13] and np.all(np.delete(g, [11, 12, 13]) == 0)


def test_restatement_lattice_ties(foracle):
    """Spacing 1.0: d2 = 1 exactly between lattice neighbours, so b = 1 links them and the next fp32 below does not."""
    g = np.arange(6, dtype=np.float32)
    X, Y, Z = np.meshgrid(g, g, g, indexing="ij")
    d = {"qx": X.ravel(), "qy": Y.ravel(), "qz": Z.ravel()}
    assert np.all(foracle.groups(d, 1.0) == 0)
    assert np.array_equal(foracle.groups(d, np.nextafter(np.float32(1), np.float32(0))), np.arange(216))


def _catalogue_loop(group, m, st, min_size):
    rows = []
    for root in sorted(set(group.tolist())):
        mem = [i for i in range(len(group)) if group[i] == root]
        if len(mem) < min_size:
            continue
        M = sum(float(m[i]) for i in mem)
        com = [sum(float(m[i]) * float(st[c][i]) for i in mem) / M for c in ("qx", "qy", "qz")]
        vel = [sum(float(m[i]) * float(st[c][i]) for i in mem) / M for c in ("vx", "vy", "vz")]
        rows.append((-len(mem), root, M, com, vel))
    rows.sort(key=lambda t: (t[0], t[1]))
    return rows


@pytest.mark.parametrize("min_size", [1, 5, 20])
def test_fof_groups_vs_loop(b200, foracle, min_size):
    d = _clumps(600, 3)
    rng = np.random.default_rng(min_size)
    st = dict(d, **{c: rng.normal(size=600).astype(np.float32) * 1e3 for c in ("vx", "vy", "vz")})
    m = (rng.random(600) * 1e22).astype(np.float32)
    group = foracle.groups(d, 3e8)
    cat = b200.fof_groups(group, m, st, min_size)
    ref = _catalogue_loop(group, m, st, min_size)
    assert len(ref) > 1 and len(cat["root"]) == len(ref)
    assert cat["root"].dtype == np.uint32 and cat["com"].shape == (len(ref), 3)
    for g, (neg, root, M, com, vel) in enumerate(ref):
        assert cat["root"][g] == root and cat["size"][g] == -neg
        assert np.isclose(cat["mass"][g], M, rtol=1e-12, atol=0)
        assert np.allclose(cat["com"][g], com, rtol=1e-12, atol=0) and np.allclose(cat["vel"][g], vel, rtol=1e-12, atol=0)


def test_fof_groups_arguments(b200):
    st = {c: np.zeros(3, np.float32) for c in ("qx", "qy", "qz", "vx", "vy", "vz")}
    g = np.array([0, 0, 2], np.uint32)
    cat = b200.fof_groups(g, np.array([0, 0, 1], np.float32), st, 1)
    assert list(cat["root"]) == [0, 2] and list(cat["size"]) == [2, 1] and np.all(np.isnan(cat["com"][0]))
    assert len(b200.fof_groups(g, np.ones(3), st, 3)["root"]) == 0
    for bad in (0, -1, 2.0, True):
        with pytest.raises(ValueError):
            b200.fof_groups(g, np.ones(3), st, bad)
    with pytest.raises(ValueError):
        b200.fof_groups(np.array([0, 3, 2]), np.ones(3), st, 1)
    with pytest.raises(ValueError):
        b200.fof_groups(g, np.ones(4), st, 1)


def test_b_checks(b200):
    check = b200.Context._fof_b
    assert check(0) == 0.0 and check(1.5) == 1.5 and check(np.float32(2)) == 2.0 and check(1.8e19) == np.float32(1.8e19)
    for bad in (-1.0, -1e-30, np.nan, np.inf, 2e19, 1e39, True, "1", None, [1.0]):
        with pytest.raises(ValueError):
            check(bad)


def test_null_context(b200):
    assert b200.lib().b200nb_fof(None, 1.0, None) == b200.EINVAL
