"""CPU checks of the nearest-neighbour feature: the fp32 restatement (tests/neighbors_oracle.c) against an independent
fp64 numpy brute force, its empty slots and sampling, and the C ABI's argument checks without a context."""
import numpy as np
import pytest

from neighbors_oracle import NONE, NeighborsOracle


@pytest.fixture(scope="module")
def noracle():
    return NeighborsOracle()


def _fp64_knn(d, targets, k, self_idx):
    """Index sets and sorted distances from fp64 distances; self_idx: body index of each target or None."""
    q = np.stack([d["qx"], d["qy"], d["qz"]]).astype(np.float64)
    r2 = np.sum((q[:, None, :] - targets.T[:, :, None]) ** 2, axis=0)
    if self_idx is not None:
        r2[np.arange(len(self_idx)), self_idx] = np.inf
    order = np.argsort(r2, axis=1, kind="stable")
    return order, np.sqrt(np.take_along_axis(r2, order, axis=1))


def _agree(idx, dist, order, r, k, n_cand):
    """The restatement's index set equals fp64's except where fp64 distances at the k-th boundary are within a relative
    1e-6 of each other; distances agree to fp32 rounding."""
    kk = min(k, n_cand)
    for t in range(idx.shape[0]):
        got = idx[t, :kk].astype(np.int64)
        if set(got) != set(order[t, :kk]):
            kth = r[t, kk - 1]
            near = np.abs(r[t] - kth) <= 1e-6 * kth
            assert set(got) ^ set(order[t, :kk]) <= set(order[t][near]), t
        assert np.allclose(dist[t, :kk], r[t, :kk], rtol=2e-6, atol=0), t
        assert np.all(idx[t, kk:] == NONE) and np.all(np.isinf(dist[t, kk:]))


@pytest.mark.parametrize("scheme,n", [("galaxy", 300), ("random", 257), ("random", 5)])
@pytest.mark.parametrize("k", [1, 6, 32])
def test_bodies_vs_fp64(oracle, noracle, scheme, n, k):
    d = oracle.init_bodies(scheme, n)
    idx, dist = noracle.bodies(d, k)
    q = np.stack([d["qx"], d["qy"], d["qz"]], axis=1).astype(np.float64)
    order, r = _fp64_knn(d, q, k, np.arange(n))
    _agree(idx, dist, order, r, k, n - 1)


@pytest.mark.parametrize("k", [1, 8, 32])
def test_points_vs_fp64(oracle, noracle, k):
    d = oracle.init_bodies("galaxy", 400)
    rng = np.random.default_rng(k)
    p = (rng.normal(size=(3, 150)) * 3e8).astype(np.float32)
    p[:, :5] = np.stack([d["qx"][:5], d["qy"][:5], d["qz"][:5]])  # points on bodies: distance 0
    idx, dist = noracle.points(d, *p, k)
    order, r = _fp64_knn(d, p.T.astype(np.float64), k, None)
    _agree(idx, dist, order, r, k, 400)
    assert np.array_equal(idx[:5, 0], np.arange(5)) and np.all(dist[:5, 0] == 0)


def test_ties_by_index_and_sampling(noracle):
    """Coincident bodies: distance 0, in index order; the self pair is excluded by index only."""
    n = 6
    d = {c: np.zeros(n, np.float32) for c in ("qx", "qy", "qz")}
    d["qx"][:] = [1.0, 5.0, 1.0, 1.0, 9.0, 5.0]
    idx, dist = noracle.bodies(d, 4)
    assert list(idx[0]) == [2, 3, 1, 5] and list(dist[0]) == [0, 0, 4, 4]
    assert list(idx[1]) == [5, 0, 2, 3]
    sub_idx, sub_dist = noracle.bodies(d, 4, np.array([4, 1], np.uint64))
    assert np.array_equal(sub_idx, idx[[4, 1]]) and np.array_equal(sub_dist, dist[[4, 1]])


def test_null_context(b200):
    L = b200.lib()
    assert L.b200nb_neighbors(None, 1, None, None) == b200.EINVAL
    assert L.b200nb_neighbors_at(None, 1, None, None, None, 1, None, None) == b200.EINVAL
