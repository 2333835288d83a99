"""CPU checks of the phase-space friends-of-friends feature: the fp32 restatement (tests/phase_fof_oracle.c) against
connected components of an independent fp64 link graph, its reduction to position friends-of-friends for a power-of-two
b_x and b_v = inf, the two-system case it exists for, the argument checks that need no context, the header declaration,
and the compiled kernels: no spills, and fof_sm100.cuh's kernels instruction for instruction what that file compiles to
alone."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components
from scipy.spatial import cKDTree
from scipy.spatial.distance import pdist, squareform

from conftest import REPO
from fof_oracle import FofOracle
from phase_fof_oracle import PhaseFofOracle

CSRC = os.path.join(REPO, "nbody-eurohpc_b200", "csrc")
NVCC = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17"]
KEYS = ("qx", "qy", "qz", "vx", "vy", "vz")


@pytest.fixture(scope="module")
def poracle():
    return PhaseFofOracle()


def _min_labels(labels):
    """component labels -> the smallest member index of each body's component"""
    first = np.full(labels.max() + 1, len(labels), np.int64)
    np.minimum.at(first, labels, np.arange(len(labels)))
    return first[labels].astype(np.uint32)


def _scaled64(d, b_x, b_v):
    q = np.stack([d[c] for c in KEYS], axis=1).astype(np.float64)
    q[:, :3] /= float(b_x)
    q[:, 3:] = q[:, 3:] / float(b_v) if np.isfinite(b_v) else 0.0
    return q


def _fp64_groups(d, b_x, b_v):
    adj = squareform(pdist(_scaled64(d, b_x, b_v))) <= 1.0
    return _min_labels(connected_components(coo_matrix(adj), directed=False)[1])


def _clear(d, b_x, b_v, links_per_body):
    """b_x, b_v scaled by one factor so that about `links_per_body` mean links result and no fp64 6D distance lies within
    a relative 1e-5 of the threshold (there fp32 and fp64 must decide every pair alike)."""
    r = np.sort(pdist(_scaled64(d, b_x, b_v)))
    k = min(int(links_per_body * len(d["qx"]) / 2), len(r) - 2)
    while not r[k + 1] > r[k] * (1 + 3e-5):
        k += 1
    f = np.sqrt(r[k] * r[k + 1])
    bx, bv = np.float32(b_x * f), np.float32(b_v * f)
    assert np.all(np.abs(pdist(_scaled64(d, bx, bv)) - 1.0) > 1e-5)
    return bx, bv


def _clumps(n, seed):
    """five clumps in space, each with two velocity streams: position FoF joins the streams, phase space need not"""
    rng = np.random.default_rng(seed)
    centres = rng.normal(size=(5, 3)) * 1e10
    q = centres[rng.integers(0, 5, n)] + rng.normal(size=(n, 3)) * 1e9 * rng.random((n, 1))
    v = rng.normal(size=(n, 3)) * 1e3 + np.where(rng.random((n, 1)) < 0.5, 2e4, -2e4)
    return {c: a.astype(np.float32) for c, a in zip(KEYS, list(q.T) + list(v.T))}


def _systems(oracle):
    return [("galaxy", oracle.init_bodies("galaxy", 300)), ("random", oracle.init_bodies("random", 257)),
            ("clumps", _clumps(700, 1))]


@pytest.mark.parametrize("links", [0.3, 2.0, 6.0, 40.0])
@pytest.mark.parametrize("ratio", [1e4, 1e5, np.inf])  # b_x / b_v in (m) / (m / s)
def test_restatement_vs_fp64_components(oracle, poracle, links, ratio):
    for name, d in _systems(oracle):
        q = np.stack([d[c] for c in ("qx", "qy", "qz")]).astype(np.float64)
        bx0 = float(np.median(np.linalg.norm(q - q.mean(axis=1, keepdims=True), axis=0)))
        b_x, b_v = _clear(d, bx0, bx0 / ratio if np.isfinite(ratio) else np.inf, links)
        got = poracle.groups(d, b_x, b_v)
        assert np.array_equal(got, _fp64_groups(d, b_x, b_v)), name
        assert np.all(got <= np.arange(len(got)))


@pytest.mark.parametrize("k", [20, 24, 27, 31, 34])
def test_power_of_two_bx_is_position_fof(oracle, poracle, k):
    """b_x = 2^k and b_v = inf: every scaling is exact, so the labels are fof_oracle's at b = b_x, whatever the ties."""
    foracle = FofOracle()
    for name, d in _systems(oracle) + [("lattice", _lattice(2.0 ** (k - 1)))]:
        b = np.float32(2.0 ** k)
        assert np.array_equal(poracle.groups(d, b, np.inf), foracle.groups(d, b)), (name, k)


def _lattice(h):
    g = np.arange(5, dtype=np.float32) * np.float32(h)
    X, Y, Z = np.meshgrid(g, g, g, indexing="ij")
    d = {"qx": X.ravel(), "qy": Y.ravel(), "qz": Z.ravel()}
    for c in ("vx", "vy", "vz"):
        d[c] = np.random.default_rng(0).normal(size=125).astype(np.float32) * 1e3
    return d


def test_restatement_extremes(poracle):
    d = _clumps(500, 2)
    n = 500
    assert np.array_equal(poracle.groups(d, 1.0, 1e-3), np.arange(n))  # no two bodies that close
    assert np.all(poracle.groups(d, np.inf, np.inf) == 0)  # both parts switched off: one group
    assert np.all(poracle.groups(d, 1e15, 1e15) == 0)
    # an overflowing scale (tiny b_v) and non-finite coordinates keep a body alone
    e = {c: d[c].copy() for c in KEYS}
    e["qx"][11], e["vy"][12], e["vz"][13] = np.nan, np.inf, -np.inf
    g = poracle.groups(e, np.inf, np.inf)
    assert list(g[11:14]) == [11, 12, 13] and np.all(np.delete(g, [11, 12, 13]) == 0)
    assert np.array_equal(poracle.groups(d, np.inf, np.float32(1e-40)), np.arange(n))


def test_ties(poracle):
    """Velocity lattice of spacing 1.0 and b_v = 1: d2 = 1 exactly between neighbours, so they link; a pair one fp32 step
    further apart does not."""
    g = np.arange(6, dtype=np.float32)
    X, Y, Z = np.meshgrid(g, g, g, indexing="ij")
    d = {"vx": X.ravel(), "vy": Y.ravel(), "vz": Z.ravel()}
    for c in ("qx", "qy", "qz"):
        d[c] = np.zeros(216, np.float32)
    assert np.all(poracle.groups(d, 1.0, 1.0) == 0)
    pair = {c: np.zeros(2, np.float32) for c in KEYS}
    pair["vx"][1] = 1.0
    assert list(poracle.groups(pair, np.inf, 1.0)) == [0, 0]
    pair["vx"][1] = np.nextafter(np.float32(1), np.float32(2))
    assert list(poracle.groups(pair, np.inf, 1.0)) == [0, 1]


def two_systems(init_bodies, n=10000):
    """Two galaxy-scheme systems (seeds 1 and 2), the second shifted by +1e8 m in x and -1e4 m/s in vx: they overlap."""
    a, b = init_bodies("galaxy", n, seed=1), init_bodies("galaxy", n, seed=2)
    b = dict(b, qx=(b["qx"] + np.float32(1e8)).astype(np.float32), vx=(b["vx"] - np.float32(1e4)).astype(np.float32))
    return {c: np.concatenate([a[c], b[c]]) for c in KEYS + ("m",)}


def test_two_overlapping_systems(oracle, poracle):
    d = two_systems(oracle.init_bodies)
    n = len(d["qx"]) // 2
    q = np.stack([d[c] for c in ("qx", "qy", "qz")], axis=1).astype(np.float64)
    b = float(np.median(cKDTree(q).query(q, 5)[0][:, 4]))
    truth = np.repeat([0, 1], n)
    pos = FofOracle().groups(d, b)
    big = np.bincount(pos).argmax()
    assert np.all(np.bincount(truth[pos == big], minlength=2) > 1000)  # position FoF mixes the systems
    for b_v in (2000.0, 3000.0):
        g = poracle.groups(d, 2 * b, b_v)
        sizes = np.bincount(g, minlength=2 * n)
        roots = np.flatnonzero(sizes >= 20)
        assert len(roots) == 2, sizes[roots]
        for r in roots:
            assert len(np.unique(truth[g == r])) == 1 and sizes[r] > 9000


def test_b_checks(b200):
    check = b200.Context._fof_phase_b
    assert check(1, "b") == 1.0 and check(np.float32(2), "b") == 2.0 and check(np.inf, "b") == np.inf
    assert check(3e38, "b") == np.float32(3e38) and check(1e-40, "b") == np.float32(1e-40)
    for bad in (0, 0.0, -0.0, -1.0, -np.inf, np.nan, 1e39, 1e-50, True, "1", None, [1.0]):
        with pytest.raises(ValueError):
            check(bad, "b")


def test_null_context(b200):
    assert b200.lib().b200nb_fof_phase(None, 1.0, 1.0, None) == b200.EINVAL


def test_header_declaration(b200):
    text = open(os.path.join(REPO, "include", "b200nb.h")).read()
    assert "int b200nb_fof_phase(b200nb_ctx *ctx, float b_x, float b_v, uint32_t *group);" in text
    assert "b200nb_fof_phase" in b200.header_functions()
    assert hasattr(ctypes.CDLL(b200.lib_path()), "b200nb_fof_phase")


def test_new_kernels_do_not_spill(tmp_path):
    src = tmp_path / "k.cu"
    src.write_text(f'#include "{os.path.join(CSRC, "phase_fof_sm100.cuh")}"\n')
    r = subprocess.run(NVCC + ["-Xptxas", "-v", "-c", str(src), "-o", str(tmp_path / "k.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    out = r.stdout + r.stderr
    props = re.findall(r"Function properties for (\S+)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads",
                       out)
    names = {p[0] for p in props if "phase_fof" in p[0]}
    assert len(names) == 2, props  # link, pack
    for name, stack, st, ld in props:
        if "phase_fof" in name:
            assert (int(stack), int(st), int(ld)) == (0, 0, 0), name
    regs = dict(re.findall(r"Compiling entry function '(\S+)' for 'sm_100a'\nptxas info\s*: Function properties for \S+\n.*\nptxas info\s*: Used (\d+) registers", out))
    link = [k for k in regs if "phase_fof_link" in k]
    assert link and int(regs[link[0]]) <= 128  # 4 CTAs of 128 threads per SM


def _sass(path):
    out = subprocess.run(["cuobjdump", "-sass", str(path)], capture_output=True, text=True, check=True).stdout
    res, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            res[cur] = []
        elif cur and re.match(r"\s*/\*[0-9a-f]{4,}\*/", line):
            res[cur].append(re.sub(r"\s+", " ", line.strip()))
    return res


@pytest.mark.parametrize("header,pattern,count", [("fof_sm100.cuh", r"_ZN6b200nb\d+fof_", 4),
                                                 ("phase_fof_sm100.cuh", r"_ZN6b200nb\d+phase_fof_", 2)])
def test_kernels_as_compiled_alone(b200, tmp_path, header, pattern, count):
    """The position friends-of-friends kernels in the library are instruction for instruction what fof_sm100.cuh compiles
    to alone, so the phase-space kernels that share its union-find changed none of their code; and the new kernels are
    what their own header compiles to."""
    src = tmp_path / "f.cu"
    src.write_text(f'#include "{os.path.join(CSRC, header)}"\n')
    obj = tmp_path / "f.o"
    subprocess.check_call(NVCC + ["-lineinfo", "-Xcompiler", "-fPIC", "-c", str(src), "-o", str(obj)])
    alone, lib = _sass(obj), _sass(b200.lib_path())
    names = [k for k in alone if re.match(pattern, k)]
    assert len(names) == count, list(alone)
    for k in names:
        assert alone[k] == lib[k], k
