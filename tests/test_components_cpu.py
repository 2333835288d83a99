"""CPU checks of the field-by-component feature: the fp64 reference (tests/components_oracle.c) against a direct numpy sum,
two point masses and the all-body field reference; the budget helper's identities (Newton's third law, zero self force and
torque, symmetric W, the energy) and its argument checks; the C ABI's argument checks; and what the compiler makes of the
new kernels (no spills) and of the field kernels beside them (unchanged)."""
import os
import re
import subprocess

import numpy as np
import pytest

from components_oracle import ComponentsOracle
from conftest import G_F32, REPO
from field_oracle import FieldOracle

G = float(G_F32)
CSRC = os.path.join(REPO, "nbody-eurohpc_b200", "csrc")
NVCC = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17"]


@pytest.fixture(scope="module")
def co():
    return ComponentsOracle()


def _direct(d, comp, C, p, soft, skip=None):
    """numpy restatement: acc [m][C][3], phi [m][C]"""
    q = np.stack([d["qx"], d["qy"], d["qz"]], 1).astype(np.float64)
    gm = G * d["m"].astype(np.float64)
    dv = q[None, :, :] - np.asarray(p, np.float64).T[:, None, :]  # [m][n][3]
    s2 = np.sum(dv * dv, axis=2) + float(np.float32(soft)) ** 2
    gi = gm[None, :] / np.sqrt(s2)
    f = gi / s2
    if skip is not None:
        f[np.arange(len(skip)), skip] = 0.0
        gi[np.arange(len(skip)), skip] = 0.0
    acc, phi = np.zeros((dv.shape[0], C, 3)), np.zeros((dv.shape[0], C))
    for h in range(C):
        sel = comp == h
        acc[:, h] = np.einsum("mj,mjk->mk", f[:, sel], dv[:, sel])
        phi[:, h] = -gi[:, sel].sum(axis=1)
    return acc, phi


def test_oracle_matches_direct_sum(oracle, co):
    n, C = 300, 3
    d = oracle.init_bodies("galaxy", n)
    rng = np.random.default_rng(0)
    comp = rng.integers(0, C, n).astype(np.uint32)
    comp[rng.random(n) < 0.1] = 0xFFFFFFFF
    p = [(rng.normal(size=25) * 3e8).astype(np.float32) for _ in range(3)]
    for soft in (2e8, 1e4):
        acc, phi, amag = co.field(d, comp, C, *p, soft=soft)
        wa, wp = _direct(d, comp, C, p, soft)
        assert np.allclose(acc, wa, rtol=1e-12, atol=1e-12 * np.max(np.abs(wa)))
        assert np.allclose(phi, wp, rtol=1e-12, atol=0)
        assert np.all(np.linalg.norm(acc, axis=2) <= amag * (1 + 1e-12))
        idx = np.array([0, 5, 299])
        acc, phi, _ = co.bodies(d, comp, C, idx, soft=soft)
        wa, wp = _direct(d, comp, C, [d[k][idx] for k in ("qx", "qy", "qz")], soft, skip=idx)
        assert np.allclose(acc, wa, rtol=1e-12, atol=1e-12 * np.max(np.abs(wa)))
        assert np.allclose(phi, wp, rtol=1e-12, atol=0)


def test_two_point_masses(co):
    """bodies 0 and 1 in components 1 and 0, a point on the x axis between them: each component's pull is its own body's"""
    d = {k: np.zeros(2, np.float32) for k in ("qx", "qy", "qz", "vx", "vy", "vz")}
    d["qx"][:] = [-1e9, 2e9]
    d["m"] = np.array([3e24, 5e23], np.float32)
    comp = np.array([1, 0], np.uint32)
    soft = 1e3
    s2 = float(np.float32(soft)) ** 2
    p = [np.array([5e8], np.float32), np.zeros(1, np.float32), np.zeros(1, np.float32)]
    acc, phi, _ = co.field(d, comp, 2, *p, soft=soft)
    for h, j in ((0, 1), (1, 0)):
        dx = float(d["qx"][j]) - 5e8
        s = np.sqrt(dx * dx + s2)
        gm = G * float(d["m"][j])
        assert np.allclose(acc[0, h], [gm * dx / s**3, 0, 0], rtol=1e-14, atol=0)
        assert np.isclose(phi[0, h], -gm / s, rtol=1e-14)
    acc, phi, _ = co.bodies(d, comp, 2, soft=soft)
    r = 3e9
    s = np.sqrt(r * r + s2)
    # body 0 (component 1) feels only component 0, body 1 only component 1; both pulled towards the other
    assert acc[0, 1].tolist() == [0, 0, 0] and phi[0, 1] == 0 and acc[1, 0].tolist() == [0, 0, 0] and phi[1, 0] == 0
    assert np.isclose(acc[0, 0, 0], G * float(d["m"][1]) * r / s**3, rtol=1e-14)
    assert np.isclose(acc[1, 1, 0], -G * float(d["m"][0]) * r / s**3, rtol=1e-14)
    assert np.isclose(phi[1, 1], -G * float(d["m"][0]) / s, rtol=1e-14)


def test_one_component_is_the_field(oracle, co):
    n = 500
    d = oracle.init_bodies("random", n)
    rng = np.random.default_rng(1)
    p = [(rng.normal(size=30) * 3e8).astype(np.float32) for _ in range(3)]
    comp = np.zeros(n, np.uint32)
    fo = FieldOracle()
    acc, phi, amag = co.field(d, comp, 1, *p)
    ax, ay, az, fphi, famag = fo.field(d, *p)
    assert np.allclose(acc[:, 0], np.stack([ax, ay, az], 1), rtol=1e-13, atol=1e-13 * np.max(famag))
    assert np.allclose(phi[:, 0], fphi, rtol=1e-13, atol=0)
    assert np.allclose(amag[:, 0], famag, rtol=1e-13, atol=0)
    _, phib, _ = co.bodies(d, comp, 1)
    assert np.allclose(phib[:, 0], fo.potential(d), rtol=1e-13, atol=0)


def _budget_inputs(oracle, co, n=400, C=3, soft=2e8, none=True):
    d = oracle.init_bodies("galaxy", n)
    rng = np.random.default_rng(2)
    comp = rng.integers(0, C, n).astype(np.uint32)
    if none:
        comp[rng.random(n) < 0.1] = 0xFFFFFFFF
    acc, phi, _ = co.bodies(d, comp, C, soft=soft)
    return d, comp, acc, phi


def test_budget_identities(b200, oracle, co):
    C = 3
    d, comp, acc, phi = _budget_inputs(oracle, co, C=C)
    m = d["m"].astype(np.float64)
    for centre in ((0.0, 0.0, 0.0), (3e8, -1e8, 2e7)):
        b = b200.component_budget(comp, C, d["m"], d, acc, phi, centre=centre)
        mem = comp != 0xFFFFFFFF
        scale = np.sum(m[mem, None] * np.linalg.norm(acc[mem], axis=2).sum(axis=1, keepdims=True))
        r = np.stack([d[k] for k in ("qx", "qy", "qz")], 1).astype(np.float64) - np.asarray(centre)
        tscale = np.sum(m[mem] * np.linalg.norm(r[mem], axis=1) * np.linalg.norm(acc[mem], axis=2).sum(axis=1))
        assert np.all(np.abs(b["force"] + np.transpose(b["force"], (1, 0, 2))) <= 1e-13 * scale)
        assert np.all(np.abs(b["torque"] + np.transpose(b["torque"], (1, 0, 2))) <= 1e-13 * tscale)
        for g in range(C):
            assert np.all(np.abs(b["force"][g, g]) <= 1e-13 * scale)
            assert np.all(np.abs(b["torque"][g, g]) <= 1e-13 * tscale)
        assert np.allclose(b["W"], b["W"].T, rtol=1e-13, atol=0)
        for g in range(C):
            sel = comp == g
            assert np.isclose(b["mass"][g], m[sel].sum(), rtol=1e-14)
            assert np.allclose(b["com"][g], (m[sel, None] * (r[sel] + centre)).sum(0) / m[sel].sum(), rtol=1e-12)
            v = np.stack([d[k] for k in ("vx", "vy", "vz")], 1).astype(np.float64)
            assert np.allclose(b["spin"][g], (m[sel, None] * np.cross(r[sel], v[sel])).sum(0), rtol=1e-12)


def test_budget_energy_is_the_total_energy(b200, oracle, co):
    """every body in a component: sum_g K_g + (1/2) sum_gh W_gh = sum m v^2 / 2 + (1/2) sum_i m_i phi_i"""
    C = 4
    d, comp, acc, phi = _budget_inputs(oracle, co, n=700, C=C, none=False)
    b = b200.component_budget(comp, C, d["m"], d, acc, phi)
    m = d["m"].astype(np.float64)
    v2 = sum(d[k].astype(np.float64) ** 2 for k in ("vx", "vy", "vz"))
    e = np.sum(0.5 * m * v2) + 0.5 * np.sum(m * FieldOracle().potential(d))
    got = b["kinetic"].sum() + 0.5 * b["W"].sum()
    assert abs(got - e) <= 1e-12 * (np.sum(0.5 * m * v2) + 0.5 * np.sum(m * np.abs(FieldOracle().potential(d))))


def test_budget_rejects_bad_input(b200, oracle, co):
    C = 2
    d, comp, acc, phi = _budget_inputs(oracle, co, n=50, C=C)
    f = b200.component_budget
    f(comp, C, d["m"], d, acc, phi)
    for bad in (0, 65, 2.0, True, None):
        with pytest.raises(ValueError):
            f(comp, bad, d["m"], d, acc, phi)
    with pytest.raises(ValueError):
        f(np.where(comp == 0, 2, comp).astype(np.uint32), C, d["m"], d, acc, phi)  # label >= n_comp
    with pytest.raises(ValueError):
        f(comp.astype(np.float32), C, d["m"], d, acc, phi)
    with pytest.raises(ValueError):
        f(comp.reshape(5, 10), C, d["m"], d, acc, phi)
    with pytest.raises(ValueError):
        f(comp, C, d["m"][:-1], d, acc, phi)
    with pytest.raises(ValueError):
        f(comp, C, d["m"], d, acc[:, :1], phi)
    with pytest.raises(ValueError):
        f(comp, C, d["m"], d, acc, phi[:, :1])
    with pytest.raises(ValueError):
        f(comp, C, d["m"], d, acc, phi, centre=(0.0, 0.0))
    # no member at all: zero budgets, NaN centres
    none = np.full(50, 0xFFFFFFFF, np.uint32)
    b = f(none, C, d["m"], d, acc, phi)
    assert np.all(b["mass"] == 0) and np.all(b["force"] == 0) and np.all(b["W"] == 0) and np.all(np.isnan(b["com"]))


def test_null_context(b200):
    L = b200.lib()
    assert L.b200nb_component_field(None, None, 1, 1, None, None, None, None, None) == b200.EINVAL
    assert L.b200nb_component_field_bodies(None, None, 1, None, None) == b200.EINVAL


def test_new_kernels_do_not_spill(tmp_path):
    src = tmp_path / "k.cu"
    src.write_text(f'#include "{os.path.join(CSRC, "components_sm100.cuh")}"\n'
                   "template __global__ void b200nb::component_field_kernel<false>(const b200nb::CompArgs);\n"
                   "template __global__ void b200nb::component_field_kernel<true>(const b200nb::CompArgs);\n")
    r = subprocess.run(NVCC + ["-Xptxas", "-v", "-c", str(src), "-o", str(tmp_path / "k.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    props = re.findall(r"Function properties for (\S+)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads",
                       r.stdout + r.stderr)
    names = {p[0] for p in props if "component" in p[0]}
    assert len(names) == 4, props  # field (points, bodies), reduce, pack
    for name, stack, st, ld in props:
        if "component" in name:
            assert (int(stack), int(st), int(ld)) == (0, 0, 0), name


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


def test_field_kernels_unchanged_beside_the_new_file(b200, tmp_path):
    """field_kernel<false> / <true> in the library are instruction for instruction what field_sm100.cuh compiles to alone,
    so sharing field_block / field_sum_rows with components_sm100.cuh changed none of their code"""
    src = tmp_path / "f.cu"
    src.write_text(f'#include "{os.path.join(CSRC, "field_sm100.cuh")}"\n'
                   "template __global__ void b200nb::field_kernel<false>(const b200nb::FieldArgs);\n"
                   "template __global__ void b200nb::field_kernel<true>(const b200nb::FieldArgs);\n")
    obj = tmp_path / "f.o"
    subprocess.check_call(NVCC + ["-lineinfo", "-Xcompiler", "-fPIC", "-c", str(src), "-o", str(obj)])
    alone, lib = _sass(obj), _sass(b200.lib_path())
    names = [k for k in alone if k.startswith("_ZN6b200nb12field_kernel")]
    assert len(names) == 2
    for k in names:
        assert alone[k] == lib[k], k
