"""CPU checks of the basis-function expansion: the long-double restatement (tests/scf_oracle.c) against an independent
scipy restatement of the definition (eval_gegenbauer, lpmv, gammaln, atan2), its gradient against finite differences, the
known Hernquist coefficients, an fp64 replay of the recurrences the kernels run (the accuracy bound of the header), the
argument checks that need no context, the header declaration, and the compiled kernels: no spills, and every kernel of
the pre-existing headers instruction for instruction what that header compiles to alone."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest
from scipy.special import eval_gegenbauer, factorial, gammaln, lpmv

from conftest import REPO
from scf_oracle import ScfOracle, packed

CSRC = os.path.join(REPO, "nbody-eurohpc_b200", "csrc")
NVCC = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17"]
A_SCALE = 1.0e17  # m; bodies stay within 50 a, below the ~1.8e19 m where the force pass's fp32 d2 overflows


@pytest.fixture(scope="module")
def so():
    return ScfOracle()


def _norm(n, l, m, a):
    K = 0.5 * n * (n + 4 * l + 3) + (l + 1) * (2 * l + 1)
    lg = (8 * l + 6) * np.log(2) + gammaln(n + 1) + np.log(n + 2 * l + 1.5) + 2 * gammaln(2 * l + 1.5) - np.log(4 * np.pi * K) - \
        gammaln(n + 4 * l + 3)
    return (2 - (m == 0)) * -np.exp(lg) * (2 * l + 1) * factorial(l - m) / factorial(l + m) / a


def _sph(q, c, a):
    d = np.stack(q, axis=1).astype(np.float64) - np.asarray(c)
    r = np.linalg.norm(d, axis=1)
    return r / a, np.where(r > 0, d[:, 2] / np.where(r > 0, r, 1), 0.0), np.arctan2(d[:, 1], d[:, 0])


def _phit(n, l, s):
    return -s ** l / (1 + s) ** (2 * l + 1) * eval_gegenbauer(n, 2 * l + 1.5, (s - 1) / (s + 1))


def scipy_coefficients(q, gm, nmax, lmax, a, c):
    s, ct, ph = _sph(q, c, a)
    S = np.zeros((nmax + 1, lmax + 1, lmax + 1))
    T = np.zeros_like(S)
    for n in range(nmax + 1):
        for l in range(lmax + 1):
            for m in range(l + 1):
                w = _norm(n, l, m, a) * gm.astype(np.float64) * _phit(n, l, s) * lpmv(m, l, ct)
                S[n, l, m], T[n, l, m] = w @ np.cos(m * ph), (w @ np.sin(m * ph) if m else 0.0)
    return S, T


def scipy_phi(S, T, a, c, p):
    s, ct, ph = _sph(p, c, a)
    out = np.zeros(len(s))
    for n in range(S.shape[0]):
        for l in range(S.shape[1]):
            for m in range(l + 1):
                out += _phit(n, l, s) * lpmv(m, l, ct) * (S[n, l, m] * np.cos(m * ph) + T[n, l, m] * np.sin(m * ph))
    return out


def hernquist_sample(n, a, seed, flatten=(1.0, 1.0, 1.0), offset=(0.0, 0.0, 0.0), rmax=50.0):
    """n bodies of a Hernquist sphere of scale a (units of a inside), optionally flattened and offset; fp32 positions"""
    rng = np.random.default_rng(seed)
    u = rng.random(n)
    s = np.sqrt(u) / (1 - np.sqrt(u))
    v = rng.normal(size=(n, 3))
    v /= np.linalg.norm(v, axis=1)[:, None]
    P = v * s[:, None] * np.asarray(flatten) + np.asarray(offset)
    P[np.linalg.norm(P, axis=1) > rmax] *= 0.5 ** 4  # keep the far tail bounded without changing n
    return [(P[:, k] * a).astype(np.float32) for k in range(3)]


def _bodies(n, seed, a=A_SCALE):
    q = hernquist_sample(n, a, seed, flatten=(1.0, 0.8, 0.5), offset=(0.15, -0.1, 0.05))
    gm = (np.random.default_rng(seed + 7).random(n) * 2e9 + 1e9).astype(np.float32)
    return q, gm


@pytest.mark.parametrize("nmax,lmax", [(0, 0), (4, 3), (8, 6)])
def test_oracle_coefficients_vs_scipy(so, nmax, lmax):
    q, gm = _bodies(300, 1)
    c = (0.1 * A_SCALE, -0.05 * A_SCALE, 0.02 * A_SCALE)
    S, T, Ss, Ts = so.coefficients(q, gm, nmax, lmax, A_SCALE, c)
    S2, T2 = scipy_coefficients(q, gm, nmax, lmax, A_SCALE, c)
    assert np.all(np.abs(S - S2) <= 1e-11 * Ss + 1e-300)
    assert np.all(np.abs(T - T2) <= 1e-11 * Ts + 1e-300)
    assert np.all(Ss[:, np.triu_indices(lmax + 1, 1)[0], np.triu_indices(lmax + 1, 1)[1]] == 0)


def test_oracle_field_vs_scipy_and_gradient(so):
    q, gm = _bodies(400, 2)
    c = (0.0, 0.0, 0.0)
    S, T, _, _ = so.coefficients(q, gm, 6, 4, A_SCALE, c)
    rng = np.random.default_rng(3)
    x = rng.normal(size=(64, 3))
    x *= (rng.uniform(0.2, 4, 64) / np.linalg.norm(x, axis=1))[:, None] * A_SCALE
    p = [x[:, k].astype(np.float32) for k in range(3)]
    ax, ay, az, phi, sa, sphi = so.field(S, T, A_SCALE, c, *p)
    assert np.all(np.abs(phi - scipy_phi(S, T, A_SCALE, c, p)) <= 1e-11 * sphi)
    # central differences of the oracle's Phi over fp32 points; step h = 2^k, about 1e-4 a
    for k, ak in enumerate((ax, ay, az)):
        h = 2.0 ** np.floor(np.log2(A_SCALE * 1e-4))
        pp = [a.copy() for a in p]
        pm = [a.copy() for a in p]
        pp[k] = (p[k].astype(np.float64) + h).astype(np.float32)
        pm[k] = (p[k].astype(np.float64) - h).astype(np.float32)
        dx = pp[k].astype(np.float64) - pm[k].astype(np.float64)
        fd = -(so.field(S, T, A_SCALE, c, *pp)[3] - so.field(S, T, A_SCALE, c, *pm)[3]) / dx
        assert np.all(np.abs(fd - ak) <= 1e-5 * (sa[k] + np.abs(ak))), k


def test_oracle_hernquist_monopole(so):
    a, n, GM = A_SCALE, 20000, 4e20
    q = hernquist_sample(n, a, 1, rmax=1e30)
    gm = np.full(n, GM / n, np.float32)
    S, T, _, _ = so.coefficients(q, gm, 2, 2, a)
    assert abs(S[0, 0, 0] / (GM / a) - 1) < 2e-2
    rest = np.abs(S).ravel()[1:]
    assert rest.max() < 5e-2 * GM / a and np.abs(T).max() < 5e-2 * GM / a
    # the exact Hernquist potential from S_000 = GM/a alone
    S1 = np.zeros((1, 1, 1))
    S1[0, 0, 0] = GM / a
    r = np.array([0.1, 1.0, 3.0, 10.0]) * a
    z = np.zeros(4, np.float32)
    phi = so.field(S1, np.zeros_like(S1), a, (0, 0, 0), r.astype(np.float32), z, z)[3]
    assert np.allclose(phi, -GM / (r.astype(np.float32).astype(np.float64) + a), rtol=1e-15)


def _tables():
    """the host tables of scf_sm100.cuh (context.cu: scf_tables), here in fp64 with numpy's long double"""
    L = np.longdouble
    ga, gb = np.zeros((16, 32)), np.zeros((16, 32))
    for l in range(16):
        al = L(2 * l) + L(1.5)
        for n in range(1, 32):
            ga[l, n] = np.float64(L(2) * (n + al - 1) / n)
            gb[l, n] = np.float64((n + 2 * al - 2) / n)
    qa, qb, qs = np.zeros((17, 17)), np.zeros((17, 17)), np.zeros(17)
    df = L(1)
    for m in range(17):
        if m:
            df *= 2 * m - 1
        qs[m] = np.float64(-df if m % 2 else df)
        for l in range(m + 1, 17):
            qa[l, m] = np.float64(L(2 * l - 1) / (l - m))
            qb[l, m] = np.float64(L(l + m - 1) / (l - m))
    return ga, gb, qa, qb, qs


def replay_coefficients(q, gm, nmax, lmax, a, c):
    """the coefficient kernel's per-body fp64 recurrences and products (sums in index order, np.float64), normalised
    with the oracle's long-double F: the accuracy that fp64 recurrences give, without a GPU"""
    ga, gb, qa, qb, qs = _tables()
    d = np.stack(q, axis=1).astype(np.float64) - np.asarray(c)
    r = np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2])
    s = r / a
    xi = (s - 1.0) / (s + 1.0)
    x = np.where(r > 0, d[:, 2] / np.where(r > 0, r, 1), 0.0)
    wr = np.where(r > 0, d[:, 0] / np.where(r > 0, r, 1), 0.0)
    wi = np.where(r > 0, d[:, 1] / np.where(r > 0, r, 1), 0.0)
    qq = 1.0 / (1.0 + s)
    t = s * qq * qq
    S = np.zeros((nmax + 1, lmax + 1, lmax + 1))
    T = np.zeros_like(S)
    rad = np.zeros((lmax + 1, nmax + 1, len(s)))
    for l in range(lmax + 1):
        P = qq.copy()
        for _ in range(l):
            P = P * t
        w = -(P * gm.astype(np.float64))
        cp, cc = np.zeros_like(s), np.ones_like(s)
        rad[l, 0] = w
        for n in range(1, nmax + 1):
            cn = ga[l, n] * xi * cc - gb[l, n] * cp
            cp, cc = cc, cn
            rad[l, n] = w * cn
    cm, sm = np.ones_like(s), np.zeros_like(s)
    for m in range(lmax + 1):
        qp, qv = np.zeros_like(s), np.full_like(s, qs[m])
        for l in range(m, lmax + 1):
            if l > m:
                qn = qa[l, m] * x * qv - qb[l, m] * qp
                qp, qv = qv, qn
            S[:, l, m] = rad[l] @ (qv * cm)
            T[:, l, m] = rad[l] @ (qv * sm) if m else 0.0
        cm, sm = cm * wr - sm * wi, cm * wi + sm * wr
    for n in range(nmax + 1):
        for l in range(lmax + 1):
            for m in range(l + 1):
                f = _norm(n, l, m, a)
                S[n, l, m] *= f
                T[n, l, m] *= f
    return S, T


def test_fp64_recurrences_within_the_bound(so):
    """the header's 1e-12 bound, for the largest expansion, against the long-double restatement"""
    q, gm = _bodies(3000, 4)
    c = (0.15 * A_SCALE, -0.1 * A_SCALE, 0.05 * A_SCALE)
    S, T, Ss, Ts = so.coefficients(q, gm, 31, 15, A_SCALE, c)
    S2, T2 = replay_coefficients(q, gm, 31, 15, A_SCALE, c)
    assert np.all(np.abs(S2 - S) <= 1e-12 * Ss)
    assert np.all(np.abs(T2 - T) <= 1e-12 * Ts)


def test_arg_checks(b200):
    check = b200.Context._scf_args
    assert check(0, 0, 1.0, (0, 0, 0))[:3] == (0, 0, 1.0)
    assert check(31, 15, 3e19, [1.0, 2.0, 3.0])[:2] == (31, 15)
    for bad in [(32, 0, 1.0, (0, 0, 0)), (0, 16, 1.0, (0, 0, 0)), (-1, 0, 1.0, (0, 0, 0)), (0, 0, 0.0, (0, 0, 0)),
                (0, 0, -1.0, (0, 0, 0)), (0, 0, np.inf, (0, 0, 0)), (0, 0, np.nan, (0, 0, 0)), (0, 0, 1.0, (0, 0)),
                (0, 0, 1.0, (0, np.nan, 0)), (0, 0, 1.0, (np.inf, 0, 0)), (1.5, 0, 1.0, (0, 0, 0)), (True, 0, 1.0, (0, 0, 0))]:
        with pytest.raises(ValueError):
            check(*bad)


def test_null_context(b200):
    L = b200.lib()
    c = (ctypes.c_double * 3)(0, 0, 0)
    S = (ctypes.c_double * 1)()
    assert L.b200nb_scf_coefficients(None, 0, 0, 1.0, c, None, 0, S, S) == b200.EINVAL
    assert L.b200nb_scf_field(None, 0, 0, 1.0, c, S, S, 0, None, None, None, None, None, None, None) == b200.EINVAL


def test_packing_roundtrip(b200):
    rng = np.random.default_rng(0)
    P = rng.normal(size=(4, 21))
    C = b200._scf_unpack(P.ravel(), 3, 5)
    assert np.all(np.triu(C[0], 1) == 0) and np.array_equal(b200._scf_pack(C), P) and np.array_equal(packed(C), P)


def test_header_declaration(b200):
    text = open(os.path.join(REPO, "include", "b200nb.h")).read()
    assert ("int b200nb_scf_coefficients(b200nb_ctx *ctx, uint32_t nmax, uint32_t lmax, double a, const double centre[3],\n"
            "                            const uint32_t *group, uint32_t label, double *S, double *T);") in text
    assert "int b200nb_scf_field(b200nb_ctx *ctx, uint32_t nmax, uint32_t lmax, double a, const double centre[3], const double *S," in text
    for f in ("b200nb_scf_coefficients", "b200nb_scf_field"):
        assert f in b200.header_functions()
        assert hasattr(ctypes.CDLL(b200.lib_path()), f)


def _compile(tmp_path, header, extra=()):
    src = tmp_path / "k.cu"
    src.write_text(f'#include "{os.path.join(CSRC, header)}"\n')
    obj = tmp_path / "k.o"
    r = subprocess.run(NVCC + list(extra) + ["-c", str(src), "-o", str(obj)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return obj, r.stdout + r.stderr


def test_new_kernels_do_not_spill(tmp_path):
    _, out = _compile(tmp_path, "scf_sm100.cuh", ["-Xptxas", "-v"])
    props = re.findall(r"Function properties for (\S+)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads",
                       out)
    names = {p[0] for p in props if "scf_" in p[0]}
    assert len(names) == 3, props  # coefficients, reduce, field
    for name, stack, st, ld in props:
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


@pytest.mark.parametrize("header", ["field_sm100.cuh", "neighbors_sm100.cuh", "fof_sm100.cuh", "phase_fof_sm100.cuh",
                                    "groups_sm100.cuh", "tidal_sm100.cuh", "components_sm100.cuh", "external_sm100.cuh",
                                    "scf_sm100.cuh"])
def test_kernels_as_compiled_alone(b200, tmp_path, header):
    """Every kernel a header compiles to on its own is, instruction for instruction, the one in the library: the new
    header and its host code changed no existing kernel, and the new kernels are what scf_sm100.cuh compiles to."""
    obj, _ = _compile(tmp_path, header, ["-lineinfo", "-Xcompiler", "-fPIC"])
    alone, lib = _sass(obj), _sass(b200.lib_path())
    names = [k for k in alone if k in lib]
    assert len(names) == len(alone), (sorted(alone), header)
    for k in names:
        assert alone[k] == lib[k], k
