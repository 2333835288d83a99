"""CPU checks of the frozen expansion as an external potential (b200nb_set_external_scf): the header declarations and
exports, the Python argument checks, the NULL-context errors, and the compiled kernels: no spills in ext_total_kernel
(both point loaders) and the three consumer instantiations that read its output, and the library's evaluator,
external-term and new kernels instruction for instruction what their headers compile to alone."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import REPO
from test_scf_cpu import CSRC, NVCC, _sass


def _coefs(nmax, lmax, seed=0):
    rng = np.random.default_rng(seed)
    S = rng.normal(size=(nmax + 1, lmax + 1, lmax + 1))
    T = rng.normal(size=S.shape)
    T[:, :, 0] = 0.0
    for C in (S, T):
        C[:, np.triu_indices(lmax + 1, 1)[0], np.triu_indices(lmax + 1, 1)[1]] = 0.0
    return S, T


def test_header_declarations(b200):
    text = open(os.path.join(REPO, "include", "b200nb.h")).read()
    assert ("int b200nb_set_external_scf(b200nb_ctx *ctx, uint32_t nmax, uint32_t lmax, double a, const double centre[3],\n"
            "                            const double *S, const double *T);") in text
    assert ("int b200nb_get_external_scf(const b200nb_ctx *ctx, uint32_t *present, uint32_t *nmax, uint32_t *lmax, double *a,\n"
            "                            double centre[3], double *S, double *T);") in text
    for f in ("b200nb_set_external_scf", "b200nb_get_external_scf"):
        assert f in b200.header_functions()
        assert hasattr(ctypes.CDLL(b200.lib_path()), f)


def test_arg_checks(b200):
    check = b200.Context._external_scf_args
    S, T = _coefs(3, 2)
    nmax, lmax, a, c, Sp, Tp = check(S, T, 2.0, (1, 2, 3))
    assert (nmax, lmax, a, tuple(c)) == (3, 2, 2.0, (1.0, 2.0, 3.0))
    assert np.array_equal(Sp, b200._scf_pack(S)) and np.array_equal(Tp, b200._scf_pack(T))
    S0, T0 = _coefs(0, 0)
    assert check(S0, T0, 1.0, (0, 0, 0))[:2] == (0, 0)
    S1, T1 = _coefs(31, 15)
    assert check(S1, T1, 1.0, (0, 0, 0))[:2] == (31, 15)
    T_nl0 = T.copy()
    T_nl0[1, 2, 0] = 1e-30
    S_nan, S_inf, T_nan = S.copy(), S.copy(), T.copy()
    S_nan[0, 1, 1] = np.nan
    S_inf[2, 0, 0] = np.inf
    T_nan[3, 2, 2] = -np.inf
    S32, T32 = _coefs(32, 0)
    S16, T16 = _coefs(0, 16)
    bad = [(S, None, 1.0, (0, 0, 0)), (None, T, 1.0, (0, 0, 0)), (S, T[:2], 1.0, (0, 0, 0)),
           (S[:, :, :2], T[:, :, :2], 1.0, (0, 0, 0)), (S[0], T[0], 1.0, (0, 0, 0)), (S32, T32, 1.0, (0, 0, 0)),
           (S16, T16, 1.0, (0, 0, 0)), (S_nan, T, 1.0, (0, 0, 0)), (S_inf, T, 1.0, (0, 0, 0)), (S, T_nan, 1.0, (0, 0, 0)),
           (S, T_nl0, 1.0, (0, 0, 0)), (S, T, 0.0, (0, 0, 0)), (S, T, None, (0, 0, 0)), (S, T, np.nan, (0, 0, 0)),
           (S, T, 1.0, (0, 0)), (S, T, 1.0, (0, np.inf, 0)), (S.astype(np.int64), T, 1.0, (0, 0, 0))]
    for i, args in enumerate(bad):
        with pytest.raises(ValueError):
            check(*args)
    # entries with m > l are not part of the expansion and are not read
    S_up = S.copy()
    S_up[0, 0, 2] = np.nan
    check(S_up, T, 1.0, (0, 0, 0))


def test_null_context(b200):
    L = b200.lib()
    c = (ctypes.c_double * 3)(0, 0, 0)
    S = (ctypes.c_double * 1)()
    u = ctypes.c_uint()
    assert L.b200nb_set_external_scf(None, 0, 0, 1.0, c, S, S) == b200.EINVAL
    assert L.b200nb_set_external_scf(None, 0, 0, 1.0, None, None, None) == b200.EINVAL
    assert L.b200nb_get_external_scf(None, ctypes.byref(u), None, None, None, None, None, None) == b200.EINVAL


def _compile(tmp_path, src_text, extra=()):
    src = tmp_path / "k.cu"
    src.write_text(src_text)
    obj = tmp_path / "k.o"
    r = subprocess.run(NVCC + list(extra) + ["-c", str(src), "-o", str(obj)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return obj, r.stdout + r.stderr


# ext_total_kernel is a template: these lines instantiate both loaders in a translation unit of its header alone
INSTANTIATE = """
namespace b200nb {
void *const ext_total_kernels[] = {(void *)ext_total_kernel<BlockedPoints>, (void *)ext_total_kernel<SoaPoints>};
}
"""


def test_ext_total_kernel_does_not_spill(tmp_path):
    _, out = _compile(tmp_path, f'#include "{os.path.join(CSRC, "external_sm100.cuh")}"\n' + INSTANTIATE, ["-Xptxas", "-v"])
    props = re.findall(r"Function properties for (\S+)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads",
                       out)
    mine = [p for p in props if "ext_total_kernel" in p[0]]
    assert len({p[0] for p in mine}) == 2, props
    for name, stack, st, ld in mine:
        assert (int(stack), int(st), int(ld)) == (0, 0, 0), name


def test_consumers_do_not_spill(tmp_path):
    """the <true, true> forms of integrate_kernel, tracer_update_kernel and energy_kernel, as the library builds them"""
    src = os.path.join(REPO, "nbody-eurohpc_b200", "csrc", "context.cu")
    r = subprocess.run(NVCC + ["-Xptxas", "-v", "-c", "-o", str(tmp_path / "ctx.o"), src], capture_output=True, text=True, cwd=REPO)
    assert r.returncode == 0, r.stderr[-2000:]
    props = dict(re.findall(r"Function properties for (\S+)\n\s*(\d+ bytes stack frame, \d+ bytes spill stores)", r.stderr))
    for name in ("integrate_kernelILb1ELb1E", "tracer_update_kernelILb1ELb1E", "energy_kernelILb1ELb1E", "ext_total_kernel"):
        hits = [v for k, v in props.items() if name in k]
        assert hits and all(v.startswith("0 bytes stack frame, 0 bytes spill") for v in hits), (name, hits)


def test_kernels_as_compiled_alone(b200, tmp_path):
    """scf_field_kernel, external_field_kernel and both ext_total_kernel loaders are, instruction for instruction, the
    kernels of the library: the step-path wiring changed none of them."""
    obj, _ = _compile(tmp_path, f'#include "{os.path.join(CSRC, "external_sm100.cuh")}"\n' + INSTANTIATE,
                      ["-lineinfo", "-Xcompiler", "-fPIC"])
    alone, lib = _sass(obj), _sass(b200.lib_path())
    for want in ("scf_field_kernel", "external_field_kernel", "ext_total_kernelINS_13BlockedPoints", "ext_total_kernelINS_9SoaPoints"):
        assert any(want in k for k in alone), (want, sorted(alone))
    names = [k for k in alone if k in lib]
    assert len(names) == len(alone), (sorted(alone), sorted(lib))
    for k in names:
        assert alone[k] == lib[k], k
