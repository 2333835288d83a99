"""ctypes view of the long-double basis-function-expansion restatement (tests/scf_oracle.c).  TEST INFRASTRUCTURE ONLY."""
import ctypes
import os
import subprocess

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FP = ctypes.POINTER(ctypes.c_float)
DP = ctypes.POINTER(ctypes.c_double)
BP = ctypes.POINTER(ctypes.c_uint8)


def _fp(a):
    return a.ctypes.data_as(FP)


def _dp(a):
    return a.ctypes.data_as(DP)


def to3(S, lmax):
    """packed [nmax+1][(lmax+1)(lmax+2)/2] -> [nmax+1][lmax+1][lmax+1], zeros where m > l"""
    S = np.asarray(S)
    out = np.zeros((S.shape[0], lmax + 1, lmax + 1))
    for l in range(lmax + 1):
        out[:, l, :l + 1] = S[:, l * (l + 1) // 2:l * (l + 1) // 2 + l + 1]
    return out


def packed(S3):
    """[nmax+1][lmax+1][lmax+1] -> packed [nmax+1][(lmax+1)(lmax+2)/2]"""
    lmax = S3.shape[1] - 1
    return np.ascontiguousarray(np.concatenate([S3[:, l, :l + 1] for l in range(lmax + 1)], axis=1), np.float64)


class ScfOracle:
    def __init__(self):
        path = os.path.join(REPO, "build", "libscforacle.so")
        if not os.path.exists(path):
            subprocess.check_call(["make", "-C", REPO, "scf_oracle"], stdout=subprocess.DEVNULL)
        L = ctypes.CDLL(path)
        L.oracle_scf_coefficients.argtypes = [ctypes.c_uint64] + [FP] * 4 + [BP, ctypes.c_int, ctypes.c_int, ctypes.c_double, DP] + [DP] * 4
        L.oracle_scf_coefficients.restype = None
        L.oracle_scf_field.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_double, DP, DP, DP, ctypes.c_uint64] + [FP] * 3 + [DP] * 4
        L.oracle_scf_field.restype = None
        self.L = L

    def coefficients(self, q, gm, nmax, lmax, a, centre=(0.0, 0.0, 0.0), member=None):
        """(S, T, S_scale, T_scale), each float64[nmax+1, lmax+1, lmax+1]; q = (qx, qy, qz) fp32, gm = the fp32 G*m."""
        q = [np.ascontiguousarray(x, np.float32) for x in q]
        gm = np.ascontiguousarray(gm, np.float32)
        n = len(gm)
        mem = np.ones(n, np.uint8) if member is None else np.ascontiguousarray(member, np.uint8)
        K = (nmax + 1) * (lmax + 1) * (lmax + 2) // 2
        out = [np.zeros(K) for _ in range(4)]
        c = np.ascontiguousarray(centre, np.float64)
        self.L.oracle_scf_coefficients(n, *[_fp(x) for x in q], _fp(gm), mem.ctypes.data_as(BP), nmax, lmax, float(a), _dp(c),
                                       *[_dp(o) for o in out])
        return tuple(to3(o.reshape(nmax + 1, -1), lmax) for o in out)

    def field(self, S, T, a, centre, px, py, pz):
        """(ax, ay, az, phi, scale_a [3, m], scale_phi) at fp32 points; S, T float64[nmax+1, lmax+1, lmax+1]."""
        nmax, lmax = S.shape[0] - 1, S.shape[1] - 1
        p = [np.ascontiguousarray(x, np.float32) for x in (px, py, pz)]
        m = len(p[0])
        acc, sa = np.zeros((3, m)), np.zeros((3, m))
        phi, sphi = np.zeros(m), np.zeros(m)
        c = np.ascontiguousarray(centre, np.float64)
        self.L.oracle_scf_field(nmax, lmax, float(a), _dp(c), _dp(packed(S)), _dp(packed(T)), m, *[_fp(x) for x in p], _dp(acc),
                                _dp(phi), _dp(sphi), _dp(sa))
        return acc[0], acc[1], acc[2], phi, sa, sphi
