"""ctypes view of the fp64 tidal-tensor reference (tests/tidal_oracle.c).  TEST INFRASTRUCTURE ONLY."""
import ctypes
import os
import subprocess

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FP = ctypes.POINTER(ctypes.c_float)
DP = ctypes.POINTER(ctypes.c_double)
G_F32 = np.float32(6.67384e-11)
IA, IB = [0, 1, 2, 0, 0, 1], [0, 1, 2, 1, 2, 2]  # the six columns xx, yy, zz, xy, xz, yz


def _fp(a):
    return np.ascontiguousarray(a, np.float32).ctypes.data_as(FP)


def matrix(t6):
    """[m][6] rows (xx, yy, zz, xy, xz, yz) -> symmetric [m][3][3]"""
    t6 = np.asarray(t6)
    t = np.empty((t6.shape[0], 3, 3), t6.dtype)
    t[:, IA, IB] = t6
    t[:, IB, IA] = t6
    return t


def six(t):
    """symmetric [m][3][3] -> [m][6] rows in the library's order"""
    return np.asarray(t)[:, IA, IB]


class TidalOracle:
    def __init__(self):
        path = os.path.join(REPO, "build", "libtidaloracle.so")
        if not os.path.exists(path):
            subprocess.check_call(["make", "-C", REPO, "tidal_oracle"], stdout=subprocess.DEVNULL)
        L = ctypes.CDLL(path)
        u64, f = ctypes.c_uint64, ctypes.c_float
        L.oracle_tidal_f64.argtypes = [u64] + [FP] * 4 + [f, f, u64] + [FP] * 3 + [DP] * 3
        L.oracle_tidal_f64.restype = None
        L.oracle_tidal_bodies_f64.argtypes = [u64] + [FP] * 4 + [f, f, ctypes.POINTER(u64), u64] + [DP] * 3
        L.oracle_tidal_bodies_f64.restype = None
        self.L = L

    def tidal(self, d, px, py, pz, G=G_F32, soft=2e8):
        """(t, amag, s5) in fp64 at the points over all bodies: t, amag [m][6]; s5 [m] = sum_j G m_j / s^5."""
        n = len(d["qx"])
        p = [np.ascontiguousarray(a, np.float32) for a in (px, py, pz)]
        M = len(p[0])
        t, amag, s5 = np.empty((M, 6)), np.empty((M, 6)), np.empty(M)
        self.L.oracle_tidal_f64(n, *[_fp(d[k]) for k in ("qx", "qy", "qz", "m")], G, soft, M,
                                *[a.ctypes.data_as(FP) for a in p], *[o.ctypes.data_as(DP) for o in (t, amag, s5)])
        return t, amag, s5

    def tidal_bodies(self, d, idx=None, G=G_F32, soft=2e8):
        """(t, amag, s5) in fp64 for bodies idx (None: all), self pair excluded by index."""
        n = len(d["qx"])
        if idx is None:
            n_idx, ip = n, None
        else:
            idx = np.ascontiguousarray(idx, np.uint64)
            n_idx, ip = len(idx), idx.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64))
        t, amag, s5 = np.empty((n_idx, 6)), np.empty((n_idx, 6)), np.empty(n_idx)
        self.L.oracle_tidal_bodies_f64(n, *[_fp(d[k]) for k in ("qx", "qy", "qz", "m")], G, soft, ip, n_idx,
                                       *[o.ctypes.data_as(DP) for o in (t, amag, s5)])
        return t, amag, s5
