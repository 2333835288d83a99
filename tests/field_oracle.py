"""ctypes view of the fp64 field reference (tests/field_oracle.c).  TEST INFRASTRUCTURE ONLY."""
import ctypes
import os
import subprocess

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FP = ctypes.POINTER(ctypes.c_float)
DP = ctypes.POINTER(ctypes.c_double)
G_F32 = np.float32(6.67384e-11)


def _fp(a):
    return np.ascontiguousarray(a, np.float32).ctypes.data_as(FP)


class FieldOracle:
    def __init__(self):
        path = os.path.join(REPO, "build", "libfieldoracle.so")
        if not os.path.exists(path):
            subprocess.check_call(["make", "-C", REPO, "field_oracle"], stdout=subprocess.DEVNULL)
        L = ctypes.CDLL(path)
        u64, f = ctypes.c_uint64, ctypes.c_float
        L.oracle_field_f64.argtypes = [u64] + [FP] * 4 + [f, f, u64] + [FP] * 3 + [DP] * 5
        L.oracle_field_f64.restype = None
        L.oracle_potential_f64.argtypes = [u64] + [FP] * 4 + [f, f, ctypes.POINTER(u64), u64, DP]
        L.oracle_potential_f64.restype = None
        self.L = L

    def field(self, d, px, py, pz, G=G_F32, soft=2e8):
        """(ax, ay, az, phi, amag) in fp64 at the points; amag = sum_j |a_ij|."""
        n = len(d["qx"])
        p = [np.ascontiguousarray(a, np.float32) for a in (px, py, pz)]
        out = [np.empty(len(p[0]), np.float64) for _ in range(5)]
        self.L.oracle_field_f64(n, *[_fp(d[k]) for k in ("qx", "qy", "qz", "m")], G, soft, len(p[0]),
                                *[a.ctypes.data_as(FP) for a in p], *[o.ctypes.data_as(DP) for o in out])
        return tuple(out)

    def potential(self, d, idx=None, G=G_F32, soft=2e8):
        """phi_i in fp64, self pair excluded by index, for bodies idx (None: all)."""
        n = len(d["qx"])
        if idx is None:
            n_idx, ip = n, None
        else:
            idx = np.ascontiguousarray(idx, np.uint64)
            n_idx, ip = len(idx), idx.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64))
        phi = np.empty(n_idx, np.float64)
        self.L.oracle_potential_f64(n, *[_fp(d[k]) for k in ("qx", "qy", "qz", "m")], G, soft, ip, n_idx,
                                    phi.ctypes.data_as(DP))
        return phi
