"""ctypes view of the fp64 field-by-component reference (tests/components_oracle.c).  TEST INFRASTRUCTURE ONLY."""
import ctypes
import os
import subprocess

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FP = ctypes.POINTER(ctypes.c_float)
DP = ctypes.POINTER(ctypes.c_double)
UP = ctypes.POINTER(ctypes.c_uint32)
G_F32 = np.float32(6.67384e-11)


def _fp(a):
    return np.ascontiguousarray(a, np.float32).ctypes.data_as(FP)


class ComponentsOracle:
    def __init__(self):
        path = os.path.join(REPO, "build", "libcomponentsoracle.so")
        if not os.path.exists(path):
            subprocess.check_call(["make", "-C", REPO, "components_oracle"], stdout=subprocess.DEVNULL)
        L = ctypes.CDLL(path)
        u64, u32, f = ctypes.c_uint64, ctypes.c_uint32, ctypes.c_float
        L.oracle_components_f64.argtypes = [u64] + [FP] * 4 + [UP, u32, f, f, u64] + [FP] * 3 + [DP] * 3
        L.oracle_components_f64.restype = None
        L.oracle_components_bodies_f64.argtypes = [u64] + [FP] * 4 + [UP, u32, f, f, ctypes.POINTER(u64), u64] + [DP] * 3
        L.oracle_components_bodies_f64.restype = None
        self.L = L

    @staticmethod
    def _args(d, comp):
        comp = np.ascontiguousarray(comp, np.uint32)
        return [_fp(d[k]) for k in ("qx", "qy", "qz", "m")] + [comp.ctypes.data_as(UP)], comp

    def field(self, d, comp, C, px, py, pz, G=G_F32, soft=2e8):
        """(acc [m][C][3], phi [m][C], amag [m][C]) in fp64 at the points; amag = sum_{j in h} |a_ij|."""
        n = len(d["qx"])
        p = [np.ascontiguousarray(a, np.float32) for a in (px, py, pz)]
        M = len(p[0])
        acc, phi, amag = np.empty((M, C, 3)), np.empty((M, C)), np.empty((M, C))
        args, keep = self._args(d, comp)
        self.L.oracle_components_f64(n, *args, C, G, soft, M, *[a.ctypes.data_as(FP) for a in p],
                                     *[o.ctypes.data_as(DP) for o in (acc, phi, amag)])
        return acc, phi, amag

    def bodies(self, d, comp, C, idx=None, G=G_F32, soft=2e8):
        """(acc, phi, amag) in fp64 for bodies idx (None: all), self pair excluded by index."""
        n = len(d["qx"])
        if idx is None:
            n_idx, ip = n, None
        else:
            idx = np.ascontiguousarray(idx, np.uint64)
            n_idx, ip = len(idx), idx.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64))
        acc, phi, amag = np.empty((n_idx, C, 3)), np.empty((n_idx, C)), np.empty((n_idx, C))
        args, keep = self._args(d, comp)
        self.L.oracle_components_bodies_f64(n, *args, C, G, soft, ip, n_idx, *[o.ctypes.data_as(DP) for o in (acc, phi, amag)])
        return acc, phi, amag
