"""ctypes view of the nearest-neighbour restatement (tests/neighbors_oracle.c).  TEST INFRASTRUCTURE ONLY."""
import ctypes
import os
import subprocess

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FP = ctypes.POINTER(ctypes.c_float)
UP = ctypes.POINTER(ctypes.c_uint32)
U64P = ctypes.POINTER(ctypes.c_uint64)
NONE = np.uint32(0xFFFFFFFF)


def _fp(a):
    return a.ctypes.data_as(FP)


class NeighborsOracle:
    def __init__(self):
        path = os.path.join(REPO, "build", "libneighborsoracle.so")
        if not os.path.exists(path):
            subprocess.check_call(["make", "-C", REPO, "neighbors_oracle"], stdout=subprocess.DEVNULL)
        L = ctypes.CDLL(path)
        u64 = ctypes.c_uint64
        L.oracle_neighbors.argtypes = [u64, FP, FP, FP, ctypes.c_int, U64P, FP, FP, FP, u64, ctypes.c_uint32, UP, FP]
        L.oracle_neighbors.restype = None
        self.L = L

    def _run(self, d, self_mode, tgt, pts, n_t, k):
        q = [np.ascontiguousarray(d[c], np.float32) for c in ("qx", "qy", "qz")]
        idx = np.empty((n_t, k), np.uint32)
        dist = np.empty((n_t, k), np.float32)
        tp = None if tgt is None else tgt.ctypes.data_as(U64P)
        pp = [None] * 3 if pts is None else [_fp(p) for p in pts]
        self.L.oracle_neighbors(len(q[0]), *[_fp(a) for a in q], int(self_mode), tp, *pp, n_t, k,
                                idx.ctypes.data_as(UP), _fp(dist))
        return idx, dist

    def bodies(self, d, k, idx=None):
        """(idx[t][k], dist[t][k]) of bodies idx (None: all), self pair excluded by index."""
        if idx is None:
            return self._run(d, True, None, None, len(d["qx"]), k)
        t = np.ascontiguousarray(idx, np.uint64)
        return self._run(d, True, t, None, len(t), k)

    def points(self, d, px, py, pz, k):
        p = [np.ascontiguousarray(a, np.float32) for a in (px, py, pz)]
        return self._run(d, False, None, p, len(p[0]), k)
