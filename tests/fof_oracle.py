"""ctypes view of the friends-of-friends restatement (tests/fof_oracle.c).  TEST INFRASTRUCTURE ONLY."""
import ctypes
import os
import subprocess

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FP = ctypes.POINTER(ctypes.c_float)
UP = ctypes.POINTER(ctypes.c_uint32)


class FofOracle:
    def __init__(self):
        path = os.path.join(REPO, "build", "libfoforacle.so")
        if not os.path.exists(path):
            subprocess.check_call(["make", "-C", REPO, "fof_oracle"], stdout=subprocess.DEVNULL)
        L = ctypes.CDLL(path)
        L.oracle_fof.argtypes = [ctypes.c_uint64, FP, FP, FP, ctypes.c_float, UP]
        L.oracle_fof.restype = None
        self.L = L

    def groups(self, d, b):
        """uint32[n]: the smallest body index of each body's group of linking length b (fp32)."""
        q = [np.ascontiguousarray(d[c], np.float32) for c in ("qx", "qy", "qz")]
        group = np.empty(len(q[0]), np.uint32)
        self.L.oracle_fof(len(q[0]), *[a.ctypes.data_as(FP) for a in q], float(np.float32(b)), group.ctypes.data_as(UP))
        return group
