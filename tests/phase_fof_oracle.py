"""ctypes view of the phase-space friends-of-friends restatement (tests/phase_fof_oracle.c).  TEST INFRASTRUCTURE ONLY."""
import ctypes
import os
import subprocess

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FP = ctypes.POINTER(ctypes.c_float)
UP = ctypes.POINTER(ctypes.c_uint32)


class PhaseFofOracle:
    def __init__(self):
        path = os.path.join(REPO, "build", "libphasefoforacle.so")
        if not os.path.exists(path):
            subprocess.check_call(["make", "-C", REPO, "phase_fof_oracle"], stdout=subprocess.DEVNULL)
        L = ctypes.CDLL(path)
        L.oracle_fof_phase.argtypes = [ctypes.c_uint64] + [FP] * 6 + [ctypes.c_float, ctypes.c_float, UP]
        L.oracle_fof_phase.restype = None
        self.L = L

    def groups(self, d, b_x, b_v):
        """uint32[n]: the smallest body index of each body's group of linking lengths b_x, b_v (fp32)."""
        q = [np.ascontiguousarray(d[c], np.float32) for c in ("qx", "qy", "qz", "vx", "vy", "vz")]
        group = np.empty(len(q[0]), np.uint32)
        self.L.oracle_fof_phase(len(q[0]), *[a.ctypes.data_as(FP) for a in q], float(np.float32(b_x)),
                                float(np.float32(b_v)), group.ctypes.data_as(UP))
        return group
