"""ctypes view of the host test-particle updates (tests/tracers_oracle.c).  TEST INFRASTRUCTURE ONLY."""
import ctypes
import os
import subprocess

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FP = ctypes.POINTER(ctypes.c_float)
KEYS = ("qx", "qy", "qz", "vx", "vy", "vz")


def _fp(a):
    assert a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(FP)


class TracersOracle:
    def __init__(self):
        path = os.path.join(REPO, "build", "libtracersoracle.so")
        if not os.path.exists(path):
            subprocess.check_call(["make", "-C", REPO, "tracers_oracle"], stdout=subprocess.DEVNULL)
        L = ctypes.CDLL(path)
        u64, f = ctypes.c_uint64, ctypes.c_float
        L.tracers_murb.argtypes = [u64] + [FP] * 9 + [f]
        L.tracers_kick_drift.argtypes = [u64] + [FP] * 9 + [f]
        L.tracers_kick.argtypes = [u64] + [FP] * 6 + [f]
        for fn in (L.tracers_murb, L.tracers_kick_drift, L.tracers_kick):
            fn.restype = None
        self.L = L

    @staticmethod
    def _a(a):
        return [np.ascontiguousarray(x, np.float32) for x in a]

    def murb(self, t, a, dt):
        """t: dict of float32 arrays qx..vz, updated in place; a: (ax, ay, az)."""
        a = self._a(a)
        self.L.tracers_murb(len(t["qx"]), *[_fp(t[k]) for k in KEYS], *[_fp(x) for x in a], dt)

    def kick_drift(self, t, a, dt):
        a = self._a(a)
        self.L.tracers_kick_drift(len(t["qx"]), *[_fp(t[k]) for k in KEYS], *[_fp(x) for x in a], dt)

    def kick(self, t, a, dt):
        a = self._a(a)
        self.L.tracers_kick(len(t["qx"]), *[_fp(t[k]) for k in KEYS[3:]], *[_fp(x) for x in a], dt)
