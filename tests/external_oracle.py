"""ctypes view of the host restatement of the external potential (tests/external_oracle.c).  TEST INFRASTRUCTURE ONLY."""
import ctypes
import os
import subprocess

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FP = ctypes.POINTER(ctypes.c_float)
DP = ctypes.POINTER(ctypes.c_double)
KEYS = ("qx", "qy", "qz", "vx", "vy", "vz")


def _fp(a):
    assert a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(FP)


class ExternalOracle:
    def __init__(self, term_type):
        path = os.path.join(REPO, "build", "libexternaloracle.so")
        if not os.path.exists(path):
            subprocess.check_call(["make", "-C", REPO, "external_oracle"], stdout=subprocess.DEVNULL)
        L = ctypes.CDLL(path)
        u32, u64 = ctypes.c_uint32, ctypes.c_uint64
        self.T = term_type
        TP = ctypes.POINTER(term_type)
        L.ext_eval.argtypes = [u32, TP, u64] + [FP] * 3 + [DP] * 4
        L.ext_steps.argtypes = [u32, TP, u64] + [FP] * 9 + [ctypes.c_float, ctypes.c_int, ctypes.c_int, ctypes.c_int]
        L.ext_eval.restype = L.ext_steps.restype = None
        self.L = L

    def _terms(self, terms):
        terms = list(terms)
        return len(terms), (self.T * max(1, len(terms)))(*terms)

    def eval(self, terms, px, py, pz):
        """(ax, ay, az, phi) in fp64 at fp32 points, in the device's operation order."""
        p = [np.ascontiguousarray(a, np.float32) for a in (px, py, pz)]
        out = [np.empty(len(p[0]), np.float64) for _ in range(4)]
        self.L.ext_eval(*self._terms(terms), len(p[0]), *[_fp(a) for a in p], *[o.ctypes.data_as(DP) for o in out])
        return out

    def steps(self, terms, t, acc, dt, integrator, n_steps, have_acc):
        """n_steps of a system without self-gravity; t: dict of float32 qx..vz and acc: [3] float32 arrays, in place."""
        self.L.ext_steps(*self._terms(terms), len(t["qx"]), *[_fp(t[k]) for k in KEYS], *[_fp(a) for a in acc], dt,
                         integrator, n_steps, int(have_acc))
