"""ctypes view of the fp64 group potential and unbinding reference (tests/groups_oracle.c).  TEST INFRASTRUCTURE ONLY."""
import ctypes
import os
import subprocess

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FP = ctypes.POINTER(ctypes.c_float)
DP = ctypes.POINTER(ctypes.c_double)
UP = ctypes.POINTER(ctypes.c_uint32)
G_F32 = np.float32(6.67384e-11)
NO_GROUP = 0xFFFFFFFF


def _fp(a):
    return a.ctypes.data_as(FP)


class GroupsOracle:
    def __init__(self):
        path = os.path.join(REPO, "build", "libgroupsoracle.so")
        if not os.path.exists(path):
            subprocess.check_call(["make", "-C", REPO, "groups_oracle"], stdout=subprocess.DEVNULL)
        L = ctypes.CDLL(path)
        u64, f = ctypes.c_uint64, ctypes.c_float
        L.oracle_group_potential_f64.argtypes = [u64] + [FP] * 4 + [f, f, UP, ctypes.POINTER(u64), u64, DP]
        L.oracle_group_potential_f64.restype = None
        L.oracle_unbind_pass_f64.argtypes = [u64] + [FP] * 7 + [f, f, UP, DP, DP]
        L.oracle_unbind_pass_f64.restype = u64
        L.oracle_unbind_f64.argtypes = [u64] + [FP] * 7 + [f, f, UP, ctypes.c_uint32, UP, DP, ctypes.POINTER(ctypes.c_int)]
        L.oracle_unbind_f64.restype = ctypes.c_uint32
        self.L = L

    @staticmethod
    def _arrays(d, keys):
        return [np.ascontiguousarray(d[k], np.float32) for k in keys]

    def potential(self, d, group, idx=None, G=G_F32, soft=2e8):
        """fp64 group potential of bodies idx (None: all)."""
        n = len(d["qx"])
        idx = np.arange(n, dtype=np.uint64) if idx is None else np.ascontiguousarray(idx, np.uint64)
        g = np.ascontiguousarray(group, np.uint32)
        a = self._arrays(d, ("qx", "qy", "qz", "m"))
        phi = np.empty(len(idx), np.float64)
        self.L.oracle_group_potential_f64(n, *[_fp(x) for x in a], G, soft, g.ctypes.data_as(UP),
                                          idx.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)), len(idx), phi.ctypes.data_as(DP))
        return phi

    def unbind_pass(self, d, group, G=G_F32, soft=2e8):
        """(phi, E) in fp64 of one unbinding pass over the member set `group`; 0 for non-members."""
        n = len(d["qx"])
        g = np.ascontiguousarray(group, np.uint32)
        a = self._arrays(d, ("qx", "qy", "qz", "m", "vx", "vy", "vz"))
        phi, E = np.empty(n, np.float64), np.empty(n, np.float64)
        self.L.oracle_unbind_pass_f64(n, *[_fp(x) for x in a], G, soft, g.ctypes.data_as(UP), phi.ctypes.data_as(DP),
                                      E.ctypes.data_as(DP))
        return phi, E

    def unbind(self, d, group, max_iter=100, G=G_F32, soft=2e8):
        """(bound, phi, n_iter, converged) of the whole fp64 loop."""
        n = len(d["qx"])
        g = np.ascontiguousarray(group, np.uint32)
        a = self._arrays(d, ("qx", "qy", "qz", "m", "vx", "vy", "vz"))
        bound, phi, conv = np.empty(n, np.uint32), np.empty(n, np.float64), ctypes.c_int()
        t = self.L.oracle_unbind_f64(n, *[_fp(x) for x in a], G, soft, g.ctypes.data_as(UP), max_iter, bound.ctypes.data_as(UP),
                                     phi.ctypes.data_as(DP), ctypes.byref(conv))
        return bound, phi, int(t), bool(conv.value)
