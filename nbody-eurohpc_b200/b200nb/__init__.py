"""b200nb — ctypes binding of libb200nb (include/b200nb.h) and a Python mirror of the MUrB plugin interface.

The product is the CUDA library; this module is plumbing so that tests and bench.py can drive the C ABI on a box that
has no copy of the reference.  The C++ glue that the `murb` CLI links is nbody-eurohpc_b200/glue/.

`SimulationNBodyB200` mirrors the reference's SimulationNBodyInterface<float>
(src/common/core/SimulationNBodyInterface.hpp:15-88): same method names, argument meaning and error behaviour
(`computeOneIteration`, `setDt`, `getDt`, `getBodies().getDataSoA()`, `getFlopsPerIte`, `getAllocatedBytes`).
There is no CPU fallback: if the shared library is missing, or no CUDA device is visible, this module raises.
"""
from __future__ import annotations

import ctypes
import os
import re
from ctypes import POINTER, byref, c_char_p, c_double, c_float, c_int, c_uint, c_uint64, c_void_p

import numpy as np

__all__ = [
    "B200Error", "Context", "SimulationNBodyB200", "B200Bodies", "init_bodies", "lib", "lib_path", "header_functions",
    "G_F32", "INTEGRATOR_MURB", "INTEGRATOR_LEAPFROG", "slice_length", "load_tab",
    "fof_groups", "NO_GROUP", "bound_groups", "component_budget", "COMPONENTS_MAX",
    "ExternalTerm", "EXTERNAL_MAX", "EXT_PLUMMER", "EXT_HERNQUIST", "EXT_NFW", "EXT_MIYAMOTO_NAGAI", "EXT_LOGARITHMIC",
    "plummer", "hernquist", "nfw", "miyamoto_nagai", "logarithmic", "SCF_NMAX", "SCF_LMAX",
]

_HERE = os.path.dirname(os.path.abspath(__file__))
_REPO = os.path.dirname(os.path.dirname(_HERE))
G_F32 = np.float32(6.67384e-11)  # SimulationNBodyInterface.hpp:18 (a float literal)
INTEGRATOR_MURB, INTEGRATOR_LEAPFROG = 0, 1
OK, EINVAL, ECUDA, ENCCL, ESTATE = 0, 1, 2, 3, 4
NO_GROUP = 0xFFFFFFFF  # B200NB_NO_GROUP: a body with this label takes no part in the group calls
COMPONENTS_MAX = 64    # n_comp of the component-field calls lies in [1, COMPONENTS_MAX]
SCF_NMAX, SCF_LMAX = 31, 15  # B200NB_SCF_NMAX, B200NB_SCF_LMAX: the largest expansion of the basis-function calls
_FP = POINTER(c_float)
_UP = POINTER(c_uint)
_DP = POINTER(c_double)

# ---- external potential (include/b200nb.h, "external potential")
EXTERNAL_MAX = 8
EXT_PLUMMER, EXT_HERNQUIST, EXT_NFW, EXT_MIYAMOTO_NAGAI, EXT_LOGARITHMIC = 0, 1, 2, 3, 4


class ExternalTerm(ctypes.Structure):
    """Mirror of b200nb_external_term (56 bytes): kind, reserved (0), gm, a, b, centre[3]; SI units, fp64."""
    _fields_ = [("kind", ctypes.c_int32), ("reserved", ctypes.c_int32), ("gm", c_double), ("a", c_double),
                ("b", c_double), ("centre", c_double * 3)]

    def __repr__(self):
        return (f"ExternalTerm(kind={self.kind}, gm={self.gm!r}, a={self.a!r}, b={self.b!r}, "
                f"centre={tuple(self.centre)!r})")


assert ctypes.sizeof(ExternalTerm) == 56 and ExternalTerm.centre.offset == 32


def _term(kind, gm, a, b, centre, rules):
    """Builds a term after checking the rules the library enforces (B200NB_EINVAL otherwise)."""
    vals = [float(gm), float(a), float(b)]
    c = [float(x) for x in centre]
    if len(c) != 3 or not all(np.isfinite(vals + c)):
        raise ValueError(f"parameters must be finite and centre three numbers, got gm={gm}, a={a}, b={b}, centre={centre}")
    if vals[0] < 0:
        raise ValueError(f"gm must be >= 0, got {gm}")
    for ok, what in rules:
        if not ok:
            raise ValueError(what)
    return ExternalTerm(kind, 0, vals[0], vals[1], vals[2], (c_double * 3)(*c))


def plummer(gm, a, centre=(0.0, 0.0, 0.0)) -> ExternalTerm:
    """Phi = -gm / sqrt(r^2 + a^2); a >= 0 (a = 0: a point mass)."""
    return _term(EXT_PLUMMER, gm, a, 0.0, centre, [(float(a) >= 0, f"Plummer needs a >= 0, got {a}")])


def hernquist(gm, a, centre=(0.0, 0.0, 0.0)) -> ExternalTerm:
    """Phi = -gm / (r + a); a > 0."""
    return _term(EXT_HERNQUIST, gm, a, 0.0, centre, [(float(a) > 0, f"Hernquist needs a > 0, got {a}")])


def nfw(gm, r_s, centre=(0.0, 0.0, 0.0)) -> ExternalTerm:
    """Phi = -gm ln(1 + r/r_s) / r with gm = G M_s = 4 pi G rho_0 r_s^3; r_s > 0."""
    return _term(EXT_NFW, gm, r_s, 0.0, centre, [(float(r_s) > 0, f"NFW needs r_s > 0, got {r_s}")])


def miyamoto_nagai(gm, a, b, centre=(0.0, 0.0, 0.0)) -> ExternalTerm:
    """Phi = -gm / sqrt(R^2 + (a + sqrt(z^2 + b^2))^2); a >= 0, b > 0."""
    return _term(EXT_MIYAMOTO_NAGAI, gm, a, b, centre,
                 [(float(a) >= 0, f"Miyamoto-Nagai needs a >= 0, got {a}"), (float(b) > 0, f"Miyamoto-Nagai needs b > 0, got {b}")])


def logarithmic(v0_sq, r_c, q, centre=(0.0, 0.0, 0.0)) -> ExternalTerm:
    """Phi = v0_sq / 2 * ln(R^2 + z^2/q^2 + r_c^2); r_c > 0, q > 0."""
    return _term(EXT_LOGARITHMIC, v0_sq, r_c, q, centre,
                 [(float(r_c) > 0, f"logarithmic needs r_c > 0, got {r_c}"), (float(q) > 0, f"logarithmic needs q > 0, got {q}")])


class B200Error(RuntimeError):
    def __init__(self, code: int, what: str, msg: str):
        super().__init__(f"{what} failed ({code}): {msg}")
        self.code = code


def lib_path() -> str:
    return os.path.join(_HERE, "libb200nb.so")


def header_functions() -> list[str]:
    """Every function declared in include/b200nb.h (used by the ABI export test)."""
    text = open(os.path.join(_REPO, "include", "b200nb.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(b200nb_[a-z0-9_]+)\s*\(", text)))


_lib = None


def lib() -> ctypes.CDLL:
    """Load libb200nb.so (built in-tree by `make lib` / __graft_entry__.build()).  Fails loudly if absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise B200Error(-1, "load", f"{path} not found: build it with `make lib` (there is no CPU fallback)")
    L = ctypes.CDLL(path)
    ctx = c_void_p
    sig = {
        "b200nb_create": (c_int, [POINTER(ctx), c_uint64, c_int, c_float, c_float]),
        "b200nb_create_sharded": (c_int, [POINTER(ctx), c_uint64, c_int, POINTER(c_int), c_float, c_float]),
        "b200nb_create_rank": (c_int, [POINTER(ctx), c_uint64, c_float, c_float, c_int, c_int, c_int, c_void_p]),
        "b200nb_comm_unique_id": (c_int, [c_void_p]),
        "b200nb_destroy": (None, [ctx]),
        "b200nb_last_error": (c_char_p, [ctx]),
        "b200nb_upload": (c_int, [ctx] + [_FP] * 7),
        "b200nb_download_state": (c_int, [ctx] + [_FP] * 6),
        "b200nb_download_slice": (c_int, [ctx] + [_FP] * 6),
        "b200nb_slice_bounds": (c_int, [ctx, c_int, POINTER(c_uint64), POINTER(c_uint64)]),
        "b200nb_download_accel": (c_int, [ctx] + [_FP] * 3),
        "b200nb_step": (c_int, [ctx, c_float, c_int, c_int]),
        "b200nb_accel": (c_int, [ctx]),
        "b200nb_integrate_host_accel": (c_int, [ctx, _FP, _FP, _FP, c_float]),
        "b200nb_energy": (c_int, [ctx, POINTER(c_double)]),
        "b200nb_metrics": (c_int, [ctx, POINTER(c_double)]),
        "b200nb_field": (c_int, [ctx, c_uint64] + [_FP] * 7),
        "b200nb_potential": (c_int, [ctx, _FP]),
        "b200nb_tidal": (c_int, [ctx, c_uint64, _FP, _FP, _FP, _FP]),
        "b200nb_tidal_bodies": (c_int, [ctx, _FP]),
        "b200nb_component_field": (c_int, [ctx, _UP, c_uint, c_uint64] + [_FP] * 5),
        "b200nb_component_field_bodies": (c_int, [ctx, _UP, c_uint, _FP, _FP]),
        "b200nb_neighbors": (c_int, [ctx, c_uint, _UP, _FP]),
        "b200nb_neighbors_at": (c_int, [ctx, c_uint64, _FP, _FP, _FP, c_uint, _UP, _FP]),
        "b200nb_fof": (c_int, [ctx, c_float, _UP]),
        "b200nb_fof_phase": (c_int, [ctx, c_float, c_float, _UP]),
        "b200nb_group_potential": (c_int, [ctx, _UP, _FP]),
        "b200nb_unbind": (c_int, [ctx, _UP, c_uint, _UP, _FP, _UP, POINTER(c_int)]),
        "b200nb_set_tracers": (c_int, [ctx, c_uint64] + [_FP] * 6),
        "b200nb_download_tracers": (c_int, [ctx] + [_FP] * 6),
        "b200nb_n_tracers": (c_uint64, [ctx]),
        "b200nb_set_external": (c_int, [ctx, c_uint, POINTER(ExternalTerm)]),
        "b200nb_get_external": (c_int, [ctx, POINTER(ExternalTerm), POINTER(c_uint)]),
        "b200nb_external_field": (c_int, [ctx, c_uint64] + [_FP] * 3 + [_DP] * 4),
        "b200nb_scf_coefficients": (c_int, [ctx, c_uint, c_uint, c_double, _DP, _UP, c_uint, _DP, _DP]),
        "b200nb_scf_field": (c_int, [ctx, c_uint, c_uint, c_double, _DP, _DP, _DP, c_uint64] + [_FP] * 3 + [_DP] * 4),
        "b200nb_set_external_scf": (c_int, [ctx, c_uint, c_uint, c_double, _DP, _DP, _DP]),
        "b200nb_get_external_scf": (c_int, [ctx, POINTER(c_uint), POINTER(c_uint), POINTER(c_uint), POINTER(c_double), _DP,
                                            _DP, _DP]),
        "b200nb_sync": (c_int, [ctx]),
        "b200nb_n_bodies": (c_uint64, [ctx]),
        "b200nb_n_local_gpus": (c_int, [ctx]),
        "b200nb_allocated_bytes": (c_uint64, [ctx]),
        "b200nb_launch_count": (c_uint64, [ctx]),
        "b200nb_kernel_name": (c_char_p, [ctx]),
        "b200nb_exchange_name": (c_char_p, [ctx]),
        "b200nb_event_record": (c_int, [ctx, c_int]),
        "b200nb_event_elapsed_ms": (c_int, [ctx, c_int, c_int, POINTER(c_float)]),
        "b200nb_profile_enable": (c_int, [ctx, c_int]),
        "b200nb_profile_get": (c_int, [ctx, POINTER(c_double), POINTER(c_uint64)]),
        "b200nb_flush_l2": (c_int, [ctx]),
        "b200nb_host_alloc": (c_int, [POINTER(c_void_p), c_uint64]),
        "b200nb_host_free": (c_int, [c_void_p]),
        "b200nb_init_bodies": (c_int, [c_int, c_uint64, c_uint] + [_FP] * 8),
        "b200nb_slice_length": (c_uint64, [c_uint64, c_int]),
        "b200nb_tab_count": (c_int, [c_char_p, POINTER(c_uint64)]),
        "b200nb_tab_load": (c_int, [c_char_p, c_uint64] + [_FP] * 8),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    _lib = L
    return L


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


def _p(a: np.ndarray | None):
    return a.ctypes.data_as(_FP) if a is not None else None


_SCHEMES = {"galaxy": 0, "random": 1}


def init_bodies(scheme: str, n: int, seed: int = 0) -> dict[str, np.ndarray]:
    """Bodies<float>(n, scheme, seed) — host only (Bodies.cpp:158-257 restated in csrc/host_ic.cpp)."""
    if scheme not in _SCHEMES:
        raise ValueError(f"scheme must be one of {list(_SCHEMES)}")
    out = {k: np.empty(n, dtype=np.float32) for k in ("qx", "qy", "qz", "vx", "vy", "vz", "m", "r")}
    rc = lib().b200nb_init_bodies(_SCHEMES[scheme], n, seed, *[_p(out[k]) for k in ("qx", "qy", "qz", "vx", "vy", "vz", "m", "r")])
    if rc != OK:
        raise B200Error(rc, "b200nb_init_bodies", "bad arguments")
    return out


def load_tab(path: str) -> dict[str, np.ndarray]:
    """Bodies<float>::initMilkyWayAndromeda (Bodies.cpp:82-153): the reference's `.tab` initial-condition file."""
    n = c_uint64()
    if lib().b200nb_tab_count(path.encode(), byref(n)) != OK:
        raise B200Error(EINVAL, "b200nb_tab_count", f"cannot read {path}")
    out = {k: np.empty(n.value, dtype=np.float32) for k in ("qx", "qy", "qz", "vx", "vy", "vz", "m", "r")}
    rc = lib().b200nb_tab_load(path.encode(), n.value, *[_p(out[k]) for k in ("qx", "qy", "qz", "vx", "vy", "vz", "m", "r")])
    if rc != OK:
        raise B200Error(rc, "b200nb_tab_load", f"parse error in {path}")
    return out


def slice_length(n: int, n_ranks: int) -> int:
    """Targets per rank (padded); rank r owns global bodies [r*L, min((r+1)*L, n))."""
    return int(lib().b200nb_slice_length(n, n_ranks))


class PinnedArrays:
    """A block of page-locked float32 arrays (cudaHostAlloc) for the end-to-end path."""

    def __init__(self, names: list[str], n: int):
        self._ptr = c_void_p()
        nbytes = 4 * n * len(names)
        rc = lib().b200nb_host_alloc(byref(self._ptr), nbytes)
        if rc != OK:
            raise B200Error(rc, "b200nb_host_alloc", lib().b200nb_last_error(None).decode())
        buf = (ctypes.c_float * (n * len(names))).from_address(self._ptr.value)
        flat = np.frombuffer(buf, dtype=np.float32)
        self.arrays = {nm: flat[i * n:(i + 1) * n] for i, nm in enumerate(names)}

    def __getitem__(self, k):
        return self.arrays[k]

    def close(self):
        if self._ptr:
            self.arrays = {}
            lib().b200nb_host_free(self._ptr)
            self._ptr = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _scf_unpack(packed: np.ndarray, nmax: int, lmax: int) -> np.ndarray:
    """the ABI's packed [nmax+1][(lmax+1)(lmax+2)/2] coefficients -> [nmax+1][lmax+1][lmax+1], zeros where m > l"""
    P = packed.reshape(nmax + 1, -1)
    out = np.zeros((nmax + 1, lmax + 1, lmax + 1))
    for l in range(lmax + 1):
        out[:, l, :l + 1] = P[:, l * (l + 1) // 2:l * (l + 1) // 2 + l + 1]
    return out


def _scf_pack(C: np.ndarray) -> np.ndarray:
    """[nmax+1][lmax+1][lmax+1] -> the ABI's packed [nmax+1][(lmax+1)(lmax+2)/2] (entries with m > l are not read)"""
    return np.ascontiguousarray(np.concatenate([C[:, l, :l + 1] for l in range(C.shape[1])], axis=1), np.float64)


class Context:
    """RAII wrapper of b200nb_ctx.  One process driving `n_gpus` devices, or one rank of a torchrun job."""

    def __init__(self, n: int, G: float = G_F32, soft: float = 2e8, n_gpus: int = 1, *, rank: int | None = None,
                 n_ranks: int = 1, device: int = 0, nccl_id: bytes | None = None, devices: list[int] | None = None):
        self._L = lib()
        self._ctx = c_void_p()
        self.n = int(n)
        if devices is not None:  # explicit placement, one shard per entry; a device may repeat (virtual shards)
            arr = (c_int * len(devices))(*devices)
            rc = self._L.b200nb_create_sharded(byref(self._ctx), n, len(devices), arr, float(G), float(soft))
            what = "b200nb_create_sharded"
        elif rank is None:
            rc = self._L.b200nb_create(byref(self._ctx), n, n_gpus, float(G), float(soft))
            what = "b200nb_create"
        else:
            idbuf = ctypes.create_string_buffer(nccl_id, 128) if nccl_id is not None else None
            rc = self._L.b200nb_create_rank(byref(self._ctx), n, float(G), float(soft), rank, n_ranks, device,
                                            ctypes.cast(idbuf, c_void_p) if idbuf is not None else None)
            what = "b200nb_create_rank"
        if rc != OK:
            raise B200Error(rc, what, self._L.b200nb_last_error(None).decode())

    @staticmethod
    def unique_id() -> bytes:
        buf = ctypes.create_string_buffer(128)
        rc = lib().b200nb_comm_unique_id(ctypes.cast(buf, c_void_p))
        if rc != OK:
            raise B200Error(rc, "b200nb_comm_unique_id", lib().b200nb_last_error(None).decode())
        return buf.raw

    def _check(self, rc: int, what: str):
        if rc != OK:
            raise B200Error(rc, what, self._L.b200nb_last_error(self._ctx).decode())

    def close(self):
        if self._ctx:
            self._L.b200nb_destroy(self._ctx)
            self._ctx = c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- state
    def upload(self, qx, qy, qz, m, vx, vy, vz):
        arrs = [_f32(a) for a in (qx, qy, qz, m, vx, vy, vz)]
        for a in arrs:
            if a.shape != (self.n,):
                raise ValueError(f"expected arrays of {self.n} floats, got {a.shape}")
        self._check(self._L.b200nb_upload(self._ctx, *[_p(a) for a in arrs]), "b200nb_upload")

    def upload_raw(self, arrs):
        """float32 C-contiguous arrays (e.g. pinned) passed without conversion: the C side reads n floats from each."""
        if len(arrs) != 7:
            raise ValueError("expected 7 arrays: qx qy qz m vx vy vz")
        for a in arrs:
            if a.dtype != np.float32 or a.shape != (self.n,) or not a.flags["C_CONTIGUOUS"]:
                raise ValueError(f"expected C-contiguous float32 arrays of {self.n} elements, got {a.dtype} {a.shape}")
        self._check(self._L.b200nb_upload(self._ctx, *[_p(a) for a in arrs]), "b200nb_upload")

    _STATE = ("qx", "qy", "qz", "vx", "vy", "vz")

    def _state_out(self, out):
        if out is None:
            return {k: np.empty(self.n, dtype=np.float32) for k in self._STATE}
        for k in self._STATE:
            a = out.get(k)
            if a is not None and (a.dtype != np.float32 or a.shape != (self.n,) or not a.flags["C_CONTIGUOUS"]):
                raise ValueError(f"{k}: expected a C-contiguous float32 array of {self.n} elements, got {a.dtype} {a.shape}")
        return out

    def download_state(self, out: dict[str, np.ndarray] | None = None) -> dict[str, np.ndarray]:
        out = self._state_out(out)
        self._check(self._L.b200nb_download_state(self._ctx, *[_p(out.get(k)) for k in self._STATE]), "b200nb_download_state")
        return out

    def download_slice(self, out: dict[str, np.ndarray] | None = None) -> dict[str, np.ndarray]:
        """Only the local shards' own bodies are written (global indexing); see slice_bounds()."""
        out = self._state_out(out)
        self._check(self._L.b200nb_download_slice(self._ctx, *[_p(out.get(k)) for k in self._STATE]), "b200nb_download_slice")
        return out

    def slice_bounds(self, local_shard: int = 0) -> tuple[int, int]:
        first, count = c_uint64(), c_uint64()
        self._check(self._L.b200nb_slice_bounds(self._ctx, local_shard, byref(first), byref(count)), "b200nb_slice_bounds")
        return first.value, count.value

    def download_accel(self) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        a = [np.empty(self.n, dtype=np.float32) for _ in range(3)]
        self._check(self._L.b200nb_download_accel(self._ctx, *[_p(x) for x in a]), "b200nb_download_accel")
        return a[0], a[1], a[2]

    # ---- hot path
    def step(self, dt: float, integrator: int = INTEGRATOR_MURB, n_steps: int = 1):
        self._check(self._L.b200nb_step(self._ctx, float(dt), integrator, n_steps), "b200nb_step")

    def accel(self):
        self._check(self._L.b200nb_accel(self._ctx), "b200nb_accel")

    def integrate_host_accel(self, ax, ay, az, dt: float):
        a = [_f32(x) for x in (ax, ay, az)]
        for x in a:
            if x.shape != (self.n,):
                raise ValueError(f"expected arrays of {self.n} floats, got {x.shape}")
        self._check(self._L.b200nb_integrate_host_accel(self._ctx, *[_p(x) for x in a], float(dt)), "b200nb_integrate_host_accel")

    def energy(self) -> float:
        e = c_double()
        self._check(self._L.b200nb_energy(self._ctx, byref(e)), "b200nb_energy")
        return e.value

    METRIC_NAMES = ("energy", "ang_x", "ang_y", "ang_z", "mass", "com_x", "com_y", "com_z", "density_x", "density_y", "density_z")

    def metrics(self) -> dict:
        """energy, angular momentum vector, total mass, centre of mass, density centre (include/b200nb.h: b200nb_metrics)."""
        out = (c_double * len(self.METRIC_NAMES))()
        self._check(self._L.b200nb_metrics(self._ctx, out), "b200nb_metrics")
        return dict(zip(self.METRIC_NAMES, list(out)))

    def field(self, px, py, pz) -> tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray]:
        """Acceleration and potential at arbitrary points, summed over every body (include/b200nb.h: b200nb_field).
        px, py, pz: 1-D arrays of equal length.  Returns (ax, ay, az, phi), float32."""
        p = [_f32(a) for a in (px, py, pz)]
        if any(a.ndim != 1 for a in p) or len({a.shape for a in p}) != 1:
            raise ValueError(f"expected three 1-D arrays of equal length, got {[a.shape for a in p]}")
        m = p[0].shape[0]
        out = [np.empty(m, dtype=np.float32) for _ in range(4)]
        self._check(self._L.b200nb_field(self._ctx, m, *[_p(a) for a in p], *[_p(a) for a in out]), "b200nb_field")
        return out[0], out[1], out[2], out[3]

    def potential(self) -> np.ndarray:
        """Per-body potential phi_i, self pair excluded (include/b200nb.h: b200nb_potential).  float32[n]."""
        phi = np.empty(self.n, dtype=np.float32)
        self._check(self._L.b200nb_potential(self._ctx, _p(phi)), "b200nb_potential")
        return phi

    # the six columns xx, yy, zz, xy, xz, yz of b200nb_tidal's rows, as (row, column) of the symmetric 3x3 matrix
    _TIDAL_IDX = ([0, 1, 2, 0, 0, 1], [0, 1, 2, 1, 2, 2])

    @classmethod
    def _tidal_matrix(cls, t6: np.ndarray) -> np.ndarray:
        t = np.empty((t6.shape[0], 3, 3), dtype=np.float32)
        r, c = cls._TIDAL_IDX
        t[:, r, c] = t6
        t[:, c, r] = t6
        return t

    def tidal(self, px, py, pz) -> np.ndarray:
        """Tidal tensor T_ab = d a_a / d p_b at arbitrary points, summed over every body (include/b200nb.h: b200nb_tidal).
        px, py, pz: 1-D arrays of equal length.  Returns float32[m, 3, 3], symmetric."""
        p = [_f32(a) for a in (px, py, pz)]
        if any(a.ndim != 1 for a in p) or len({a.shape for a in p}) != 1:
            raise ValueError(f"expected three 1-D arrays of equal length, got {[a.shape for a in p]}")
        m = p[0].shape[0]
        t6 = np.empty((m, 6), dtype=np.float32)
        self._check(self._L.b200nb_tidal(self._ctx, m, *[_p(a) for a in p], _p(t6)), "b200nb_tidal")
        return self._tidal_matrix(t6)

    def tidal_bodies(self) -> np.ndarray:
        """Tidal tensor of every body, self pair excluded (include/b200nb.h: b200nb_tidal_bodies).  float32[n, 3, 3]."""
        t6 = np.empty((self.n, 6), dtype=np.float32)
        self._check(self._L.b200nb_tidal_bodies(self._ctx, _p(t6)), "b200nb_tidal_bodies")
        return self._tidal_matrix(t6)

    NEIGHBORS_K_MAX = 32

    def _k(self, k) -> int:
        if isinstance(k, bool) or not isinstance(k, (int, np.integer)) or not 1 <= int(k) <= self.NEIGHBORS_K_MAX:
            raise ValueError(f"k must be an integer in [1, {self.NEIGHBORS_K_MAX}], got {k!r}")
        return int(k)

    def neighbors(self, k) -> tuple[np.ndarray, np.ndarray]:
        """k nearest other bodies of every body (include/b200nb.h: b200nb_neighbors).  Returns (idx uint32[n, k],
        dist float32[n, k]), each row sorted by (distance, index); empty slots are (0xFFFFFFFF, inf)."""
        k = self._k(k)
        idx = np.empty((self.n, k), dtype=np.uint32)
        dist = np.empty((self.n, k), dtype=np.float32)
        self._check(self._L.b200nb_neighbors(self._ctx, k, idx.ctypes.data_as(_UP), _p(dist)), "b200nb_neighbors")
        return idx, dist

    def neighbors_at(self, px, py, pz, k) -> tuple[np.ndarray, np.ndarray]:
        """k nearest bodies of arbitrary points (include/b200nb.h: b200nb_neighbors_at).  px, py, pz: 1-D arrays of equal
        length m.  Returns (idx uint32[m, k], dist float32[m, k])."""
        k = self._k(k)
        p = [_f32(a) for a in (px, py, pz)]
        if any(a.ndim != 1 for a in p) or len({a.shape for a in p}) != 1:
            raise ValueError(f"expected three 1-D arrays of equal length, got {[a.shape for a in p]}")
        m = p[0].shape[0]
        idx = np.empty((m, k), dtype=np.uint32)
        dist = np.empty((m, k), dtype=np.float32)
        self._check(self._L.b200nb_neighbors_at(self._ctx, m, *[_p(a) for a in p], k, idx.ctypes.data_as(_UP), _p(dist)),
                    "b200nb_neighbors_at")
        return idx, dist

    @staticmethod
    def _fof_b(b) -> float:
        """b as the fp32 value the library uses; ValueError unless b >= 0 with b * b finite in fp32."""
        ok = not isinstance(b, bool) and isinstance(b, (int, float, np.integer, np.floating))
        if ok:
            with np.errstate(over="ignore", invalid="ignore"):
                b32 = np.float32(b)
                ok = bool(b32 >= 0) and bool(np.isfinite(b32 * b32))
        if not ok:
            raise ValueError(f"b must be a real number >= 0 with b * b finite in fp32, got {b!r}")
        return float(b32)

    def fof(self, b) -> np.ndarray:
        """Friends-of-friends groups of linking length b (include/b200nb.h: b200nb_fof).  Returns uint32[n]: the
        smallest body index of each body's group."""
        b = self._fof_b(b)
        group = np.empty(self.n, dtype=np.uint32)
        self._check(self._L.b200nb_fof(self._ctx, b, group.ctypes.data_as(_UP)), "b200nb_fof")
        return group

    @staticmethod
    def _fof_phase_b(b, name) -> float:
        """b as the fp32 value the library uses; ValueError unless b > 0 in fp32 (+inf allowed, a finite b that
        overflows fp32 is not)."""
        ok = not isinstance(b, bool) and isinstance(b, (int, float, np.integer, np.floating))
        if ok:
            with np.errstate(over="ignore"):
                b32 = np.float32(b)
            ok = bool(b32 > 0) and (bool(np.isfinite(b32)) or not np.isfinite(float(b)))
        if not ok:
            raise ValueError(f"{name} must be a real number > 0 in fp32 (+inf allowed), got {b!r}")
        return float(b32)

    def fof_phase(self, b_x, b_v) -> np.ndarray:
        """Phase-space friends-of-friends groups of linking lengths b_x (positions, m) and b_v (velocities, m/s)
        (include/b200nb.h: b200nb_fof_phase).  b = inf switches that part of the metric off.  Returns uint32[n]: the
        smallest body index of each body's group, which fof_groups and bound_groups take as they take fof's."""
        b_x, b_v = self._fof_phase_b(b_x, "b_x"), self._fof_phase_b(b_v, "b_v")
        group = np.empty(self.n, dtype=np.uint32)
        self._check(self._L.b200nb_fof_phase(self._ctx, b_x, b_v, group.ctypes.data_as(_UP)), "b200nb_fof_phase")
        return group

    def _labels(self, group) -> np.ndarray:
        """group as the uint32[n] labels the library reads; ValueError unless 1-D, n long, integer, in [0, 2^32 - 1]."""
        g = np.asarray(group)
        if g.ndim != 1 or g.shape[0] != self.n or g.dtype.kind not in "ui":
            raise ValueError(f"group must be a 1-D integer array of {self.n} labels, got {g.dtype} {g.shape}")
        if len(g) and (int(g.min()) < 0 or int(g.max()) > NO_GROUP):
            raise ValueError("labels must lie in [0, 2^32 - 1]")
        return np.ascontiguousarray(g, np.uint32)

    def group_potential(self, group) -> np.ndarray:
        """Potential of every body from the members of its own label only (include/b200nb.h: b200nb_group_potential).
        group: uint32 labels, NO_GROUP for none.  Returns float32[n]; +0 for NO_GROUP bodies and lone members."""
        g = self._labels(group)
        phi = np.empty(self.n, dtype=np.float32)
        self._check(self._L.b200nb_group_potential(self._ctx, g.ctypes.data_as(_UP), _p(phi)), "b200nb_group_potential")
        return phi

    def unbind(self, group, max_iter=100) -> tuple[np.ndarray, np.ndarray, int, bool]:
        """Iterative removal of the members whose energy in their group's frame is not negative (include/b200nb.h:
        b200nb_unbind).  Returns (bound uint32[n]: the label of every body still bound, NO_GROUP for the others;
        phi float32[n]: the group potential of the last pass; passes run; converged)."""
        g = self._labels(group)
        if isinstance(max_iter, bool) or not isinstance(max_iter, (int, np.integer)) or not 1 <= int(max_iter) <= NO_GROUP:
            raise ValueError(f"max_iter must be an integer in [1, 2^32 - 1], got {max_iter!r}")
        bound = np.empty(self.n, dtype=np.uint32)
        phi = np.empty(self.n, dtype=np.float32)
        n_iter, conv = c_uint(), c_int()
        self._check(self._L.b200nb_unbind(self._ctx, g.ctypes.data_as(_UP), int(max_iter), bound.ctypes.data_as(_UP), _p(phi),
                                          byref(n_iter), byref(conv)), "b200nb_unbind")
        return bound, phi, int(n_iter.value), bool(conv.value)

    def _components(self, comp, n_comp) -> tuple[np.ndarray, int]:
        """(labels, n_comp) as the library reads them; ValueError unless n_comp is an integer in [1, COMPONENTS_MAX] and
        every label is < n_comp or NO_GROUP."""
        if isinstance(n_comp, bool) or not isinstance(n_comp, (int, np.integer)) or not 1 <= int(n_comp) <= COMPONENTS_MAX:
            raise ValueError(f"n_comp must be an integer in [1, {COMPONENTS_MAX}], got {n_comp!r}")
        g = self._labels(comp)
        if np.any((g >= n_comp) & (g != NO_GROUP)):
            raise ValueError(f"every label must be < n_comp = {int(n_comp)} or NO_GROUP")
        return g, int(n_comp)

    def component_field(self, comp, n_comp, px, py, pz) -> tuple[np.ndarray, np.ndarray]:
        """Acceleration and potential at arbitrary points from each source component (include/b200nb.h:
        b200nb_component_field).  comp: uint32 labels in [0, n_comp) or NO_GROUP; px, py, pz: 1-D arrays of equal length m.
        Returns (acc float32[m, n_comp, 3], phi float32[m, n_comp])."""
        g, C = self._components(comp, n_comp)
        p = [_f32(a) for a in (px, py, pz)]
        if any(a.ndim != 1 for a in p) or len({a.shape for a in p}) != 1:
            raise ValueError(f"expected three 1-D arrays of equal length, got {[a.shape for a in p]}")
        m = p[0].shape[0]
        acc = np.empty((m, C, 3), dtype=np.float32)
        phi = np.empty((m, C), dtype=np.float32)
        self._check(self._L.b200nb_component_field(self._ctx, g.ctypes.data_as(_UP), C, m, *[_p(a) for a in p], _p(acc), _p(phi)),
                    "b200nb_component_field")
        return acc, phi

    def component_field_bodies(self, comp, n_comp) -> tuple[np.ndarray, np.ndarray]:
        """Acceleration and potential of every body from each source component, self pair excluded (include/b200nb.h:
        b200nb_component_field_bodies).  Returns (acc float32[n, n_comp, 3], phi float32[n, n_comp])."""
        g, C = self._components(comp, n_comp)
        acc = np.empty((self.n, C, 3), dtype=np.float32)
        phi = np.empty((self.n, C), dtype=np.float32)
        self._check(self._L.b200nb_component_field_bodies(self._ctx, g.ctypes.data_as(_UP), C, _p(acc), _p(phi)),
                    "b200nb_component_field_bodies")
        return acc, phi

    def set_tracers(self, qx, qy, qz, vx, vy, vz):
        """Replaces the massless test particles (include/b200nb.h: b200nb_set_tracers): six 1-D arrays of equal length
        M, positions and velocities.  Empty arrays remove them."""
        t = [_f32(a) for a in (qx, qy, qz, vx, vy, vz)]
        if any(a.ndim != 1 for a in t) or len({a.shape for a in t}) != 1:
            raise ValueError(f"expected six 1-D arrays of equal length, got {[a.shape for a in t]}")
        m = t[0].shape[0]
        ptrs = [_p(a) for a in t] if m else [None] * 6
        self._check(self._L.b200nb_set_tracers(self._ctx, m, *ptrs), "b200nb_set_tracers")

    def download_tracers(self) -> dict[str, np.ndarray]:
        """Positions and velocities of every tracer after the steps enqueued so far: keys qx .. vz, float32[M]."""
        out = {k: np.empty(self.n_tracers, dtype=np.float32) for k in self._STATE}
        self._check(self._L.b200nb_download_tracers(self._ctx, *[_p(out[k]) for k in self._STATE]), "b200nb_download_tracers")
        return out

    @property
    def n_tracers(self) -> int:
        return int(self._L.b200nb_n_tracers(self._ctx))

    def set_external(self, terms):
        """Replaces the static external potential (include/b200nb.h: b200nb_set_external): a sequence of at most
        EXTERNAL_MAX terms made by plummer, hernquist, nfw, miyamoto_nagai or logarithmic.  An empty sequence removes it."""
        terms = list(terms)
        if len(terms) > EXTERNAL_MAX:
            raise ValueError(f"at most {EXTERNAL_MAX} external terms, got {len(terms)}")
        arr = (ExternalTerm * max(1, len(terms)))(*terms)
        self._check(self._L.b200nb_set_external(self._ctx, len(terms), arr if terms else None), "b200nb_set_external")

    @property
    def external(self) -> list[ExternalTerm]:
        """The current external terms, in order."""
        arr, n = (ExternalTerm * EXTERNAL_MAX)(), c_uint()
        self._check(self._L.b200nb_get_external(self._ctx, arr, byref(n)), "b200nb_get_external")
        return [arr[i] for i in range(n.value)]

    def external_field(self, px, py, pz) -> tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray]:
        """Acceleration and potential of the external terms at fp32 points, evaluated on the device: bit for bit what the
        step adds there (include/b200nb.h: b200nb_external_field).  Returns (ax, ay, az, phi), float64."""
        p = [_f32(a) for a in (px, py, pz)]
        if any(a.ndim != 1 for a in p) or len({a.shape for a in p}) != 1:
            raise ValueError(f"expected three 1-D arrays of equal length, got {[a.shape for a in p]}")
        m = p[0].shape[0]
        out = [np.empty(m, dtype=np.float64) for _ in range(4)]
        self._check(self._L.b200nb_external_field(self._ctx, m, *[_p(a) for a in p], *[o.ctypes.data_as(_DP) for o in out]),
                    "b200nb_external_field")
        return out[0], out[1], out[2], out[3]

    @staticmethod
    def _scf_args(nmax, lmax, a, centre) -> tuple[int, int, float, np.ndarray]:
        """(nmax, lmax, a, centre) as the library reads them; ValueError unless nmax in [0, SCF_NMAX], lmax in
        [0, SCF_LMAX], a finite and > 0 and the centre three finite numbers."""
        for name, v, hi in (("nmax", nmax, SCF_NMAX), ("lmax", lmax, SCF_LMAX)):
            if isinstance(v, bool) or not isinstance(v, (int, np.integer)) or not 0 <= int(v) <= hi:
                raise ValueError(f"{name} must be an integer in [0, {hi}], got {v!r}")
        if isinstance(a, bool) or not isinstance(a, (int, float, np.integer, np.floating)) or not (np.isfinite(a) and a > 0):
            raise ValueError(f"a must be a finite number > 0, got {a!r}")
        c = np.ascontiguousarray(centre, dtype=np.float64)
        if c.shape != (3,) or not np.all(np.isfinite(c)):
            raise ValueError(f"centre must be three finite numbers, got {centre!r}")
        return int(nmax), int(lmax), float(a), c

    def scf_coefficients(self, nmax, lmax, a, centre=(0.0, 0.0, 0.0), group=None, label=0) -> tuple[np.ndarray, np.ndarray]:
        """Hernquist-Ostriker basis-function expansion of the bodies with group == label (group None: every body) about
        `centre` with scale radius a (include/b200nb.h: b200nb_scf_coefficients).  Returns (S, T), float64[nmax+1, lmax+1,
        lmax+1] in m^2/s^2, zero where m > l (gala's layout)."""
        nmax, lmax, a, c = self._scf_args(nmax, lmax, a, centre)
        g = None if group is None else self._labels(group)
        if isinstance(label, bool) or not isinstance(label, (int, np.integer)) or not 0 <= int(label) <= NO_GROUP:
            raise ValueError(f"label must be an integer in [0, 2^32 - 1], got {label!r}")
        K = (nmax + 1) * (lmax + 1) * (lmax + 2) // 2
        S, T = np.empty(K), np.empty(K)
        self._check(self._L.b200nb_scf_coefficients(self._ctx, nmax, lmax, a, c.ctypes.data_as(_DP),
                                                    None if g is None else g.ctypes.data_as(_UP), int(label),
                                                    S.ctypes.data_as(_DP), T.ctypes.data_as(_DP)), "b200nb_scf_coefficients")
        return _scf_unpack(S, nmax, lmax), _scf_unpack(T, nmax, lmax)

    def scf_field(self, S, T, a, centre, px, py, pz) -> tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray]:
        """Acceleration and potential of an expansion (S, T float64[nmax+1, lmax+1, lmax+1], as scf_coefficients returns
        them) at fp32 points (include/b200nb.h: b200nb_scf_field).  Returns (ax, ay, az, phi), float64."""
        S, T = np.asarray(S), np.asarray(T)
        if S.ndim != 3 or S.shape != T.shape or S.shape[1] != S.shape[2] or S.dtype.kind != "f" or T.dtype.kind != "f":
            raise ValueError(f"S and T must be float arrays of one shape (nmax+1, lmax+1, lmax+1), got {S.shape}, {T.shape}")
        nmax, lmax, a, c = self._scf_args(S.shape[0] - 1, S.shape[1] - 1, a, centre)
        p = [_f32(x) for x in (px, py, pz)]
        if any(x.ndim != 1 for x in p) or len({x.shape for x in p}) != 1:
            raise ValueError(f"expected three 1-D arrays of equal length, got {[x.shape for x in p]}")
        m = p[0].shape[0]
        out = [np.empty(m, dtype=np.float64) for _ in range(4)]
        Sp, Tp = _scf_pack(S), _scf_pack(T)
        self._check(self._L.b200nb_scf_field(self._ctx, nmax, lmax, a, c.ctypes.data_as(_DP), Sp.ctypes.data_as(_DP),
                                             Tp.ctypes.data_as(_DP), m, *[_p(x) for x in p],
                                             *[o.ctypes.data_as(_DP) for o in out]), "b200nb_scf_field")
        return out[0], out[1], out[2], out[3]

    @staticmethod
    def _external_scf_args(S, T, a, centre) -> tuple[int, int, float, np.ndarray, np.ndarray, np.ndarray]:
        """(nmax, lmax, a, centre, packed S, packed T) as b200nb_set_external_scf reads them; ValueError for a bad shape,
        nmax or lmax out of range, a or the centre (as scf_field), a non-finite entry or T[n, l, 0] != 0."""
        if S is None or T is None:
            raise ValueError("S and T must both be given (or both None to remove the expansion)")
        S, T = np.asarray(S), np.asarray(T)
        if S.ndim != 3 or S.shape != T.shape or S.shape[1] != S.shape[2] or S.dtype.kind != "f" or T.dtype.kind != "f":
            raise ValueError(f"S and T must be float arrays of one shape (nmax+1, lmax+1, lmax+1), got {S.shape}, {T.shape}")
        nmax, lmax, a, c = Context._scf_args(S.shape[0] - 1, S.shape[1] - 1, a, centre)
        Sp, Tp = _scf_pack(S), _scf_pack(T)
        if not (np.all(np.isfinite(Sp)) and np.all(np.isfinite(Tp))):
            raise ValueError("S and T must be finite where m <= l")
        if np.any(T[:, :, 0] != 0):
            raise ValueError("T[n, l, 0] must be 0 (scf_coefficients returns 0 there)")
        return nmax, lmax, a, c, Sp, Tp

    def set_external_scf(self, S, T=None, a=None, centre=(0.0, 0.0, 0.0)):
        """Installs (or replaces) a frozen basis-function expansion as part of the external potential (include/b200nb.h:
        b200nb_set_external_scf).  S, T float64[nmax+1, lmax+1, lmax+1] as scf_coefficients returns them, scale radius a,
        centre.  set_external_scf(None) removes it; the analytic terms of set_external are not affected."""
        if S is None and T is None:
            self._check(self._L.b200nb_set_external_scf(self._ctx, 0, 0, 0.0, None, None, None), "b200nb_set_external_scf")
            return
        nmax, lmax, a, c, Sp, Tp = self._external_scf_args(S, T, a, centre)
        self._check(self._L.b200nb_set_external_scf(self._ctx, nmax, lmax, a, c.ctypes.data_as(_DP), Sp.ctypes.data_as(_DP),
                                                    Tp.ctypes.data_as(_DP)), "b200nb_set_external_scf")

    @property
    def external_scf(self):
        """None, or the expansion as set: (S, T, a, centre), S and T float64[nmax+1, lmax+1, lmax+1], centre a tuple."""
        present, nmax, lmax, a = c_uint(), c_uint(), c_uint(), c_double()
        c = np.zeros(3)
        self._check(self._L.b200nb_get_external_scf(self._ctx, byref(present), byref(nmax), byref(lmax), byref(a),
                                                    c.ctypes.data_as(_DP), None, None), "b200nb_get_external_scf")
        if not present.value:
            return None
        K = (nmax.value + 1) * (lmax.value + 1) * (lmax.value + 2) // 2
        S, T = np.empty(K), np.empty(K)
        self._check(self._L.b200nb_get_external_scf(self._ctx, byref(present), None, None, None, None, S.ctypes.data_as(_DP),
                                                    T.ctypes.data_as(_DP)), "b200nb_get_external_scf")
        return (_scf_unpack(S, nmax.value, lmax.value), _scf_unpack(T, nmax.value, lmax.value), a.value,
                tuple(float(x) for x in c))

    def sync(self):
        self._check(self._L.b200nb_sync(self._ctx), "b200nb_sync")

    # ---- introspection / measurement
    @property
    def n_local_gpus(self) -> int:
        return self._L.b200nb_n_local_gpus(self._ctx)

    @property
    def allocated_bytes(self) -> int:
        return self._L.b200nb_allocated_bytes(self._ctx)

    @property
    def launch_count(self) -> int:
        return self._L.b200nb_launch_count(self._ctx)

    @property
    def kernel_name(self) -> str:
        return self._L.b200nb_kernel_name(self._ctx).decode()

    @property
    def exchange_name(self) -> str:
        """'none' | 'p2p-push' | 'nccl-allgather' (include/b200nb.h: b200nb_exchange_name)."""
        return self._L.b200nb_exchange_name(self._ctx).decode()

    def event_record(self, slot: int):
        self._check(self._L.b200nb_event_record(self._ctx, slot), "b200nb_event_record")

    def event_elapsed_ms(self, a: int, b: int) -> float:
        ms = c_float()
        self._check(self._L.b200nb_event_elapsed_ms(self._ctx, a, b, byref(ms)), "b200nb_event_elapsed_ms")
        return ms.value

    def flush_l2(self):
        self._check(self._L.b200nb_flush_l2(self._ctx), "b200nb_flush_l2")

    def profile_enable(self, on: bool = True):
        self._check(self._L.b200nb_profile_enable(self._ctx, int(on)), "b200nb_profile_enable")

    def profile_get(self) -> tuple[float, int]:
        ms, n = c_double(), c_uint64()
        self._check(self._L.b200nb_profile_get(self._ctx, byref(ms), byref(n)), "b200nb_profile_get")
        return ms.value, n.value


def fof_groups(group, m, state, min_size: int = 20) -> dict[str, np.ndarray]:
    """Catalogue of the friends-of-friends groups of at least `min_size` members (host, O(N)).

    group: the labels of Context.fof or Context.fof_phase; m: the masses; state: positions and velocities as
    Context.download_state returns them.  Groups come sorted by size, largest first, then by root.  Returns arrays with one entry per group:
      root uint32 (the smallest body index), size int64, mass float64, com float64[g, 3] (centre of mass),
      vel float64[g, 3] (mass-weighted mean velocity; both NaN for a group of zero mass).
    Sums are fp64 np.bincount sums, accumulated in body order, so the catalogue is reproducible."""
    group = np.asarray(group)
    if group.ndim != 1 or group.dtype.kind not in "ui" or (len(group) and (group.min() < 0 or group.max() >= len(group))):
        raise ValueError("group must be a 1-D integer array of body indices")
    n = len(group)
    if isinstance(min_size, bool) or not isinstance(min_size, (int, np.integer)) or min_size < 1:
        raise ValueError(f"min_size must be an integer >= 1, got {min_size!r}")
    m = np.asarray(m, dtype=np.float64)
    if m.shape != (n,):
        raise ValueError(f"expected {n} masses, got {m.shape}")
    size = np.bincount(group, minlength=n)
    roots = np.flatnonzero(size >= min_size)
    roots = roots[np.lexsort((roots, -size[roots]))]
    mass = np.bincount(group, weights=m, minlength=n)[roots]

    def mean(keys):
        cols = [np.bincount(group, weights=m * np.asarray(state[k], dtype=np.float64), minlength=n)[roots] for k in keys]
        with np.errstate(invalid="ignore", divide="ignore"):
            return np.stack(cols, axis=1) / mass[:, None] if len(roots) else np.zeros((0, 3))

    return {"root": roots.astype(np.uint32), "size": size[roots].astype(np.int64), "mass": mass,
            "com": mean(("qx", "qy", "qz")), "vel": mean(("vx", "vy", "vz"))}


def bound_groups(bound, m, state, phi, min_size: int = 20) -> dict[str, np.ndarray]:
    """Catalogue of the bound groups of Context.unbind (host, O(N)).

    bound: the labels Context.unbind returns (NO_GROUP: not bound); m: the masses; state: positions and velocities as
    Context.download_state returns them; phi: the group potential Context.unbind returns.  Labels with at least
    `min_size` bound members come sorted by size, largest first, then by label.  Returns arrays with one entry per group:
      label uint32, size int64, mass float64, com float64[g, 3] (centre of mass), vel float64[g, 3] (mass-weighted mean
      velocity V; both NaN for a group of zero mass), kinetic float64 (sum m |v - V|^2 / 2), potential float64
      (sum m phi / 2, each pair counted once).
    Sums are fp64 np.bincount sums, accumulated in body order, so the catalogue is reproducible."""
    bound = np.asarray(bound)
    if bound.ndim != 1 or bound.dtype.kind not in "ui" or (len(bound) and (int(bound.min()) < 0 or int(bound.max()) > NO_GROUP)):
        raise ValueError("bound must be a 1-D integer array of labels in [0, 2^32 - 1]")
    n = len(bound)
    if isinstance(min_size, bool) or not isinstance(min_size, (int, np.integer)) or min_size < 1:
        raise ValueError(f"min_size must be an integer >= 1, got {min_size!r}")
    m = np.asarray(m, dtype=np.float64)
    phi = np.asarray(phi, dtype=np.float64)
    if m.shape != (n,) or phi.shape != (n,):
        raise ValueError(f"expected {n} masses and potentials, got {m.shape} and {phi.shape}")
    members = np.flatnonzero(bound.astype(np.uint64) != NO_GROUP)
    labels, gid = np.unique(bound[members].astype(np.uint64), return_inverse=True)
    ng = len(labels)
    size = np.bincount(gid, minlength=ng)
    keep = np.flatnonzero(size >= min_size)
    keep = keep[np.lexsort((labels[keep], -size[keep]))]
    mm = m[members]
    mass = np.bincount(gid, weights=mm, minlength=ng)

    def mean(keys):
        cols = [np.bincount(gid, weights=mm * np.asarray(state[k], dtype=np.float64)[members], minlength=ng) for k in keys]
        with np.errstate(invalid="ignore", divide="ignore"):
            return np.stack(cols, axis=1) / mass[:, None] if ng else np.zeros((0, 3))

    com, vel = mean(("qx", "qy", "qz")), mean(("vx", "vy", "vz"))
    kin = np.zeros(ng)
    for k, key in enumerate(("vx", "vy", "vz")):
        dv = np.asarray(state[key], dtype=np.float64)[members] - vel[gid, k]
        kin += np.bincount(gid, weights=0.5 * mm * dv * dv, minlength=ng)
    pot = np.bincount(gid, weights=0.5 * mm * phi[members], minlength=ng)
    return {"label": labels[keep].astype(np.uint32), "size": size[keep].astype(np.int64), "mass": mass[keep],
            "com": com[keep].reshape(-1, 3), "vel": vel[keep].reshape(-1, 3), "kinetic": kin[keep], "potential": pot[keep]}


def component_budget(comp, n_comp, m, state, acc, phi, centre=(0.0, 0.0, 0.0)) -> dict[str, np.ndarray]:
    """Mass, momentum, energy and torque budget of the source components (host, O(N * n_comp)).

    comp, n_comp: the labels of Context.component_field_bodies (NO_GROUP bodies belong to no component and are left out);
    m: the masses; state: positions and velocities as Context.download_state returns them; acc, phi: the rows
    Context.component_field_bodies returns (float[n, n_comp, 3] and float[n, n_comp]); centre: the point about which spins
    and torques are taken.  With r_i, v_i the body's position and velocity and c the centre, returns for each component g:
      mass float64[C], com float64[C, 3] (centre of mass), vel float64[C, 3] (mass-weighted mean velocity; both NaN for a
      component of zero mass), kinetic float64[C] (sum m |v|^2 / 2), spin float64[C, 3] (sum m (r - c) x v),
    and for each pair (g, h), the action of the sources h on the bodies of g:
      force float64[C, C, 3] = sum_{i in g} m_i a_i^h, torque float64[C, C, 3] = sum_{i in g} m_i (r_i - c) x a_i^h,
      W float64[C, C] = sum_{i in g} m_i phi_i^h (the interaction energy for g != h is W[g, h] = W[h, g]).
    The total potential energy of the components is (1/2) sum_gh W[g, h], so sum_g kinetic[g] + (1/2) sum_gh W[g, h] is
    their total energy; Newton's third law makes force and torque antisymmetric in (g, h), with force[g, g] = 0 and
    torque[g, g] = 0 up to rounding.  Sums are fp64 np.bincount sums, accumulated in body order, so the budget is
    reproducible."""
    if isinstance(n_comp, bool) or not isinstance(n_comp, (int, np.integer)) or not 1 <= int(n_comp) <= COMPONENTS_MAX:
        raise ValueError(f"n_comp must be an integer in [1, {COMPONENTS_MAX}], got {n_comp!r}")
    C = int(n_comp)
    comp = np.asarray(comp)
    if comp.ndim != 1 or comp.dtype.kind not in "ui":
        raise ValueError("comp must be a 1-D integer array of labels")
    n = len(comp)
    lab = comp.astype(np.int64)
    if n and np.any(((lab < 0) | (lab >= C)) & (lab != NO_GROUP)):
        raise ValueError(f"every label must lie in [0, {C}) or be NO_GROUP")
    m = np.asarray(m, dtype=np.float64)
    acc = np.asarray(acc, dtype=np.float64)
    phi = np.asarray(phi, dtype=np.float64)
    if m.shape != (n,) or acc.shape != (n, C, 3) or phi.shape != (n, C):
        raise ValueError(f"expected m[{n}], acc[{n}, {C}, 3] and phi[{n}, {C}], got {m.shape}, {acc.shape} and {phi.shape}")
    c = np.asarray(centre, dtype=np.float64)
    if c.shape != (3,):
        raise ValueError(f"centre must be 3 numbers, got shape {c.shape}")
    members = np.flatnonzero(lab != NO_GROUP)
    gid = lab[members]
    mm = m[members]
    r = np.stack([np.asarray(state[k], dtype=np.float64)[members] for k in ("qx", "qy", "qz")], axis=1) - c
    v = np.stack([np.asarray(state[k], dtype=np.float64)[members] for k in ("vx", "vy", "vz")], axis=1)

    def gsum(w):  # per-component sums of the columns of w[members, ...]
        w = w.reshape(len(members), int(np.prod(w.shape[1:])))
        return np.stack([np.bincount(gid, weights=w[:, k], minlength=C) for k in range(w.shape[1])], axis=1)

    mass = np.bincount(gid, weights=mm, minlength=C)
    with np.errstate(invalid="ignore", divide="ignore"):
        com = gsum(mm[:, None] * (r + c)) / mass[:, None]
        vel = gsum(mm[:, None] * v) / mass[:, None]
    ma = mm[:, None, None] * acc[members]  # [members, C, 3]
    return {"mass": mass, "com": com, "vel": vel,
            "kinetic": np.bincount(gid, weights=0.5 * mm * np.einsum("ik,ik->i", v, v), minlength=C),
            "spin": gsum(mm[:, None] * np.cross(r, v)),
            "force": gsum(ma).reshape(C, C, 3),
            "torque": gsum(np.cross(r[:, None, :], ma)).reshape(C, C, 3),
            "W": gsum(mm[:, None] * phi[members])}


class B200Bodies:
    """Mirror of the glue's B200Bodies : Bodies<float> — host SoA mirror with lazy device -> host copy
    (pattern: CUDABodies::getDataSoA, src/common/core/CUDABodies.cu:63-93)."""

    def __init__(self, n: int, scheme: str = "galaxy", randInit: int = 0):
        self.n = int(n)
        self.scheme = scheme
        self.dataSoA = init_bodies(scheme, n, randInit)
        self._ctx: Context | None = None
        self._host_current = True

    def getN(self) -> int:
        return self.n

    def bind(self, G, soft, n_gpus=1, **rank_kw):
        if self._ctx is not None:
            self.getDataSoA()
            self._ctx.close()
        self._ctx = Context(self.n, G, soft, n_gpus, **rank_kw)
        d = self.dataSoA
        self._ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
        self._host_current = True

    def context(self) -> Context:
        if self._ctx is None:
            self.bind(G_F32, 1.0)
        return self._ctx

    def invalidateDataSoA(self):
        self._host_current = False

    def getDataSoA(self) -> dict[str, np.ndarray]:
        if not self._host_current and self._ctx is not None:
            self._ctx.download_state(self.dataSoA)
            self._host_current = True
        return self.dataSoA

    def updatePositionsAndVelocities(self, ax, ay, az, dt: float):
        self.context().integrate_host_accel(ax, ay, az, dt)
        self.invalidateDataSoA()


class SimulationNBodyB200:
    """Mirror of SimulationNBodyB200 : SimulationNBodyInterface<float> (glue/SimulationNBodyB200.hpp)."""

    def __init__(self, n: int, scheme: str = "galaxy", soft: float = 2e8, leapfrog: bool = False, n_gpus: int = 1,
                 randInit: int = 0, **rank_kw):
        self.G = G_F32
        self.soft = np.float32(soft)
        self.dt = np.float32(np.inf)  # SimulationNBodyInterface.cpp:12
        self.integrator = INTEGRATOR_LEAPFROG if leapfrog else INTEGRATOR_MURB
        self.bodies = B200Bodies(n, scheme, randInit)
        self.bodies.bind(self.G, self.soft, n_gpus, **rank_kw)
        self.flopsPerIte = np.float32(20.0) * np.float32(n) * np.float32(n)  # SimulationNBodyNaive.cpp:15

    def getBodies(self) -> B200Bodies:
        return self.bodies

    def setDt(self, dt: float):
        self.dt = np.float32(dt)

    def getDt(self) -> float:
        return float(self.dt)

    def getFlopsPerIte(self) -> float:
        return float(self.flopsPerIte)

    def getAllocatedBytes(self) -> float:
        return float(self.bodies.context().allocated_bytes + 8 * 2 * 4 * self.bodies.n)

    def computeOneIteration(self):
        ctx = self.bodies.context()
        ctx.step(self.dt, self.integrator, 1)
        if ctx.n_local_gpus > 1:
            ctx.sync()
        self.bodies.invalidateDataSoA()

    def computeAccelerationsOnly(self):
        self.bodies.context().accel()

    def getAccSoA(self):
        return self.bodies.context().download_accel()

    def computeEnergy(self) -> float:
        return self.bodies.context().energy()
