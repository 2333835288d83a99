"""CPU checks of the test-particle feature: the host restatement of the tracer updates (tests/tracers_oracle.c) against
the pinned oracle's integrators, and the C ABI's argument checks."""
import numpy as np

from conftest import DT
from tracers_oracle import KEYS, TracersOracle


def _bits(d):
    return [np.asarray(d[k]).view(np.uint32).copy() for k in KEYS]


def _f32_accel(oracle, d):
    return [a.astype(np.float32) for a in oracle.accel_f64(d)]


def test_helper_reproduces_oracle_integrators(oracle):
    """Fed the oracle's fp64 accelerations rounded to fp32, the helper steps the bodies exactly as
    oracle_run_f64force does, for both integrators."""
    to = TracersOracle()
    dt = np.float32(DT)
    for integrator in (0, 1):
        for scheme, n in (("galaxy", 600), ("random", 257)):
            ref = oracle.init_bodies(scheme, n)
            d = {k: v.copy() for k, v in ref.items()}
            steps = 3
            oracle.run_f64force(ref, steps, integrator)
            if integrator == 0:
                for _ in range(steps):
                    to.murb(d, _f32_accel(oracle, d), dt)
            else:
                a = _f32_accel(oracle, d)
                for _ in range(steps):
                    to.kick_drift(d, a, dt)
                    a = _f32_accel(oracle, d)
                    to.kick(d, a, dt)
            for k, (x, y) in zip(KEYS, zip(_bits(d), _bits(ref))):
                assert np.array_equal(x, y), (integrator, scheme, k)


def test_murb_helper_equals_oracle_integrate(oracle):
    to = TracersOracle()
    rng = np.random.default_rng(0)
    n = 5000
    d = {k: (rng.normal(size=n) * s).astype(np.float32) for k, s in zip(KEYS, (1e10, 1e10, 1e9, 3e4, 3e4, 1e3))}
    a = [(rng.normal(size=n) * 1e-3).astype(np.float32) for _ in range(3)]
    ref = {k: v.copy() for k, v in d.items()}
    for dt in (np.float32(DT), np.float32(0.37)):
        to.murb(d, a, dt)
        oracle.integrate_murb(ref, *a, dt)
        assert all(np.array_equal(x, y) for x, y in zip(_bits(d), _bits(ref)))


def test_null_context(b200):
    L = b200.lib()
    assert L.b200nb_set_tracers(None, 0, *[None] * 6) == b200.EINVAL
    assert L.b200nb_set_tracers(None, 5, *[None] * 6) == b200.EINVAL
    assert L.b200nb_download_tracers(None, *[None] * 6) == b200.EINVAL
    assert L.b200nb_n_tracers(None) == 0
