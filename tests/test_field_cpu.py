"""CPU checks of the field / potential feature: the fp64 field reference (tests/field_oracle.c) against the pinned oracle,
and the C ABI's argument checks."""
import numpy as np

from conftest import G_F32, SOFT
from field_oracle import FieldOracle


def test_field_at_bodies_equals_fp64_accel(oracle):
    d = oracle.init_bodies("galaxy", 1500)
    ref = oracle.accel_f64(d)
    ax, ay, az, phi, amag = FieldOracle().field(d, d["qx"], d["qy"], d["qz"])
    scale = np.linalg.norm(np.stack(ref), axis=0)
    assert np.all(np.linalg.norm(np.stack([ax, ay, az]) - np.stack(ref), axis=0) <= 1e-12 * scale)
    assert np.all(amag >= scale * (1 - 1e-12))
    # at a body the field's potential carries the self term that the per-body potential leaves out
    pot = FieldOracle().potential(d)
    self_term = float(G_F32) * d["m"].astype(np.float64) / SOFT
    assert np.allclose(phi, pot - self_term, rtol=1e-12, atol=0)


def test_potential_energy_matches_oracle_energy(oracle):
    d = oracle.init_bodies("random", 1200)
    for soft in (SOFT, 1e4):
        phi = FieldOracle().potential(d, soft=soft)
        m = d["m"].astype(np.float64)
        kin = 0.5 * np.sum(m * sum(d[k].astype(np.float64) ** 2 for k in ("vx", "vy", "vz")))
        e = oracle.energy(d, soft=soft)
        assert abs(kin + 0.5 * np.sum(m * phi) - e) <= 1e-12 * abs(e)


def test_potential_sampled_indices(oracle):
    d = oracle.init_bodies("galaxy", 700)
    fo = FieldOracle()
    idx = np.array([0, 5, 699], np.uint64)
    assert np.array_equal(fo.potential(d, idx), fo.potential(d)[idx.astype(np.int64)])


def test_null_context(b200):
    L = b200.lib()
    assert L.b200nb_field(None, 1, None, None, None, None, None, None, None) == b200.EINVAL
    assert L.b200nb_potential(None, None) == b200.EINVAL
