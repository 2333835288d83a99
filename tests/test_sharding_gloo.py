"""The N>1 path on CPU: world_size-2 `gloo` processes run the sharded algorithm of csrc/context.cu (own-slice targets,
replicated positions, one all-gather of the updated slice per step) with the ORACLE force in place of the CUDA kernel,
and must reproduce the unsharded oracle trajectory bit for bit.  Also covers the unique-id broadcast bench.py uses."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import DT, G_F32, REPO, SOFT, Oracle


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, n, steps, out_dir):
    sys.path.insert(0, os.path.join(REPO, "nbody-eurohpc_b200"))
    sys.path.insert(0, os.path.join(REPO, "tests"))
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port),
                      CUDA_VISIBLE_DEVICES="")  # a CPU-only job: ranks must not bind GPUs, which a host may have fewer of
    from b200nb import dist as bdist, slice_length
    d = bdist.init_process_group("gloo")
    token = bdist.broadcast_bytes(d, bytes(range(128)) if rank == 0 else None)
    assert token == bytes(range(128))
    oracle = Oracle(os.path.join(REPO, "oracle", "liboracle.so"))
    s = oracle.init_bodies("galaxy", n)          # every rank holds the full (replicated) state, like the MPI reference
    L = slice_length(n, world)
    first, last = bdist.slice_bounds(n, rank, world)
    assert first == min(rank * L, n) and last - first <= L
    idx = np.arange(first, last, dtype=np.uint64)
    for _ in range(steps):
        a = [x.astype(np.float32) for x in oracle.accel_f64(s, idx)]          # force on the own targets only
        own = {k: s[k][first:last].copy() for k in ("qx", "qy", "qz", "vx", "vy", "vz")}
        oracle.integrate_murb(own, a[0], a[1], a[2], DT)                      # integrate the own slice only
        for k in ("qx", "qy", "qz", "vx", "vy", "vz"):                        # padded all-gather, slice layout [rank][L]
            send = torch.zeros(L, dtype=torch.float32)
            send[: last - first] = torch.from_numpy(own[k])
            recv = [torch.zeros(L, dtype=torch.float32) for _ in range(world)]
            d.all_gather(recv, send)
            s[k] = torch.cat(recv).numpy()[:n].copy()
    if rank == 0:
        np.savez(os.path.join(out_dir, "sharded.npz"), **{k: s[k] for k in ("qx", "qy", "qz", "vx", "vy", "vz")})
    d.barrier()
    d.destroy_process_group()


@pytest.mark.parametrize("n", [3000, 1024])
def test_two_rank_sharding_matches_unsharded(oracle, tmp_path, n):
    steps, world = 3, 2
    mp.spawn(_worker, args=(world, _free_port(), n, steps, str(tmp_path)), nprocs=world, join=True)
    got = np.load(tmp_path / "sharded.npz")
    ref = oracle.init_bodies("galaxy", n)
    oracle.run_f64force(ref, steps, 0)
    for k in ("qx", "qy", "qz", "vx", "vy", "vz"):
        assert np.array_equal(got[k].view(np.uint32), ref[k].view(np.uint32)), k


def test_slice_bounds_tile_the_bodies(b200):
    from b200nb import dist as bdist
    for n in (1, 1023, 1024, 1025, 200000, 4194304):
        for world in (1, 2, 3, 4, 8):
            spans = [bdist.slice_bounds(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            assert b200.slice_length(n, world) % 256 == 0  # whole AoSoA blocks; the launch rounds up to target tiles itself
