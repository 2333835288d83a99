"""Multi-process worker of tests/test_scf.py::test_torchrun_ranks (launched with `python -m torch.distributed.run
--nproc-per-node P`): every rank owns one GPU and one shard.  b200nb_scf_coefficients is not collective: each rank computes
it on its own device straight after two asynchronous steps, and must get, bit for bit, what a one-GPU context gives for
the positions those steps left."""
import os
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "nbody-eurohpc_b200"))
import b200nb  # noqa: E402
from b200nb import dist as bdist  # noqa: E402

SOFT, DT, A = 2e8, 3600.0, 3e19


def main():
    rank, world, local_rank = bdist.env_rank()
    dist = bdist.init_process_group()
    ok = True
    for scheme, n in (("galaxy", 20011), ("random", 70000)):
        d = b200nb.init_bodies(scheme, n)
        a = A if scheme == "random" else 1e9
        nccl_id = bdist.broadcast_bytes(dist, b200nb.Context.unique_id() if rank == 0 else None)
        ctx = b200nb.Context(n, b200nb.G_F32, SOFT, rank=rank, n_ranks=world, device=local_rank, nccl_id=nccl_id)
        ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
        ctx.step(DT, 0, 2)  # asynchronous: the pass must wait for the position exchange
        got = ctx.scf_coefficients(10, 6, a)  # not collective
        st = ctx.download_state()  # collective
        ctx.close()
        with b200nb.Context(n, b200nb.G_F32, SOFT, rank=0, n_ranks=1, device=local_rank) as one:
            one.upload(st["qx"], st["qy"], st["qz"], d["m"], st["vx"], st["vy"], st["vz"])
            want = one.scf_coefficients(10, 6, a)
        good = all(np.array_equal(x.view(np.uint64), y.view(np.uint64)) for x, y in zip(got, want))
        ok &= good
        print(f"rank {rank} {scheme} n={n}: coefficients identical to one GPU, ok={good}", flush=True)
    dist.barrier()
    dist.destroy_process_group()
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
