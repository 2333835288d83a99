"""Multi-process worker of tests/test_phase_fof.py::test_torchrun_ranks (launched with `python -m torch.distributed.run
--nproc-per-node P`): every rank owns one GPU and one shard; b200nb_fof_phase is collective and every rank receives all
labels.  Rank 0 compares them with a single-GPU context after the same two steps."""
import os
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "nbody-eurohpc_b200"))
import b200nb  # noqa: E402
from b200nb import dist as bdist  # noqa: E402

SOFT, DT = 2e8, 3600.0


def main():
    rank, world, local_rank = bdist.env_rank()
    dist = bdist.init_process_group()
    ok = True
    for scheme, n in (("galaxy", 20011), ("random", 70000)):
        d = b200nb.init_bodies(scheme, n)
        nccl_id = bdist.broadcast_bytes(dist, b200nb.Context.unique_id() if rank == 0 else None)
        ctx = b200nb.Context(n, b200nb.G_F32, SOFT, rank=rank, n_ranks=world, device=local_rank, nccl_id=nccl_id)
        ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
        ctx.step(DT, 0, 2)  # asynchronous: the pack must wait for the position exchange
        dist6 = ctx.neighbors(6)[1]  # collective
        sig = float(np.std(d["vx"]))
        bs = [(float(np.median(dist6[:, 5])), np.inf), (float(np.median(dist6[:, 5])), sig), (2 * float(np.median(dist6[:, 5])), 0.3 * sig)]
        got = [ctx.fof_phase(*b) for b in bs]  # collective
        ctx.close()
        if rank == 0:
            with b200nb.Context(n, b200nb.G_F32, SOFT, rank=0, n_ranks=1, device=local_rank) as one:
                one.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
                one.step(DT, 0, 2)
                want = [one.fof_phase(*b) for b in bs]
            good = all(np.array_equal(x, y) for x, y in zip(got, want))
            ok &= good
            print(f"{scheme} n={n} (b_x, b_v)={bs}: groups identical to one GPU, ok={good}", flush=True)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0 and not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
