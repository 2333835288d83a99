"""Multi-process worker of tests/test_groups.py::test_torchrun_ranks (launched with `python -m torch.distributed.run
--nproc-per-node P`): every rank owns one GPU and one shard; b200nb_group_potential and b200nb_unbind are collective and
every rank receives every result.  Rank 0 compares them bit for bit with a single-GPU context after the same two steps."""
import os
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "nbody-eurohpc_b200"))
import b200nb  # noqa: E402
from b200nb import dist as bdist  # noqa: E402

SOFT, DT = 2e8, 3600.0


def run(ctx, d):
    ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
    ctx.step(DT, 0, 2)  # asynchronous: the group calls must wait for the position exchange
    dist6 = ctx.neighbors(6)[1]  # collective
    g = ctx.fof(float(np.median(dist6[:, 5])))  # collective
    return [g, ctx.group_potential(g), *ctx.unbind(g)[:2], *ctx.unbind(g, 2)[:2]]


def main():
    rank, world, local_rank = bdist.env_rank()
    dist = bdist.init_process_group()
    ok = True
    for scheme, n in (("galaxy", 20011), ("random", 70000)):
        d = b200nb.init_bodies(scheme, n)
        rng = np.random.default_rng(n)
        for c in ("vx", "vy", "vz"):
            d[c] = (d[c] + rng.normal(size=n) * 3e4).astype(np.float32)
        nccl_id = bdist.broadcast_bytes(dist, b200nb.Context.unique_id() if rank == 0 else None)
        ctx = b200nb.Context(n, b200nb.G_F32, SOFT, rank=rank, n_ranks=world, device=local_rank, nccl_id=nccl_id)
        got = run(ctx, d)
        ctx.close()
        if rank == 0:
            with b200nb.Context(n, b200nb.G_F32, SOFT, rank=0, n_ranks=1, device=local_rank) as one:
                want = run(one, d)
            good = all(np.array_equal(x.view(np.uint32), y.view(np.uint32)) for x, y in zip(got, want))
            ok &= good
            print(f"{scheme} n={n}: group potential and unbinding identical to one GPU, ok={good}", flush=True)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0 and not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
