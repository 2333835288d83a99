"""Multi-process worker of tests/test_components.py::test_bitwise_torchrun_ranks (launched with `python -m
torch.distributed.run --nproc-per-node P`): every rank owns one GPU and one shard; b200nb_component_field and
b200nb_component_field_bodies are collective and every rank receives every row.  Rank 0 compares them bit for bit with a
single-GPU context after the same two steps."""
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
    for n, m, C in ((20011, 3001, 3), (70000, 65536 + 129, 64)):
        d = b200nb.init_bodies("galaxy", n)
        rng = np.random.default_rng(n)
        p = [(rng.normal(size=m) * 2e8).astype(np.float32) for _ in range(3)]
        comp = rng.integers(0, C, n).astype(np.uint32)
        comp[::11] = b200nb.NO_GROUP
        nccl_id = bdist.broadcast_bytes(dist, b200nb.Context.unique_id() if rank == 0 else None)
        ctx = b200nb.Context(n, b200nb.G_F32, SOFT, rank=rank, n_ranks=world, device=local_rank, nccl_id=nccl_id)
        ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
        ctx.step(DT, 0, 2)  # asynchronous: the component calls must wait for the position exchange
        got = ctx.component_field(comp, C, *p) + ctx.component_field_bodies(comp, C)  # collective
        ctx.close()
        if rank == 0:
            with b200nb.Context(n, b200nb.G_F32, SOFT, rank=0, n_ranks=1, device=local_rank) as one:
                one.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
                one.step(DT, 0, 2)
                want = one.component_field(comp, C, *p) + one.component_field_bodies(comp, C)
            good = all(np.array_equal(a.view(np.uint32), b.view(np.uint32)) for a, b in zip(got, want))
            ok &= good
            print(f"n={n} points={m} C={C}: component fields bit-identical to one GPU, ok={good}", flush=True)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0 and not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
