"""Multi-process worker of tests/test_external_scf.py::test_torchrun_ranks (launched with `python -m torch.distributed.run
--nproc-per-node P`): every rank owns one GPU and one shard and sets the same analytic terms and the same expansion.
Rank 0 compares the bodies and tracers bit for bit with a single-GPU context after the same steps."""
import os
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "nbody-eurohpc_b200"))
import b200nb  # noqa: E402
from b200nb import dist as bdist  # noqa: E402

SOFT, DT = 2e8, 3600.0
KEYS = ("qx", "qy", "qz", "vx", "vy", "vz")
GM = float(b200nb.G_F32) * 2.51e24
TERMS = [b200nb.hernquist(2 * GM, 5e7), b200nb.nfw(5 * GM, 4e8, (1e6, 0, 0))]
A, CENTRE = 1e8, (1e6, -2e6, 5e5)


def expansion():
    """a lopsided (12, 6) expansion with every coefficient set, from a fixed seed (identical on every rank)"""
    rng = np.random.default_rng(12)
    S = rng.normal(size=(13, 7, 7)) * 1e-2 * GM / A
    T = rng.normal(size=S.shape) * 1e-2 * GM / A
    S[0, 0, 0] = 3 * GM / A
    T[:, :, 0] = 0.0
    return S, T


def run(ctx, d, t, integrator):
    ctx.set_external(TERMS)
    ctx.set_external_scf(*expansion(), A, CENTRE)
    ctx.upload(d["qx"], d["qy"], d["qz"], d["m"], d["vx"], d["vy"], d["vz"])
    ctx.set_tracers(*[t[k] for k in KEYS])  # collective
    ctx.step(DT, integrator, 5)  # asynchronous
    return ctx.download_tracers(), ctx.download_state()  # collective


def main():
    rank, world, local_rank = bdist.env_rank()
    dist = bdist.init_process_group()
    ok = True
    n, m = 20011, 3001
    d = b200nb.init_bodies("galaxy", n)
    rng = np.random.default_rng(n)
    t = {k: (rng.normal(size=m) * (2e8 if k[0] == "q" else 2e4)).astype(np.float32) for k in KEYS}
    for integrator in (0, 1):
        nccl_id = bdist.broadcast_bytes(dist, b200nb.Context.unique_id() if rank == 0 else None)
        ctx = b200nb.Context(n, b200nb.G_F32, SOFT, rank=rank, n_ranks=world, device=local_rank, nccl_id=nccl_id)
        tr, st = run(ctx, d, t, integrator)
        ctx.close()
        if rank == 0:
            with b200nb.Context(n, b200nb.G_F32, SOFT, rank=0, n_ranks=1, device=local_rank) as one:
                tr1, st1 = run(one, d, t, integrator)
            good = all(np.array_equal(a[k].view(np.uint32), b[k].view(np.uint32)) for a, b in ((tr, tr1), (st, st1)) for k in KEYS)
            ok &= good
            print(f"n={n} tracers={m} integrator={integrator} with terms and an expansion: bit-identical to one GPU, ok={good}",
                  flush=True)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0 and not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
