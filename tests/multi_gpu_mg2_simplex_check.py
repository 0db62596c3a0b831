"""Run under torchrun on a multi-GPU box: "cg.mg2.simplex" (polOrder-2 multigrid on the ALU ladder, replicated vertex
hierarchy) on N ranks, the subdomains dealt out in contiguous slabs, against the oracle solution on every rank and against
the iteration count of the same solve on one rank.
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29534 tests/multi_gpu_mg2_simplex_check.py
"""
import os
import sys

import numpy as np
import scipy.sparse.linalg as spla
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import dune_hdd_b200 as hdd  # noqa: E402
from oracle import oracle as o  # noqa: E402


def main():
    rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(lr)
    dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
    comm = hdd.parallel.init_comm(rank, world, lr)
    opts = {"type": "cg.mg2.simplex", "precision": 1e-13, "max_iter": 500}
    for n, parts in ((4, (2, 2)), (8, (4, 4)), (16, (8, 8))):
        g = hdd.grids.simplex(n, partitions=parts)
        prob = hdd.problems.ESV2007()
        roff = hdd.parallel.rank_cell_offsets(g, world)
        rng = (int(roff[rank]), int(roff[rank + 1]))
        d = hdd.BlockSWIPDG(g, prob, polorder=2, device=lr, cell_range=rng, comm=comm)
        d.init()
        m = o.Mesh(o.SIMPLEX, g.xy, g.cell_verts, g.cell_neigh).with_polorder(2)
        rp, col = o.pattern(m)
        A = o.assemble_lhs(m, o.const(1.0), None, rp, col)
        u_ref = spla.spsolve(o.to_scipy(rp, col, A).tocsc(), o.assemble_rhs(m, o.esv2007_force()))
        q0, q1 = rng[0] * 6, rng[1] * 6
        u, info = d.solve(opts, return_info=True)
        assert info["converged"], "cg.mg2.simplex converged"
        assert np.abs(u - u_ref[q0:q1]).max() <= 1e-8 * np.abs(u_ref).max(), "cg.mg2.simplex solution"
        # the same solve on one rank (this rank's device, no communicator): the reductions are summed in another order,
        # which may move the last iteration across the threshold, nothing more
        d1 = hdd.BlockSWIPDG(g, prob, polorder=2, device=lr)
        d1.init()
        u1, info1 = d1.solve(opts, return_info=True)
        assert np.abs(u1 - u_ref).max() <= 1e-8 * np.abs(u_ref).max(), "cg.mg2.simplex solution on one rank"
        assert abs(info["iterations"] - info1["iterations"]) <= 1, ("iterations", info["iterations"], info1["iterations"])
        if rank == 0:
            print("cg.mg2.simplex iterations", n, "world", world, info["iterations"], "one rank", info1["iterations"])
            print("multi-GPU cg.mg2.simplex check ok:", n, "world", world)
        del d, d1
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
