"""Times the row-partitioned multiplicative V-cycle (MULT, csrc/dist.cu dist_vcycle) beside the partitioned synchronous Multadd
cycle on the same problem: a 7-pt Laplacian on an n x n x (n * GPUs) grid, one z-slab of n^3 rows per GPU (bench.py --gpus N's
weak-scaling partition).  One JSON line per solver:

    torchrun --nproc-per-node 1 tools/dist_mult_time.py --edge 128
    torchrun --nproc-per-node 2 tools/dist_mult_time.py --edge 128

cycles: to ||r|| / ||r0|| < 1e-9; s_per_cycle and solve_s: CUDA events around the solve loop (amgb_dist_solve_sync), mean over
--steps solves after one warm-up solve, maximum over the ranks; halo_bytes_per_cycle (summed over the ranks) and
collectives_per_cycle (one rank's halo exchanges, all-gathers and all-reduces): the difference between solves of 3 and 2 cycles.
MULT: V(pre, post) with weighted Jacobi (weight 0.8), plain P and R = P^T, num_pre + num_post sweeps on the coarsest level.
Multadd: as bench.py's multi-GPU leg (symmetrised Jacobi, weight 0.9, factorised level-0 transfers)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import async_multigrid_b200 as amg  # noqa: E402
from async_multigrid_b200 import hierarchy as H, partition as PT  # noqa: E402

TOL = 1e-9


def gpu_info(device):
    """name, power limit and max SM clock of the card (read-only query)"""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or None
    except Exception:
        return None


def measure(s, f, steps, reduce_max, reduce_sum):
    s.set_rhs(f)
    hist, _ = s.solve_sync(TOL, 200)                    # warm-up (the one-rank graph is captured here)
    times = []
    for _ in range(steps):
        hist, secs = s.solve_sync(TOL, 200)
        times.append(secs)
    per = []
    for k in (2, 3):
        hb0, c0 = s.stats()
        s.solve_sync(0.0, k)
        hb1, c1 = s.stats()
        per.append((hb1 - hb0, c1 - c0))
    cycles = len(hist) - 1
    solve_s = reduce_max(float(np.mean(times)))
    return {"cycles": cycles, "final_relres": float(hist[-1]), "s_per_cycle": solve_s / max(cycles, 1), "solve_s": solve_s,
            "halo_bytes_per_cycle": int(reduce_sum(float(per[1][0] - per[0][0]))), "collectives_per_cycle": per[1][1] - per[0][1]}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--edge", type=int, default=128, help="grid edge n: n^3 rows per GPU (named so that torchrun does not take it for one of its own options)")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--num-pre", type=int, default=1)
    ap.add_argument("--num-post", type=int, default=1)
    ap.add_argument("--min-rows-per-rank", type=int, default=4096)
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if not torch.cuda.is_available():
        raise SystemExit("dist_mult_time.py measures on the GPU: no CUDA device")
    dist.init_process_group("gloo", rank=rank, world_size=world)

    def reduce(v, op):
        t = torch.tensor([v], dtype=torch.float64)
        dist.all_reduce(t, op=op)
        return float(t[0])

    reduce_max = lambda v: reduce(v, dist.ReduceOp.MAX)     # noqa: E731
    reduce_sum = lambda v: reduce(v, dist.ReduceOp.SUM)     # noqa: E731
    n = args.edge
    dims = (n, n, n * world)
    t0 = time.time()
    A = H.laplacian("7pt", *dims)
    h = H.amg_setup(A)
    b = H.rand_rhs(A.nrows)
    setup_s = time.time() - t0
    gpu = gpu_info(local)
    runs = [("MULT", H.MULT, 0.8, dict(num_pre=args.num_pre, num_post=args.num_post), {}),
            ("Multadd", H.MULTADD, 0.9, dict(num_pre=1, num_post=1, factor_level0=True), dict(factor_level0=True))]
    for name, solver, w, kw, bt in runs:
        h.build_transfers(solver, w, **bt)
        plan = PT.RankPlan(h, world, rank, plane=n * n, min_rows_per_rank=args.min_rows_per_rank)
        uid = [amg.solver.dist_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        s = amg.DistSolver(plan, uid[0], w, solver=solver, device=local, **kw)
        l0 = plan.layouts[0]
        rec = measure(s, b[l0.row_start:l0.row_start + l0.n_owned], args.steps, reduce_max, reduce_sum)
        s.close()
        if rank == 0:
            rec = dict(solver=name, gpus=world, grid=list(dims), rows_per_gpu=n ** 3, levels=h.num_levels, num_dist=plan.num_dist,
                       graph=world == 1, host_setup_s=round(setup_s, 1), gpu=gpu, **rec)
            print(json.dumps(rec), flush=True)
        dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
