"""bench.py's multi-GPU leg: the row-partitioned synchronous Multadd solve (DMEM_Add replacement,
csrc/dist.cu) on N GPUs of one box, one process per GPU (torchrun), NCCL for the data path.

Workload (BASELINE.json configs[4] family): weak-scaling series with n^3 rows per GPU (n x n x nN grid, one z-slab of n planes
per GPU; N = 8, n = 256 has the size of the 512^3 problem: 134 M rows); and, beside it, the STRONG-scaling record of
configs[4]: the fixed 512^3 problem on N GPUs, E(P) = t(1) / (P t(P)).
Rank 0 builds the global hierarchy on the host (as DMEM_Setup's hypre does on all ranks), cuts it into
per-rank row blocks and hands them over through /dev/shm; the timed region is the solve only.
"""
import json
import os
import shutil
import sys
import time

import numpy as np

from . import hierarchy as H
from . import partition as PT
from . import solver as S


def _log(*a):
    print(*a, file=sys.stderr, flush=True)


def _save_csr(d, name, m):
    np.save(os.path.join(d, name + "_ip.npy"), m.indptr)
    np.save(os.path.join(d, name + "_ix.npy"), m.indices)
    np.save(os.path.join(d, name + "_dv.npy"), m.data)
    np.save(os.path.join(d, name + "_sh.npy"), np.asarray([m.nrows, m.ncols], dtype=np.int64))


def _load_csr(d, name):
    sh = np.load(os.path.join(d, name + "_sh.npy"))
    ip = np.load(os.path.join(d, name + "_ip.npy"), mmap_mode="r")
    ix = np.load(os.path.join(d, name + "_ix.npy"), mmap_mode="r")
    dv = np.load(os.path.join(d, name + "_dv.npy"), mmap_mode="r")
    m = H.CSR.__new__(H.CSR)
    m.nrows, m.ncols = int(sh[0]), int(sh[1])
    m.indptr, m.indices, m.data = np.ascontiguousarray(ip), ix, dv   # indices / data stay memory-mapped (no copy)
    m.nnz = int(m.indptr[-1])
    return m


class _PlanFromDisk:
    """RankPlan look-alike rebuilt from the files rank 0 wrote"""

    def __init__(self, d, rank, nranks):
        meta = json.load(open(os.path.join(d, "meta.json")))
        self.rank, self.nranks = rank, nranks
        self.num_levels = meta["num_levels"]
        self.num_dist = meta["num_dist"]
        self.all_counts = [np.asarray(c, dtype=np.int64) for c in meta["all_counts"]]
        self.layouts = [PT.LevelLayout(*x) for x in meta["layouts"][rank]]
        rd = os.path.join(d, "rank%d" % rank)
        sd = os.path.join(d, "shared")
        self.A, self.P, self.R = [], [], []
        for l in range(self.num_levels):
            src = rd if self.layouts[l].distributed else sd
            self.A.append(_load_csr(src, "A%d" % l))
            if l < self.num_levels - 1:
                self.P.append(_load_csr(src, "P%d" % l))
                self.R.append(_load_csr(src, "R%d" % l))
        self.b = np.load(os.path.join(rd, "b.npy"))
        self.info = meta["info"]


def _fact0(args):
    """level-0 transfers in factorised form (amgb_options.factor_level0): symmetrised Jacobi only"""
    return not getattr(args, "no_factor_level0", False) and args.num_post > 0


def weak_dims(n, world):
    """grid of the weak-scaling series, n^3 rows per GPU: n x n x (n * world), one z-slab of n planes per GPU (round 1's series,
    so the rounds stay comparable; the slab shape -- and with it the halo size and the cycle count, 36 -> 38 -- stays put as N
    grows, which the cube-doubling alternative does not: 512^3 needs 43 cycles)"""
    return (n, n, n * world)


def _build_and_scatter(args, world, d, dims):
    """rank 0: global problem -> plan -> per-rank blocks on /dev/shm (freed level by level)"""
    t0 = time.time()
    nx, ny, nz = dims
    H.set_host_threads(os.cpu_count() or 1)      # the other ranks idle at the barrier meanwhile
    A = H.laplacian("7pt", nx, ny, nz)
    h = H.amg_setup(A, theta=args.theta)
    fact0 = _fact0(args)
    h.build_transfers(H.MULTADD, args.smooth_weight, num_pre=1, num_post=args.num_post, factor_level0=fact0)
    b = H.rand_rhs(A.nrows)
    info = {"levels": h.num_levels, "n": [int(x) for x in h.n], "nnz_A": [int(a.nnz) for a in h.A],
            "operator_complexity": round(h.operator_complexity(), 3),
            "bytes_per_cycle": int(H.bytes_sync_multadd_cycle_factored(h, factor_restriction=False) if fact0 else H.bytes_sync_multadd_cycle(h, args.num_post > 0)),
            "host_setup_s": round(time.time() - t0, 1)}
    _log("[bench] global hierarchy %dx%dx%d: %d levels, n=%s, host setup %.1fs" % (nx, ny, nz, h.num_levels, h.n, time.time() - t0))
    starts, num_dist, halos = PT.plan_layouts(h, world, plane=nx * ny, min_rows_per_rank=args.min_rows_per_rank)
    layouts = [PT.rank_layouts(h, world, r, starts, num_dist, halos) for r in range(world)]
    os.makedirs(os.path.join(d, "shared"), exist_ok=True)
    for r in range(world):
        os.makedirs(os.path.join(d, "rank%d" % r), exist_ok=True)
        l0 = layouts[r][0]
        np.save(os.path.join(d, "rank%d" % r, "b.npy"), b[l0.row_start:l0.row_start + l0.n_owned])
    L = h.num_levels
    from concurrent.futures import ThreadPoolExecutor

    def cut(l, r):
        lay, rd = layouts[r][l], os.path.join(d, "rank%d" % r)
        _save_csr(rd, "A%d" % l, PT._block(h.A[l], lay.row_start, lay.row_start + lay.n_owned, lay.base, lay.n_ext))
        if l < L - 1:
            nxt = layouts[r][l + 1]
            _save_csr(rd, "P%d" % l, PT._block(h.P[l], lay.row_start, lay.row_start + lay.n_owned, nxt.base, nxt.n_ext))
            _save_csr(rd, "R%d" % l, PT._block(h.R[l], nxt.row_start, nxt.row_start + nxt.n_owned, lay.base, lay.n_ext))

    for l in range(L):
        if l < num_dist:
            with ThreadPoolExecutor(max_workers=min(world, 8)) as ex:      # numpy slicing / np.save release the GIL
                list(ex.map(lambda r: cut(l, r), range(world)))
        else:
            sd = os.path.join(d, "shared")
            _save_csr(sd, "A%d" % l, h.A[l])
            if l < L - 1:
                _save_csr(sd, "P%d" % l, h.P[l])
                _save_csr(sd, "R%d" % l, h.R[l])
        # free the global copies of this level as soon as they are on /dev/shm
        h.A[l] = None
        if l < L - 1:
            h.P[l] = h.R[l] = None
            h.P_plain[l] = None
    meta = {"num_levels": L, "num_dist": num_dist, "all_counts": [[int(x) for x in np.diff(s)] for s in starts],
            "layouts": [[[x.n_global, x.row_start, x.n_owned, x.halo_lo, x.halo_hi, x.distributed, x.send_lo, x.send_hi]
                         for x in layouts[r]] for r in range(world)], "info": info}
    json.dump(meta, open(os.path.join(d, "meta.json"), "w"))
    _log("[bench] plan: %d distributed + %d replicated levels, blocks on %s after %.1fs" % (num_dist, L - num_dist, d, time.time() - t0))


STRONG_T1 = os.path.join(os.environ.get("TMPDIR", "/tmp"), "amgb_strong_t1.json")


def _leg(args, rank, world, local, dims, tag, steps, warmup, sampler=None, want_async=False):
    """one partitioned solve series on the grid `dims` (z-slabs): returns the measurements (valid on every rank)"""
    import torch
    import torch.distributed as dist
    from bench import TOL
    base = "/dev/shm" if os.path.isdir("/dev/shm") else "/tmp"
    d = os.path.join(base, "amgb_plan_%s_%s" % (os.environ.get("MASTER_PORT", "0"), tag))
    if rank == 0:
        shutil.rmtree(d, ignore_errors=True)
        _build_and_scatter(args, world, d, dims)
    dist.barrier()
    plan = _PlanFromDisk(d, rank, world)
    uid = [S.dist_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    t0 = time.time()
    s = S.DistSolver(plan, uid[0], args.smooth_weight, num_pre=1, num_post=args.num_post, use_sell=not args.no_sell,
                     factor_level0=_fact0(args), device=local, lean_storage=True,
                     sell_uniform=0 if getattr(args, "no_sell_uniform", False) else 1)
    upload_s = time.time() - t0
    _log("[bench] rank %d (%s): upload + device setup %.1fs, owned rows per level %s" % (rank, tag, upload_s, [x.n_owned for x in plan.layouts]))
    dist.barrier()
    if rank == 0:
        shutil.rmtree(d, ignore_errors=True)
    f_t = torch.empty(plan.layouts[0].n_owned, dtype=torch.float64).pin_memory()
    u_t = torch.empty_like(f_t).pin_memory()
    f_host, u_host = f_t.numpy(), u_t.numpy()
    f_host[:] = plan.b
    s.set_rhs(f_host)

    def sync_all():
        torch.cuda.synchronize()
        dist.barrier()

    for _ in range(warmup):
        hist, secs = s.solve_sync(TOL, args.max_cycles)
    if sampler is not None and rank == 0:
        sampler.start()
    launches0 = s.launch_count()
    sync_all()
    times = []
    for _ in range(steps):
        hist, secs = s.solve_sync(TOL, args.max_cycles)
        times.append(secs)
    sync_all()
    launches = s.launch_count() - launches0
    t = torch.tensor([float(np.mean(times))], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    solve_s = float(t.item())
    # end to end: host f slice in, host u slice out, per rank; wall clock, max over ranks
    e2e = []
    for _ in range(steps + 1):
        sync_all()
        w0 = time.perf_counter()
        s.set_rhs(f_host)
        s.solve_sync(TOL, args.max_cycles)
        s.get_solution(u_host)
        e2e.append(time.perf_counter() - w0)
    t = torch.tensor([float(np.mean(e2e[1:]))], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    hb, ops = s.stats()
    hbt = torch.tensor([float(hb)], dtype=torch.float64, device="cuda")
    dist.all_reduce(hbt)
    clocks = sampler.stop() if (sampler is not None and rank == 0) else None
    out = {"solve_s": solve_s, "e2e_s": e2e_s, "cycles": len(hist) - 1, "final_relres": float(hist[-1]), "launches": int(launches),
           "halo_bytes": float(hbt.item()), "nccl_ops": int(ops), "info": plan.info, "num_dist": plan.num_dist, "clocks": clocks,
           "upload_s": round(upload_s, 1), "graph": bool(int(os.environ.get("AMGB_DIST_GRAPH", "1" if world == 1 else "0")))}
    if want_async:
        out["async"] = _async_on(s, plan, args, world, out["cycles"], min(steps, 3))
    s.close()
    dist.barrier()
    return out


def _calibrate_corrections(one, sync_cycles, tol, max_tries=5):
    """The LOCAL stop rule takes the correction count as an input (as the reference's -num_cycles): the smallest count that
    reaches the tolerance, searched from the synchronous solve's cycle count -- downwards in steps of 2 while the solve still
    converges with a margin (the asynchronous result varies a little from run to run), else upwards in steps of 4.
    one(K) -> (corrections per level, relres, seconds).  -> (K, [tries])"""
    K, tried = int(sync_cycles), []
    cor, rel, secs = one(K)
    tried.append({"corrections": K, "relres": rel, "seconds": secs})
    if rel < tol:
        while K > 4 and len(tried) < max_tries:
            cor, rel, secs = one(K - 2)
            tried.append({"corrections": K - 2, "relres": rel, "seconds": secs})
            if rel >= 0.7 * tol:
                break
            K -= 2
    else:
        while rel >= tol and len(tried) < max_tries:
            K += 4
            cor, rel, secs = one(K)
            tried.append({"corrections": K, "relres": rel, "seconds": secs})
    return K, tried


def _async_on(s, plan, args, world, sync_cycles, steps):
    """the ROW-PARTITIONED asynchronous Multadd solve (csrc/dist_async.cu, DMEM_Add's asynchronous loop) on the solver the
    synchronous leg just used: from x0 = 0, every level group of every rank performs K corrections (LOCAL stop rule); K from
    _calibrate_corrections.  Every rank returns the same record (the ranks
    fail together or not at all: amgb_dist_solve_async agrees on errors before it returns)."""
    import torch
    import torch.distributed as dist
    from bench import TOL

    def one(K):
        s.zero_solution()
        torch.cuda.synchronize()
        dist.barrier()
        cor, rel, secs = s.DMEM_Add_async(K)
        t = torch.tensor([secs], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [int(x) for x in cor], float(rel), float(t.item())

    try:
        K, tried = _calibrate_corrections(one, int(sync_cycles), TOL)
        times = []
        for _ in range(max(int(steps), 1)):
            cor, rel, secs = one(K)
            times.append(secs)
        cb, gt = s.async_groups()
        hb, _ = s.stats()
        return {"solver": "asynchronous Multadd, row-partitioned: one persistent kernel per GPU, level groups exchange boundaries by stores "
                          "over NVLink with per-group step flags, groups asynchronous to one another (LOCAL stop rule)",
                "corrections_per_level": cor, "relres": rel, "converged": bool(rel < TOL), "value": float(np.mean(times)), "unit": "s",
                "timing": "kernel seconds, max over ranks (CUDA events around each rank's launch), mean of %d solves" % len(times),
                "ms_per_correction_round": float(np.mean(times)) * 1e3 / K, "calibration": tried,
                "cta_groups_rank0": [int(x) for x in np.diff(cb)], "group_seconds_rank0": [round(float(x), 4) for x in gt],
                "sync_cycles": int(sync_cycles)}
    except Exception as e:      # (the synchronous records of this line must survive a failure here)
        return {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}


def run(args, rank, world, local):
    import torch
    import torch.distributed as dist
    from bench import ClockSampler, METRIC, load_peaks
    torch.cuda.set_device(local)
    dist.init_process_group("cpu:gloo,cuda:nccl", rank=rank, world_size=world)
    if args.solver != "multadd" or args.smoother != "j":
        raise SystemExit("bench.py --gpus N>1 runs the synchronous Multadd / weighted-Jacobi path")
    n = args.n
    wd = weak_dims(n, world)
    sn = args.strong_n
    # the asynchronous solve runs on the strong-scaling problem (512^3, BASELINE.json configs[4]) -- the weak leg when that IS it
    aleg = getattr(args, "async_leg", "strong")
    strong_is_weak = wd == (sn, sn, sn)
    weak = _leg(args, rank, world, local, wd, "weak", args.steps, args.warmup, ClockSampler(local),
                want_async=aleg == "weak" or (aleg == "strong" and strong_is_weak and not args.no_strong))
    strong = None
    if not args.no_strong:
        if wd == (sn, sn, sn):
            strong = dict(weak)            # at this rank count the weak-series grid IS the strong-scaling problem
            strong["same_run_as_weak"] = True
        else:
            strong = _leg(args, rank, world, local, (sn, sn, sn), "strong", min(args.steps, 3), min(args.warmup, 3), want_async=aleg == "strong")
    if rank == 0:
        peak, peak_src = load_peaks()
        info = weak["info"]
        cycles = weak["cycles"]
        solve_s = weak["solve_s"]
        solve_bytes = info["bytes_per_cycle"] * cycles
        n0 = info["n"][0]
        line = {
            "metric": METRIC, "value": solve_s, "unit": "s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": solve_s * 1e3, "higher_is_better": False, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "3D 7pt Laplacian %dx%dx%d (n=%d) in %d z-slabs of %d rows, sync Multadd, smoother j w=%.2f, tol 1e-9"
                       % (wd[0], wd[1], wd[2], n0, world, n0 // world, args.smooth_weight),
                       "levels": info["levels"], "distributed_levels": weak["num_dist"],
                       "level0_transfers": "factorised (amgb_options.factor_level0)" if _fact0(args) else "explicit Pbar_0 / Rbar_0",
                       "operator_complexity": info["operator_complexity"],
                       "cycles_to_tol": int(cycles), "final_relres": weak["final_relres"], "rows_per_s": n0 / solve_s,
                       "l2": "per-GPU inputs exceed the 126 MB L2; no explicit flush",
                       "exchange": "NCCL send/recv halo with row-neighbours per SpMV input, all-gather of the first replicated level, all-reduce of the norm; "
                                   "the whole cycle (kernels + NCCL operations) is one CUDA graph per iteration" if weak["graph"] else
                                   "NCCL send/recv halo with row-neighbours per SpMV input, all-gather of the first replicated level, all-reduce of the norm",
                       "coarse_levels": "levels below %d rows per rank are REPLICATED on every GPU after one all-gather and computed redundantly "
                                        "(instead of agglomerating them onto one GPU: no second exchange on the way up)" % args.min_rows_per_rank,
                       "host_setup_s": info["host_setup_s"], "upload_s": weak["upload_s"]},
            "e2e": {"value": weak["e2e_s"], "unit": "s", "h2d_bytes_per_step": int(8 * n0), "d2h_bytes_per_step": int(8 * n0)},
            "gpu_launches": int(weak["launches"]) * world,
            "clocks": weak["clocks"],
            "roofline": {"bound": "hbm", "kernel": "whole cycle (all k_spmv launches), aggregate over ranks", "achieved": solve_bytes / solve_s / 1e9,
                         "peak": peak * world, "unit": "GB/s", "frac": solve_bytes / solve_s / 1e9 / (peak * world),
                         "peak_source": peak_src + " x n_gpus", "traffic": None},
            "comm": {"halo_bytes_sent_all_ranks": weak["halo_bytes"], "nccl_ops_per_rank": weak["nccl_ops"]},
        }
        if strong is not None:
            si = strong["info"]
            sb = si["bytes_per_cycle"] * strong["cycles"]
            rec = {"workload": "3D 7pt Laplacian %d^3 (n=%d) in %d z-slabs, sync Multadd, smoother j w=%.2f, tol 1e-9 (BASELINE.json configs[4] problem)"
                               % (sn, si["n"][0], world, args.smooth_weight),
                   "scaling": "strong", "n_gpus": world, "value": strong["solve_s"], "unit": "s", "e2e": strong["e2e_s"],
                   "cycles_to_tol": int(strong["cycles"]), "ms_per_cycle": strong["solve_s"] * 1e3 / max(strong["cycles"], 1),
                   "final_relres": strong["final_relres"], "levels": si["levels"], "distributed_levels": strong["num_dist"],
                   "roofline_frac": sb / strong["solve_s"] / 1e9 / (peak * world), "host_setup_s": si["host_setup_s"],
                   "upload_s": strong["upload_s"], "same_run_as_weak": bool(strong.get("same_run_as_weak", False))}
            try:
                t1 = json.load(open(STRONG_T1))
                if int(t1.get("n", 0)) == sn:
                    rec["t1_seconds"] = t1["value"]
                    rec["t1_cycles"] = t1["cycles"]
                    rec["parallel_efficiency"] = t1["value"] / (world * strong["solve_s"])
                    rec["parallel_efficiency_per_cycle"] = (t1["value"] / t1["cycles"]) / (world * strong["solve_s"] / max(strong["cycles"], 1))
                    rec["efficiency_definition"] = "E(P) = t(1) / (P t(P)) on solve seconds of the same %d^3 problem; t(1) from `bench.py --gpus 1` on this box" % sn
            except Exception:
                rec["parallel_efficiency"] = None
                rec["note"] = "t(1) not found on this box (%s): run `bench.py --gpus 1` first" % STRONG_T1
            if "async" in strong:
                rec["async"] = strong["async"]
            line["strong"] = rec
        if "async" in weak and not (strong is not None and strong.get("same_run_as_weak")):
            line["async"] = weak["async"]
        print(json.dumps(line), flush=True)
    dist.barrier()
    dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------
# asynchronous additive solve across GPUs: a GPU plays one grid's rank group of DMEM_Add (BASELINE.json configs[4])
# ---------------------------------------------------------------------------------------------------------------
def _assign_levels(h, world):
    """working levels (all but the coarsest) -> ranks, longest-processing-time first on the algorithmic bytes of a
    level's chain (the reference sizes its rank groups by the same kind of work model, src/DMEM_Setup.cpp:1678-1736)"""
    work = [(H.bytes_async_chain(h, k, True), k) for k in range(h.num_levels - 1)]
    load, owner = [0] * world, {}
    for w, k in sorted(work, reverse=True):
        r = int(np.argmin(load))
        owner[k] = r
        load[r] += w
    return owner


def run_async(args, rank, world, local):
    import torch
    import torch.distributed as dist
    from bench import ClockSampler, METRIC, TOL, load_peaks
    torch.cuda.set_device(local)
    dist.init_process_group("cpu:gloo,cuda:nccl", rank=rank, world_size=world)
    tag = os.environ.get("MASTER_PORT", "0")
    base = "/dev/shm" if os.path.isdir("/dev/shm") else "/tmp"
    d = os.path.join(base, "amgb_async_%s" % tag)
    n = args.n
    if rank == 0:
        shutil.rmtree(d, ignore_errors=True)
        os.makedirs(d)
        t0 = time.time()
        H.set_host_threads(os.cpu_count() or 1)
        A = H.laplacian("7pt", n)
        h0 = H.amg_setup(A, theta=args.theta)
        h0.build_transfers(H.MULTADD, args.smooth_weight, num_pre=1, num_post=args.num_post)
        for l in range(h0.num_levels):
            _save_csr(d, "A%d" % l, h0.A[l])
            if l < h0.num_levels - 1:
                _save_csr(d, "P%d" % l, h0.P[l])
                _save_csr(d, "R%d" % l, h0.R[l])
        np.save(os.path.join(d, "b.npy"), H.rand_rhs(A.nrows))
        json.dump({"L": h0.num_levels, "host_setup_s": round(time.time() - t0, 1)}, open(os.path.join(d, "meta.json"), "w"))
        del h0, A
    dist.barrier()
    meta = json.load(open(os.path.join(d, "meta.json")))
    L = meta["L"]
    h = H.Hierarchy([_load_csr(d, "A%d" % l) for l in range(L)], [])
    h.P = [_load_csr(d, "P%d" % l) for l in range(L - 1)]
    h.R = [_load_csr(d, "R%d" % l) for l in range(L - 1)]
    b = np.load(os.path.join(d, "b.npy"))
    s = S.Solver(h, H.MULTADD, H.JACOBI, args.smooth_weight, num_pre=1, num_post=args.num_post, use_sell=not args.no_sell, device=local)
    dist.barrier()
    if rank == 0:
        shutil.rmtree(d, ignore_errors=True)
    f_t = torch.empty(h.n[0], dtype=torch.float64).pin_memory()
    u_t = torch.empty_like(f_t).pin_memory()
    f_host, u_host = f_t.numpy(), u_t.numpy()
    f_host[:] = b
    s.set_rhs(f_host)
    s.set_solution(None)
    handles = [None] * world
    dist.all_gather_object(handles, s.ipc_export_solution())
    s.ipc_open_peers([handles[o] for o in range(world) if o != rank])
    owner = _assign_levels(h, world)
    mine = sorted(k for k, r in owner.items() if r == rank)
    bnorm = float(np.linalg.norm(b))

    def solve(nc, e2e=False):
        """x0 = 0; `nc` corrections of every level; returns (max-over-ranks seconds, relres seen by rank 0)"""
        s.synchronize()
        dist.barrier()
        s.set_solution(None)
        s.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        if e2e:
            s.set_rhs(f_host)
        for _ in range(nc):
            for q in mine:
                s.async_dist_correct(q)
        s.synchronize()
        dist.barrier()                       # every peer's reductions have landed
        if e2e and rank == 0:
            s.get_solution(u_host)
        secs = time.perf_counter() - t0
        t = torch.tensor([secs], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        rel = torch.tensor([s.residual_norm() / bnorm if rank == 0 else 0.0], dtype=torch.float64, device="cuda")
        dist.broadcast(rel, src=0)
        return float(t.item()), float(rel.item())

    num = None
    for nc in range(15, args.max_cycles + 1, 5):
        secs, rel = solve(nc)
        if rank == 0:
            _log("[bench] cross-GPU async calibration: %d corrections/level -> relres %.3e (%.4fs)" % (nc, rel, secs))
        if rel < TOL * 0.5:
            num = nc
            break
    if num is None:
        num = args.max_cycles
    for _ in range(args.warmup):
        solve(num)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = s.launch_count()
    runs = [solve(num) for _ in range(args.steps)]
    launches = s.launch_count() - launches0
    e2e = [solve(num, e2e=True) for _ in range(args.steps)]
    clocks = sampler.stop() if rank == 0 else None
    lt = torch.tensor([float(launches)], dtype=torch.float64, device="cuda")
    dist.all_reduce(lt)
    if rank == 0:
        peak, peak_src = load_peaks()
        solve_s = float(np.mean([r[0] for r in runs]))
        bytes_round = sum(H.bytes_async_chain(h, k, True) for k in range(L - 1))
        line = {
            "metric": METRIC, "value": solve_s, "unit": "s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": solve_s * 1e3, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "3D 7-pt Laplacian %d^3 (n=%d), ASYNCHRONOUS Multadd across %d GPUs (a GPU = one grid's rank group of DMEM_Add), "
                                   "smoother j w=%.2f, tol 1e-9, x0=0" % (n, h.n[0], world, args.smooth_weight),
                       "levels": L, "level_owner": {str(k): int(r) for k, r in sorted(owner.items())},
                       "corrections_per_level": int(num), "final_relres": float(np.max([r[1] for r in runs])),
                       "exchange": "fp64 red.global.add into every peer's IPC-mapped solution vector over NVLink; no collective, no waiting",
                       "l2": "per-GPU inputs exceed the 126 MB L2; no explicit flush", "host_setup_s": meta["host_setup_s"],
                       "timing": "host clock between barriers around enqueue + stream synchronize, max over ranks"},
            "e2e": {"value": float(np.mean([r[0] for r in e2e])), "unit": "s", "h2d_bytes_per_step": int(8 * h.n[0] * world),
                    "d2h_bytes_per_step": int(8 * h.n[0])},
            "gpu_launches": int(lt.item()),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "all chains of one correction round, aggregate over ranks", "achieved": bytes_round * num / solve_s / 1e9,
                         "peak": peak * world, "unit": "GB/s", "frac": bytes_round * num / solve_s / 1e9 / (peak * world),
                         "peak_source": peak_src + " x n_gpus", "traffic": None},
        }
        print(json.dumps(line), flush=True)
    dist.barrier()
    s.close()
    dist.barrier()
    dist.destroy_process_group()
