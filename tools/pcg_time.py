"""Times the cycle-preconditioned conjugate-gradient solve (amgb_solve_pcg) beside the stationary and Chebyshev-accelerated
iterations of the same cycles on one GPU, one JSON record per solver:

    python tools/pcg_time.py --problem 7pt --n 256     stationary Multadd, Multadd-PCG, Chebyshev-BPX, BPX-PCG
    python tools/pcg_time.py --problem beam --ex 560   BPX-PCG and Multadd-PCG on the elasticity beam of bench.py's c4 leg
                                                        (num_functions = 3, lean storage; host set-up takes minutes)

bytes_per_iter is the algorithmic traffic of one iteration (SURVEY.md 8d): the cycle, for PCG also q = A_0 p and the vector
passes of the dot products, k_pcg_dir and k_pcg_update.  frac_of_6555GBps = bytes_per_iter / (seconds per iteration) over
6555.5 GB/s, the copy bandwidth SURVEY.md measured on a B200."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import async_multigrid_b200 as amg  # noqa: E402
from async_multigrid_b200 import hierarchy as H  # noqa: E402

HBM_GBPS = 6555.5


def bytes_bpx_cycle(h, sweeps=1):
    """restriction chain, (sweeps of) Jacobi from a zero guess on every level, prolongation chain"""
    L = h.num_levels
    tot = 0
    for l in range(L - 1):
        tot += H.bytes_spmv(h.R[l], False) + H.bytes_spmv(h.P[l], True)
    for l in range(L):
        tot += 24 * h.n[l] + (sweeps - 1) * (H.bytes_spmv(h.A[l], True) + 16 * h.n[l])
    return tot


def bytes_cycle(h, solver):
    """the cycle alone (bytes_sync_multadd_cycle counts the stationary solve's residual on A_0 as well)"""
    if solver == H.BPX:
        return bytes_bpx_cycle(h)
    return H.bytes_sync_multadd_cycle(h) - H.bytes_spmv(h.A[0], True)


def bytes_pcg_iteration(h, solver):
    n0 = h.n[0]
    # (r, z) fused: + r;  k_pcg_dir: z, p -> p;  q = A p with (p, q): + p;  k_pcg_update: p, q, u, r -> u, r
    return bytes_cycle(h, solver) + 8 * n0 + 24 * n0 + H.bytes_spmv(h.A[0], False) + 8 * n0 + 48 * n0


def record(name, iters, seconds, relres, bytes_iter, **extra):
    per = seconds / max(iters, 1)
    rec = {"solver": name, "iters": iters, "seconds": seconds, "ms_per_iter": 1e3 * per, "final_true_relres": relres,
           "bytes_per_iter": bytes_iter, "frac_of_6555GBps": (bytes_iter / per / 1e9 / HBM_GBPS) if iters else None}
    rec.update(extra)
    print(json.dumps(rec), flush=True)


def pcg(s, h, solver, name, rhs, max_iters, reps=3):
    out = None
    for _ in range(reps):
        s.set_rhs(rhs)
        s.set_solution(None)
        out = s.solve_pcg(1e-9, max_iters)
    record(name, out["iters"], out["seconds"], out["relres"], bytes_pcg_iteration(h, solver))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--problem", choices=["7pt", "beam"], default="7pt")
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--ex", type=int, default=560)
    ap.add_argument("--max-iters", type=int, default=1000)
    a = ap.parse_args()
    print(json.dumps({"gpu": gpu_info(), "problem": a.problem, "n": a.n if a.problem == "7pt" else a.ex}), flush=True)
    t0 = time.time()
    if a.problem == "7pt":
        A = H.laplacian("7pt", a.n)
        rhs = H.rand_rhs(A.nrows)
        h = H.amg_setup(A)
        hb = H.Hierarchy(h.A, h.P_plain)
        h.build_transfers(H.MULTADD, 0.9)
        hb.build_transfers(H.BPX, 0.9)
        print(json.dumps({"rows": h.n, "levels": h.num_levels, "host_setup_s": round(time.time() - t0, 1)}), flush=True)
        s = amg.Solver(h, H.MULTADD, H.JACOBI, 0.9)
        for _ in range(3):
            s.set_rhs(rhs)
            s.set_solution(None)
            hist, secs = s.solve_sync(1e-9, a.max_iters)
        # (the stationary history is the true residual)
        record("multadd_stationary", len(hist) - 1, secs, float(hist[-1]), bytes_cycle(h, H.MULTADD) + H.bytes_spmv(h.A[0], True))
        pcg(s, h, H.MULTADD, "multadd_pcg", rhs, a.max_iters)
        s.close()
        s = amg.Solver(hb, H.BPX, H.JACOBI, 0.9)
        s.set_rhs(rhs)
        mu, delta, lo, hi = s.ChebySetup(20)
        for _ in range(3):
            s.set_solution(None)
            hist, secs = s.solve_sync(1e-9, a.max_iters, cheby=(mu, delta))
        record("bpx_chebyshev_20_power_steps", len(hist) - 1, secs, float(hist[-1]),
               bytes_cycle(hb, H.BPX) + H.bytes_spmv(hb.A[0], True) + 48 * hb.n[0], eig=[lo, hi])
        pcg(s, hb, H.BPX, "bpx_pcg", rhs, a.max_iters)
        s.close()
    else:
        A, rhs = H.elasticity_beam(a.ex)
        h = H.amg_setup(A, theta=0.5, num_functions=3)
        hm = H.Hierarchy(h.A, h.P_plain)
        h.build_transfers(H.BPX, 0.6)
        hm.build_transfers(H.MULTADD, 0.6)
        print(json.dumps({"rows": h.n, "levels": h.num_levels, "host_setup_s": round(time.time() - t0, 1)}), flush=True)
        s = amg.Solver(h, H.BPX, H.JACOBI, 0.6, lean_storage=True)
        pcg(s, h, H.BPX, "bpx_pcg", rhs, a.max_iters, reps=1)
        s.close()
        s = amg.Solver(hm, H.MULTADD, H.JACOBI, 0.6, lean_storage=True)
        pcg(s, hm, H.MULTADD, "multadd_pcg", rhs, a.max_iters, reps=1)
        s.close()
    print(json.dumps({"gpu_after": gpu_info()}), flush=True)


if __name__ == "__main__":
    main()
