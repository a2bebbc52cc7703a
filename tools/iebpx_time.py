"""Times the implicit extended-system BPX solver (amgb_solve_extended) next to Chebyshev-accelerated BPX (amgb_solve_sync)
on the same hierarchy and bounds:  python tools/iebpx_time.py --n 128
--async adds the asynchronous implicit form (amgb_solve_extended_implicit_async) on the same hierarchy and bounds."""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import async_multigrid_b200 as amg  # noqa: E402
from async_multigrid_b200 import hierarchy as H  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=128)
    ap.add_argument("--w", type=float, default=0.8)
    ap.add_argument("--eig-iters", type=int, default=60, help="power-iteration steps (the reference's default 20 underestimates "
                    "the largest eigenvalue at 128^3 and the Chebyshev iteration then diverges -- in the reference's own loop too)")
    ap.add_argument("--eig-inflate", type=float, default=1.1, help="safety factor on the largest eigenvalue estimate")
    ap.add_argument("--async", dest="run_async", action="store_true", help="also time the asynchronous implicit form")
    ap.add_argument("--async-cap", type=int, default=20000, help="num_cycles of the asynchronous form")
    a = ap.parse_args()
    t0 = time.time()
    A = H.laplacian("7pt", a.n)
    h = H.amg_setup(A)
    h.build_transfers(H.BPX, a.w)
    b = H.rand_rhs(A.nrows)
    setup_s = time.time() - t0
    s = amg.Solver(h, H.BPX, H.JACOBI, a.w)
    s.set_rhs(b)
    _, _, lo, hi = s.ChebySetup(a.eig_iters)
    hi *= a.eig_inflate
    mu, delta = (hi + lo) / (hi - lo), 2.0 / (hi + lo)
    out = None
    for _ in range(3):
        l0 = s.launch_count()
        out = s.SMEM_ExtendedSystemSolve(b, 1e-9, 1000, mu, delta)
        launches = s.launch_count() - l0
    bpx = None
    for _ in range(3):
        s.set_solution(None)
        hist, secs = s.solve_sync(1e-9, 1000, cheby=(mu, delta))
        bpx = dict(cycles=len(hist) - 1, seconds=secs, relres=float(hist[-1]))
    res = {"n": a.n, "rows": h.n, "levels": h.num_levels, "host_setup_s": round(setup_s, 1), "eig": [lo, hi],
           "iebpx": {"iters": out["iters"], "seconds": out["seconds"], "ms_per_iter": 1e3 * out["seconds"] / max(out["iters"] - 1, 1),
                     "ext_relres": out["ext_relres"], "relres": out["relres"], "launches": launches},
           "bpx_cheby": bpx}
    if a.run_async:
        runs = [s.SMEM_ExtendedSystemSolve_async(b, 1e-9, a.async_cap, mu, delta) for _ in range(3)]
        ao = runs[-1]
        res["async_iebpx"] = {"seconds": ao["seconds"], "iters": [int(k) for k in ao["iters"]],
                              "group_seconds": [float(t) for t in ao["group_seconds"]], "ext_relres": ao["ext_relres"],
                              "relres": ao["relres"], "seconds_all_runs": [r["seconds"] for r in runs]}
    print(json.dumps(res))
    s.close()


if __name__ == "__main__":
    main()
