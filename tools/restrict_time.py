"""The synchronous Multadd solve with the explicit restrictions Rbar_l against the factorised ones (amgb_options.factor_restriction)
on ONE hierarchy, alternated in one process so that both forms see the same card and the same moment:

    python tools/restrict_time.py --n 256 --rounds 3 --solves 5

Per round and form: `--solves` resident solves (device seconds, cycles).  Then the event-timed operators of every level that
differs: y = Rbar_l x against y = P_l^T x, and the explicit cycle's one-pass symmetrised smoother against the factorised
form's pass that also writes t_l (amgb_time_spmv modes 2 and 3).  The last record carries the card's name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import async_multigrid_b200 as amg  # noqa: E402
from async_multigrid_b200 import hierarchy as H  # noqa: E402

MAT_A, MAT_R = 0, 2


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--problem", default="7pt")
    ap.add_argument("--w", type=float, default=0.9)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--solves", type=int, default=5)
    ap.add_argument("--reps", type=int, default=50, help="launches per event-timed operator")
    a = ap.parse_args()
    t0 = time.time()
    h = H.amg_setup(H.laplacian(a.problem, a.n))
    h.build_transfers(H.MULTADD, a.w, factor_level0=True)
    b = H.rand_rhs(h.n[0])
    print(json.dumps({"rows": [int(x) for x in h.n], "host_setup_s": round(time.time() - t0, 1)}), flush=True)
    forms = {"explicit": amg.Solver(h, H.MULTADD, H.JACOBI, a.w, factor_level0=True, factor_restriction=False),
             "factorised": amg.Solver(h, H.MULTADD, H.JACOBI, a.w, factor_level0=True, factor_restriction=True)}
    for s in forms.values():
        s.set_rhs(b)
        s.set_solution(None)
        s.solve_sync(1e-9, 200)                                   # warm-up: graph capture, first launches
    seconds = {k: [] for k in forms}
    for r in range(a.rounds):
        for name, s in forms.items():
            for _ in range(a.solves):
                s.set_solution(None)
                hist, secs = s.solve_sync(1e-9, 200)
                seconds[name].append(secs)
            print(json.dumps({"round": r, "form": name, "cycles": len(hist) - 1, "final_relres": float(hist[-1]),
                              "seconds": [round(x, 5) for x in seconds[name][-a.solves:]]}), flush=True)
    ops = []
    last_r = h.num_levels - 2
    for l in range(1, last_r):
        if h.n[l] < 20000:
            break
        ex, fa = forms["explicit"], forms["factorised"]
        ops.append({"level": l, "Rbar_l_ms": ex.time_spmv(MAT_R, l, False, a.reps), "Rbar_l_nnz": int(h.R[l].nnz),
                    "PlT_ms": fa.time_spmv(MAT_R, l, False, a.reps), "PlT_nnz": int(h.plain_restriction(l).nnz),
                    "smoother_pass_ms": ex.time_spmv(MAT_A, l, 2, a.reps), "dual_pass_ms": fa.time_spmv(MAT_A, l, 3, a.reps),
                    "A_l_sell": bool(fa.is_sell(MAT_A, l))})
        print(json.dumps(ops[-1]), flush=True)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    med = {k: float(np.median(v)) for k, v in seconds.items()}
    print(json.dumps({"summary": True, "median_s": med, "min_s": {k: min(v) for k, v in seconds.items()},
                      "max_s": {k: max(v) for k, v in seconds.items()}, "speedup": med["explicit"] / med["factorised"],
                      "gpu": q.stdout.strip()}), flush=True)
    for s in forms.values():
        s.close()


if __name__ == "__main__":
    main()
