"""The synchronous Multadd solve with the SELL-C-sigma epilogue applied in row order (amgb_options.sell_window_epilogue = 1, the
default) against the epilogue at the sorted slot (0), on ONE hierarchy, alternated in one process so that both forms see the
same card and the same moment:

    python tools/sell_epilogue_time.py --n 256 --rounds 3 --solves 5

Per round and form: `--solves` resident solves (device seconds, cycles).  Then the event-timed SELL-C-sigma operators in the
forms the cycle launches them: P_0 and R_0 plain, the factorised restriction's DUAL pass over A_l (amgb_time_spmv mode 3) and
the prolongation e_l += P_l e_{l+1} (mode 4).  The last record carries the card's name, power limit and SM clock."""
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

MAT_A, MAT_P, MAT_R = 0, 1, 2
FORMS = {"slot": False, "window": True}


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
    solvers = {k: amg.Solver(h, H.MULTADD, H.JACOBI, a.w, factor_level0=True, sell_window_epilogue=v) for k, v in FORMS.items()}
    hists = {}
    for name, s in solvers.items():
        s.set_rhs(b)
        s.set_solution(None)
        hists[name], _ = s.solve_sync(1e-9, 200)                   # warm-up: graph capture, first launches
    same = bool(np.array_equal(np.asarray(hists["slot"]), np.asarray(hists["window"])))
    print(json.dumps({"relres_history_bitwise_equal": same, "cycles": len(hists["window"]) - 1}), flush=True)
    seconds = {k: [] for k in solvers}
    for r in range(a.rounds):
        for name, s in solvers.items():
            for _ in range(a.solves):
                s.set_solution(None)
                hist, secs = s.solve_sync(1e-9, 200)
                seconds[name].append(secs)
            print(json.dumps({"round": r, "form": name, "cycles": len(hist) - 1, "final_relres": float(hist[-1]),
                              "seconds": [round(x, 5) for x in seconds[name][-a.solves:]]}), flush=True)
    # the operators of the cycle stored as SELL-C-sigma, in the forms enq_cycle launches them
    ops = [("P_0 plain", MAT_P, 0, 0), ("R_0 plain", MAT_R, 0, 0)]
    for l in range(1, h.num_levels - 1):
        ops += [("A_%d dual" % l, MAT_A, l, 3), ("Pbar_%d e += P e" % l, MAT_P, l, 4)]
    for name, kind, l, mode in ops:
        if not solvers["window"].is_sell(kind, l):
            continue
        rec = {"op": name, "rows": int({MAT_A: h.A, MAT_P: h.P, MAT_R: h.R}[kind][l].nrows)}
        for r in range(2):                                        # alternated twice
            for form, s in solvers.items():
                rec.setdefault(form + "_ms", []).append(round(s.time_spmv(kind, l, mode, a.reps), 4))
        print(json.dumps(rec), flush=True)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    med = {k: float(np.median(v)) for k, v in seconds.items()}
    print(json.dumps({"summary": True, "median_s": med, "min_s": {k: min(v) for k, v in seconds.items()},
                      "max_s": {k: max(v) for k, v in seconds.items()}, "speedup": med["slot"] / med["window"],
                      "gpu": q.stdout.strip()}), flush=True)
    for s in solvers.values():
        s.close()


if __name__ == "__main__":
    main()
