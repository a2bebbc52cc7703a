#!/usr/bin/env python
"""Probe of the DEFAULT synchronous Multadd cycle (bench.py's configuration: level-0 transfers factorised) for profiling:
builds the hierarchy, runs `--cycles` cycles and prints the event-timed SpMV of every large operator against its
algorithmic bytes (SURVEY.md 8d).  Under ncu this is the command whose launch list / --set full capture goes to profiles/.

    python tools/cycle_probe.py --n 256 --cycles 2 [--explicit] [--no-factor-restriction] [--problem 27pt]"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import async_multigrid_b200 as amg  # noqa: E402
from async_multigrid_b200 import hierarchy as H  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--problem", default="7pt")
    ap.add_argument("--cycles", type=int, default=2)
    ap.add_argument("--w", type=float, default=0.9)
    ap.add_argument("--explicit", action="store_true", help="explicit Pbar_0 / Rbar_0 instead of the factorised level-0 transfers")
    ap.add_argument("--no-factor-restriction", action="store_true",
                    help="explicit Rbar_l on the levels l >= 1 instead of the factorised restriction (amgb_options.factor_restriction)")
    ap.add_argument("--time-ops", action="store_true", help="event-time every large operator (skip under ncu)")
    ap.add_argument("--peak", type=float, default=6555.5)
    a = ap.parse_args()
    t0 = time.time()
    A = H.laplacian(a.problem, a.n)
    h = H.amg_setup(A)
    fact = not a.explicit
    h.build_transfers(H.MULTADD, a.w, factor_level0=fact)
    b = H.rand_rhs(A.nrows)
    host_s = time.time() - t0
    s = amg.Solver(h, H.MULTADD, H.JACOBI, a.w, factor_level0=fact, factor_restriction=False if a.no_factor_restriction else None)
    s.set_rhs(b)
    s.set_solution(None)
    hist, secs = s.solve_sync(1e-300, a.cycles)
    out = {"n": a.n, "rows": [int(x) for x in h.n], "nnz_A": [int(m.nnz) for m in h.A], "cycles": a.cycles, "seconds": secs,
           "ms_per_cycle": secs * 1e3 / max(a.cycles, 1), "hist": [float(x) for x in hist], "host_setup_s": round(host_s, 1)}
    if a.time_ops:
        ops = {}
        for l in range(h.num_levels - 1):
            if h.A[l].nrows < 20000:
                break
            for name, kind, sval in (("A%d" % l, 0, False), ("A%d*" % l, 0, True), ("P%d" % l, 1, False), ("R%d" % l, 2, False)):
                m = (h.A, h.P, h.R)[kind][l]
                ms = s.time_spmv(kind, l, sval, 20)
                gbs = H.bytes_spmv(m, False) / (ms * 1e-3) / 1e9
                ops[name] = {"rows": int(m.nrows), "nnz": int(m.nnz), "ms": round(ms, 4), "GBps": round(gbs), "frac": round(gbs / a.peak, 3),
                             "sell": bool(s.is_sell(kind, l))}
        out["ops"] = ops
    s.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
