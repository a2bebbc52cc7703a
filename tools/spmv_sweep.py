#!/usr/bin/env python
"""Tuning harness: event-timed y = M x for every large matrix of the 7-pt hierarchy in every storage layout:
`stream` (the warp-stream CSR kernel), `csr` (vector-per-row CSR, use_stream=False) and `sellN` (SELL-C-sigma with
sigma = N); sliced ELL with sigma = 1 stays on where the upload picks it.  Prints achieved GB/s on the ALGORITHMIC
bytes of SURVEY.md 8d.  Run on a B200:  python tools/spmv_sweep.py --n 256"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import async_multigrid_b200 as amg  # noqa: E402
from async_multigrid_b200 import hierarchy as H  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--layouts", default="stream,csr,sell128")
    ap.add_argument("--levels", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    A = H.laplacian("7pt", args.n)
    h = H.amg_setup(A)
    h.build_transfers(H.MULTADD, 0.9)
    mats = []
    for l in range(min(args.levels, h.num_levels - 1)):
        mats += [("A%d" % l, 0, l, False), ("A%d*" % l, 0, l, True), ("P%d" % l, 1, l, False), ("R%d" % l, 2, l, False)]
    rows = {}
    for v in args.layouts.split(","):
        if v == "csr":
            kw = dict(use_stream=False, sell_sigma=0)
        elif v.startswith("sell"):
            kw = dict(sell_sigma=int(v[4:]))
        elif v == "stream":
            kw = dict(sell_sigma=0)
        else:
            raise SystemExit("unknown layout %r (stream, csr, sellN)" % v)
        s = amg.Solver(h, H.MULTADD, H.JACOBI, 0.9, **kw)
        out = {}
        for name, kind, l, sval in mats:
            m = (h.A, h.P, h.R)[kind][l]
            ms = s.time_spmv(kind, l, sval, args.reps)
            out[name] = round(H.bytes_spmv(m, False) / (ms * 1e-3) / 1e9, 0)
        rows[v] = out
        print("layout %-7s  " % v + "  ".join("%s %5.0f" % (k, x) for k, x in out.items()), flush=True)
        s.close()
    print(json.dumps({"n": args.n, "unit": "GB/s (algorithmic bytes)", "nnz_per_row": {name: round(((h.A, h.P, h.R)[k][l]).nnz / ((h.A, h.P, h.R)[k][l]).nrows, 1) for name, k, l, _ in mats}, "results": rows}))


if __name__ == "__main__":
    main()
