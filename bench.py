#!/usr/bin/env python
"""bench.py -- the reference's headline measurement on B200: fp64 additive-AMG (Multadd) solve of the
3-D 7-point Laplacian to 1e-9 relative residual, solve seconds + achieved HBM GB/s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--n 256] [--solver ...]

One "step" = one complete solve (x0 = 0 -> ||r||/||r0|| < 1e-9) of the same synthetic problem
(srand(0) right-hand side, the reference's SMEM convention).  `value` = device-timed seconds of the
cycle loop with f, u and the hierarchy resident in HBM (the reference times exactly this loop,
src/SMEM_Solve.cpp:107,245); `e2e` = the same solve through the drop-in C-ABI call amgb_smem_solve
with HOST buffers (pinned f in, u out), copies inside the timed region.  The hierarchy (A_l, P_l, R_l)
is built on the host before the timed region, as the reference's SMEM_Setup does.

--impl reference times the reference's own OpenMP solve phase (oracle/_ref/libref_smem.so: the
unmodified translation units of /root/reference/src compiled by oracle/build_ref.sh) on the host
cores, on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "fp64 Multadd solve sec to 1e-9 rel resid, 3D 7pt Laplacian; SpMV HBM GB/s"
TOL = 1e-9


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device=0):
        self.device, self.proc, self.lines = device, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power)}


SOLVERS = {"mult": 0, "multadd": 2, "afacx": 1, "bpx": 3, "async_multadd": 6, "async_afacx": 5}
SMOOTHERS = {"j": 0, "hybrid_jgs": 2, "L1j": 6}


def factor_level0(args):
    """level-0 transfers in factorised form (amgb_options.factor_level0): synchronous / asynchronous Multadd, symmetrised Jacobi"""
    return (not args.no_factor_level0 and args.solver in ("multadd", "async_multadd") and args.smoother in ("j", "L1j")
            and args.num_post > 0 and args.impl == "b200" and int(os.environ.get("WORLD_SIZE", "1")) == 1)


def build_problem(args, H, fact0=None):
    t0 = time.time()
    if args.problem == "5pt":
        A = H.laplacian("5pt", args.n)
    else:
        A = H.laplacian(args.problem, args.n, args.n, args.nz or args.n)
    h = H.amg_setup(A, theta=args.theta)
    sv = SOLVERS[args.solver]
    base = H.MULTADD if sv in (H.MULTADD, H.ASYNC_MULTADD) else sv
    if sv == H.ASYNC_AFACX:
        base = H.AFACX
    h.build_transfers(base, args.smooth_weight, num_pre=1, num_post=args.num_post,
                      factor_level0=factor_level0(args) if fact0 is None else fact0)
    b = H.rand_rhs(A.nrows)
    log("[bench] hierarchy: %d levels, n=%s, nnz(A)=%s, opcx=%.2f, host setup %.1fs" %
        (h.num_levels, h.n, [a.nnz for a in h.A], h.operator_complexity(), time.time() - t0))
    return h, b


def workload_string(args, h):
    """the SAME string in both arms (the driver compares the arms' `config`)"""
    dims = "%d^2" % args.n if args.problem == "5pt" else ("%d^3" % args.n if not args.nz else "%dx%dx%d" % (args.n, args.n, args.nz))
    return ("%s %s Laplacian %s (n=%d, nnz=%d), %s%s, smoother %s w=%.2f, tol 1e-9, x0=0, b=srand(0) RandDouble(-1,1)"
            % ("2D" if args.problem == "5pt" else "3D", args.problem, dims, h.n[0], h.A[0].nnz, args.solver,
               " + Chebyshev acceleration" if args.cheby else "", args.smoother, args.smooth_weight))


def base_config(args, h, cycles):
    """config keys common to both arms"""
    return {"workload": workload_string(args, h), "levels": h.num_levels, "operator_complexity": round(h.operator_complexity(), 3),
            "cycles_to_tol": int(cycles),
            "hierarchy": "host classical AMG stand-in for hypre BoomerAMG (PMIS, direct interp + 1 Jacobi step, Pmax 4)"}


def ref_hist_path(args, h):
    import hashlib
    key = hashlib.sha1(workload_string(args, h).encode()).hexdigest()[:16]
    return os.path.join(os.environ.get("TMPDIR", "/tmp"), "amgb_ref_hist_%s.json" % key)


def pinned(n):
    import torch
    t = torch.empty(n, dtype=torch.float64).pin_memory()
    return t, t.numpy()


DUMP_SAMPLE = 1 << 21      # solution entries kept by --dump-outputs: with their indices 32 MB, inside the 64 MB the dump may take


def dump_outputs(d, s, hist, corr, rel):
    """--dump-outputs: what the last timed solve handed back, as d/<name>.npy (float64), so that two builds can be compared
    output for output on the same inputs.  Synchronous solvers: the relative residual history; asynchronous ones: the
    corrections per level and the final relative residual.  The solution whole when it has at most DUMP_SAMPLE entries, else
    a fixed sample of it (seed 0, ascending rows) and the sampled row indices."""
    os.makedirs(d, exist_ok=True)
    out = {}
    if hist is not None:
        out["relres_history"] = np.asarray(hist, dtype=np.float64)
    else:
        out["corrections_per_level"] = np.asarray(corr, dtype=np.float64)
        out["final_relres"] = np.asarray([rel], dtype=np.float64)
    u = s.get_solution()
    if u.size <= DUMP_SAMPLE:
        out["solution"] = u
    else:
        rows = np.sort(np.random.default_rng(0).choice(u.size, DUMP_SAMPLE, replace=False))
        out["solution_sample"] = u[rows]
        out["solution_sample_rows"] = rows.astype(np.float64)
    for name, a in out.items():
        np.save(os.path.join(d, name + ".npy"), a)
    log("[bench] outputs of the last timed step written to %s: %s" % (d, ", ".join("%s%s" % (k, v.shape) for k, v in out.items())))


# ------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import async_multigrid_b200 as amg
    from async_multigrid_b200 import hierarchy as H
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 path has no CPU fallback")
    if world > 1:
        if args.dump_outputs:
            raise SystemExit("bench.py: --dump-outputs covers the single-GPU solve only")
        from async_multigrid_b200 import dist_bench
        if args.solver == "async_multadd":
            return dist_bench.run_async(args, rank, world, local)     # BASELINE.json configs[4]: asynchronous across GPUs
        return dist_bench.run(args, rank, world, local)
    torch.cuda.set_device(local)
    peak, peak_src = load_peaks()
    h, b = build_problem(args, H)
    sv, sm = SOLVERS[args.solver], SMOOTHERS[args.smoother]
    is_async = sv in (H.ASYNC_MULTADD, H.ASYNC_AFACX)
    fact0 = factor_level0(args)
    t0 = time.time()
    s = amg.Solver(h, sv, sm, args.smooth_weight, num_pre=1, num_post=args.num_post, jgs_block_rows=args.jgs_block_rows,
                   use_sell=not args.no_sell, factor_level0=fact0, sell_uniform=0 if args.no_sell_uniform else 1,
                   async_type=args.async_type, res_compute_type=args.res_compute_type, read_type=args.read_type)
    log("[bench] upload + device setup %.1fs" % (time.time() - t0))
    f_t, f_host = pinned(h.n[0])
    u_t, u_host = pinned(h.n[0])
    f_host[:] = b
    max_cycles = args.max_cycles

    # async: the stop rule is a correction count (src/SMEM_Async_AMG.cpp:317-322); find the smallest count
    # (multiple of 5) that reaches the tolerance, untimed
    num_cycles = max_cycles
    if is_async:
        for nc in range(10, max_cycles + 1, 5):
            out = s.SMEM_Solve(f_host, TOL, nc)
            log("[bench] async calibration: %d corrections/level -> relres %.3e (%.4fs)" % (nc, out["relres"], out["seconds"]))
            if out["relres"] < TOL * 0.5:
                num_cycles = nc
                break

    cheby = None
    if args.cheby:
        # ChebySetup (EigsPower, 20 steps) is setup, outside the timed region as in the reference (src/SMEM_Setup.cpp:173-175)
        s.set_rhs(f_host)
        mu, delta, alpha, beta = s.ChebySetup(args.cheby_eig_max_iters)
        cheby = (mu, delta)
        log("[bench] ChebySetup: eig min %.4f, eig max %.4f, mu %.4f, delta %.4f" % (alpha, beta, mu, delta))

    def one_solve_resident():
        s.set_solution(None)
        if is_async:
            corr, rel, secs = s.solve_async(num_cycles)
            return secs, num_cycles, rel, corr, None
        hist, secs = s.solve_sync(TOL, max_cycles, cheby=cheby)
        return secs, len(hist) - 1, hist[-1], None, hist

    def one_solve_e2e():
        if cheby is None:
            return s.SMEM_Solve(f_host, TOL, num_cycles if is_async else max_cycles, u_out=u_host)
        s.set_rhs(f_host)
        s.set_solution(None)
        hist, _ = s.solve_sync(TOL, max_cycles, cheby=cheby)
        s.get_solution(u_host)
        return {"relres": hist[-1]}

    s.set_rhs(f_host)
    for _ in range(args.warmup):
        one_solve_resident()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = s.launch_count()
    torch.cuda.synchronize()
    secs_list, cycles, rel, hist = [], 0, 0.0, None
    for _ in range(args.steps):
        secs, cycles, rel, corr, hist = one_solve_resident()
        secs_list.append(secs)
    torch.cuda.synchronize()
    launches = s.launch_count() - launches0
    solve_s = float(np.mean(secs_list))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, s, hist, corr, rel)

    # end to end through the drop-in call with host buffers
    one_solve_e2e()
    e2e_list = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        out = one_solve_e2e()
        e2e_list.append(time.perf_counter() - t0)
    e2e_s = float(np.mean(e2e_list))

    # per-kernel picture of one cycle: every large operator event-timed on the solver's stream (y = M x, plain epilogue),
    # against its ALGORITHMIC bytes (SURVEY.md 8d: 12 nnz + 4 (m+1) + 8 n + 8 m, defined on CSR whatever the storage)
    kernels = []
    for l in range(h.num_levels - 1):
        if h.A[l].nrows < 50000:
            break
        for name, kind, sval in (("A%d" % l, 0, False), ("P%d" % l, 1, False), ("R%d" % l, 2, False)):
            m = (h.A, h.P, h.R)[kind][l]
            ms = s.time_spmv(kind, l, sval, 20)
            gbs = H.bytes_spmv(m, False) / (ms * 1e-3) / 1e9
            kernels.append({"op": "y = %s x" % name, "rows": int(m.nrows), "nnz": int(m.nnz), "ms": round(ms, 4),
                            "achieved": round(gbs, 1), "frac": round(gbs / peak, 3)})
    res_ms = s.time_residual(50)
    clocks = sampler.stop()
    res_bytes = H.bytes_spmv(h.A[0], True)
    res_gbs = res_bytes / (res_ms * 1e-3) / 1e9
    su_slices, su_groups = s.sellu_stats()
    symmetric = sm != H.HYBRID_JACOBI_GAUSS_SEIDEL and args.num_post > 0
    if is_async:
        cyc_bytes = sum(H.bytes_async_chain(h, k, symmetric, fact0) for k in range(h.num_levels))
    else:
        cyc_bytes = H.bytes_sync_multadd_cycle_factored(h) if fact0 else H.bytes_sync_multadd_cycle(h, symmetric)
    solve_bytes = cyc_bytes * cycles
    solve_gbs = solve_bytes / solve_s / 1e9
    true_rel = float(out["relres"])
    cfg = base_config(args, h, cycles)
    line = {
        "metric": METRIC, "value": solve_s, "unit": "s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": solve_s * 1e3, "higher_is_better": False, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": cfg,
        "details": {"final_relres": float(rel),
                    "l2": "inputs (A_0 alone %.2f GB as CSR) exceed the 126 MB L2; no explicit flush" % (12e-9 * h.A[0].nnz),
                    "level0_transfers": ("factorised: plain P_0 / R_0, smoothing factors applied on the fly (amgb_options.factor_level0); "
                                         "bytes_per_cycle counts that form") if fact0 else "explicit Pbar_0 / Rbar_0",
                    "sell_uniform": {"slices_encoded": int(su_slices), "groups": int(su_groups),
                                     "note": "SELL-U: lossless (delta, mask, value) groups replace the column / value streams of the "
                                             "stencil level; its kernels are flagged `exceeds_csr_roofline` below"}},
        "e2e": {"value": e2e_s, "unit": "s", "h2d_bytes_per_step": int(8 * h.n[0]), "d2h_bytes_per_step": int(8 * h.n[0]),
                "final_relres": true_rel},
        "gpu_launches": int(launches),
        "clocks": clocks,
        # time-weighted over EVERY kernel of the timed region: algorithmic bytes of all cycles / device seconds of the solve
        "roofline": {"bound": "hbm", "kernel": "all kernels of the timed solve, time-weighted (algorithmic bytes of %d cycles / device seconds)" % cycles,
                     "achieved": solve_gbs, "peak": peak, "unit": "GB/s", "frac": solve_gbs / peak, "frac_of_8000_spec": solve_gbs / 8000.0,
                     "peak_source": peak_src, "bytes_per_cycle": int(cyc_bytes), "cycles": int(cycles),
                     "traffic": None,      # no ncu pass runs inside bench.py; per-kernel DRAM bytes are in profiles/r2_ncu_*.csv
                     "kernels": kernels,
                     "fine_residual": {"kernel": "k_spmv<1,0>, r = f - A_0 u" + (" (SELL-U encoding)" if su_slices else ""),
                                       "ms_per_launch": res_ms, "bytes_per_launch": int(res_bytes), "achieved": res_gbs,
                                       "frac": res_gbs / peak,
                                       "exceeds_csr_roofline": bool(res_gbs > peak),
                                       "actual_traffic_model_bytes": int(32 * h.n[0]) if su_slices else int(res_bytes)}},
    }
    if hist is not None:
        line["details"]["hist_check"] = hist_check(args, h, hist)
    if corr is not None:
        line["details"]["corrections_per_level"] = [int(x) for x in corr]
        line["details"]["async_group_seconds"] = [round(float(x), 4) for x in s.async_group_times()]
        line["details"]["async_cta_groups"] = [int(x) for x in s.async_groups()[0]]
        used, cap = s.l2_arena_bytes()
        line["details"]["l2_persisting_window_bytes"] = int(used)
    s.close()
    if not is_async and not args.no_async and sv == H.MULTADD:
        # the asynchronous member of BASELINE.json configs[1] on the same problem (persistent cooperative kernel),
        # reported beside the synchronous headline: smallest correction count (multiple of 5) that reaches 1e-9
        sa = amg.Solver(h, H.ASYNC_MULTADD, sm, args.smooth_weight, num_pre=1, num_post=args.num_post,
                        jgs_block_rows=args.jgs_block_rows, use_sell=not args.no_sell, factor_level0=fact0,
                        sell_uniform=0 if args.no_sell_uniform else 1)
        res = None
        for nc in range(25, max_cycles + 1, 5):
            out = sa.SMEM_Solve(f_host, TOL, nc, u_out=u_host)
            if out["relres"] < TOL:
                t0 = time.perf_counter()
                out = sa.SMEM_Solve(f_host, TOL, nc, u_out=u_host)
                ab = int(sum(H.bytes_async_chain(h, k, symmetric, fact0) for k in range(h.num_levels)))
                res = {"solver": "async_multadd", "corrections_per_level": [int(x) for x in out["corrections"]],
                       "value": out["seconds"], "e2e": time.perf_counter() - t0, "unit": "s", "final_relres": float(out["relres"]),
                       "bytes_per_correction_round": ab,
                       "roofline": {"achieved": ab * nc / out["seconds"] / 1e9, "frac": ab * nc / out["seconds"] / 1e9 / peak, "unit": "GB/s"},
                       "group_seconds": [round(float(x), 4) for x in sa.async_group_times()],
                       "cta_groups": [int(x) for x in sa.async_groups()[0]],
                       "l2_persisting_window_bytes": int(sa.l2_arena_bytes()[0]), "gpu_launches": 1}
                break
        line["async"] = res
        sa.close()
    default_leg = sv == H.MULTADD and sm == H.JACOBI and args.problem == "7pt" and not args.cheby
    extras = set(x for x in args.extras.split(",") if x) if default_leg else set()
    if extras:
        try:
            line["configs"] = extra_configs(args, amg, H, h, b, extras)
        except Exception as e:      # the headline line must survive a failure of an extra leg
            line["configs"] = {"failed": "%s: %s" % (type(e).__name__, e)}
    if not args.no_strong and default_leg:
        line["strong"] = strong_leg_single(args, amg, H, peak)
    if not args.no_cpu_baseline:
        if fact0:
            # the reference's own code takes the explicit products (src/SMEM_Setup.cpp:1173-1254)
            h.build_transfers(H.MULTADD, args.smooth_weight, num_pre=1, num_post=args.num_post)
        line["cpu_baseline"] = cpu_baseline(args, h, b, cycles if not is_async else num_cycles)
        if hist is not None and "hist" in line["cpu_baseline"]:
            rh = np.asarray(line["cpu_baseline"].pop("hist"))
            k = min(len(rh), len(hist))
            d = np.abs(np.asarray(hist[:k]) - rh[:k])
            line["details"]["hist_check_sample"] = {"against": "cpu_baseline sample (reference object code, same run)", "cycles_compared": int(k - 1),
                                                    "max_abs_diff": float(np.max(d)), "max_rel_diff": float(np.max(d / np.maximum(rh[:k], 1e-300)))}
    print(json.dumps(line), flush=True)


def strong_leg_single(args, amg, H, peak):
    """t(1) of the strong-scaling record (BASELINE.json configs[4]): the 512^3 problem on ONE GPU (lean storage: sliced ELL
    only), written to a temp file so that the `--gpus N` runs on the same box can form E(P) = t(1) / (P t(P))"""
    import gc
    import torch
    sn = args.strong_n
    try:
        import psutil
        ram = psutil.virtual_memory().available / 2 ** 30
    except Exception:
        ram = 1e9
    need = 110.0 * (sn / 512.0) ** 3
    if ram < need:
        return {"skipped": "host has %.0f GiB available; building the %d^3 hierarchy takes about %.0f GiB" % (ram, sn, need)}
    try:
        t0 = time.time()
        A = H.laplacian("7pt", sn)
        h = H.amg_setup(A, theta=args.theta)
        h.build_transfers(H.MULTADD, args.smooth_weight, num_pre=1, num_post=args.num_post, factor_level0=True)
        b = H.rand_rhs(A.nrows)
        host_s = time.time() - t0
        log("[bench] strong leg: %d^3 hierarchy %s, host setup %.1fs" % (sn, h.n, host_s))
        t0 = time.time()
        s = amg.Solver(h, H.MULTADD, H.JACOBI, args.smooth_weight, num_pre=1, num_post=args.num_post, factor_level0=True,
                       lean_storage=True, sell_uniform=0 if args.no_sell_uniform else 1)
        upload_s = time.time() - t0
        bytes_cycle = H.bytes_sync_multadd_cycle_factored(h)
        n0, levels = h.n[0], h.num_levels
        s.set_rhs(b)
        times, hist = [], None
        for k in range(1 + min(args.steps, 3)):
            s.set_solution(None)
            hist, secs = s.solve_sync(TOL, args.max_cycles)
            if k > 0:
                times.append(secs)
        t0 = time.perf_counter()
        out = s.SMEM_Solve(b, TOL, args.max_cycles)
        e2e = time.perf_counter() - t0
        s.close()
        del s, h, A, b
        gc.collect()
        torch.cuda.empty_cache()
        v = float(np.mean(times))
        cycles = len(hist) - 1
        rec = {"workload": "3D 7pt Laplacian %d^3 (n=%d) on 1 GPU, sync Multadd, smoother j w=%.2f, tol 1e-9 (BASELINE.json configs[4] problem)"
                           % (sn, n0, args.smooth_weight),
               "scaling": "strong", "n_gpus": 1, "value": v, "unit": "s", "e2e": e2e, "cycles_to_tol": int(cycles),
               "ms_per_cycle": v * 1e3 / max(cycles, 1), "final_relres": float(hist[-1]), "levels": levels,
               "roofline_frac": bytes_cycle * cycles / v / 1e9 / peak, "host_setup_s": round(host_s, 1), "upload_s": round(upload_s, 1),
               "parallel_efficiency": 1.0, "storage": "lean (sliced ELL only, no CSR copy)"}
        try:
            from async_multigrid_b200.dist_bench import STRONG_T1
            json.dump({"n": sn, "value": v, "cycles": int(cycles)}, open(STRONG_T1, "w"))
        except Exception as e:
            rec["note"] = "could not write t(1) for the multi-GPU runs: %s" % e
        return rec
    except Exception as e:      # the headline line must survive a failure of this extra leg
        return {"failed": "%s: %s" % (type(e).__name__, e)}


def _solve_record(s, f_host, is_async, max_cycles, cheby=None, steps=2):
    """resident solve(s) of one extra configuration -> dict (value = device seconds of the best of `steps`)"""
    s.set_rhs(f_host)
    if is_async:
        for nc in range(20, max_cycles + 1, 10):
            out = s.SMEM_Solve(f_host, TOL, nc)
            if not np.isfinite(out["relres"]) or out["relres"] > 1e6:
                return {"diverged": True, "corrections_tried": nc, "relres": float(out["relres"])}
            if out["relres"] < TOL:
                best = min(s.SMEM_Solve(f_host, TOL, nc)["seconds"] for _ in range(steps))
                return {"value": best, "unit": "s", "corrections_per_level": int(nc), "final_relres": float(out["relres"])}
        return {"not_converged": True, "corrections_tried": max_cycles, "relres": float(out["relres"])}
    best, hist = None, None
    for _ in range(steps):
        s.set_solution(None)
        hist, secs = s.solve_sync(TOL, max_cycles, cheby=cheby)
        best = secs if best is None else min(best, secs)
    ok = bool(np.isfinite(hist[-1]) and hist[-1] < TOL)
    rec = {"value": best, "unit": "s", "cycles": int(len(hist) - 1), "final_relres": float(hist[-1])}
    if not ok:
        rec["not_converged"] = True
    return rec


def extra_configs(args, amg, H, h, b, which):
    """the other members of BASELINE.json `configs` at their stated sizes, as extra keys of the line (device seconds of the solve,
    hierarchy resident; same stand-in hierarchy provider).  `which`: set of {c1, c2, c3, c4}."""
    out = {}
    w = args.smooth_weight
    if "c1" in which:
        # configs[0]: SMEM sync Multadd, 2-D 5-point 512 x 512, weighted Jacobi (L2-resident on a B200: not an HBM test)
        t0 = time.time()
        A = H.laplacian("5pt", 512)
        h1 = H.amg_setup(A, theta=args.theta)
        h1.build_transfers(H.MULTADD, w, factor_level0=True)
        s = amg.Solver(h1, H.MULTADD, H.JACOBI, w, factor_level0=True)
        rec = _solve_record(s, H.rand_rhs(A.nrows), False, args.max_cycles, steps=3)
        s.close()
        rec.update({"workload": "2D 5pt Laplacian 512^2 (n=%d), sync Multadd, smoother j w=%.2f" % (A.nrows, w), "levels": h1.num_levels,
                    "host_setup_s": round(time.time() - t0, 1)})
        out["c1_5pt_512"] = rec
    if "c2" in which:
        # configs[1]: async Multadd + AFACx, 7pt 256^3, hybrid JGS smoother.  Hybrid JGS with w = 1 diverges asynchronously in the
        # reference's own object code too (DESIGN.md section 4); reported: async Multadd with hybrid JGS (pre 1 / post 0, w = 0.7),
        # sync and async AFACx with weighted Jacobi
        hh = H.Hierarchy(h.A, h.P_plain)
        hh.cpts = h.cpts
        hh.build_transfers(H.MULTADD, 0.7, num_pre=1, num_post=0)
        s = amg.Solver(hh, H.ASYNC_MULTADD, H.HYBRID_JACOBI_GAUSS_SEIDEL, 0.7, num_pre=1, num_post=0, jgs_block_rows=args.jgs_block_rows)
        rec = _solve_record(s, b, True, 150)
        s.close()
        rec["workload"] = "3D 7pt Laplacian %d^3, ASYNC Multadd, hybrid JGS (blocks of %d rows), w=0.70, pre 1 / post 0" % (args.n, args.jgs_block_rows)
        out["c2_async_multadd_hybrid_jgs"] = rec
        hh.build_transfers(H.AFACX, 0.5)
        for tag, sv, asy in (("c2_afacx", H.AFACX, False), ("c2_async_afacx", H.ASYNC_AFACX, True)):
            s = amg.Solver(hh, sv, H.JACOBI, 0.5)
            rec = _solve_record(s, b, asy, 200 if asy else args.max_cycles)
            s.close()
            rec["workload"] = "3D 7pt Laplacian %d^3, %s AFACx, smoother j w=0.50" % (args.n, "ASYNC" if asy else "sync")
            out[tag] = rec
    if "c3" in which:
        # configs[2]: 27-point 256^3, Chebyshev-accelerated Multadd, sync vs async (EigsPower on the device supplies mu, delta)
        t0 = time.time()
        A = H.laplacian("27pt", args.n)
        h3 = H.amg_setup(A, theta=args.theta)
        h3.build_transfers(H.MULTADD, w, factor_level0=True)
        b3 = H.rand_rhs(A.nrows)
        host_s = time.time() - t0
        s = amg.Solver(h3, H.MULTADD, H.JACOBI, w, factor_level0=True, lean_storage=True)
        plain = _solve_record(s, b3, False, args.max_cycles)
        s.set_rhs(b3)
        mu, delta, alpha, beta = s.ChebySetup(args.cheby_eig_max_iters)
        acc = _solve_record(s, b3, False, args.max_cycles, cheby=(mu, delta))
        acc["cheby"] = {"eig_min": alpha, "eig_max": beta, "mu": mu, "delta": delta, "power_iterations": args.cheby_eig_max_iters}
        s.close()
        sa = amg.Solver(h3, H.ASYNC_MULTADD, H.JACOBI, w, factor_level0=True, lean_storage=True)
        asy = _solve_record(sa, b3, True, 150)
        sa.close()
        wl = "3D 27pt Laplacian %d^3 (n=%d, nnz=%d)" % (args.n, A.nrows, A.nnz)
        out["c3_27pt"] = {"workload": wl, "levels": h3.num_levels, "host_setup_s": round(host_s, 1), "sync_multadd": plain,
                          "sync_multadd_chebyshev": acc, "async_multadd": asy}
    if "c4" in which:
        # configs[3]: linear elasticity, 3 unknowns per node, ~8 M DOF, BPX (+ Chebyshev acceleration: plain BPX does not converge);
        # MFEM is absent: Q1 hexahedra on an 8:1:1 two-material beam from the host assembler (DESIGN.md section 7)
        t0 = time.time()
        ex = args.elasticity_ex
        A, rhs = H.elasticity_beam(ex)
        h4 = H.amg_setup(A, theta=args.theta, num_functions=3)
        h4.build_transfers(H.BPX, 0.8)
        host_s = time.time() - t0
        s = amg.Solver(h4, H.BPX, H.JACOBI, 0.8, lean_storage=True)
        s.set_rhs(rhs)
        mu, delta, alpha, beta = s.ChebySetup(args.elasticity_eig_iters)
        beta *= 1.05
        mu, delta = (beta + alpha) / (beta - alpha), 2.0 / (beta + alpha)
        rec = _solve_record(s, rhs, False, args.elasticity_max_cycles, cheby=(mu, delta), steps=1)
        ms = s.time_spmv(0, 0, False, 10)
        s.close()
        rec.update({"workload": "Q1 linear elasticity beam %dx%dx%d elements (n=%d DOF, nnz=%d), BPX + Chebyshev acceleration, smoother j w=0.80"
                                % (ex, max(1, ex // 8), max(1, ex // 8), A.nrows, A.nnz), "levels": h4.num_levels,
                    "host_setup_s": round(host_s, 1), "cheby": {"eig_min": alpha, "eig_max": beta, "mu": mu, "delta": delta},
                    "A0_spmv_ms": ms, "A0_spmv_GBps": H.bytes_spmv(A, False) / (ms * 1e-3) / 1e9})
        out["c4_elasticity_bpx"] = rec
    return out


def hist_check(args, h, hist):
    """max |hist_gpu - hist_ref| against the FULL solve of the reference arm (bench.py --impl reference writes its history to
    a temp file; the driver runs that arm first on the same box)"""
    p = ref_hist_path(args, h)
    if not os.path.exists(p):
        return {"against": None, "note": "no history file from `bench.py --impl reference` on this box (%s)" % p}
    try:
        ref = np.asarray(json.load(open(p))["hist"], dtype=np.float64)
    except Exception as e:
        return {"against": None, "note": "unreadable reference history: %s" % e}
    k = min(len(ref), len(hist))
    d = np.abs(np.asarray(hist[:k]) - ref[:k])
    return {"against": "full solve of the reference arm (oracle/_ref object code), all cycles", "cycles_ref": int(len(ref) - 1),
            "cycles_gpu": int(len(hist) - 1), "max_abs_diff": float(np.max(d)),
            "max_rel_diff": float(np.max(d / np.maximum(ref[:k], 1e-300)))}


# ------------------------------------------------------------------------------------------------
_REF = {}


def cpu_baseline(args, h, b, cycles_to_tol, sample_cycles=None, full=False):
    """The reference's own OpenMP solve phase (oracle/_ref) -- or the oracle port when _ref is absent --
    on the host cores, on a bounded sample: `sample_cycles` cycles, scaled to the cycle count of the full
    solve (every cycle costs the same)."""
    from async_multigrid_b200 import hierarchy as H
    from oracle import oracle as O
    sv, sm = SOLVERS[args.solver], SMOOTHERS[args.smoother]
    cores = os.cpu_count() or 1
    threads = max(h.num_levels, min(cores, args.cpu_threads or cores))
    sample = sample_cycles or args.cpu_sample_cycles
    if full:
        sample = args.max_cycles
    use_ref = O.ref_lib() is not None and not args.cpu_port
    t0 = time.time()
    ref_hist, stock = None, None
    if use_ref:
        # one driver object per process: its setup (allocating and zeroing ~20 GB of per-group vectors) is not the solve phase
        rs = _REF.get("rs")
        if rs is None:
            rs = _REF["rs"] = O.RefSolver(h, sv, sm, b, args.smooth_weight, num_pre=1, num_post=args.num_post, num_threads=threads)
        if sv in (H.ASYNC_MULTADD, H.ASYNC_AFACX):
            out = rs.solve(sample, TOL if full else 1e-300)
            secs, done, rel = out["seconds"], sample, out["relres"]
        elif sv in (H.MULTADD, H.AFACX):
            # SMEM_Solve's loop with ONE added barrier between the cycle's "u += e" and the residual
            # (oracle/ref_driver.cpp ref_solve_sync_det): as shipped, the grouped synchronous cycle races on u
            # (SURVEY.md 5.9b) and does not reach 1e-9; cycle, smoothers and SpMV are the reference's object code
            if not full:
                # untimed pass first, as the reference's own -warmup run does (src/SMEM_Main.cpp:691-693): the first
                # touch of the ~20 GB of per-group vectors would otherwise be charged to the sample
                rs.solve_sync_det(sample, 1e-300)
            out = rs.solve_sync_det(sample, TOL if full else 1e-300)
            secs, done, rel = out["seconds"], out["cycles"], out["hist"][-1]      # omp_get_wtime around the cycle loop
            ref_hist = [float(x) for x in out["hist"]]
            if not full:
                # the STOCK loop beside it (SMEM_Solve exactly as shipped: no added barrier, no lock), same sample: shows what the
                # added barrier + lock cost (its iterates race, SURVEY.md 5.9b, so only its time is used)
                so = rs.solve(sample, 1e-300, async_type=0)
                stock = so["seconds"] / max(so["cycles"], 1)
        else:
            out = rs.solve(sample, TOL if full else 1e-300, async_type=0)
            secs, done, rel = out["seconds"], out["cycles"], out["relres"]
        kind = "reference"
    else:
        O.lib().orc_set_threads(threads)
        base = {H.ASYNC_MULTADD: H.MULTADD, H.ASYNC_AFACX: H.AFACX}.get(sv, sv)
        pb = O.Problem(h, base, sm, args.smooth_weight, num_pre=1, num_post=args.num_post, jgs_blocks=[H.uniform_blocks(m, args.jgs_block_rows) for m in h.n])
        _, hist, secs = pb.solve_sync(b, TOL if full else 1e-300, sample)
        done, rel = len(hist) - 1, hist[-1]
        ref_hist = [float(x) for x in hist]
        kind = "port"
    per_cycle = secs / max(done, 1)
    total = cycles_to_tol if cycles_to_tol else done
    log("[bench] cpu %s: %d cycles in %.2fs (%d threads, wall incl. setup %.1fs), relres after sample %.3e" %
        (kind, done, secs, threads, time.time() - t0, rel))
    out = {"value": per_cycle * total, "unit": "s", "cores": threads, "kind": kind,
           "sample": "%d cycles of the same solve timed (%.3fs, %.4fs/cycle), scaled to the %d cycles of the full solve"
                     % (done, secs, per_cycle, total),
           "seconds_per_cycle": per_cycle, "cycles": int(total), "relres_after_sample": float(rel)}
    if kind == "reference" and sv in (H.MULTADD, H.AFACX):
        out["timed_loop"] = ("SMEM_Solve's k-loop with ONE added omp barrier + the reference's SEMI_ASYNC lock (oracle/ref_driver.cpp "
                             "ref_solve_sync_det): the stock grouped cycle races on u; cycle / smoother / SpMV are the reference's object code")
        if stock is not None:
            out["stock_loop_seconds_per_cycle"] = stock
    if ref_hist is not None:
        out["hist"] = ref_hist
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from async_multigrid_b200 import hierarchy as H
    h, b = build_problem(args, H)
    sv = SOLVERS[args.solver]
    # warm-up 1: the full solve to the tolerance (gives the cycle count); further warm-ups and the timed
    # steps: a bounded sample of cycles each
    full = cpu_baseline(args, h, b, None, full=True)
    cycles = int(full["cycles"])
    if "hist" in full:
        try:        # the b200 arm (run after this one on the same box) compares its history with this full solve
            json.dump({"workload": workload_string(args, h), "hist": full["hist"]}, open(ref_hist_path(args, h), "w"))
        except Exception as e:
            log("[bench] could not write the reference history: %s" % e)
    for _ in range(max(0, args.warmup - 1)):
        cpu_baseline(args, h, b, cycles)
    vals = [cpu_baseline(args, h, b, cycles) for _ in range(args.steps)]
    v = float(np.mean([x["value"] for x in vals]))
    cb = dict(vals[-1])
    cb.pop("hist", None)
    cb["value"] = v
    cb["full_solve_seconds_measured_once"] = full["value"]
    cb["timing"] = ("value = seconds/cycle of a %d-cycle sample (after an untimed pass) x the %d cycles of the full solve; the full solve "
                    "itself was run once to the tolerance (full_solve_seconds_measured_once)" % (args.cpu_sample_cycles, cycles))
    cfg = base_config(args, h, cycles)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": v * 1e3, "higher_is_better": False, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": cb,
        "e2e": {"value": v, "unit": "s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if args.gpus > 1:
        line["same_workload_as_b200_arm"] = False
        line["note"] = ("the reference arm solves the 1-GPU-sized problem (%d^3) on the host cores; at --gpus %d the b200 arm solves %d x "
                        "the rows (weak scaling) -- the ratio of the two arms is NOT a same-workload speed-up" % (args.n, args.gpus, args.gpus))
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", "--grid", dest="n", type=int, default=256, help="grid points per dimension (per GPU slab)")
    ap.add_argument("--nz", type=int, default=0)
    ap.add_argument("--problem", default="7pt", choices=["7pt", "27pt", "5pt"],
                    help="stencil: BASELINE.json configs[1] (7pt) / configs[2] (27pt) / configs[0] (5pt, 2-D n x n)")
    ap.add_argument("--solver", default="multadd", choices=sorted(SOLVERS))
    ap.add_argument("--smoother", default="j", choices=sorted(SMOOTHERS))
    ap.add_argument("--smooth-weight", type=float, default=0.9)
    ap.add_argument("--theta", type=float, default=0.25)
    ap.add_argument("--cheby", action="store_true", help="Chebyshev acceleration of the cycle (-cheby, src/SMEM_Solve.cpp:169-188)")
    ap.add_argument("--cheby-eig-max-iters", type=int, default=20)
    ap.add_argument("--num-post", type=int, default=1, help="-num_post_smooth_sweeps: 0 = plain P + non-symmetrised smoother")
    ap.add_argument("--max-cycles", type=int, default=200)
    ap.add_argument("--jgs-block-rows", type=int, default=8)
    ap.add_argument("--no-sell", action="store_true")
    ap.add_argument("--no-sell-uniform", action="store_true", help="keep the regular sliced-ELL encoding on the stencil levels (no SELL-U)")
    ap.add_argument("--async-type", type=int, default=0, help="asynchronous solver: 0 full (default), 1 semi (-async_type)")
    ap.add_argument("--res-compute-type", type=int, default=0, help="asynchronous solver: 0 local (default), 1 global (-res_compute_type)")
    ap.add_argument("--read-type", type=int, default=0, help="asynchronous solver: 0 sol (default), 1 res (-read_type)")
    ap.add_argument("--min-rows-per-rank", type=int, default=16384,
                    help="multi-GPU: levels with fewer owned rows per rank are replicated, not partitioned")
    ap.add_argument("--extras", default="c1,c2", help="other members of BASELINE.json `configs` reported as extra keys: c1 (5pt 512^2), "
                    "c2 (async Multadd hybrid JGS + AFACx at 256^3), c3 (27pt 256^3, Chebyshev, sync vs async), c4 (elasticity ~8 M DOF, BPX); "
                    "c3 and c4 add minutes of host set-up, so the default runs c1,c2 only")
    ap.add_argument("--elasticity-ex", type=int, default=560, help="c4: elements along the beam (560 -> 561 x 71 x 71 nodes, 8.5 M DOF)")
    ap.add_argument("--elasticity-eig-iters", type=int, default=300)
    ap.add_argument("--elasticity-max-cycles", type=int, default=3000)
    ap.add_argument("--strong-n", type=int, default=512, help="grid of the strong-scaling record (BASELINE.json configs[4]: 512^3)")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling record (512^3 on --gpus N GPUs)")
    ap.add_argument("--async-leg", default="strong", choices=["strong", "weak", "none"],
                    help="--gpus N>1: which problem the row-partitioned ASYNCHRONOUS Multadd solve runs on after the synchronous one "
                         "(strong = the 512^3 problem of BASELINE.json configs[4])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-async", action="store_true", help="skip the asynchronous solve reported beside the headline")
    ap.add_argument("--no-factor-level0", action="store_true",
                    help="upload the explicit products Pbar_0 / Rbar_0 instead of applying the level-0 smoothing factors on the fly")
    ap.add_argument("--cpu-port", action="store_true", help="time the oracle port instead of oracle/_ref")
    ap.add_argument("--cpu-sample-cycles", type=int, default=3)
    ap.add_argument("--cpu-threads", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (residual history or correction counts, the "
                         "solution or a fixed sample of it) to DIR/<name>.npy; single-GPU b200 arm only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm's timed solve")
    if args.warmup < 3 and args.impl == "b200":
        log("[bench] note: fewer than 3 warm-up steps requested")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
