"""Host-side mirror of the reference's solve-phase interface on top of the C ABI
(include/amg_b200.h, libamg_b200.so).  Python only marshals pointers; all arithmetic runs in
the sm_100a kernels.  There is no CPU fallback: constructing a solver without a CUDA device
(or without the built extension) raises.

Names follow the reference: SMEM_Solve, SMEM_Sync_Add_Vcycle (-> cycle), SMEM_Async_Add_AMG,
SMEM_MatVec/SMEM_Residual (-> spgemv), SMEM_Smooth (-> smooth)."""
import ctypes as C
import os

import numpy as np

from . import build as _build
from . import hierarchy as H

DP = C.POINTER(C.c_double)
IP = C.POINTER(C.c_int)

MAT_A, MAT_P, MAT_R = 0, 1, 2
CONVERGE_LOCAL, CONVERGE_GLOBAL = 0, 1

ABI_SYMBOLS = [
    "amgb_default_options", "amgb_create", "amgb_destroy", "amgb_last_error", "amgb_launch_count",
    "amgb_set_num_levels", "amgb_set_matrix", "amgb_set_options", "amgb_setup",
    "amgb_set_rhs", "amgb_set_solution", "amgb_get_solution", "amgb_get_residual",
    "amgb_spgemv", "amgb_spgemv_transpose", "amgb_smooth", "amgb_set_jgs_blocks", "amgb_norm2", "amgb_cycle", "amgb_eigs_power", "amgb_solve_sync", "amgb_solve_async",
    "amgb_async_groups", "amgb_solve_extended", "amgb_solve_extended_async", "amgb_smooth_transfer", "amgb_host_csr_free", "amgb_smem_solve", "amgb_time_residual", "amgb_level_storage", "amgb_time_spmv", "amgb_spmv_probe", "amgb_l2_arena_bytes", "amgb_sellu_stats",
    "amgb_sellu_encode_host", "amgb_host_free", "amgb_async_program", "amgb_async_group_times",
    "amgb_solve_extended_implicit_async", "amgb_ext_async_program", "amgb_solve_pcg",
    "amgb_dist_unique_id", "amgb_dist_init", "amgb_dist_set_level", "amgb_dist_setup", "amgb_dist_set_rhs",
    "amgb_dist_get_solution", "amgb_dist_solve_sync", "amgb_dist_solve_sync_accel", "amgb_dist_stats", "amgb_dist_eigs_power",
    "amgb_dist_solve_async", "amgb_dist_async_groups", "amgb_dist_async_plan",
    "amgb_dist_ipc_export_solution", "amgb_dist_ipc_open_neighbours", "amgb_dist_async_smooth", "amgb_dist_residual_norm",
    "amgb_dist_zero_solution",
    "amgb_ipc_export_solution", "amgb_ipc_open_peers", "amgb_async_dist_correct", "amgb_residual_norm", "amgb_stream_synchronize",
]


class Options(C.Structure):
    _fields_ = [("solver", C.c_int), ("smoother", C.c_int), ("smooth_weight", C.c_double),
                ("num_pre_smooth_sweeps", C.c_int), ("num_post_smooth_sweeps", C.c_int),
                ("num_fine_smooth_sweeps", C.c_int), ("num_coarse_smooth_sweeps", C.c_int),
                ("jgs_block_rows", C.c_int), ("use_sell", C.c_int), ("l2_persist", C.c_int), ("use_stream", C.c_int),
                ("factor_level0", C.c_int), ("coarse_solve", C.c_int), ("sell_sigma", C.c_int), ("stream_variant", C.c_int),
                ("sell_uniform", C.c_int), ("async_type", C.c_int), ("res_compute_type", C.c_int), ("read_type", C.c_int),
                ("lean_storage", C.c_int), ("factor_restriction", C.c_int), ("sell_window_epilogue", C.c_int)]


class HostCSR(C.Structure):
    _fields_ = [("nrows", C.c_int), ("ncols", C.c_int), ("nnz", C.c_int),
                ("row_ptr", IP), ("col_idx", IP), ("values", DP)]


_lib = None


def load_library():
    """dlopen libamg_b200.so (building it in-tree if the sources are newer)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.CUDA_LIB
    if not os.path.exists(path):
        _build.build_cuda()
    L = C.CDLL(path)
    L.amgb_last_error.restype = C.c_char_p
    L.amgb_last_error.argtypes = [C.c_void_p]
    L.amgb_launch_count.restype = C.c_longlong
    L.amgb_launch_count.argtypes = [C.c_void_p]
    L.amgb_create.argtypes = [C.POINTER(C.c_void_p), C.c_int]
    L.amgb_destroy.argtypes = [C.c_void_p]
    L.amgb_default_options.argtypes = [C.POINTER(Options)]
    L.amgb_default_options.restype = None
    L.amgb_set_num_levels.argtypes = [C.c_void_p, C.c_int]
    L.amgb_set_matrix.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, IP, IP, DP]
    L.amgb_set_options.argtypes = [C.c_void_p, C.POINTER(Options)]
    L.amgb_setup.argtypes = [C.c_void_p]
    L.amgb_set_rhs.argtypes = [C.c_void_p, DP]
    L.amgb_set_solution.argtypes = [C.c_void_p, DP]
    L.amgb_get_solution.argtypes = [C.c_void_p, DP]
    L.amgb_get_residual.argtypes = [C.c_void_p, DP]
    L.amgb_spgemv.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, DP, C.c_double, DP, DP]
    L.amgb_spgemv_transpose.argtypes = [C.c_void_p, C.c_int, C.c_int, DP, DP]
    L.amgb_smooth.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, DP, DP]
    L.amgb_norm2.argtypes = [C.c_void_p, DP, C.c_int, DP]
    L.amgb_cycle.argtypes = [C.c_void_p, DP, DP]
    L.amgb_eigs_power.argtypes = [C.c_void_p, C.c_int, DP, DP]
    L.amgb_set_jgs_blocks.argtypes = [C.c_void_p, C.c_int, C.c_int, IP]
    L.amgb_solve_sync.argtypes = [C.c_void_p, C.c_double, C.c_int, C.c_int, C.c_double, C.c_double, DP, IP, DP]
    L.amgb_solve_pcg.argtypes = [C.c_void_p, C.c_double, C.c_int, DP, IP, DP, DP]
    L.amgb_solve_async.argtypes = [C.c_void_p, C.c_int, C.c_int, IP, DP, DP]
    L.amgb_solve_extended.argtypes = [C.c_void_p, C.c_double, C.c_int, C.c_double, C.c_double, DP, IP, DP, DP, DP]
    L.amgb_solve_extended_async.argtypes = [C.c_void_p, C.c_double, C.c_int, C.c_double, C.c_double, IP, IP, DP, DP]
    L.amgb_solve_extended_implicit_async.argtypes = [C.c_void_p, C.c_double, C.c_int, C.c_double, C.c_double, IP, DP, DP, DP, DP]
    L.amgb_ext_async_program.argtypes = [C.POINTER(Options), C.c_int, C.c_void_p, C.c_int, IP]
    L.amgb_smooth_transfer.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_int, IP, IP, DP, C.c_int, IP, IP, DP,
                                       C.POINTER(HostCSR), C.POINTER(HostCSR)]
    L.amgb_host_csr_free.argtypes = [C.POINTER(HostCSR)]
    L.amgb_host_csr_free.restype = None
    L.amgb_smem_solve.argtypes = [C.c_void_p, DP, DP, C.c_double, C.c_int, DP, IP, IP, DP, DP]
    L.amgb_time_residual.argtypes = [C.c_void_p, C.c_int, DP]
    L.amgb_level_storage.argtypes = [C.c_void_p, C.c_int, C.c_int, IP]
    L.amgb_time_spmv.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, DP]
    L.amgb_spmv_probe.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, DP, DP, DP, DP, DP, DP, DP, DP, C.c_int, DP, DP, DP, IP]
    L.amgb_l2_arena_bytes.argtypes = [C.c_void_p, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]
    L.amgb_sellu_stats.argtypes = [C.c_void_p, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]
    L.amgb_async_groups.argtypes = [C.c_void_p, IP, IP]
    L.amgb_async_group_times.argtypes = [C.c_void_p, DP]
    L.amgb_async_program.argtypes = [C.POINTER(Options), C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, IP]
    L.amgb_ipc_export_solution.argtypes = [C.c_void_p, C.c_char_p]
    L.amgb_ipc_open_peers.argtypes = [C.c_void_p, C.c_int, C.c_char_p]
    L.amgb_async_dist_correct.argtypes = [C.c_void_p, C.c_int]
    L.amgb_residual_norm.argtypes = [C.c_void_p, DP]
    L.amgb_stream_synchronize.argtypes = [C.c_void_p]
    L.amgb_dist_unique_id.argtypes = [C.c_char_p]
    L.amgb_dist_init.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int]
    L.amgb_dist_set_level.argtypes = [C.c_void_p] + [C.c_int] * 9 + [IP]
    L.amgb_dist_setup.argtypes = [C.c_void_p]
    L.amgb_dist_set_rhs.argtypes = [C.c_void_p, DP]
    L.amgb_dist_get_solution.argtypes = [C.c_void_p, DP]
    L.amgb_dist_solve_sync.argtypes = [C.c_void_p, C.c_double, C.c_int, DP, IP, DP]
    L.amgb_dist_solve_sync_accel.argtypes = [C.c_void_p, C.c_double, C.c_int, C.c_int, C.c_double, C.c_double, DP, IP, DP]
    L.amgb_dist_stats.argtypes = [C.c_void_p, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]
    L.amgb_dist_eigs_power.argtypes = [C.c_void_p, C.c_int, DP, DP, DP]
    L.amgb_dist_solve_async.argtypes = [C.c_void_p, C.c_int, IP, DP, DP]
    L.amgb_dist_async_groups.argtypes = [C.c_void_p, IP, DP]
    L.amgb_dist_async_plan.argtypes = [C.POINTER(Options), C.c_int, C.c_int, C.c_int, IP, C.c_int, C.c_int, C.c_void_p, C.c_int, IP,
                                       C.POINTER(C.c_longlong), IP, IP, C.c_int, IP]
    L.amgb_dist_ipc_export_solution.argtypes = [C.c_void_p, C.c_char_p]
    L.amgb_dist_ipc_open_neighbours.argtypes = [C.c_void_p, C.c_char_p, C.c_longlong, C.c_char_p]
    L.amgb_dist_async_smooth.argtypes = [C.c_void_p, C.c_int]
    L.amgb_dist_residual_norm.argtypes = [C.c_void_p, DP]
    L.amgb_dist_zero_solution.argtypes = [C.c_void_p]
    _lib = L
    return L


def _dp(a):
    return a.ctypes.data_as(DP)


def _ip(a):
    return a.ctypes.data_as(IP)


class AmgError(RuntimeError):
    pass


class Solver:
    """One hierarchy resident on one B200.  `h` is a hierarchy.Hierarchy whose transfers were
    built for `solver` (build_transfers)."""

    def __init__(self, h, solver=H.MULTADD, smoother=H.JACOBI, smooth_weight=1.0, num_pre=1, num_post=1,
                 fine_sweeps=1, coarse_sweeps=1, jgs_block_rows=8, use_sell=True, l2_persist=True, use_stream=True,
                 sell_sigma=None, coarse_solve=False, factor_level0=False, device=0, jgs_blocks=None,
                 sell_uniform=None, async_type=0, res_compute_type=0, read_type=0, lean_storage=False, factor_restriction=None,
                 sell_window_epilogue=None):
        """factor_restriction (amgb_options.factor_restriction): None = on exactly where amgb_setup accepts it, i.e. with
        factor_level0 for the synchronous Multadd cycle with the symmetrised (L1-)Jacobi smoother and one fine sweep; the
        plain P_l^T (Hierarchy.plain_restriction) is then uploaded for the levels l >= 1 in place of h.R[l], which stays as it is.
        sell_window_epilogue (amgb_options.sell_window_epilogue): None = the library's default (on); False = the SELL-C-sigma
        products apply their epilogue at the sorted slot instead of in row order (same results, for A/B timing)"""
        self.L = load_library()
        self.h = h
        self.ctx = C.c_void_p()
        rc = self.L.amgb_create(C.byref(self.ctx), device)
        if rc != 0:
            raise AmgError("amgb_create failed (%d): no CUDA device / driver -- there is no CPU fallback" % rc)
        if solver == H.PAR_BPX:          # same cycle as BPX with the weight applied twice (hierarchy.par_bpx_equivalent)
            solver, smoother, smooth_weight = H.par_bpx_equivalent(smoother, smooth_weight)
        o = Options()
        self.L.amgb_default_options(C.byref(o))
        o.solver, o.smoother, o.smooth_weight = solver, smoother, smooth_weight
        o.num_pre_smooth_sweeps, o.num_post_smooth_sweeps = num_pre, num_post
        o.num_fine_smooth_sweeps, o.num_coarse_smooth_sweeps = fine_sweeps, coarse_sweeps
        o.jgs_block_rows, o.use_sell, o.l2_persist = jgs_block_rows, int(use_sell), int(l2_persist)
        o.use_stream = int(use_stream)
        o.coarse_solve = int(coarse_solve)
        o.factor_level0 = int(factor_level0)
        if sell_sigma is not None:
            o.sell_sigma = int(sell_sigma)
        elif "AMGB_SELL_SIGMA" in os.environ:
            o.sell_sigma = int(os.environ["AMGB_SELL_SIGMA"])
        if sell_uniform is not None:
            o.sell_uniform = int(sell_uniform)
        elif "AMGB_SELL_UNIFORM" in os.environ:
            o.sell_uniform = int(os.environ["AMGB_SELL_UNIFORM"])
        o.async_type, o.res_compute_type, o.read_type = int(async_type), int(res_compute_type), int(read_type)
        o.lean_storage = int(lean_storage)
        if factor_restriction is None:
            factor_restriction = (factor_level0 and solver == H.MULTADD and smoother in (H.JACOBI, H.L1_JACOBI) and num_pre > 0
                                  and num_post > 0 and fine_sweeps == 1)
        o.factor_restriction = int(factor_restriction)
        if sell_window_epilogue is not None:
            o.sell_window_epilogue = int(sell_window_epilogue)
        self.options = o
        self._ck(self.L.amgb_set_options(self.ctx, C.byref(o)))
        self._ck(self.L.amgb_set_num_levels(self.ctx, h.num_levels))
        for l in range(h.num_levels):
            self._set(MAT_A, l, h.A[l])
            if l < h.num_levels - 1:
                self._set(MAT_P, l, h.P[l])
                self._set(MAT_R, l, h.plain_restriction(l) if factor_restriction and l >= 1 else h.R[l])
        self._ck(self.L.amgb_setup(self.ctx))
        self.n0 = h.n[0]
        if jgs_blocks is not None:
            for l, b in enumerate(jgs_blocks):
                self.set_jgs_blocks(l, b)

    def set_jgs_blocks(self, level, bounds):
        """explicit Gauss-Seidel blocks of the hybrid smoother on `level` (the reference's blocks are thread row ranges,
        src/SMEM_Setup.cpp:954-959: hierarchy.nnz_balanced_bounds); None / empty: back to uniform jgs_block_rows blocks"""
        if bounds is None or len(bounds) == 0:
            self._ck(self.L.amgb_set_jgs_blocks(self.ctx, level, 0, None))
            return
        b = np.ascontiguousarray(bounds, dtype=np.int32)
        self._ck(self.L.amgb_set_jgs_blocks(self.ctx, level, len(b) - 1, _ip(b)))

    def _ck(self, rc):
        if rc != 0:
            raise AmgError("amg_b200 error %d: %s" % (rc, self.L.amgb_last_error(self.ctx).decode()))

    def _set(self, kind, l, m):
        self._ck(self.L.amgb_set_matrix(self.ctx, kind, l, m.nrows, m.ncols, m.nnz, _ip(m.indptr), _ip(m.indices), _dp(m.data)))

    def close(self):
        if self.ctx:
            self.L.amgb_destroy(self.ctx)
            self.ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- vectors -------------------------------------------------------------------------------
    def set_rhs(self, f):
        f = np.ascontiguousarray(f, dtype=np.float64)
        assert f.shape[0] == self.n0
        self._ck(self.L.amgb_set_rhs(self.ctx, _dp(f)))

    def set_solution(self, u=None):
        if u is None:
            self._ck(self.L.amgb_set_solution(self.ctx, None))
        else:
            u = np.ascontiguousarray(u, dtype=np.float64)
            self._ck(self.L.amgb_set_solution(self.ctx, _dp(u)))

    def get_solution(self, out=None):
        u = np.empty(self.n0) if out is None else out
        self._ck(self.L.amgb_get_solution(self.ctx, _dp(u)))
        return u

    # -- per-op ----------------------------------------------------------------------------------
    def spgemv(self, kind, level, alpha, x, beta=0.0, b=None):
        m = (self.h.A, self.h.P, self.h.R)[kind][level]
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.empty(m.nrows)
        bb = None if b is None else np.ascontiguousarray(b, dtype=np.float64)
        self._ck(self.L.amgb_spgemv(self.ctx, kind, level, alpha, _dp(x), beta, None if bb is None else _dp(bb), _dp(y)))
        return y

    def spgemv_transpose(self, kind, level, x):
        """y = M^T x (SMEM_MatVecT; restriction through P with -no_construct_R)"""
        m = (self.h.A, self.h.P, self.h.R)[kind][level]
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.empty(m.ncols)
        self._ck(self.L.amgb_spgemv_transpose(self.ctx, kind, level, _dp(x), _dp(y)))
        return y

    def smooth(self, level, f, sweeps=1, symmetric=False, zero_guess=True, u0=None):
        n = self.h.n[level]
        f = np.ascontiguousarray(f, dtype=np.float64)
        u = np.zeros(n) if u0 is None else np.array(u0, dtype=np.float64)
        self._ck(self.L.amgb_smooth(self.ctx, level, self.options.smoother, int(symmetric), sweeps, int(zero_guess), _dp(f), _dp(u)))
        return u

    def norm2(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        out = C.c_double(0)
        self._ck(self.L.amgb_norm2(self.ctx, _dp(x), len(x), C.byref(out)))
        return out.value

    # -- cycles / solves ---------------------------------------------------------------------------
    def cycle(self, r):
        r = np.ascontiguousarray(r, dtype=np.float64)
        c = np.empty(self.n0)
        self._ck(self.L.amgb_cycle(self.ctx, _dp(r), _dp(c)))
        return c

    def SMEM_ExtendedSystemSolve(self, f, tol=1e-9, num_cycles=100, mu=1.0, delta=1.0):
        """`-solver iebpx` (src/SMEM_ExtendedSystem.cpp): hierarchy built for BPX.  -> dict(x, iters, ext_hist, ext_relres,
        relres, seconds)"""
        self.set_rhs(f)
        hist = np.zeros(max(num_cycles, 2) + 1)
        it = C.c_int(0)
        er, rr, secs = C.c_double(0), C.c_double(0), C.c_double(0)
        self._ck(self.L.amgb_solve_extended(self.ctx, tol, int(num_cycles), mu, delta, _dp(hist), C.byref(it), C.byref(er),
                                            C.byref(rr), C.byref(secs)))
        return dict(x=self.get_solution(), iters=it.value, ext_hist=hist[:it.value], ext_relres=er.value, relres=rr.value,
                    seconds=secs.value)

    def SMEM_ExtendedSystemSolve_async(self, f, tol=1e-9, num_cycles=100, mu=1.0, delta=1.0):
        """`-solver async_iebpx` (amgb_solve_extended_implicit_async): the implicit form with every level's group iterating
        asynchronously in one persistent kernel.  -> dict(x, iters (every group's loc_iters), ext_relres, relres,
        group_seconds, seconds)"""
        self.set_rhs(f)
        it = np.zeros(self.h.num_levels, dtype=np.int32)
        gs = np.zeros(self.h.num_levels)
        er, rr, secs = C.c_double(0), C.c_double(0), C.c_double(0)
        self._ck(self.L.amgb_solve_extended_implicit_async(self.ctx, tol, int(num_cycles), mu, delta, _ip(it), C.byref(er), C.byref(rr),
                                                           _dp(gs), C.byref(secs)))
        return dict(x=self.get_solution(), iters=it, ext_relres=er.value, relres=rr.value, group_seconds=gs, seconds=secs.value)

    def ChebySetup(self, iters=20):
        """EigsPower + ChebySetup (src/SMEM_Cheby.cpp:28-60,410-518): returns (mu, delta, alpha, beta)"""
        a, b = C.c_double(0), C.c_double(0)
        self._ck(self.L.amgb_eigs_power(self.ctx, iters, C.byref(a), C.byref(b)))
        alpha, beta = a.value, b.value
        return (beta + alpha) / (beta - alpha), 2.0 / (beta + alpha), alpha, beta

    def solve_sync(self, tol=1e-9, max_cycles=100, cheby=None):
        """resident f,u -> (relres history, seconds)"""
        hist = np.zeros(max_cycles + 1)
        n = C.c_int(0)
        secs = C.c_double(0)
        mu, delta = cheby if cheby else (1.0, 1.0)
        self._ck(self.L.amgb_solve_sync(self.ctx, tol, max_cycles, 1 if cheby else 0, mu, delta, _dp(hist), C.byref(n), C.byref(secs)))
        return hist[:n.value + 1], secs.value

    def solve_pcg(self, tol=1e-9, max_iters=200):
        """conjugate gradients preconditioned by the context's Multadd / BPX cycle on the resident f, u (amgb_solve_pcg; the
        reference's -hypre_pcg).  -> dict(iters, hist (recurrence residual, hist[0] = 1), relres (true final residual),
        seconds); the solution stays in u (get_solution)"""
        hist = np.zeros(max(int(max_iters), 0) + 1)
        it = C.c_int(0)
        rel, secs = C.c_double(0), C.c_double(0)
        self._ck(self.L.amgb_solve_pcg(self.ctx, tol, int(max_iters), _dp(hist), C.byref(it), C.byref(rel), C.byref(secs)))
        return dict(iters=it.value, hist=hist[:it.value + 1], relres=rel.value, seconds=secs.value)

    def solve_async(self, num_cycles, converge=CONVERGE_LOCAL):
        corr = np.zeros(self.h.num_levels, dtype=np.int32)
        rel, secs = C.c_double(0), C.c_double(0)
        self._ck(self.L.amgb_solve_async(self.ctx, num_cycles, converge, _ip(corr), C.byref(rel), C.byref(secs)))
        return corr, rel.value, secs.value

    def SMEM_Solve(self, f_host, tol=1e-9, num_cycles=100, u_out=None):
        """Drop-in for one SMEM_Solve call with host buffers (src/SMEM_Main.cpp:694-757):
        returns dict(u, hist, cycles, corrections, relres, seconds).  u_out: optional caller-owned
        (e.g. pinned) result buffer."""
        f = np.ascontiguousarray(f_host, dtype=np.float64)
        u = np.empty(self.n0) if u_out is None else u_out
        assert u.dtype == np.float64 and u.shape[0] == self.n0 and u.flags["C_CONTIGUOUS"]
        hist = np.zeros(num_cycles + 1)
        n = C.c_int(0)
        corr = np.zeros(self.h.num_levels, dtype=np.int32)
        rel, secs = C.c_double(0), C.c_double(0)
        self._ck(self.L.amgb_smem_solve(self.ctx, _dp(f), _dp(u), tol, num_cycles, _dp(hist), C.byref(n), _ip(corr),
                                        C.byref(rel), C.byref(secs)))
        return dict(u=u, hist=hist[:n.value + 1], cycles=n.value, corrections=corr, relres=rel.value, seconds=secs.value)

    # -- asynchronous solve across GPUs (a GPU plays one grid's rank group of DMEM_Add) ------------------
    def ipc_export_solution(self):
        buf = C.create_string_buffer(64)
        self._ck(self.L.amgb_ipc_export_solution(self.ctx, buf))
        return buf.raw

    def ipc_open_peers(self, handles):
        """handles: list of 64-byte IPC handles of the OTHER ranks' solution vectors"""
        blob = b"".join(handles)
        self._ck(self.L.amgb_ipc_open_peers(self.ctx, len(handles), blob if handles else None))

    def async_dist_correct(self, level):
        self._ck(self.L.amgb_async_dist_correct(self.ctx, level))

    def residual_norm(self):
        v = C.c_double(0)
        self._ck(self.L.amgb_residual_norm(self.ctx, C.byref(v)))
        return v.value

    def synchronize(self):
        self._ck(self.L.amgb_stream_synchronize(self.ctx))

    # -- introspection --------------------------------------------------------------------------------
    def launch_count(self):
        return int(self.L.amgb_launch_count(self.ctx))

    def time_residual(self, reps=20):
        ms = C.c_double(0)
        self._ck(self.L.amgb_time_residual(self.ctx, reps, C.byref(ms)))
        return ms.value

    def time_spmv(self, kind, level, use_sval=False, reps=20):
        ms = C.c_double(0)
        self._ck(self.L.amgb_time_spmv(self.ctx, kind, level, int(use_sval), reps, C.byref(ms)))
        return ms.value

    def spmv_probe(self, kind, level, x, alpha=1.0, b=None, beta=0.0, c=None, gamma=0.0, rs=None, b2=None, beta2=0.0,
                   xs=None, xself=0.0, use_sval=False, norm=False, dot_w=None, dual_s2=None):
        """y = gamma c + rs o (beta b + beta2 b2 + alpha M x) + xself xs through the solve's SpMV kernels (amgb_spmv_probe).
        norm: also sum y_i^2; dot_w: also sum y_i dot_w_i; dual_s2 (column-scaled values, b given): also y2 = dual_s2 o (b + y).
        Returns (y, y2 or None, sum or None, whether the window-staged SELL-C-sigma kernel ran)."""
        m = {MAT_A: self.h.A, MAT_P: self.h.P, MAT_R: self.h.R}[kind][level]
        vec = lambda v: None if v is None else np.ascontiguousarray(v, dtype=np.float64)
        x, b, c, rs, b2, xs = vec(x), vec(b), vec(c), vec(rs), vec(b2), vec(xs)
        w = vec(dot_w if dot_w is not None else dual_s2)
        mode = 3 if dual_s2 is not None else (2 if dot_w is not None else (1 if norm else 0))
        coef = np.array([alpha, beta, gamma, beta2, xself], dtype=np.float64)
        y = np.empty(m.nrows)
        y2 = np.empty(m.nrows) if mode == 3 else None
        ss, win = C.c_double(0), C.c_int(0)
        p = lambda v: None if v is None else _dp(v)
        self._ck(self.L.amgb_spmv_probe(self.ctx, kind, level, int(use_sval), _dp(coef), _dp(x), p(b), p(c), p(rs), p(b2), p(xs),
                                        p(w), mode, _dp(y), p(y2), C.byref(ss), C.byref(win)))
        return y, y2, (ss.value if mode in (1, 2) else None), bool(win.value)

    def l2_arena_bytes(self):
        a, b = C.c_longlong(0), C.c_longlong(0)
        self._ck(self.L.amgb_l2_arena_bytes(self.ctx, C.byref(a), C.byref(b)))
        return a.value, b.value

    def sellu_stats(self):
        """(slices stored in the SELL-U encoding, groups) over the whole hierarchy"""
        a, b = C.c_longlong(0), C.c_longlong(0)
        self._ck(self.L.amgb_sellu_stats(self.ctx, C.byref(a), C.byref(b)))
        return a.value, b.value

    def is_sell(self, kind, level):
        v = C.c_int(0)
        self._ck(self.L.amgb_level_storage(self.ctx, kind, level, C.byref(v)))
        return bool(v.value)

    def async_group_times(self):
        """seconds every level group spent inside the last launch of the persistent kernel"""
        t = np.zeros(self.h.num_levels)
        self._ck(self.L.amgb_async_group_times(self.ctx, _dp(t)))
        return t

    def async_groups(self):
        cb = np.zeros(self.h.num_levels + 1, dtype=np.int32)
        g = C.c_int(0)
        self._ck(self.L.amgb_async_groups(self.ctx, _ip(cb), C.byref(g)))
        return cb, g.value


class AsyncOpSym(C.Structure):
    """csrc/launch.h AsyncOpSym: one operation of a level group's program (symbolic)"""
    _fields_ = [(k, C.c_int) for k in ("type", "mat_kind", "mat_level", "sval", "range", "barrier", "x", "y", "b", "c", "rs", "b2",
                                       "xs", "red", "red_copy", "acc", "level", "sweeps", "zero", "locked")] + \
               [(k, C.c_double) for k in ("alpha", "beta", "gamma", "beta2", "xself", "red_scale")]


def async_program(num_levels, solver, smoother=H.JACOBI, symmetric=True, factor_level0=False, fine_sweeps=1, coarse_sweeps=1,
                  async_type=0, res_compute_type=0, read_type=0, coarse_solve=False):
    """the programs the persistent asynchronous kernel interprets (amgb_async_program; host-only, no GPU needed):
    list over the level groups of lists of AsyncOpSym"""
    L = load_library()
    o = Options()
    L.amgb_default_options(C.byref(o))
    o.solver, o.smoother = solver, smoother
    o.num_fine_smooth_sweeps, o.num_coarse_smooth_sweeps = fine_sweeps, coarse_sweeps
    o.async_type, o.res_compute_type, o.read_type = async_type, res_compute_type, read_type
    o.coarse_solve = int(coarse_solve)
    ops = (AsyncOpSym * 4096)()
    ob = np.zeros(num_levels + 1, dtype=np.int32)
    rc = L.amgb_async_program(C.byref(o), num_levels, int(symmetric), int(factor_level0), ops, 4096, _ip(ob))
    if rc != 0:
        raise AmgError("amgb_async_program failed (%d): unsupported combination of asynchronous options" % rc)
    return [[ops[i] for i in range(ob[q], ob[q + 1])] for q in range(num_levels)]


def ext_async_program(num_levels, smoother=H.JACOBI):
    """the programs of the asynchronous implicit extended-system solver (amgb_ext_async_program; host-only, no GPU needed):
    list over the level groups of lists of AsyncOpSym"""
    L = load_library()
    o = Options()
    L.amgb_default_options(C.byref(o))
    o.solver, o.smoother = H.IMPLICIT_EXTENDED_SYSTEM_BPX, smoother
    ops = (AsyncOpSym * 4096)()
    ob = np.zeros(max(num_levels, 0) + 1, dtype=np.int32)
    rc = L.amgb_ext_async_program(C.byref(o), num_levels, ops, 4096, _ip(ob))
    if rc != 0:
        raise AmgError("amgb_ext_async_program failed (%d): the asynchronous extended-system solver runs with weighted or L1 "
                       "Jacobi on at most 32 levels" % rc)
    return [[ops[i] for i in range(ob[q], ob[q + 1])] for q in range(num_levels)]


class DistAsyncOp(C.Structure):
    """csrc/launch.h DistAsyncOp: one operation of a level group's program on one rank of the row-partitioned asynchronous
    solve; operands are (slot, elem): slot >= 0 an arena slot, -1 none, -2 f (owned rows), -3 u (level-0 layout),
    -100 - l the smoother's scale vector of level l (level layout)"""
    ROLES = ("x", "y", "b", "c", "rs", "b2", "xs", "red", "red_copy", "acc")
    _fields_ = [(k, C.c_int) for k in ("type", "mat_kind", "mat_level", "sval", "barrier", "level", "count", "dst_rank")] + \
               [("slot", C.c_int * 10), ("elem", C.c_longlong * 10)] + \
               [(k, C.c_double) for k in ("alpha", "beta", "gamma", "beta2", "xself", "red_scale")]


def dist_async_plan(layouts, rank, solver, smoother=H.JACOBI, symmetric=True, factor_level0=False, fine_sweeps=1, coarse_sweeps=1,
                    coarse_solve=False):
    """planning of amgb_dist_solve_async for `rank` (host-only).  layouts[p][l]: partition.LevelLayout of rank p.
    -> (programs: list over the level groups of lists of DistAsyncOp, slot_off (doubles, len num_slots + 1), slot_group, slot_vec)"""
    L = load_library()
    o = Options()
    L.amgb_default_options(C.byref(o))
    o.solver, o.smoother = solver, smoother
    o.num_fine_smooth_sweeps, o.num_coarse_smooth_sweeps = fine_sweeps, coarse_sweeps
    o.coarse_solve = int(coarse_solve)
    nranks, nl = len(layouts), len(layouts[0])
    tab = np.zeros((nranks, nl, 8), dtype=np.int32)
    for p in range(nranks):
        for l, a in enumerate(layouts[p]):
            tab[p, l] = (a.n_global, a.row_start, a.n_owned, a.halo_lo, a.halo_hi, int(a.distributed), a.send_lo, a.send_hi)
    ops = (DistAsyncOp * 8192)()
    ob = np.zeros(nl + 1, dtype=np.int32)
    so = np.zeros(1025, dtype=np.int64)
    sg, sv = np.zeros(1024, dtype=np.int32), np.zeros(1024, dtype=np.int32)
    ns = C.c_int(0)
    rc = L.amgb_dist_async_plan(C.byref(o), nl, nranks, rank, _ip(tab), int(symmetric), int(factor_level0), ops, 8192, _ip(ob),
                                so.ctypes.data_as(C.POINTER(C.c_longlong)), _ip(sg), _ip(sv), 1024, C.byref(ns))
    if rc != 0:
        raise AmgError("amgb_dist_async_plan failed (%d): unsupported options or inconsistent layouts" % rc)
    n = ns.value
    return [[ops[i] for i in range(ob[q], ob[q + 1])] for q in range(nl)], so[:n + 1].copy(), sg[:n].copy(), sv[:n].copy()


def dist_unique_id():
    """128-byte NCCL unique id (rank 0 creates it, everybody receives it through the launcher's channel)"""
    L = load_library()
    buf = C.create_string_buffer(128)
    rc = L.amgb_dist_unique_id(buf)
    if rc != 0:
        raise AmgError("amgb_dist_unique_id failed (%d)" % rc)
    return buf.raw


class DistSolver:
    """One rank of the row-partitioned synchronous solve -- Multadd, AFACx or BPX with weighted / L1 Jacobi (DMEM_Add /
    DMEM_SyncAdd replacement).  `plan` is a
    partition.RankPlan; `uid` the 128-byte id from dist_unique_id() of rank 0."""

    def __init__(self, plan, uid, smooth_weight=1.0, num_pre=1, num_post=1, use_sell=True, use_stream=True,
                 coarse_solve=False, solver=H.MULTADD, factor_level0=False, device=0, smoother=H.JACOBI, sell_uniform=None,
                 lean_storage=False):
        self.L = load_library()
        self.plan = plan
        self.ctx = C.c_void_p()
        rc = self.L.amgb_create(C.byref(self.ctx), device)
        if rc != 0:
            raise AmgError("amgb_create failed (%d): no CUDA device / driver -- there is no CPU fallback" % rc)
        self._ck(self.L.amgb_dist_init(self.ctx, uid, plan.rank, plan.nranks))
        o = Options()
        self.L.amgb_default_options(C.byref(o))
        o.solver, o.smoother, o.smooth_weight = solver, smoother, smooth_weight
        o.num_pre_smooth_sweeps, o.num_post_smooth_sweeps = num_pre, num_post
        o.use_sell, o.use_stream = int(use_sell), int(use_stream)
        o.coarse_solve = int(coarse_solve)
        o.factor_level0 = int(factor_level0)
        o.lean_storage = int(lean_storage)
        if sell_uniform is not None:
            o.sell_uniform = int(sell_uniform)
        elif "AMGB_SELL_UNIFORM" in os.environ:
            o.sell_uniform = int(os.environ["AMGB_SELL_UNIFORM"])
        self._ck(self.L.amgb_set_options(self.ctx, C.byref(o)))
        nl = plan.num_levels
        self._ck(self.L.amgb_set_num_levels(self.ctx, nl))
        for l in range(nl):      # all layouts first: a matrix's interior / boundary split needs its input level's layout
            lay = plan.layouts[l]
            counts = np.ascontiguousarray(plan.all_counts[l], dtype=np.int32)
            self._ck(self.L.amgb_dist_set_level(self.ctx, l, lay.n_global, lay.row_start, lay.n_owned, lay.halo_lo,
                                                lay.halo_hi, int(lay.distributed), lay.send_lo, lay.send_hi, _ip(counts)))
        for l in range(nl):
            self._set(MAT_A, l, plan.A[l])
            if l < nl - 1:
                self._set(MAT_P, l, plan.P[l])
                self._set(MAT_R, l, plan.R[l])
        self._ck(self.L.amgb_setup(self.ctx))
        self._ck(self.L.amgb_dist_setup(self.ctx))
        self.n_owned = plan.layouts[0].n_owned

    _ck = Solver._ck
    _set = Solver._set
    close = Solver.close
    launch_count = Solver.launch_count

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_rhs(self, f_owned):
        f = np.ascontiguousarray(f_owned, dtype=np.float64)
        assert f.shape[0] == self.n_owned
        self._ck(self.L.amgb_dist_set_rhs(self.ctx, _dp(f)))

    def get_solution(self, out=None):
        u = np.empty(self.n_owned) if out is None else out
        self._ck(self.L.amgb_dist_get_solution(self.ctx, _dp(u)))
        return u

    def solve_sync(self, tol=1e-9, max_cycles=100, accel=0, mu=1.0, delta=1.0):
        """accel: 0 none, 1 Chebyshev, 2 second-order Richardson (DMEM_ChebyUpdate)"""
        hist = np.zeros(max_cycles + 1)
        n, secs = C.c_int(0), C.c_double(0)
        self._ck(self.L.amgb_dist_solve_sync_accel(self.ctx, tol, max_cycles, accel, mu, delta, _dp(hist), C.byref(n), C.byref(secs)))
        return hist[:n.value + 1], secs.value

    def stats(self):
        hb, ops = C.c_longlong(0), C.c_longlong(0)
        self._ck(self.L.amgb_dist_stats(self.ctx, C.byref(hb), C.byref(ops)))
        return hb.value, ops.value

    def DMEM_PowerMult(self, iters=20, u0_owned=None):
        """DMEM_PowerMult + DMEM's ChebySetup (src/DMEM_Eig.cpp:10-104, src/DMEM_Setup.cpp:1901-1914): (mu, delta, alpha, beta) with
        B = this context's partitioned additive cycle; collective"""
        a, b = C.c_double(0), C.c_double(0)
        u0 = None if u0_owned is None else np.ascontiguousarray(u0_owned, dtype=np.float64)
        self._ck(self.L.amgb_dist_eigs_power(self.ctx, int(iters), None if u0 is None else _dp(u0), C.byref(a), C.byref(b)))
        alpha, beta = a.value, b.value
        return (beta + alpha) / (beta - alpha), 2.0 / (beta + alpha), alpha, beta

    def DMEM_Add_async(self, num_cycles):
        """DMEM_Add's asynchronous loop on the row-partitioned hierarchy (amgb_dist_solve_async): every level group of every
        rank performs num_cycles corrections; collective.  -> (corrections per level on this rank, global relres, this rank's
        kernel seconds)"""
        cor = np.zeros(self.plan.num_levels, dtype=np.int32)
        rel, secs = C.c_double(0), C.c_double(0)
        self._ck(self.L.amgb_dist_solve_async(self.ctx, int(num_cycles), _ip(cor), C.byref(rel), C.byref(secs)))
        return cor, rel.value, secs.value

    def async_groups(self):
        cb = np.zeros(self.plan.num_levels + 1, dtype=np.int32)
        t = np.zeros(self.plan.num_levels)
        self._ck(self.L.amgb_dist_async_groups(self.ctx, _ip(cb), _dp(t)))
        return cb, t

    # ---- DMEM_AsyncSmooth: asynchronous (L1-)Jacobi on the fine grid across GPUs (src/DMEM_Smooth.cpp:16-313) ----
    def ipc_export_solution(self):
        buf = C.create_string_buffer(64)
        self._ck(self.L.amgb_dist_ipc_export_solution(self.ctx, buf))
        return buf.raw

    def ipc_open_neighbours(self, handle_lo, handle_hi):
        """handles exported by rank-1 / rank+1 (None where there is no such rank)"""
        off = 0
        if handle_lo is not None:
            lo, _ = self.plan.halos[0][self.plan.rank - 1]
            off = int(lo) + int(self.plan.all_counts[0][self.plan.rank - 1])
        self._ck(self.L.amgb_dist_ipc_open_neighbours(self.ctx, handle_lo, off, handle_hi))

    def DMEM_AsyncSmooth(self, sweeps):
        """enqueue `sweeps` own relaxations; returns without waiting for the GPU or for any peer"""
        self._ck(self.L.amgb_dist_async_smooth(self.ctx, int(sweeps)))

    def zero_solution(self):
        self._ck(self.L.amgb_dist_zero_solution(self.ctx))

    def synchronize(self):
        self._ck(self.L.amgb_stream_synchronize(self.ctx))

    def residual_norm(self):
        """global ||f - A_0 x||_2 (collective)"""
        v = C.c_double(0)
        self._ck(self.L.amgb_dist_residual_norm(self.ctx, C.byref(v)))
        return v.value


def smooth_transfer_device(A, P, smooth_interp_type=H.JACOBI, smooth_weight=1.0, want_P=True, want_R=True, device=0):
    """EXPERIMENTAL (not yet validated on hardware): SmoothTransfer (src/SMEM_Setup.cpp:1173-1254) on the device --
    (Pbar, Rbar) = (G P, P^T GT) as hierarchy.CSR in the reference's product layout; None for an output not asked for."""
    L = load_library()
    ctx = C.c_void_p()
    if L.amgb_create(C.byref(ctx), device) != 0:
        raise AmgError("amgb_create failed: no CUDA device / driver -- there is no CPU fallback")
    pb, rb = HostCSR(), HostCSR()
    try:
        rc = L.amgb_smooth_transfer(ctx, smooth_interp_type, smooth_weight, A.nrows, _ip(A.indptr), _ip(A.indices), _dp(A.data),
                                    P.ncols, _ip(P.indptr), _ip(P.indices), _dp(P.data),
                                    C.byref(pb) if want_P else None, C.byref(rb) if want_R else None)
        if rc != 0:
            raise AmgError("amg_b200 error %d: %s" % (rc, L.amgb_last_error(ctx).decode()))
        out = []
        for want, m in ((want_P, pb), (want_R, rb)):
            if not want:
                out.append(None)
                continue
            ip = np.ctypeslib.as_array(m.row_ptr, shape=(m.nrows + 1,)).copy()
            ix = np.ctypeslib.as_array(m.col_idx, shape=(max(m.nnz, 1),))[:m.nnz].copy()
            dv = np.ctypeslib.as_array(m.values, shape=(max(m.nnz, 1),))[:m.nnz].copy()
            out.append(H.CSR(m.nrows, m.ncols, ip, ix, dv))
        return tuple(out)
    finally:
        L.amgb_host_csr_free(C.byref(pb))
        L.amgb_host_csr_free(C.byref(rb))
        L.amgb_destroy(ctx)


class ExtendedExplicitSolver:
    """`-solver eebpx`: SMEM_ExtendedSystemSolve with EXPLICIT_EXTENDED_SYSTEM_BPX (src/SMEM_ExtendedSystem.cpp:84-110,295-365,
    finish :736-775).  `h`: hierarchy with the plain transfers of BPX.  The extended matrix AA is assembled on the host
    (hierarchy.extended_system = BuildExtendedMatrix, src/SMEM_Setup.cpp:1426-1521) and lives in a one-level context; the
    right-hand side bb = (f, R_0 f, ...) and the final x = sum_l P^{0<-l} x_l are computed on the device through the
    hierarchy's own context."""

    def __init__(self, h, device=0, **kw):
        self.h = h
        self.AA, self.disp = H.extended_system(h)
        h1 = H.Hierarchy([self.AA], [])
        h1.P, h1.R = [], []
        self.ext = Solver(h1, H.IMPLICIT_EXTENDED_SYSTEM_BPX, H.JACOBI, 1.0, device=device, **kw)
        self.hs = Solver(h, H.BPX, H.JACOBI, 1.0, device=device, **kw)

    def extended_rhs(self, f):
        parts = [np.ascontiguousarray(f, dtype=np.float64)]
        for l in range(self.h.num_levels - 1):
            parts.append(self.hs.spgemv(MAT_R, l, 1.0, parts[-1], 0.0, None))
        return np.concatenate(parts)

    def SMEM_ExtendedSystemSolve(self, f, tol=1e-9, num_cycles=100, mu=1.0, delta=1.0):
        """-> dict(x, xx, iters, ext_hist, ext_relres, relres, seconds)"""
        bb = self.extended_rhs(f)
        out = self.ext.SMEM_ExtendedSystemSolve(bb, tol, num_cycles, mu, delta)
        xx, d, L = out["x"], self.disp, self.h.num_levels
        v = np.ascontiguousarray(xx[d[L - 1]:d[L]])
        for l in range(L - 2, -1, -1):
            v = self.hs.spgemv(MAT_P, l, 1.0, v, 1.0, np.ascontiguousarray(xx[d[l]:d[l + 1]]))
        r = self.hs.spgemv(MAT_A, 0, -1.0, v, 1.0, np.ascontiguousarray(f, dtype=np.float64))
        rel = self.hs.norm2(r) / self.hs.norm2(np.ascontiguousarray(f, dtype=np.float64))
        return dict(x=v, xx=xx, iters=out["iters"], ext_hist=out["ext_hist"], ext_relres=out["relres"], relres=rel,
                    seconds=out["seconds"])

    def SMEM_ExtendedSystemSolve_async(self, f, tol=1e-9, num_cycles=100, mu=1.0, delta=1.0):
        """`-solver async_eebpx`: the same system relaxed asynchronously (amgb_solve_extended_async) -> dict(x, xx, iters_min,
        iters_max, ext_relres, relres, seconds)"""
        bb = self.extended_rhs(f)
        self.ext.set_rhs(bb)
        lo, hi = C.c_int(0), C.c_int(0)
        er, secs = C.c_double(0), C.c_double(0)
        self.ext._ck(self.ext.L.amgb_solve_extended_async(self.ext.ctx, tol, int(num_cycles), mu, delta, C.byref(lo), C.byref(hi),
                                                          C.byref(er), C.byref(secs)))
        xx, d, L = self.ext.get_solution(), self.disp, self.h.num_levels
        v = np.ascontiguousarray(xx[d[L - 1]:d[L]])
        for l in range(L - 2, -1, -1):
            v = self.hs.spgemv(MAT_P, l, 1.0, v, 1.0, np.ascontiguousarray(xx[d[l]:d[l + 1]]))
        r = self.hs.spgemv(MAT_A, 0, -1.0, v, 1.0, np.ascontiguousarray(f, dtype=np.float64))
        rel = self.hs.norm2(r) / self.hs.norm2(np.ascontiguousarray(f, dtype=np.float64))
        return dict(x=v, xx=xx, iters_min=lo.value, iters_max=hi.value, ext_relres=er.value, relres=rel, seconds=secs.value)

    def close(self):
        self.ext.close()
        self.hs.close()
