"""GPU tests of the factorised restriction (amgb_options.factor_restriction): the synchronous Multadd cycle whose levels
l >= 1 restrict through the plain P_l^T after the smoother's pass over A_l wrote t_l beside e_l, against the oracle's cycle
with the explicit products Rbar_l, in every storage layout an A_l can take; coexistence with the explicit form, the launch
count, the refusals, and the solvers built on the same cycle (PCG, ChebySetup)."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

import async_multigrid_b200 as amg
from async_multigrid_b200 import hierarchy as H
from async_multigrid_b200 import partition as PT
from conftest import assert_hist_close
from oracle import oracle as O
from pcg_reference import OK, solve_pcg
from test_gpu_parity import _check_hist, _rel

pytestmark = pytest.mark.gpu

EINVAL = -1
MAT_A = 0


def _pair(h, smoother, w, **dkw):
    """(oracle problem with the explicit products, device solver with the factorised transfers) on one hierarchy"""
    sit = H.L1_JACOBI if smoother == H.L1_JACOBI else H.JACOBI
    h.build_transfers(H.MULTADD, w, smooth_interp_type=sit)
    pb = O.Problem(h, H.MULTADD, smoother, w)
    hf = H.Hierarchy(h.A, h.P_plain)
    hf.cpts = h.cpts
    hf.build_transfers(H.MULTADD, w, smooth_interp_type=sit, factor_level0=True)
    s = amg.Solver(hf, H.MULTADD, smoother, w, factor_level0=True, **dkw)
    return pb, hf, s


@pytest.mark.parametrize("prob,n", [("7pt", 16), ("5pt", 48), ("27pt", 10)])
@pytest.mark.parametrize("smoother", [H.JACOBI, H.L1_JACOBI], ids=["j", "L1j"])
def test_cycle_and_history_match_explicit_products(prob, n, smoother):
    h = H.amg_setup(H.laplacian(prob, n))
    assert h.num_levels >= 4                      # at least one level l >= 1 below last_r = L - 2
    pb, _, s = _pair(h, smoother, 0.9)
    assert s.options.factor_restriction == 1      # on by default with factor_level0
    b = H.rand_rhs(h.n[0])
    assert _rel(s.cycle(b), pb.cycle(b)) <= 1e-12
    _, want, _ = pb.solve_sync(b, 1e-9, 100)
    _check_hist(s.SMEM_Solve(b, 1e-9, 100)["hist"], want)
    s.close()


def _geometric_hierarchy(n, levels):
    """7-point Laplacians on nested grids with piecewise-constant interpolation: constant-coefficient stencils on the coarse
    levels too, so A_1 takes the SELL-U encoding"""
    As, Ps = [], []
    for l in range(levels):
        m = n >> l
        As.append(H.laplacian("7pt", m))
        if l < levels - 1:
            p1 = sp.csr_matrix((np.ones(m), (np.arange(m), np.arange(m) // 2)), shape=(m, m // 2))
            Ps.append(H.CSR.from_scipy(sp.kron(sp.kron(p1, p1), p1).tocsr()))
    return H.Hierarchy(As, Ps)


LAYOUTS = [
    ("default", {}),
    ("no_sellu", dict(sell_uniform=0)),
    ("sell_sigma_off", dict(sell_sigma=0)),
    ("warp_stream", dict(use_sell=False)),
    ("csr_per_row", dict(use_sell=False, use_stream=False)),
]


@pytest.mark.parametrize("layout", LAYOUTS, ids=[c[0] for c in LAYOUTS])
def test_every_storage_layout(layout):
    h = H.amg_setup(H.laplacian("7pt", 24))
    pb, _, s = _pair(h, H.JACOBI, 0.9, **layout[1])
    b = H.rand_rhs(h.n[0])
    assert _rel(s.cycle(b), pb.cycle(b)) <= 1e-12
    s.close()


def test_retired_stream_variant_is_refused():
    """amgb_options.stream_variant only keeps its place in the struct: 8 (the default, the warp-stream kernel) is accepted,
    any other value is an error rather than a silent fall-back to another kernel"""
    L = amg.solver.load_library()
    ctx = C.c_void_p()
    assert L.amgb_create(C.byref(ctx), 0) == 0
    try:
        o = amg.solver.Options()
        L.amgb_default_options(C.byref(o))
        assert o.stream_variant == 8
        for v in (0, 3, 11, 13, -1):
            o.stream_variant = v
            assert L.amgb_set_options(ctx, C.byref(o)) == EINVAL, v
            assert b"stream_variant" in L.amgb_last_error(ctx)
        o.stream_variant = 8
        assert L.amgb_set_options(ctx, C.byref(o)) == 0
    finally:
        L.amgb_destroy(ctx)


def test_sell_sigma_level():
    """a level-1 operator with >= 262144 rows, where the upload may sort rows by length (SELL-C-sigma)"""
    h = H.amg_setup(H.laplacian("7pt", 100))
    assert h.n[1] >= 262144
    pb, _, s = _pair(h, H.JACOBI, 0.9)
    b = H.rand_rhs(h.n[0])
    assert _rel(s.cycle(b), pb.cycle(b)) <= 1e-12
    s.close()


def test_sellu_coarse_level():
    h = _geometric_hierarchy(32, 4)
    pb, _, s = _pair(h, H.JACOBI, 0.9)
    assert s.is_sell(MAT_A, 1)
    slices, _ = s.sellu_stats()
    assert slices > h.n[0] // 32                  # level 1 is encoded too, not only level 0
    b = H.rand_rhs(h.n[0])
    assert _rel(s.cycle(b), pb.cycle(b)) <= 1e-12
    s.close()


def test_on_and_off_in_one_process_with_graph_replay():
    w = 0.9
    h = H.amg_setup(H.laplacian("7pt", 20))
    pb, hf, on = _pair(h, H.JACOBI, w)
    off = amg.Solver(hf, H.MULTADD, H.JACOBI, w, factor_level0=True, factor_restriction=False)
    assert hf.R[1].nnz > hf.plain_restriction(1).nnz          # the hierarchy keeps the explicit products for other solvers
    b = H.rand_rhs(h.n[0])
    _, want, _ = pb.solve_sync(b, 1e-9, 100)
    hists = {}
    for name, s in (("on", on), ("off", off), ("on2", on), ("off2", off)):
        s.set_rhs(b)
        s.set_solution(None)
        hists[name], _ = s.solve_sync(1e-9, 100)            # the second solve of each replays the captured graph
        _check_hist(hists[name], want)
    assert np.array_equal(hists["on"], hists["on2"]) and np.array_equal(hists["off"], hists["off2"])
    on.close()
    off.close()


def test_launches_per_cycle_unchanged():
    w = 0.9
    h = H.amg_setup(H.laplacian("7pt", 20))
    _, hf, on = _pair(h, H.JACOBI, w)
    off = amg.Solver(hf, H.MULTADD, H.JACOBI, w, factor_level0=True, factor_restriction=False)
    b = H.rand_rhs(h.n[0])
    counts = []
    for s in (on, off):
        k0 = s.launch_count()
        s.cycle(b)
        k1 = s.launch_count()
        s.set_rhs(b)
        s.set_solution(None)
        hist, _ = s.solve_sync(1e-9, 100)
        counts.append((k1 - k0, len(hist), s.launch_count() - k1))
    assert counts[0] == counts[1], counts
    on.close()
    off.close()


REFUSED = [
    ("no_factor_level0", H.MULTADD, H.JACOBI, dict(factor_level0=False)),
    ("afacx", H.AFACX, H.JACOBI, {}),
    ("bpx", H.BPX, H.JACOBI, {}),
    ("hybrid_jgs", H.MULTADD, H.HYBRID_JACOBI_GAUSS_SEIDEL, {}),
    ("no_post_smoothing", H.MULTADD, H.JACOBI, dict(num_post=0)),
    ("two_fine_sweeps", H.MULTADD, H.JACOBI, dict(fine_sweeps=2)),
    ("async_multadd", H.ASYNC_MULTADD, H.JACOBI, {}),
]


@pytest.mark.parametrize("case", REFUSED, ids=[c[0] for c in REFUSED])
def test_refusals(case):
    _, solver, smoother, kw = case
    h = H.amg_setup(H.laplacian("7pt", 12))
    h.build_transfers(H.MULTADD, 0.9, factor_level0=True)
    kw = dict(dict(factor_level0=True), **kw)
    with pytest.raises(amg.solver.AmgError, match="factor_restriction"):
        amg.Solver(h, solver, smoother, 0.9, factor_restriction=True, **kw)
    if case[0] in ("no_factor_level0", "two_fine_sweeps", "async_multadd"):
        s = amg.Solver(h, solver, smoother, 0.9, **kw)          # left to the default, the option stays off here
        assert s.options.factor_restriction == 0
        s.close()


def test_refused_on_a_distributed_context():
    w = 0.9
    h = H.amg_setup(H.laplacian("7pt", 12))
    h.build_transfers(H.MULTADD, w, factor_level0=True)
    plan = PT.RankPlan(h, 1, 0)
    L = amg.solver.load_library()
    ctx = C.c_void_p()
    assert L.amgb_create(C.byref(ctx), 0) == 0
    try:
        assert L.amgb_dist_init(ctx, amg.solver.dist_unique_id(), 0, 1) == 0
        o = amg.solver.Options()
        L.amgb_default_options(C.byref(o))
        o.smooth_weight, o.factor_level0, o.factor_restriction = w, 1, 1
        assert L.amgb_set_options(ctx, C.byref(o)) == 0
        assert L.amgb_set_num_levels(ctx, plan.num_levels) == 0
        for l in range(plan.num_levels):
            lay = plan.layouts[l]
            counts = np.ascontiguousarray(plan.all_counts[l], dtype=np.int32)
            assert L.amgb_dist_set_level(ctx, l, lay.n_global, lay.row_start, lay.n_owned, lay.halo_lo, lay.halo_hi,
                                         int(lay.distributed), lay.send_lo, lay.send_hi, counts.ctypes.data_as(amg.solver.IP)) == 0
        for l in range(plan.num_levels):
            mats = [(0, plan.A[l])] + ([(1, plan.P[l]), (2, plan.R[l])] if l < plan.num_levels - 1 else [])
            for kind, m in mats:
                assert L.amgb_set_matrix(ctx, kind, l, m.nrows, m.ncols, m.nnz, m.indptr.ctypes.data_as(amg.solver.IP),
                                         m.indices.ctypes.data_as(amg.solver.IP), m.data.ctypes.data_as(amg.solver.DP)) == 0
        assert L.amgb_setup(ctx) == EINVAL
        assert b"factor_restriction" in L.amgb_last_error(ctx)
    finally:
        L.amgb_destroy(ctx)


def test_cross_gpu_correction_refused():
    h = H.amg_setup(H.laplacian("7pt", 12))
    _, _, s = _pair(h, H.JACOBI, 0.9)
    with pytest.raises(amg.solver.AmgError, match="factor_restriction"):
        s.async_dist_correct(1)
    s.close()


def test_pcg_and_cheby_setup_follow_the_cycle():
    w = 0.9
    h = H.amg_setup(H.laplacian("7pt", 20))
    pb, hf, on = _pair(h, H.JACOBI, w)
    off = amg.Solver(hf, H.MULTADD, H.JACOBI, w, factor_level0=True, factor_restriction=False)
    f = H.rand_rhs(h.n[0])
    _, want, final_ref, status = solve_pcg(pb, f, 1e-9, 200)
    assert status == OK
    on.set_rhs(f)
    on.set_solution(None)
    out = on.solve_pcg(1e-9, 200)
    assert out["iters"] == len(want) - 1
    assert_hist_close(out["hist"], want)
    assert abs(out["relres"] - final_ref) <= 1e-13
    for s in (on, off):
        s.set_rhs(f)
    e_on, e_off = on.ChebySetup(20), off.ChebySetup(20)
    assert np.allclose(e_on, e_off, rtol=1e-10, atol=0.0), (e_on, e_off)
    on.close()
    off.close()
