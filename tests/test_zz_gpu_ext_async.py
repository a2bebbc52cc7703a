"""GPU tests of the asynchronous implicit extended-system BPX solver (`-solver async_iebpx`;
amgb_solve_extended_implicit_async, csrc/extended.cu, k_async_amg<false, true> in csrc/async.cu).  Its programs are checked
against the oracle on the CPU (tests/test_ext_async_program.py); here the device kernel runs them.

With one level there is one group, the iteration is deterministic and must be the oracle's synchronous one.  With several
levels the groups run chaotically: the solver must reach the tolerance on the solution the synchronous form finds."""
import ctypes as C
import os

import numpy as np
import pytest

import async_multigrid_b200 as amg
from async_multigrid_b200 import hierarchy as H
from conftest import GOLDEN, HIST_TOL, hierarchy_from_golden
from oracle import oracle as O

pytestmark = pytest.mark.gpu


def _check_one_group(out, want):
    assert list(out["iters"]) == [want["iters"]], (out["iters"], want["iters"])
    assert abs(out["ext_relres"] - want["ext_relres"]) <= HIST_TOL
    assert abs(out["relres"] - want["relres"]) <= HIST_TOL
    assert np.max(np.abs(out["x"] - want["x"])) <= 1e-11 * np.max(np.abs(want["x"]))


def test_one_group_is_the_explicit_reference():
    """one-level context holding the assembled extended matrix AA (weight 1, as ExtendedExplicitSolver builds it): the one
    group's iteration is the synchronous one on AA -- the oracle and the reference fixture's explicit entries"""
    g = dict(np.load(os.path.join(GOLDEN, "iebpx.npz")))
    name = "lap7pt_n12"
    h, d = hierarchy_from_golden(name)
    h.build_transfers(H.BPX, 1.0)
    AA, disp, bb = H.extended_system(h, d["b"])
    h1 = H.Hierarchy([AA], [])
    h1.P, h1.R = [], []
    pb = O.Problem(h1, H.BPX, H.JACOBI, 1.0)
    s = amg.Solver(h1, H.IMPLICIT_EXTENDED_SYSTEM_BPX, H.JACOBI, 1.0)
    for nc in (2, 7, 300):
        k = "%s_explicit_nc%d_" % (name, nc)
        mu, delta = g[k + "mu_delta"]
        out = s.SMEM_ExtendedSystemSolve_async(bb, 1e-9, nc, mu, delta)
        want = pb.solve_iebpx(bb, 1e-9, nc, mu, delta)
        _check_one_group(out, want)
        assert want["iters"] == int(g[k + "iters"])
        assert abs(out["ext_relres"] - g[k + "norms"][0]) <= HIST_TOL
    s.close()


def test_one_group_l1_jacobi_equals_the_oracle():
    A = H.laplacian("5pt", 32)
    h = H.amg_setup(A, max_levels=1)
    h.build_transfers(H.BPX, 0.8)
    b = H.rand_rhs(A.nrows)
    pb = O.Problem(h, H.BPX, H.L1_JACOBI, 0.8)
    lo, hi = pb.eigs_power(20)
    hi *= 1.1                          # (the 20-step estimate is below the largest eigenvalue here: the iteration would diverge)
    mu, delta = (hi + lo) / (hi - lo), 2.0 / (hi + lo)
    s = amg.Solver(h, H.BPX, H.L1_JACOBI, 0.8)
    for nc in (2, 7, 300, 3000):
        _check_one_group(s.SMEM_ExtendedSystemSolve_async(b, 1e-9, nc, mu, delta), pb.solve_iebpx(b, 1e-9, nc, mu, delta))
    s.close()


def _setup(prob, n, sm, w=0.8):
    A = H.laplacian(prob, n)
    h = H.amg_setup(A)
    h.build_transfers(H.BPX, w)
    b = H.rand_rhs(A.nrows)
    s = amg.Solver(h, H.BPX, sm, w)
    if A.nrows <= 5000:
        lo, hi = O.Problem(h, H.BPX, sm, w).eigs_power(20)
    else:
        s.set_rhs(b)
        _, _, lo, hi = s.ChebySetup(60)
        hi *= 1.1
    return h, b, s, (hi + lo) / (hi - lo), 2.0 / (hi + lo)


@pytest.mark.parametrize("prob,n,sm", [("7pt", 16, H.JACOBI), ("5pt", 48, H.L1_JACOBI), ("27pt", 10, H.JACOBI), ("7pt", 64, H.JACOBI)])
def test_converges_to_the_synchronous_solution(prob, n, sm):
    h, b, s, mu, delta = _setup(prob, n, sm)
    L = h.num_levels
    sync = s.SMEM_ExtendedSystemSolve(b, 1e-9, 1000, mu, delta)
    cap = 5000
    out = s.SMEM_ExtendedSystemSolve_async(b, 1e-9, cap, mu, delta)
    true = O.norm2(O.spgemv(h.A[0], out["x"], b, -1.0, 1.0)) / O.norm2(b)
    assert abs(true - out["relres"]) <= 1e-12
    assert out["relres"] < 1e-8 and out["ext_relres"] < 1e-8, out
    assert np.max(np.abs(out["x"] - sync["x"])) <= 1e-6 * np.max(np.abs(sync["x"]))
    assert len(out["iters"]) == L and np.all(out["iters"] >= 2) and np.all(out["iters"] < cap), out["iters"]
    assert np.all(out["group_seconds"] > 0.0), out["group_seconds"]
    print("async iebpx %s n=%d L=%d: iters per group %s, ext relres %.2e, relres %.2e, %.4f s, group seconds %s "
          "(sync: %d iterations, %.4f s)" % (prob, n, L, list(out["iters"]), out["ext_relres"], out["relres"], out["seconds"],
                                             np.round(out["group_seconds"], 5).tolist(), sync["iters"], sync["seconds"]))
    s.close()


def test_count_rule():
    """tol = 0: no group ever converges, each is done at num_cycles, the last to get there stops exactly there"""
    h, b, s, mu, delta = _setup("7pt", 16, H.JACOBI)
    out = s.SMEM_ExtendedSystemSolve_async(b, 0.0, 12, mu, delta)
    assert min(out["iters"]) == 12, out["iters"]
    s.close()


def test_no_iteration():
    h, b, s, mu, delta = _setup("7pt", 16, H.JACOBI)
    for nc in (0, 1):
        out = s.SMEM_ExtendedSystemSolve_async(b, 1e-9, nc, mu, delta)
        want = s.SMEM_ExtendedSystemSolve(b, 1e-9, nc, mu, delta)
        assert list(out["iters"]) == [1] * h.num_levels and want["iters"] == 1
        assert np.max(np.abs(out["x"] - want["x"])) <= 1e-13 * np.max(np.abs(want["x"]))
        assert abs(out["relres"] - want["relres"]) <= 1e-13
    s.close()


def test_coexists_with_the_synchronous_solver():
    h, b, s, mu, delta = _setup("27pt", 10, H.JACOBI)
    first = s.SMEM_ExtendedSystemSolve(b, 1e-9, 400, mu, delta)
    out = s.SMEM_ExtendedSystemSolve_async(b, 1e-9, 3000, mu, delta)
    again = s.SMEM_ExtendedSystemSolve(b, 1e-9, 400, mu, delta)
    assert out["relres"] < 1e-8
    assert first["iters"] == again["iters"] and np.array_equal(first["x"], again["x"])
    assert np.array_equal(first["ext_hist"], again["ext_hist"]) and first["relres"] == again["relres"]
    s.close()


def _refused(obj, n_levels):
    it = np.zeros(n_levels, dtype=np.int32)
    gs = np.zeros(n_levels)
    d = C.c_double(0)
    before = obj.launch_count()
    with pytest.raises(amg.solver.AmgError):
        obj._ck(obj.L.amgb_solve_extended_implicit_async(obj.ctx, 1e-9, 50, 2.0, 1.0, it.ctypes.data_as(C.POINTER(C.c_int)),
                                                         C.byref(d), C.byref(d), gs.ctypes.data_as(C.POINTER(C.c_double)),
                                                         C.byref(d)))
    assert obj.launch_count() == before


def test_refusals():
    from async_multigrid_b200 import partition as PT
    A = H.laplacian("7pt", 12)
    b = H.rand_rhs(A.nrows)
    h = H.amg_setup(A)
    h.build_transfers(H.BPX, 0.8)
    s = amg.Solver(h, H.BPX, H.HYBRID_JACOBI_GAUSS_SEIDEL, 0.8)
    s.set_rhs(b)
    _refused(s, h.num_levels)
    s.close()
    hm = H.amg_setup(A)
    hm.build_transfers(H.MULTADD, 0.9)
    s = amg.Solver(hm, H.MULTADD, H.JACOBI, 0.9)
    s.set_rhs(b)
    _refused(s, hm.num_levels)
    s.close()
    d = amg.DistSolver(PT.RankPlan(h, 1, 0), amg.solver.dist_unique_id(), 0.8, solver=H.BPX)
    d.set_rhs(b)
    _refused(d, h.num_levels)
    d.close()
