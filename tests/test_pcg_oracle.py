"""CPU: the statement of the cycle-preconditioned conjugate-gradient solve (tests/pcg_reference.py, the meaning
amgb_solve_pcg follows) against scipy's CG with the oracle's cycle as the preconditioner.  From a zero start vector the
two stop on the same test (||r_k|| < tol ||f||), so they must take the same number of iterations to the same iterate."""
import numpy as np
import pytest
import scipy.sparse.linalg as sla

from async_multigrid_b200 import hierarchy as H
from conftest import hierarchy_from_golden
from oracle import oracle as O
from pcg_reference import OK, negated, solve_pcg

# (name, solver, smoother, weight, problem keywords, build_transfers keywords)
CASES = [
    ("multadd_symmetrised", H.MULTADD, H.JACOBI, 0.9, {}, {}),
    ("multadd_plain_jacobi", H.MULTADD, H.JACOBI, 0.9, dict(num_pre=0, num_post=0), dict(num_pre=0, num_post=0)),
    ("bpx_jacobi", H.BPX, H.JACOBI, 0.8, {}, {}),
    ("bpx_l1", H.BPX, H.L1_JACOBI, 1.0, {}, {}),
    ("multadd_coarse_solve", H.MULTADD, H.JACOBI, 0.9, dict(coarse_solve=1), {}),
]


def _scipy_cg(pb, A, f, tol, maxiter):
    n = A.shape[0]
    M = sla.LinearOperator((n, n), matvec=lambda r: pb.cycle(np.asarray(r).ravel()), dtype=np.float64)
    count = [0]

    def cb(_):
        count[0] += 1

    x, info = sla.cg(A, f, rtol=tol, atol=0.0, maxiter=maxiter, M=M, callback=cb)
    return x, info, count[0]


@pytest.mark.parametrize("golden_name", ["lap5pt_n32", "lap7pt_n12"])
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_pcg_equals_scipy_cg(golden_name, case):
    _, solver, smoother, w, pkw, tkw = case
    h, _ = hierarchy_from_golden(golden_name)
    h.build_transfers(solver, w, **tkw)
    pb = O.Problem(h, solver, smoother, w, **pkw)
    A = h.A[0].to_scipy()
    f = H.rand_rhs(A.shape[0])
    tol = 1e-9
    u, hist, final, status = solve_pcg(pb, f, tol, 200)
    assert status == OK, status
    x, info, its = _scipy_cg(pb, A, f, tol, 200)
    assert info == 0
    assert len(hist) - 1 == its, (len(hist) - 1, its)
    assert np.linalg.norm(u - x) <= 1e-10 * np.linalg.norm(x)
    assert hist[-1] < tol and final < 10 * tol
    assert np.all(np.diff(np.log(hist[1:])) < 2.0)      # no wild excursions of the recurrence residual


def test_beam_bpx_reaches_tolerance():
    """the 24x3x3 elasticity beam with the BPX cycle (omega 0.6): the stationary and Chebyshev iterations diverge here;
    PCG reaches 1e-9 (130 iterations when this was written)"""
    A, b = H.elasticity_beam(24, 3, 3)
    h = H.amg_setup(A, num_functions=3, theta=0.5)
    h.build_transfers(H.BPX, 0.6)
    pb = O.Problem(h, H.BPX, H.JACOBI, 0.6)
    u, hist, final, status = solve_pcg(pb, b, 1e-9, 200)
    assert status == OK, status
    assert len(hist) - 1 <= 200 and hist[-1] < 1e-9
    assert final < 1e-9, final


def test_start_vector_and_trivial_cases():
    h, _ = hierarchy_from_golden("lap7pt_n12")
    h.build_transfers(H.MULTADD, 0.9)
    pb = O.Problem(h, H.MULTADD, H.JACOBI, 0.9)
    A = h.A[0].to_scipy()
    f = H.rand_rhs(A.shape[0])
    u_ref, _, _, _ = solve_pcg(pb, f, 1e-12, 200)
    # a start vector: the solve continues from it to the same solution
    u0 = H.rand_rhs(A.shape[0], seed=3)
    u, hist, final, status = solve_pcg(pb, f, 1e-9, 200, u0=u0)
    assert status == OK and hist[-1] < 1e-9
    assert np.linalg.norm(u - u_ref) <= 1e-7 * np.linalg.norm(u_ref)
    # f = 0 from zero: no iteration, no NaN
    u, hist, final, status = solve_pcg(pb, np.zeros_like(f), 1e-9, 200)
    assert list(hist) == [1.0] and final == 0.0 and not np.any(u)
    # max_iters = 0: the start vector is left alone
    u, hist, final, status = solve_pcg(pb, f, 1e-9, 0, u0=u0)
    assert list(hist) == [1.0] and np.array_equal(u, u0) and final == 1.0


def test_breakdown_on_negative_definite():
    """-A with the BPX / L1-Jacobi cycle: the l1 norms are those of A, so B stays positive definite, rho > 0 and the first
    sigma = (p, -A p) < 0"""
    h, _ = hierarchy_from_golden("lap5pt_n32")
    neg = negated(h)
    neg.build_transfers(H.BPX, 1.0)
    f = H.rand_rhs(h.n[0])
    pb = O.Problem(neg, H.BPX, H.L1_JACOBI, 1.0)
    u, hist, final, status = solve_pcg(pb, f, 1e-9, 50)
    assert status.startswith("breakdown: sigma") and status.endswith("iteration 1"), status
    assert list(hist) == [1.0] and not np.any(u) and final == 1.0
