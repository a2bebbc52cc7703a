"""CPU statement of amgb_solve_pcg -- test infrastructure: conjugate gradients preconditioned by the oracle's additive cycle
(oracle.Problem.cycle = orc_cycle, the cycle from a zero guess).  The device solver (csrc/pcg.cu) follows this order of
operations exactly:

    r = f - A u                      (u = the start vector; zero unless one is given)
    r0 = ||r||_2; hist[0] = 1;  r0 == 0 -> 0 iterations
    for k = 1 .. max_iters:
        z = B r                      (B = the cycle from a zero guess)
        rho = (r, z)                 rho <= 0 or not finite -> breakdown
        beta = 0 if k == 1 else rho / rho_old;  p = z + beta p;  rho_old = rho
        q = A p;  sigma = (p, q)     sigma <= 0 or not finite -> breakdown
        alpha = rho / sigma;  u += alpha p;  r -= alpha q
        hist[k] = ||r||_2 / r0       (recurrence residual); stop when hist[k] < tol
    final_relres = ||f - A u||_2 / r0 (true residual, recomputed once)

On the first iteration beta is 0 and p is set to z outright (0 * p would carry a NaN left from an earlier solve).  On a
breakdown nothing of that iteration reaches u: the history and u hold the iterations completed before it.

The reference reaches this through hypre's PCG with its additive cycles as the preconditioner (-hypre_pcg,
src/DMEM_Setup.cpp:129-167).  hypre is not vendored, so parity with hypre_PCGSolve (its stop test, its two-norm
options, its restarts) is not pinned by any reference object code: the meaning above is the one this project defines."""
import numpy as np

from async_multigrid_b200 import hierarchy as H

OK, BREAKDOWN = "ok", "breakdown"


def solve_pcg(pb, f, tol=1e-9, max_iters=200, u0=None):
    """pb: oracle.Problem.  -> (u, hist[0..iters], final_relres, status); status is "ok" or "breakdown: <what> at
    iteration k" (hist then ends at iteration k - 1)"""
    A = pb.h.A[0].to_scipy()
    f = np.asarray(f, dtype=np.float64)
    u = np.zeros(A.shape[0]) if u0 is None else np.array(u0, dtype=np.float64)
    r = f - A @ u
    r0 = float(np.sqrt(r @ r))
    hist = [1.0]
    status = OK
    if r0 == 0.0:
        return u, np.asarray(hist), 0.0, status
    p = None
    rho_old = None
    for k in range(1, max_iters + 1):
        z = pb.cycle(r)
        rho = float(r @ z)
        if not (np.isfinite(rho) and rho > 0.0):
            status = "%s: rho = %r at iteration %d" % (BREAKDOWN, rho, k)
            break
        p = z.copy() if k == 1 else z + (rho / rho_old) * p
        rho_old = rho
        q = A @ p
        sigma = float(p @ q)
        if not (np.isfinite(sigma) and sigma > 0.0):
            status = "%s: sigma = %r at iteration %d" % (BREAKDOWN, sigma, k)
            break
        alpha = rho / sigma
        u += alpha * p
        r -= alpha * q
        hist.append(float(np.sqrt(r @ r)) / r0)
        if hist[-1] < tol:
            break
    final = float(np.linalg.norm(f - A @ u)) / r0
    return u, np.asarray(hist), final, status


def negated(h):
    """the hierarchy of -A (same plain interpolation): a negative definite operator, for the breakdown tests"""
    return H.Hierarchy([H.CSR(a.nrows, a.ncols, a.indptr, a.indices, -a.data) for a in h.A], h.P_plain)
