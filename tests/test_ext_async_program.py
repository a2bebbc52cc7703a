"""The per-group programs of the asynchronous implicit extended-system solver (`-solver async_iebpx`; csrc/async.cu
async_build_ext_program, run by k_async_amg<false, true> from amgb_solve_extended_implicit_async), interpreted on the CPU.

The interpreter below executes the operation lists the host hands the device kernel, one list per level group, and lets the
groups interleave in several legal orders.  With every group reading the others' vectors as they were at the start of a round
(lock step) the asynchronous method IS the synchronous one, so the programs must reproduce the oracle's `solve_iebpx`
(pinned by the reference's object code, tests/test_oracle_golden.py): iteration counts, residual history, final norms and
iterate.  With the groups taking turns in other orders or at unequal rates the method must still converge to the same
solution."""
import numpy as np
import pytest
import scipy.sparse as sp

import async_multigrid_b200 as amg  # noqa: F401
from async_multigrid_b200 import hierarchy as H
from async_multigrid_b200 import solver as S
from conftest import HIST_TOL
from oracle import oracle as O

SPMV, EXT_RESID, EXT_CHEBY, EXT_STOP = 0, 13, 14, 15
MAT_A, MAT_P, MAT_R = 0, 1, 2
V_WS, V_INVL1, V_XF, V_XU, V_XY, V_XE, V_XZ1, V_XZ2, V_XR = 10, 11, 12, 13, 14, 15, 16, 17, 18
SHARED = (V_XF, V_XU, V_XY, V_XE)
PRIVATE = (V_XZ1, V_XZ2, V_XR)
READ_ONLY = (V_WS, V_INVL1)


class ExtInterp:
    """CPU model of one launch: the shared per-level vectors f, u, y, e, every group's private chain vectors, its omega and
    loc_iters, the published contributions, the converge flag and the count of groups that are done.  The stop operation is
    split into the memory steps its group root performs (publish and count, the flag test of group 0, the decision), so that
    a schedule can interleave other groups between them as the device may."""

    def __init__(self, h, progs, b, smoother, w, mu, delta, tol, num_cycles):
        self.h, self.progs, self.L = h, progs, h.num_levels
        L = self.L
        self.A = [m.to_scipy() for m in h.A]
        self.P = [m.to_scipy() for m in h.P]
        self.R = [m.to_scipy() for m in h.R]
        self.rs = {V_WS: [w / a.diagonal() for a in self.A], V_INVL1: [1.0 / x for x in h.l1_norms()]}
        self.b = np.asarray(b, dtype=np.float64)
        self.mu22, self.delta, self.tol, self.num_cycles = (2.0 * mu) ** 2, delta, tol, num_cycles
        f = [self.b.copy()]
        for l in range(L - 1):
            f.append(self.R[l] @ f[l])
        self.r0, self.r0_ext = np.linalg.norm(self.b), np.sqrt(sum(np.dot(x, x) for x in f))
        u = [delta * f[l] / self.A[l].diagonal() for l in range(L)]
        self.shared = {V_XF: f, V_XU: u, V_XY: [np.zeros_like(x) for x in u], V_XE: [self.A[l] @ u[l] for l in range(L)]}
        self.priv = [{} for _ in range(L)]
        self.omega, self.it = [2.0] * L, [1] * L
        self.contrib, self.flag, self.done = [1e300] * L, False, 0
        self.stopped = [num_cycles <= 1] * L          # (no launch at all for num_cycles <= 1)
        self.last_ss = [0.0] * L

    def vec(self, q, vid):
        if vid < 0:
            return None
        kind, l = vid // 64, vid % 64
        if kind in SHARED:
            return self.shared[kind][l]
        if kind in READ_ONLY:
            return self.rs[kind][l]
        assert kind in PRIVATE, kind
        return self.priv[q].setdefault((kind, l), np.zeros(self.h.n[l]))

    def run_op(self, q, op):
        if op.type in (SPMV, EXT_RESID):
            M = (self.A, self.P, self.R)[op.mat_kind][op.mat_level]
            t = op.alpha * (M @ self.vec(q, op.x))
            if op.b >= 0:
                t = t + op.beta * self.vec(q, op.b)
            if op.b2 >= 0:
                t = t + op.beta2 * self.vec(q, op.b2)
            assert op.rs < 0 and op.c < 0 and op.xs < 0 and op.red < 0 and op.acc < 0
            self.vec(q, op.y)[:] = t
            if op.type == EXT_RESID:
                self.last_ss[q] = float(np.dot(t, t))
        elif op.type == EXT_CHEBY:
            u, yv, r, rs = self.vec(q, op.y), self.vec(q, op.c), self.vec(q, op.x), self.vec(q, op.rs)
            uo = u.copy()
            u[:] = yv + self.omega[q] * (self.delta * (rs * r) + uo - yv)
            yv[:] = uo
            self.omega[q] = 1.0 / (1.0 - self.omega[q] / self.mu22)
        else:
            raise AssertionError("operation %d" % op.type)

    # the three memory steps of EXT_STOP
    def stop_publish(self, q):
        if self.it[q] > 1:
            self.contrib[q] = self.last_ss[q]
        if self.it[q] + 1 == self.num_cycles:
            self.done += 1
        self.it[q] += 1

    def stop_check(self, q):
        if q == 0 and not self.flag and np.sqrt(sum(self.contrib)) / self.r0_ext < self.tol:
            self.flag = True

    def stop_decide(self, q):
        self.stopped[q] = self.flag or self.done >= self.L

    def body(self, q):
        return [op for op in self.progs[q] if op.type != EXT_STOP]

    def iteration(self, q):
        """one whole iteration of group q on its own"""
        for op in self.body(q):
            self.run_op(q, op)
        self.stop_publish(q)
        self.stop_check(q)
        self.stop_decide(q)

    def run(self, schedule, rng=None, max_rounds=100000):
        """schedule: 'lockstep', 'up', 'down', 'random' (a seeded permutation per round) or a list of iterations per round
        and group (unequal rates).  -> residual history of lock step (sum over the groups of this round's |r_k|^2)"""
        L, hist = self.L, []
        for _ in range(max_rounds):
            live = [q for q in range(L) if not self.stopped[q]]
            if not live:
                break
            if schedule == "lockstep":
                # every group's reads (chains, residual) before any group's writes, then every group's writes, then the stop
                # operations: publish everywhere, group 0's test, the decisions
                nread = {q: [op.type for op in self.body(q)].index(EXT_CHEBY) for q in live}
                for q in live:
                    for op in self.body(q)[:nread[q]]:
                        self.run_op(q, op)
                for q in live:
                    for op in self.body(q)[nread[q]:]:
                        self.run_op(q, op)
                for q in live:
                    self.stop_publish(q)
                hist.append(np.sqrt(sum(self.last_ss)) / self.r0_ext)
                for q in live:
                    self.stop_check(q)
                for q in live:
                    self.stop_decide(q)
            else:
                if schedule == "up":
                    order = [(q, 1) for q in range(L)]
                elif schedule == "down":
                    order = [(q, 1) for q in reversed(range(L))]
                elif schedule == "random":
                    order = [(int(q), 1) for q in rng.permutation(L)]
                else:
                    order = [(q, schedule[q]) for q in range(L)]
                for q, k in order:
                    for _ in range(k):
                        if not self.stopped[q]:
                            self.iteration(q)
        else:
            raise AssertionError("no stop after %d rounds" % max_rounds)
        return hist

    def finish(self):
        """the synchronous finish: extended residual of the final iterate, x = sum_l P^{0<-l} u_l, relres"""
        L, u, e, f = self.L, self.shared[V_XU], self.shared[V_XE], self.shared[V_XF]
        z1 = [None] * L
        z1[L - 1] = u[L - 1]
        for k in range(L - 2, -1, -1):
            z1[k] = self.P[k] @ z1[k + 1] + u[k]
        z2 = [np.zeros(self.h.n[0])]
        for k in range(L - 1):
            z2.append(self.R[k] @ (z2[k] + e[k]))
        ss = sum(np.sum((f[k] - (self.A[k] @ z1[k] + z2[k])) ** 2) for k in range(L))
        x = u[L - 1].copy()
        for k in range(L - 2, -1, -1):
            x = self.P[k] @ x + u[k]
        relres = np.linalg.norm(self.b - self.A[0] @ x) / self.r0
        return x, np.sqrt(ss) / self.r0_ext, relres


PROBLEMS = [("7pt", 16, H.JACOBI), ("5pt", 48, H.L1_JACOBI), ("27pt", 10, H.JACOBI)]
_cache = {}


def _problem(prob, n, sm, w=0.8):
    key = (prob, n, sm)
    if key not in _cache:
        A = H.laplacian(prob, n)
        h = H.amg_setup(A)
        h.build_transfers(H.BPX, w)
        b = H.rand_rhs(A.nrows)
        pb = O.Problem(h, H.BPX, sm, w)
        lo, hi = pb.eigs_power(20)
        _cache[key] = (h, b, pb, (hi + lo) / (hi - lo), 2.0 / (hi + lo))
    return _cache[key]


@pytest.mark.parametrize("sm", [H.JACOBI, H.L1_JACOBI])
@pytest.mark.parametrize("L", [1, 2, 3, 4, 5, 6])
def test_program_structure(L, sm):
    progs = S.ext_async_program(L, sm)
    assert len(progs) == L
    rs_kind = V_INVL1 if sm == H.L1_JACOBI else V_WS
    for k, prog in enumerate(progs):
        spmv = [op for op in prog if op.type in (SPMV, EXT_RESID)]
        assert sorted(op.mat_level for op in spmv if op.mat_kind == MAT_P) == list(range(k, L - 1))
        assert sorted(op.mat_level for op in spmv if op.mat_kind == MAT_R) == list(range(k))
        a = [op for op in spmv if op.mat_kind == MAT_A]
        assert all(op.mat_level == k for op in a) and len(a) == (2 if k < L - 1 else 1)
        assert [op.type for op in prog].count(EXT_RESID) == 1
        assert [op.type for op in prog].count(EXT_CHEBY) == 1
        assert [op.type for op in prog].count(EXT_STOP) == 1 and prog[-1].type == EXT_STOP
        for op in prog:
            writes = [op.y] + ([op.c] if op.type == EXT_CHEBY else [])
            reads = [op.x, op.b, op.b2, op.rs] + ([] if op.type == EXT_CHEBY else [op.c])
            for v in writes:
                if v < 0:
                    continue
                kind, l = v // 64, v % 64
                assert kind in PRIVATE or (kind in (V_XU, V_XY, V_XE) and l == k), (k, op.type, kind, l)
            for v in reads:
                if v < 0:
                    continue
                kind, l = v // 64, v % 64
                ok = (kind in PRIVATE or (kind == V_XU and l >= k) or (kind == V_XE and l < k) or (kind == V_XF and l == k)
                      or (kind == V_XY and l == k and op.type == EXT_CHEBY) or (kind == rs_kind and l == k))
                assert ok, (k, op.type, kind, l)
            assert op.red < 0 and op.red_copy < 0 and op.acc < 0 and op.xs < 0


@pytest.mark.parametrize("prob,n,sm", PROBLEMS)
def test_lock_step_equals_the_synchronous_solver(prob, n, sm):
    h, b, pb, mu, delta = _problem(prob, n, sm)
    progs = S.ext_async_program(h.num_levels, sm)
    for nc in (1, 2, 3, 12, 400):
        want = pb.solve_iebpx(b, 1e-9, nc, mu, delta)
        e = ExtInterp(h, progs, b, sm, 0.8, mu, delta, 1e-9, nc)
        hist = e.run("lockstep")
        x, ext_relres, relres = e.finish()
        assert e.it == [want["iters"]] * h.num_levels, (nc, e.it, want["iters"])
        k = want["iters"]
        assert len(hist) == k - 1
        if k > 1:
            assert np.max(np.abs(np.asarray(hist) - want["ext_hist"][1:k])) <= HIST_TOL
        assert abs(ext_relres - want["ext_relres"]) <= HIST_TOL
        assert abs(relres - want["relres"]) <= HIST_TOL
        assert np.max(np.abs(x - want["x"])) <= 1e-12 * np.max(np.abs(want["x"]))


@pytest.mark.parametrize("prob,n,sm", PROBLEMS)
@pytest.mark.parametrize("schedule", ["up", "down", "random", "rates"])
def test_chaotic_interleavings_converge(prob, n, sm, schedule):
    h, b, pb, mu, delta = _problem(prob, n, sm)
    L = h.num_levels
    want = pb.solve_iebpx(b, 1e-9, 400, mu, delta)
    progs = S.ext_async_program(L, sm)
    e = ExtInterp(h, progs, b, sm, 0.8, mu, delta, 1e-9, 3000)
    # unequal rates: group k does k + 1 iterations per round
    e.run([k + 1 for k in range(L)] if schedule == "rates" else schedule, rng=np.random.default_rng(7))
    x, ext_relres, relres = e.finish()
    true = np.linalg.norm(b - e.A[0] @ x) / np.linalg.norm(b)
    assert abs(true - relres) <= 1e-14
    assert true < 1e-8, (schedule, true, e.it)
    assert np.max(np.abs(x - want["x"])) <= 1e-7 * np.max(np.abs(want["x"])), schedule
    assert min(e.it) >= 2 and max(e.it) < 3000
    assert e.flag


def test_count_rule_without_tolerance():
    """tol = 0: the flag never rises, every group is done at num_cycles, the slowest one stops exactly there"""
    h, b, pb, mu, delta = _problem("7pt", 16, H.JACOBI)
    L = h.num_levels
    e = ExtInterp(h, S.ext_async_program(L, H.JACOBI), b, H.JACOBI, 0.8, mu, delta, 0.0, 12)
    e.run([k + 1 for k in range(L)])
    assert not e.flag and min(e.it) == 12 and e.it[0] == 12


def test_unsupported_options_are_refused():
    with pytest.raises(S.AmgError):
        S.ext_async_program(4, H.HYBRID_JACOBI_GAUSS_SEIDEL)
    with pytest.raises(S.AmgError):
        S.ext_async_program(33, H.JACOBI)
