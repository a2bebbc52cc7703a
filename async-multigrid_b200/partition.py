"""Row partition of an AMG hierarchy over the GPUs of one box (the DMEM replacement's host logic).

The reference's DMEM path lets hypre's ParCSR matrices carry the partition (row ranges per rank,
`diag`/`offd` blocks, `comm_pkg` send maps; /root/reference/src/DMEM_Setup.cpp:216-292,1160-1264) and
moves vector slices with DMEM_Comm (src/DMEM_Comm.cpp:81-382).  Here every level's rows are cut into
contiguous ranges (z-slabs on level 0; coarse points follow their fine points, so the slabs persist down
the hierarchy) and every rank's row block is renumbered into its *extended* index space

        [ ghost_lo | owned | ghost_hi ]

so that a halo exchange is two contiguous send/recv pairs with the immediate neighbours and the SpMV
kernels are the single-GPU ones.  Levels that are too small to be worth cutting (or whose halo would
reach beyond the immediate neighbour) are REPLICATED: the first such level's residual is all-gathered
and every rank computes the coarse part of the cycle redundantly.

This module is pure host logic (numpy); `dist_emulator` below executes the distributed cycle with numpy
kernels over torch.distributed (gloo) so that the plan is testable without GPUs; csrc/dist.cu executes the
same plan with the sm_100a kernels over NCCL.
"""
import numpy as np

from . import hierarchy as H


class LevelLayout:
    """Vector layout of one level on one rank."""

    def __init__(self, n_global, row_start, n_owned, halo_lo, halo_hi, distributed, send_lo, send_hi):
        self.n_global = int(n_global)
        self.row_start = int(row_start)      # first owned global row (also defined for replicated levels)
        self.n_owned = int(n_owned)
        self.halo_lo = int(halo_lo)          # ghost entries received from rank-1 (0 when replicated)
        self.halo_hi = int(halo_hi)          # ghost entries received from rank+1
        self.distributed = bool(distributed)
        self.send_lo = int(send_lo)          # my first send_lo owned entries go to rank-1 (= its halo_hi)
        self.send_hi = int(send_hi)          # my last send_hi owned entries go to rank+1 (= its halo_lo)

    @property
    def n_ext(self):
        return self.halo_lo + self.n_owned + self.halo_hi if self.distributed else self.n_global

    @property
    def base(self):
        """global index of extended entry 0"""
        return self.row_start - self.halo_lo if self.distributed else 0


def row_starts(h, nranks, plane=None):
    """starts[l][p] = first row of rank p on level l (length nranks+1).  Level 0: equal contiguous
    ranges, rounded to whole planes of `plane` rows when given (z-slabs); level l+1: coarse point j
    belongs to the rank that owns its fine point cpts[l][j]."""
    n0 = h.n[0]
    if plane:
        nplanes = n0 // plane
        s0 = np.array([plane * ((nplanes * p) // nranks) for p in range(nranks + 1)], dtype=np.int64)
        s0[-1] = n0
    else:
        s0 = np.array([(n0 * p) // nranks for p in range(nranks + 1)], dtype=np.int64)
    starts = [s0]
    for l in range(h.num_levels - 1):
        if h.cpts is None:
            raise ValueError("hierarchy has no coarse-point map (cpts); cannot derive the coarse partitions")
        starts.append(np.searchsorted(h.cpts[l], starts[l], side="left").astype(np.int64))
        starts[-1][-1] = h.n[l + 1]
    return starts


def _col_range(m, r0, r1):
    """(min, max) column index over rows [r0, r1) of CSR m; (None, None) when empty"""
    a, b = int(m.indptr[r0]), int(m.indptr[r1])
    if b <= a:
        return None, None
    seg = m.indices[a:b]
    return int(seg.min()), int(seg.max())


def plan_layouts(h, nranks, plane=None, min_rows_per_rank=4096):
    """Returns (starts, num_dist, halos) where halos[l][p] = (lo, hi) ghost widths of rank p on
    distributed level l.  Level l is distributed iff every rank owns >= min_rows_per_rank rows, every finer
    level is distributed, and every ghost range fits inside the immediate neighbour's owned range."""
    starts = row_starts(h, nranks, plane)
    L = h.num_levels
    halos = []
    num_dist = 0
    if nranks == 1:
        return starts, 0, halos
    for l in range(L):
        own = np.diff(starts[l])
        if l > 0 and own.min() < min_rows_per_rank:
            break
        # matrices whose INPUT vector lives on level l: A_l (rows of l), R_l (rows of l+1), P_{l-1} (rows of l-1)
        readers = [(h.A[l], starts[l])]
        if l < L - 1:
            readers.append((h.R[l], starts[l + 1]))
        if l > 0:
            readers.append((h.P[l - 1], starts[l - 1]))
        w = []
        ok = True
        for p in range(nranks):
            lo_col, hi_col = int(starts[l][p]), int(starts[l][p + 1]) - 1
            for m, rs in readers:
                cmin, cmax = _col_range(m, int(rs[p]), int(rs[p + 1]))
                if cmin is not None:
                    lo_col, hi_col = min(lo_col, cmin), max(hi_col, cmax)
            lo = int(starts[l][p]) - lo_col
            hi = hi_col - (int(starts[l][p + 1]) - 1)
            if (lo > 0 and (p == 0 or lo > own[p - 1])) or (hi > 0 and (p == nranks - 1 or hi > own[p + 1])):
                ok = False
            w.append((lo, hi))
        if not ok:
            if l == 0:
                raise ValueError("level-0 halo reaches beyond the immediate neighbour: too many ranks for this problem")
            break
        halos.append(w)
        num_dist = l + 1
    # a level's P reads level l+1: if l+1 is distributed its halo already covers P_l (it was a reader there)
    return starts, num_dist, halos


def rank_layouts(h, nranks, rank, starts, num_dist, halos):
    out = []
    for l in range(h.num_levels):
        rs, re = int(starts[l][rank]), int(starts[l][rank + 1])
        if l < num_dist:
            lo, hi = halos[l][rank]
            send_lo = halos[l][rank - 1][1] if rank > 0 else 0
            send_hi = halos[l][rank + 1][0] if rank < nranks - 1 else 0
            out.append(LevelLayout(h.n[l], rs, re - rs, lo, hi, True, send_lo, send_hi))
        else:
            out.append(LevelLayout(h.n[l], rs, re - rs, 0, 0, False, 0, 0))
    return out


def _block(m, r0, r1, col_base, ncols):
    """rows [r0,r1) of CSR m with columns shifted by -col_base into an ncols-wide index space"""
    a, b = int(m.indptr[r0]), int(m.indptr[r1])
    ip = (m.indptr[r0:r1 + 1] - m.indptr[r0]).astype(np.int32)
    ix = (m.indices[a:b].astype(np.int64) - col_base).astype(np.int32)
    if ix.size and (ix.min() < 0 or ix.max() >= ncols):
        raise AssertionError("column outside the extended range")
    return H.CSR(r1 - r0, ncols, ip, ix, m.data[a:b].copy())


class RankPlan:
    """Everything one rank needs: layouts + local matrix blocks in extended numbering."""

    def __init__(self, h, nranks, rank, plane=None, min_rows_per_rank=4096, plan=None):
        self.nranks, self.rank = nranks, rank
        self.num_levels = h.num_levels
        starts, num_dist, halos = plan if plan is not None else plan_layouts(h, nranks, plane, min_rows_per_rank)
        self.starts, self.num_dist, self.halos = starts, num_dist, halos
        self.layouts = rank_layouts(h, nranks, rank, starts, num_dist, halos)
        self.all_counts = [np.diff(s).astype(np.int64) for s in starts]
        L = h.num_levels
        self.A, self.P, self.R = [], [], []
        for l in range(L):
            lay = self.layouts[l]
            if lay.distributed:
                self.A.append(_block(h.A[l], lay.row_start, lay.row_start + lay.n_owned, lay.base, lay.n_ext))
            else:
                self.A.append(h.A[l])
            if l < L - 1:
                nxt = self.layouts[l + 1]
                # P_l: rows of level l, input vector on level l+1
                if lay.distributed:
                    self.P.append(_block(h.P[l], lay.row_start, lay.row_start + lay.n_owned, nxt.base, nxt.n_ext))
                else:
                    self.P.append(h.P[l])
                # R_l: rows of level l+1 (owned range, also when l+1 is the first replicated level), input on level l
                if lay.distributed:
                    self.R.append(_block(h.R[l], nxt.row_start, nxt.row_start + nxt.n_owned, lay.base, lay.n_ext))
                else:
                    self.R.append(h.R[l])

    def local_hierarchy(self):
        """the rank's blocks packaged as a hierarchy.Hierarchy (what amgb_set_matrix receives)"""
        hh = H.Hierarchy(self.A, [])
        hh.P, hh.R = self.P, self.R
        return hh


# ---------------------------------------------------------------------------------------------------
# numpy / gloo executor of the distributed synchronous cycles (tests; mirrors csrc/dist.cu)
# ---------------------------------------------------------------------------------------------------
class DistEmulator:
    """Runs the plan with numpy kernels; communication through a `comm` object with
    sendrecv(send_lo, send_hi, n_lo, n_hi) -> (from_lo, from_hi), allgatherv(x, counts) and allreduce_sum(v).
    solver: Multadd, AFACx or BPX (`cycle`, one sweep per level) or MULT (`vcycle`, num_pre / num_post sweeps, coarse_solve:
    direct solve on the replicated coarsest level).  `counts` tallies the halo exchanges (of distributed levels), all-gathers
    and all-reduces; `per_cycle` the collectives of every iteration of the last `solve` (cycle + residual norm)."""

    def __init__(self, plan, comm, smooth_weight, solver=H.MULTADD, smoother=H.JACOBI, symmetric=True, num_pre=1, num_post=1,
                 coarse_solve=False):
        import scipy.sparse as sp
        self.pl, self.comm, self.w = plan, comm, smooth_weight
        self.solver, self.smoother = solver, smoother
        self.symmetric = bool(symmetric) and solver == H.MULTADD
        self.num_pre, self.num_post = int(num_pre), int(num_post)
        self.coarse_solve = bool(coarse_solve) and plan.num_levels > 1
        if self.coarse_solve and plan.layouts[-1].distributed:
            raise ValueError("coarse_solve needs a replicated coarsest level")
        self.counts = {"halo": 0, "allgather": 0, "allreduce": 0}
        self.per_cycle = []
        self.sp = sp
        self.A = [m.to_scipy() for m in plan.A]
        self.P = [m.to_scipy() for m in plan.P]
        self.R = [m.to_scipy() for m in plan.R]
        self.Ac = self.A[-1].toarray() if self.coarse_solve else None
        # omega/d (1/l1 for L1-Jacobi: the row sums of a local row block are the global ones) in the level's vector
        # layout (ghosts filled by one halo exchange at setup)
        self.ws = []
        self.e = [self.new_vec(l) for l in range(plan.num_levels)]     # level iterates of the V-cycle (l >= 1)
        for l, lay in enumerate(plan.layouts):
            v = self.new_vec(l)
            if smoother == H.L1_JACOBI:
                self.owned(l, v)[:] = 1.0 / np.add.reduceat(np.abs(plan.A[l].data), plan.A[l].indptr[:-1])
            else:
                self.owned(l, v)[:] = smooth_weight / plan.A[l].data[plan.A[l].indptr[:-1]]
            self.halo(l, v)
            self.ws.append(v)
        self.counts["halo"] = 0

    def new_vec(self, l):
        return np.zeros(self.pl.layouts[l].n_ext)

    def owned(self, l, v):
        lay = self.pl.layouts[l]
        return v[lay.halo_lo:lay.halo_lo + lay.n_owned] if lay.distributed else v

    def halo(self, l, v):
        lay = self.pl.layouts[l]
        if not lay.distributed:
            return
        self.counts["halo"] += 1
        o = self.owned(l, v)
        lo, hi = self.comm.sendrecv(o[:lay.send_lo].copy(), o[lay.n_owned - lay.send_hi:].copy(), lay.halo_lo, lay.halo_hi)
        v[:lay.halo_lo] = lo
        v[lay.halo_lo + lay.n_owned:] = hi

    def smooth_symmetric(self, l, r):
        """e = s o (2 r - A (s o r)) on the owned rows, s = w/d or 1/l1; r must have valid ghosts"""
        ws = self.ws[l]
        t = self.A[l] @ (ws * r)
        e = self.new_vec(l)
        self.owned(l, e)[:] = self.owned(l, ws) * (2.0 * self.owned(l, r) - t)
        return e

    def smooth_plain(self, l, r):
        """one (L1-)Jacobi sweep from a zero guess: e = s o r on the owned rows"""
        e = self.new_vec(l)
        self.owned(l, e)[:] = self.owned(l, self.ws[l]) * self.owned(l, r)
        return e

    def restrict(self, l, v):
        """R_l v (ghosts of v) as a level-(l+1) vector, owned part valid; all-gathered whole at the first replicated level"""
        self.halo(l, v)
        y = self.R[l] @ v
        out = self.new_vec(l + 1)
        if self.pl.layouts[l + 1].distributed or not self.pl.layouts[l].distributed:
            self.owned(l + 1, out)[:] = y
        else:
            self.counts["allgather"] += 1
            out[:] = self.comm.allgatherv(y, self.pl.all_counts[l + 1])
        return out

    def sweeps(self, l, f, u, k):
        """k (L1-)Jacobi sweeps u <- u + s o (f - A_l u) on the owned rows, in place; ghosts refreshed before every sweep"""
        s = self.owned(l, self.ws[l])
        for _ in range(k):
            self.halo(l, u)
            self.owned(l, u)[:] = self.owned(l, u) + s * (f - self.A[l] @ u)

    def vcycle(self, f, u):
        """one multiplicative V-cycle (SMEM_Sync_Parfor_Vcycle, src/SMEM_Sync_AMG.cpp:8-145; DMEM_MultCycle with coarse_solve) on
        f (owned rows of level 0) and u (level-0 layout, updated in place).  The first pre-sweep of levels 1..L-2 starts from
        zero, the coarsest level's sweeps continue from the previous cycle's iterate.  Mirrors dist_vcycle of csrc/dist.cu."""
        L = self.pl.num_levels
        pre, post = self.num_pre, self.num_post
        fs, us = [np.asarray(f, dtype=np.float64)] + [None] * (L - 1), [u] + self.e[1:]
        for l in range(L - 1):
            if l > 0 and pre > 0:
                self.owned(l, us[l])[:] = self.owned(l, self.ws[l]) * fs[l]
                self.sweeps(l, fs[l], us[l], pre - 1)
            else:
                self.sweeps(l, fs[l], us[l], pre)
            self.halo(l, us[l])
            w = self.new_vec(l)
            self.owned(l, w)[:] = fs[l] - self.A[l] @ us[l]
            fs[l + 1] = self.owned(l + 1, self.restrict(l, w))
        c = L - 1
        if self.coarse_solve:
            us[c][:] = np.linalg.solve(self.Ac, fs[c])
        else:
            self.sweeps(c, fs[c], us[c], pre + post)
        for l in range(L - 2, -1, -1):
            self.halo(l + 1, us[l + 1])
            self.owned(l, us[l])[:] += self.P[l] @ us[l + 1]
            self.sweeps(l, fs[l], us[l], post)

    def cycle(self, r0):
        """one synchronous additive cycle -- Multadd (symmetrised or plain Jacobi), AFACx or BPX, one sweep per level --
        on the residual r0 (level-0 layout, owned part valid); returns the correction in level-0 layout (owned part
        valid).  Mirrors dist_cycle of csrc/dist.cu."""
        pl = self.pl
        L = pl.num_levels
        afacx, bpx = self.solver == H.AFACX, self.solver == H.BPX
        top = L if bpx else L - 1                   # levels that contribute a correction
        last_r = L - 1 if afacx else top - 1        # coarsest residual the cycle reads
        r = [r0] + [None] * (L - 1)
        for l in range(last_r):
            r[l + 1] = self.restrict(l, r[l])
        if self.symmetric and L >= 2:
            self.halo(L - 2, r[L - 2])
        if afacx:
            # src/SEQ_AMG.cpp:172-208: u_c = S_{l+1} r_{l+1}; e = P_l u_c; r_f = r_l - A_l e; u_f = S_l r_f
            e = []
            for l in range(L - 1):
                uc = self.smooth_plain(l + 1, r[l + 1])
                self.halo(l + 1, uc)
                t = self.new_vec(l)
                self.owned(l, t)[:] = self.P[l] @ uc
                self.halo(l, t)
                rf = self.new_vec(l)
                self.owned(l, rf)[:] = self.owned(l, r[l]) - self.A[l] @ t
                e.append(self.smooth_plain(l, rf))
        elif self.symmetric:
            e = [self.smooth_symmetric(l, r[l]) for l in range(top)]
        else:
            e = [self.smooth_plain(l, r[l]) for l in range(top)]
        for l in range(top - 2, -1, -1):
            self.halo(l + 1, e[l + 1])
            self.owned(l, e[l])[:] += self.P[l] @ e[l + 1]
        return e[0]

    def async_smooth_lockstep(self, f_owned, sweeps):
        """DMEM_AsyncSmooth (src/DMEM_Smooth.cpp:16-313; csrc/dist.cu amgb_dist_async_smooth) in the one interleaving that is
        reproducible: every rank's boundary values reach its neighbours before their next sweep.  x_own += s o (f - A_0
        [ghosts | x_own]); this is global (L1-)Jacobi.  Returns the owned part of x."""
        u = self.new_vec(0)
        f = np.asarray(f_owned, dtype=np.float64)
        so = self.owned(0, self.ws[0])
        for _ in range(sweeps):
            self.halo(0, u)
            self.owned(0, u)[:] += so * (f - self.A[0] @ u)
        return self.owned(0, u).copy()

    def solve(self, f_owned, tol, max_cycles):
        l0 = self.pl.layouts[0]
        u = self.new_vec(0)
        f = np.asarray(f_owned, dtype=np.float64)

        def residual():
            self.halo(0, u)
            r = self.new_vec(0)
            self.owned(0, r)[:] = f - self.A[0] @ u
            self.counts["allreduce"] += 1
            return r, np.sqrt(self.comm.allreduce_sum(float(np.dot(self.owned(0, r), self.owned(0, r)))))
        r, r0n = residual()
        hist = [1.0]
        for v in self.e:
            v[:] = 0.0
        self.per_cycle = []
        for _ in range(max_cycles):
            before = sum(self.counts.values())
            if self.solver == H.MULT:
                self.vcycle(f, u)
            else:
                c = self.cycle(r)
                self.owned(0, u)[:] += self.owned(0, c)
            r, rn = residual()
            self.per_cycle.append(sum(self.counts.values()) - before)
            hist.append(rn / r0n)
            if hist[-1] < tol:
                break
        return self.owned(0, u).copy(), np.asarray(hist)


class LoopbackComm:
    """single-process stand-in: a list of LoopbackComm objects exchanging through shared python lists
    is not needed for tests (they use gloo); this class serves nranks == 1."""

    def sendrecv(self, send_lo, send_hi, n_lo, n_hi):
        return np.zeros(n_lo), np.zeros(n_hi)

    def allgatherv(self, x, counts):
        return x

    def allreduce_sum(self, v):
        return v


class TorchComm:
    """torch.distributed (gloo on CPU) implementation of the emulator's communication"""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank, self.n = dist.get_rank(), dist.get_world_size()

    def sendrecv(self, send_lo, send_hi, n_lo, n_hi):
        t, d = self.torch, self.dist
        ops, lo, hi = [], t.zeros(n_lo, dtype=t.float64), t.zeros(n_hi, dtype=t.float64)
        if self.rank > 0:
            if len(send_lo):
                ops.append(d.P2POp(d.isend, t.from_numpy(send_lo), self.rank - 1))
            if n_lo:
                ops.append(d.P2POp(d.irecv, lo, self.rank - 1))
        if self.rank < self.n - 1:
            if len(send_hi):
                ops.append(d.P2POp(d.isend, t.from_numpy(send_hi), self.rank + 1))
            if n_hi:
                ops.append(d.P2POp(d.irecv, hi, self.rank + 1))
        if ops:
            for w in d.batch_isend_irecv(ops):
                w.wait()
        return lo.numpy(), hi.numpy()

    def allgatherv(self, x, counts):
        t, d = self.torch, self.dist
        parts = [t.zeros(int(c), dtype=t.float64) for c in counts]
        d.all_gather(parts, t.from_numpy(np.ascontiguousarray(x))) if len(set(int(c) for c in counts)) == 1 else None
        if len(set(int(c) for c in counts)) != 1:
            for p in range(self.n):
                buf = t.from_numpy(np.ascontiguousarray(x)) if p == self.rank else parts[p]
                d.broadcast(buf, src=p)
                if p == self.rank:
                    parts[p] = buf
        return np.concatenate([p.numpy() for p in parts])

    def allreduce_sum(self, v):
        x = self.torch.tensor([v], dtype=self.torch.float64)
        self.dist.all_reduce(x)
        return float(x[0])
