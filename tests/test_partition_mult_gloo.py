"""Host logic of the row-partitioned multiplicative V-cycle (MULT; csrc/dist.cu dist_vcycle), on CPU: the numpy emulator
(partition.DistEmulator.vcycle) over torch.distributed (gloo, world_size 2 and 3) must reproduce the GLOBAL oracle's
V-cycle history, and with the direct coarse solve the reference's DMEM_Mult object code (tests/golden/dmem_mult.npz)."""
import os
import socket
import sys

import numpy as np
import pytest

from conftest import assert_hist_close, hierarchy_from_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def cpts_from_injection(h):
    """coarse-point map of a hierarchy read from a fixture: coarse point j of level l+1 is the fine row of P_l that injects it
    (a single entry 1.0 in column j)"""
    cpts = []
    for P in h.P_plain:
        c = np.full(P.ncols, -1, dtype=np.int64)
        for i in range(P.nrows):
            a = P.indptr[i]
            if P.indptr[i + 1] - a == 1 and P.data[a] == 1.0:
                c[P.indices[a]] = i
        assert np.all(c >= 0) and np.all(np.diff(c) > 0)
        cpts.append(c)
    return cpts


def _problem(H, prob, n, w):
    A = H.laplacian(prob, n)
    h = H.amg_setup(A)
    h.build_transfers(H.MULT, w)
    return h, H.rand_rhs(A.nrows), (n * n if prob == "7pt" else n)


def _golden(H, name):
    h, d = hierarchy_from_golden(name)
    h.cpts = cpts_from_injection(h)
    h.build_transfers(H.MULT, 0.8)
    return h, d["b"], (144 if name == "lap7pt_n12" else 32)


def _worker(rank, world, port, case, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    os.environ["OMP_NUM_THREADS"] = "1"
    import torch.distributed as dist
    import async_multigrid_b200 as amg  # noqa: F401
    from async_multigrid_b200 import hierarchy as H, partition as PT
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        prob, n, min_rows, smoother, w, pre, post, cs = case
        h, b, plane = _golden(H, prob) if prob.startswith("lap") else _problem(H, prob, n, w)
        plan = PT.RankPlan(h, world, rank, plane=plane, min_rows_per_rank=min_rows)
        l0 = plan.layouts[0]
        em = PT.DistEmulator(plan, PT.TorchComm(), w, H.MULT, smoother, num_pre=pre, num_post=post, coarse_solve=cs)
        u, hist = em.solve(b[l0.row_start:l0.row_start + l0.n_owned], 1e-9, 100)
        q.put((rank, plan.num_dist, plan.num_levels, hist, u, l0.row_start, em.per_cycle))
    finally:
        dist.destroy_process_group()


def _run(world, case):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, case, q)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        res = sorted([q.get(timeout=240) for _ in range(world)], key=lambda x: x[0])
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join(timeout=10)
    return res


# (problem, n, min_rows_per_rank, smoother, weight, pre, post, coarse_solve)
CASES = [("7pt", 16, 64, 0, 0.8, 1, 1, 0), ("7pt", 16, 64, 0, 0.8, 2, 2, 1), ("7pt", 16, 64, 6, 0.8, 1, 0, 0),
         ("5pt", 48, 100, 6, 0.8, 1, 1, 1), ("5pt", 48, 100, 0, 0.8, 1, 0, 1), ("5pt", 48, 100, 0, 0.8, 2, 2, 0)]


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("case", CASES, ids=lambda c: "%s-sm%d-%d%d-cs%d" % (c[0], c[3], c[5], c[6], c[7]))
def test_partitioned_vcycle_reproduces_global_oracle(world, case):
    sys.path.insert(0, ROOT)
    from async_multigrid_b200 import hierarchy as H
    from oracle import oracle as O
    prob, n, _, smoother, w, pre, post, cs = case
    h, b, _ = _problem(H, prob, n, w)
    _, want, _ = O.Problem(h, H.MULT, smoother, w, num_pre=pre, num_post=post, coarse_solve=cs).solve_sync(b, 1e-9, 100)
    assert want[-1] < 1e-9
    res = _run(world, case)
    for rank, num_dist, L, hist, _, _, per_cycle in res:
        assert num_dist >= 2, num_dist              # at least two levels are really partitioned
        assert num_dist < L                          # and the coarse tail is replicated
        assert len(hist) == len(want)
        assert np.max(np.abs(hist - want) / np.maximum(want, 1.0)) <= 1e-10
        assert_hist_close(hist, want)
        assert len(set(per_cycle)) == 1              # the same collectives in every cycle
    assert all(r[6] == res[0][6] for r in res)        # on every rank


@pytest.mark.parametrize("name", ["lap5pt_n32", "lap7pt_n12"])
@pytest.mark.parametrize("world", [1, 2])
def test_partitioned_vcycle_matches_dmem_mult_fixture(name, world):
    """coarse_solve = 1 (DMEM_MultCycle's direct solve on the replicated coarsest level): the reference's DMEM_Mult object code"""
    sys.path.insert(0, ROOT)
    from async_multigrid_b200 import hierarchy as H, partition as PT
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "dmem_mult.npz")))
    if world == 1:
        h, b, _ = _golden(H, name)
        em = PT.DistEmulator(PT.RankPlan(h, 1, 0), PT.LoopbackComm(), 0.8, H.MULT, H.JACOBI, coarse_solve=True)
        u, hist = em.solve(b, 1e-9, 100)
    else:
        res = _run(world, (name, 0, 64, H.JACOBI, 0.8, 1, 1, 1))
        assert all(r[1] >= 2 for r in res)
        hist = res[0][3]
        assert all(np.array_equal(r[3], hist) for r in res)
        u = np.concatenate([r[4] for r in res])
    assert_hist_close(hist, g[name + "_hist"])
    assert np.max(np.abs(u - g[name + "_x"])) <= 1e-11 * np.max(np.abs(u))


def test_direct_coarse_solve_needs_a_replicated_coarsest_level():
    """with a small enough min_rows_per_rank every level of lap5pt_n32 is cut over two ranks: the direct coarse solve is refused"""
    sys.path.insert(0, ROOT)
    from async_multigrid_b200 import hierarchy as H, partition as PT
    h, _, plane = _golden(H, "lap5pt_n32")
    plan = PT.RankPlan(h, 2, 0, plane=plane, min_rows_per_rank=1)
    assert plan.num_dist == plan.num_levels
    with pytest.raises(ValueError, match="replicated coarsest"):
        PT.DistEmulator(plan, PT.LoopbackComm(), 0.8, H.MULT, H.JACOBI, coarse_solve=True)
