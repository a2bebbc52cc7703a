"""GPU tests of the row-partitioned multiplicative V-cycle (MULT; csrc/dist.cu dist_vcycle) through DistSolver.  One GPU: a
one-rank communicator against the oracle, the single-GPU MULT solver and the reference's DMEM_Mult object code
(tests/golden/dmem_mult.npz), the captured graph, the collective counts and the refusals.  Two GPUs: two processes, one z-slab
each, against the GLOBAL oracle and the numpy emulator of the same plan (partition.DistEmulator over gloo)."""
import os
import socket
import sys

import numpy as np
import pytest

import async_multigrid_b200 as amg
from async_multigrid_b200 import hierarchy as H, partition as PT
from conftest import assert_hist_close, hierarchy_from_golden
from oracle import oracle as O
from test_partition_mult_gloo import cpts_from_injection

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EINVAL = -1


def _problem(prob, n, w=0.8):
    A = H.laplacian(prob, n)
    h = H.amg_setup(A)
    h.build_transfers(H.MULT, w)
    return h, H.rand_rhs(A.nrows)


def _dist(h, **kw):
    return amg.DistSolver(PT.RankPlan(h, 1, 0), amg.solver.dist_unique_id(), kw.pop("w", 0.8), solver=H.MULT, **kw)


@pytest.mark.parametrize("use_sell", [True, False])
@pytest.mark.parametrize("coarse_solve", [0, 1])
@pytest.mark.parametrize("pre,post", [(1, 1), (2, 2), (1, 0)])
@pytest.mark.parametrize("prob,n,smoother", [("7pt", 16, H.JACOBI), ("5pt", 48, H.L1_JACOBI)])
def test_single_rank_vcycle_matches_oracle_and_single_gpu(prob, n, smoother, pre, post, coarse_solve, use_sell):
    w = 0.8
    h, b = _problem(prob, n, w)
    _, want, _ = O.Problem(h, H.MULT, smoother, w, num_pre=pre, num_post=post, coarse_solve=coarse_solve).solve_sync(b, 1e-9, 100)
    s = _dist(h, w=w, smoother=smoother, num_pre=pre, num_post=post, coarse_solve=bool(coarse_solve), use_sell=use_sell)
    s.set_rhs(b)
    hist, _ = s.solve_sync(1e-9, 100)
    assert_hist_close(hist, want)
    u = s.get_solution()
    true = O.norm2(O.spgemv(h.A[0], u, b, -1.0, 1.0)) / O.norm2(b)
    assert abs(true - hist[-1]) <= 1e-12
    s.close()
    g = amg.Solver(h, H.MULT, smoother, w, num_pre=pre, num_post=post, coarse_solve=bool(coarse_solve), use_sell=use_sell)
    assert_hist_close(hist, g.SMEM_Solve(b, 1e-9, 100)["hist"])
    g.close()


@pytest.mark.parametrize("name", ["lap5pt_n32", "lap7pt_n12"])
def test_single_rank_vcycle_matches_dmem_mult_fixture(name):
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "dmem_mult.npz")))
    h, d = hierarchy_from_golden(name)
    h.cpts = cpts_from_injection(h)
    h.build_transfers(H.MULT, 0.8)
    s = _dist(h, coarse_solve=True)
    s.set_rhs(d["b"])
    hist, _ = s.solve_sync(1e-9, 100)
    assert_hist_close(hist, g[name + "_hist"])
    u = s.get_solution()
    assert np.max(np.abs(u - g[name + "_x"])) <= 1e-11 * np.max(np.abs(u))
    s.close()


def test_single_rank_graph_replay_and_a_second_context():
    """the second solve replays the captured V-cycle: bit-identical history; a partitioned Multadd solve on another context of
    the same process is unaffected"""
    h, b = _problem("7pt", 16)
    hm = H.Hierarchy(h.A, h.P_plain)
    hm.cpts = h.cpts
    hm.build_transfers(H.MULTADD, 0.9)
    add = amg.DistSolver(PT.RankPlan(hm, 1, 0), amg.solver.dist_unique_id(), 0.9)
    add.set_rhs(b)
    add_hist, _ = add.solve_sync(1e-9, 100)
    s = _dist(h)
    s.set_rhs(b)
    h1, _ = s.solve_sync(1e-9, 100)
    l1 = s.launch_count()
    h2, _ = s.solve_sync(1e-9, 100)
    assert np.array_equal(h1, h2)
    assert s.launch_count() - l1 > 0
    add2, _ = add.solve_sync(1e-9, 100)
    assert np.array_equal(add_hist, add2)
    _, want, _ = O.Problem(hm, H.MULTADD, H.JACOBI, 0.9).solve_sync(b, 1e-9, 100)
    assert_hist_close(add2, want)
    s.close()
    add.close()


def _per_cycle_collectives(s):
    """collectives of one iteration (V-cycle + residual norm) from the stats() deltas of solves of 1, 2, 3 cycles"""
    d = []
    for k in (1, 2, 3):
        _, c0 = s.stats()
        hist, _ = s.solve_sync(0.0, k)
        assert len(hist) == k + 1
        _, c1 = s.stats()
        d.append(c1 - c0)
    return d[1] - d[0], d[2] - d[1]


def test_single_rank_collectives_per_cycle_equal_the_emulator():
    h, b = _problem("7pt", 16)
    s = _dist(h)
    s.set_rhs(b)
    c1, c2 = _per_cycle_collectives(s)
    s.close()
    em = PT.DistEmulator(PT.RankPlan(h, 1, 0), PT.LoopbackComm(), 0.8, H.MULT)
    em.solve(b, 0.0, 3)
    assert c1 == c2 and [c1] * 3 == em.per_cycle


def _expect_einval(call, word):
    with pytest.raises(amg.AmgError) as ei:
        call()
    msg = str(ei.value)
    assert ("error %d:" % EINVAL) in msg and word in msg, msg


def test_refusals():
    h, b = _problem("7pt", 12)
    # set-up refusals: the factorised transfers (amgb_setup refuses them for every solver but Multadd) and hybrid JGS
    for kw, word in ((dict(factor_level0=True), "factor_level0"), (dict(smoother=H.HYBRID_JACOBI_GAUSS_SEIDEL), "hybrid JGS")):
        s = amg.DistSolver.__new__(amg.DistSolver)
        _expect_einval(lambda: s.__init__(PT.RankPlan(h, 1, 0), amg.solver.dist_unique_id(), 0.8, solver=H.MULT, **kw), word)
        s.close()
    # solve-time refusals, before any launch
    s = _dist(h)
    s.set_rhs(b)
    n0 = s.launch_count()
    for call, word in ((lambda: s.solve_sync(1e-9, 10, accel=1, mu=2.0, delta=1.0), "accel 1"),
                       (lambda: s.solve_sync(1e-9, 10, accel=2, mu=2.0, delta=1.0), "accel 2"),
                       (lambda: s.DMEM_PowerMult(10), "DMEM_PowerMult"),
                       (lambda: s.DMEM_Add_async(10), "asynchronous MULT")):
        _expect_einval(call, word)
        assert s.launch_count() == n0
    hist, _ = s.solve_sync(1e-9, 100)                   # the context is still usable
    assert hist[-1] < 1e-9
    s.close()
    # a direct coarse solve on a distributed coarsest level needs two ranks: see test_two_gpus_match_global_oracle


_LIVE = []


@pytest.fixture(autouse=True)
def _reap_workers():
    yield
    for p in _LIVE:
        if p.is_alive():
            p.kill()
            p.join(timeout=10)
    del _LIVE[:]


def _worker(rank, world, port, uid_q, res_q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    import torch.distributed as dist
    import async_multigrid_b200 as amg2
    from async_multigrid_b200 import hierarchy as H2, partition as PT2
    from conftest import hierarchy_from_golden as hfg
    from test_partition_mult_gloo import cpts_from_injection as cfi
    n, w = 32, 0.8
    A = H2.laplacian("7pt", n)
    h = H2.amg_setup(A)
    h.build_transfers(H2.MULT, w)
    b = H2.rand_rhs(A.nrows)
    plan = PT2.RankPlan(h, world, rank, plane=n * n, min_rows_per_rank=256)
    if rank == 0:
        uids = [amg2.solver.dist_unique_id() for _ in range(2)]
        for _ in range(world - 1):
            uid_q.put(uids)
    else:
        uids = uid_q.get(timeout=120)
    s = amg2.DistSolver(plan, uids[0], w, solver=H2.MULT, device=rank)
    l0 = plan.layouts[0]
    f = b[l0.row_start:l0.row_start + l0.n_owned]
    s.set_rhs(f)
    hist, secs = s.solve_sync(1e-9, 100)
    u = s.get_solution()
    hb, _ = s.stats()
    per = _per_cycle_collectives(s)
    s.close()
    # the same plan in numpy over gloo: the collectives of one iteration
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        em = PT2.DistEmulator(plan, PT2.TorchComm(), w, H2.MULT)
        em.solve(f, 0.0, 2)
        em_per = em.per_cycle
    finally:
        dist.destroy_process_group()
    # every level of lap5pt_n32 cut over the two ranks: a direct coarse solve is refused
    hg, _ = hfg("lap5pt_n32")
    hg.cpts = cfi(hg)
    hg.build_transfers(H2.MULT, w)
    pg = PT2.RankPlan(hg, world, rank, plane=32, min_rows_per_rank=1)
    refused = ""
    try:
        amg2.DistSolver(pg, uids[1], w, solver=H2.MULT, coarse_solve=True, device=rank).close()
    except amg2.AmgError as e:
        refused = str(e)
    res_q.put((rank, hist, u, plan.num_dist, plan.num_levels, hb, per, em_per, pg.num_dist == pg.num_levels, refused))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_two_gpus_match_global_oracle():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    uid_q, res_q = ctx.Queue(), ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, uid_q, res_q)) for r in range(2)]
    _LIVE.extend(procs)
    for p in procs:
        p.start()
    res = sorted([res_q.get(timeout=300) for _ in range(2)], key=lambda x: x[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    h, b = _problem("7pt", 32)
    want_u, want, _ = O.Problem(h, H.MULT, H.JACOBI, 0.8).solve_sync(b, 1e-9, 100)
    u = np.concatenate([r[2] for r in res])
    for rank, hist, _, num_dist, L, hb, per, em_per, all_dist, refused in res:
        assert 2 <= num_dist < L and hb > 0
        assert len(hist) == len(want)
        assert np.max(np.abs(hist - want) / np.maximum(want, 1.0)) <= 1e-10
        assert_hist_close(hist, want)
        assert per[0] == per[1] and em_per == [per[0]] * 2
        assert all_dist and ("error %d:" % EINVAL) in refused and "coarse_solve" in refused, refused
    assert np.max(np.abs(u - want_u)) <= 1e-10 * np.max(np.abs(want_u))
