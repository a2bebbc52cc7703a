"""GPU tests of the window-staged SELL-C-sigma epilogue (amgb_options.sell_window_epilogue): the products with a matrix stored
as SELL-C-sigma park every row sum in shared memory and apply the epilogue in row order.  The row arithmetic is the one of the
slot-order path (same entries, same order, same epilogue code), so y and y2 must be bitwise equal between the two paths; only
the fused per-CTA partial sums (norm, dot) are added in another order.

The matrix is a one-level "hierarchy" whose A_0 reaches the SELL-C-sigma storage: more than 262144 rows, random row lengths
1-40 (natural-order sliced ELL pads ~90 %, so sigma = 1 is refused; sigma = 128 pads ~23 %, under the 25 % limit), the row
count not a multiple of 256 (a partial last window, padding slots)."""
import numpy as np
import pytest
import scipy.sparse as sp

import async_multigrid_b200 as amg
from async_multigrid_b200 import hierarchy as H

pytestmark = pytest.mark.gpu

MAT_A = 0
N = 262144 + 3 * 32 + 13
W = 0.7


@pytest.fixture(scope="module")
def problem():
    rng = np.random.default_rng(20261021)
    lens = rng.integers(1, 41, N)
    rows = np.repeat(np.arange(N), lens)
    cols = rng.integers(0, N, rows.size)
    first = np.concatenate(([0], np.cumsum(lens)[:-1]))
    cols = np.where(cols == rows, (cols + 1) % N, cols)         # one diagonal entry per row ...
    cols[first] = np.arange(N)                                  # ... and first (amgb_set_matrix checks it)
    vals = rng.standard_normal(rows.size)
    vals[first] = 40.0 + rng.random(N)
    # keep the generated entry order (duplicates stay separate entries), diagonal first in every row
    m = sp.csr_matrix((vals, cols, np.concatenate(([0], np.cumsum(lens)))), shape=(N, N))
    A = H.CSR(N, N, m.indptr.astype(np.int32), m.indices.astype(np.int32), m.data.astype(np.float64))
    h = H.Hierarchy([A], [])
    h.P, h.R = [], []
    vec = lambda: rng.standard_normal(N)
    v = dict(x=vec(), b=vec(), c=vec(), rs=rng.random(N) + 0.5, b2=vec(), xs=vec(), w=vec(), s2=rng.random(N) + 0.5)
    return h, m, v


@pytest.fixture(scope="module")
def solvers(problem):
    h = problem[0]
    out = {flag: amg.Solver(h, H.MULTADD, H.JACOBI, W, sell_window_epilogue=flag) for flag in (True, False)}
    yield out
    for s in out.values():
        s.close()


def _ref(m, v, a):
    """scipy: y = gamma c + rs o (beta b + beta2 b2 + alpha M x) + xself xs"""
    mat = m
    if a.get("use_sval"):
        mat = m @ sp.diags(W / m.diagonal())                    # the column-scaled values A diag(w/d)
    t = a.get("alpha", 1.0) * (mat @ v["x"])
    if "b" in a: t = t + a["beta"] * v["b"]
    if "b2" in a: t = t + a["beta2"] * v["b2"]
    if "rs" in a: t = t * v["rs"]
    if "c" in a: t = t + a["gamma"] * v["c"]
    if "xs" in a: t = t + a["xself"] * v["xs"]
    return t


FORMS = {
    "plain": dict(),
    "b": dict(alpha=-1.0, b=1, beta=1.0),
    "c": dict(c=1, gamma=1.0),
    "rs": dict(alpha=-1.0, b=1, beta=2.0, rs=1),
    "b2_xs": dict(alpha=-1.0, b=1, beta=1.0, b2=1, beta2=1.0, rs=1, c=1, gamma=1.0, xs=1, xself=1.0),
    "norm": dict(alpha=-1.0, b=1, beta=1.0, norm=True),
    "dot": dict(alpha=1.0, c=1, gamma=1.0, dot=True),
    "dual": dict(alpha=-1.0, b=1, beta=1.0, use_sval=True, dual=True),
}


def _run(s, v, a):
    kw = {k: v[k] for k in ("b", "c", "rs", "b2", "xs") if k in a}
    kw.update({k: a[k] for k in ("alpha", "beta", "gamma", "beta2", "xself") if k in a})
    return s.spmv_probe(MAT_A, 0, v["x"], use_sval=a.get("use_sval", False), norm=a.get("norm", False),
                        dot_w=v["w"] if a.get("dot") else None, dual_s2=v["s2"] if a.get("dual") else None, **kw)


def test_matrix_reaches_sell_sigma(solvers):
    for s in solvers.values():
        assert s.is_sell(MAT_A, 0)


@pytest.mark.parametrize("form", list(FORMS))
def test_window_epilogue_equals_slot_order(problem, solvers, form):
    _, m, v = problem
    a = FORMS[form]
    y1, y21, s1, win1 = _run(solvers[True], v, a)
    y0, y20, s0, win0 = _run(solvers[False], v, a)
    assert win1 and not win0
    assert np.array_equal(y1.view(np.int64), y0.view(np.int64))                     # bitwise
    ref = _ref(m, v, a)
    assert np.max(np.abs(y1 - ref)) <= 1e-13 * np.max(np.abs(ref))
    if a.get("dual"):
        assert np.array_equal(y21.view(np.int64), y20.view(np.int64))
        r2 = v["s2"] * (v["b"] + ref)
        assert np.max(np.abs(y21 - r2)) <= 1e-13 * np.max(np.abs(r2))
    if a.get("norm") or a.get("dot"):
        want = float(ref @ ref) if a.get("norm") else float(ref @ v["w"])
        scale = float(np.abs(ref) @ (np.abs(ref) if a.get("norm") else np.abs(v["w"])))
        assert abs(s1 - s0) <= 1e-13 * scale                                         # partial sums in another order
        assert abs(s1 - want) <= 1e-13 * scale


def test_sigma_not_dividing_the_cta_declines(problem):
    """sigma = 512 does not divide the 256 slots a CTA takes per iteration: the product stays on the slot-order path"""
    h, m, v = problem
    s = amg.Solver(h, H.MULTADD, H.JACOBI, W, sell_sigma=512)
    try:
        assert s.is_sell(MAT_A, 0)
        a = FORMS["b2_xs"]
        y, _, _, win = _run(s, v, a)
        assert not win
        ref = _ref(m, v, a)
        assert np.max(np.abs(y - ref)) <= 1e-13 * np.max(np.abs(ref))
    finally:
        s.close()
