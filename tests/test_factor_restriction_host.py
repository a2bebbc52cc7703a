"""CPU checks of the factorised restriction (amgb_options.factor_restriction): the algebra the device cycle relies on,
Rbar_l r = P_l^T (r - A_l diag(s) r) with the smoother's scale s, on every level of the host hierarchies, and the byte model
bench.py reports for that cycle."""
import numpy as np
import pytest

from async_multigrid_b200 import hierarchy as H


def _hierarchy(prob, n, smooth_interp_type, w):
    h = H.amg_setup(H.laplacian(prob, n))
    h.build_transfers(H.MULTADD, w, smooth_interp_type=smooth_interp_type)
    return h


@pytest.mark.parametrize("prob,n", [("7pt", 16), ("5pt", 48), ("27pt", 10)])
@pytest.mark.parametrize("sit", [H.JACOBI, H.L1_JACOBI], ids=["j", "L1j"])
def test_plain_restriction_of_t_equals_explicit_product(prob, n, sit):
    w = 0.9
    h = _hierarchy(prob, n, sit, w)
    rng = np.random.default_rng(7)
    assert h.num_levels >= 3
    for l in range(h.num_levels - 1):
        A = h.A[l].to_scipy()
        s = w / A.diagonal() if sit == H.JACOBI else 1.0 / np.asarray(abs(A).sum(axis=1)).ravel()
        r = rng.uniform(-1, 1, h.n[l])
        t = r - A @ (s * r)
        R = h.plain_restriction(l).to_scipy()
        assert (R != h.P_plain[l].to_scipy().T).nnz == 0
        got = R @ t
        want = h.R[l].to_scipy() @ r
        mag = abs(R) @ (np.abs(r) + abs(A) @ (s * np.abs(r)))
        assert np.max(np.abs(got - want) / np.maximum(mag, 1e-300)) <= 1e-13, l


def test_plain_restriction_is_built_once():
    h = _hierarchy("7pt", 12, H.JACOBI, 0.9)
    assert h.plain_restriction(1) is h.plain_restriction(1)


def _spmv(nnz, rows, cols, with_b=False):
    return 12 * nnz + 4 * (rows + 1) + 8 * cols + 8 * rows + (8 * rows if with_b else 0)


def test_byte_model_counts_the_factorised_cycle():
    h = H.amg_setup(H.laplacian("7pt", 16))
    h.build_transfers(H.MULTADD, 0.9, factor_level0=True)
    L, n = h.num_levels, h.n
    assert L >= 4
    A, P, R = h.A, h.P, h.R
    level0 = (3 * _spmv(A[0].nnz, n[0], n[0], True) + 24 * n[0]
              + _spmv(R[0].nnz, R[0].nrows, R[0].ncols) + _spmv(P[0].nnz, P[0].nrows, P[0].ncols))
    smooth = [_spmv(A[l].nnz, n[l], n[l]) + 8 * n[l] for l in range(L)]
    prolong = [_spmv(P[l].nnz, P[l].nrows, P[l].ncols, True) for l in range(L - 1)]
    # P_l^T t_l: P_l's entries, n_{l+1} rows, n_l columns; then the t_l store of the smoother's pass
    plain = sum(_spmv(h.P_plain[l].nnz, n[l + 1], n[l]) + 8 * n[l] + smooth[l] + prolong[l] for l in range(1, L - 1))
    explicit = sum(_spmv(R[l].nnz, n[l + 1], n[l]) + smooth[l] + prolong[l] for l in range(1, L - 1))
    assert H.bytes_sync_multadd_cycle_factored(h) == level0 + plain
    assert H.bytes_sync_multadd_cycle_factored(h, factor_restriction=False) == level0 + explicit
    assert H.bytes_sync_multadd_cycle_factored(h) < H.bytes_sync_multadd_cycle_factored(h, factor_restriction=False)
