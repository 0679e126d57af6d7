"""The oracle judges every GPU route, so its handling of stored zeros is pinned here against a closed
form: a stored zero is an observed interaction of confidence 0.  It adds nothing to the row's Gram,
adds bias * y (bias = alpha0 under the ORIGINAL loss) to b and counts in nnz, which sets the ridge
reg * (alpha0 * n_other + nnz)^nu."""
import numpy as np
import pytest
import scipy.sparse as sps

import oracle
from parity import np_cholesky_step, row_reg


def _matrix_with_stored_zeros():
    rng = np.random.default_rng(21)
    X = sps.random(40, 30, density=0.25, random_state=3, format="csr", dtype=np.float64)
    X.data[:] = rng.integers(1, 4, X.nnz)
    X.data[rng.random(X.nnz) < 0.2] = 0.0
    X.data[X.indptr[4]:X.indptr[5]] = 0.0  # a row of stored zeros only
    assert X.indptr[5] > X.indptr[4]
    return X


@pytest.mark.parametrize("nu", [0.0, 0.5, 2.0])
@pytest.mark.parametrize("loss", ["ORIGINAL", "IALSPP"])
def test_step_cholesky_counts_stored_zeros(loss, nu):
    X = _matrix_with_stored_zeros()
    K, alpha0, reg = 6, 0.3, 0.02
    rng = np.random.default_rng(5)
    other = rng.standard_normal((X.shape[1], K))
    target = rng.standard_normal((X.shape[0], K))
    lt = oracle.LOSS_ORIGINAL if loss == "ORIGINAL" else oracle.LOSS_IALSPP
    got = target.copy()
    oracle.step_cholesky(got, X, other, oracle.gram(other, alpha0), alpha0, reg, nu, lt)
    want = np_cholesky_step(target, X, other, alpha0, reg, nu, loss)
    np.testing.assert_allclose(got, want, rtol=1e-10, atol=1e-12)
    # the zeros count: dropping them changes the answer, except under the IALSPP loss at nu = 0,
    # where a zero adds neither to b nor to the ridge
    Xe = X.copy()
    Xe.eliminate_zeros()
    rows = np.diff(Xe.indptr) > 0
    dropped = np_cholesky_step(target[rows], Xe[rows], other, alpha0, reg, nu, loss)
    kept = want[rows]
    if loss == "ORIGINAL" or nu != 0:
        assert np.abs(dropped - kept).max() > 1e-6  # far above the 1e-10 agreement above
    else:
        np.testing.assert_allclose(dropped, kept, rtol=1e-10, atol=1e-12)
    # the row of stored zeros only: b = bias * sum y, ridge with nnz = its stored count
    u, s, e = 4, X.indptr[4], X.indptr[5]
    Y = other[X.indices[s:e]]
    A = alpha0 * other.T @ other + row_reg(e - s, X.shape[1], alpha0, reg, nu) * np.eye(K)
    b = (alpha0 if loss == "ORIGINAL" else 0.0) * Y.sum(axis=0)
    np.testing.assert_allclose(got[u], np.linalg.solve(A, b), rtol=1e-10, atol=1e-12)
