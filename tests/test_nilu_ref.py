"""The restatements tests/test_nilu_gpu.py holds csrc/nilu.cu (pc = 7, ILU(0) in the caller's order) against, on their own (no GPU):
oracle/pilu_ref.pilu0 with colour = arange(n) is ILU(0) in natural order, and tests/_nilu_ref.depth counts the sweeps' levels."""
import numpy as np
import pytest
import scipy.sparse as sps

import _nilu_ref
from oracle import pilu_ref


def _dense_ilu0(A):
    """ILU(0), IKJ variant (Saad alg. 10.4) on a dense array, rows in natural order, written out longhand: the unit lower factor's
    multipliers below the diagonal and U on and above it, both on the nonzero pattern of A."""
    n = A.shape[0]
    nz = A != 0
    W = A.astype(np.float64).copy()
    for i in range(1, n):
        for k in range(i):
            if not nz[i, k]:
                continue
            W[i, k] = W[i, k] / W[k, k]
            for j in range(k + 1, n):
                if nz[i, j]:
                    W[i, j] = W[i, j] - W[i, k] * W[k, j]
    return W


def _random_pattern_matrix(n, density, seed):
    rng = np.random.default_rng(seed)
    A = sps.random(n, n, density=density, random_state=rng, format="csr")
    A = A + A.T + sps.diags(rng.uniform(n, 2 * n, n))          # symmetric pattern, diagonally dominant: no pivot breaks down
    A = sps.csr_matrix(A)
    A.sort_indices()
    return A


@pytest.mark.parametrize("n,density,seed", [(6, 0.4, 0), (17, 0.2, 1), (40, 0.08, 2), (40, 0.3, 3)])
def test_pilu0_in_natural_order_is_the_dense_ikj_ilu0(n, density, seed):
    A = _random_pattern_matrix(n, density, seed)
    W = _dense_ilu0(A.toarray())
    order, L, U, udiag = pilu_ref.pilu0(A.indptr, A.indices, A.data, np.arange(n))
    assert np.array_equal(order, np.arange(n))
    for i in range(n):
        lc, lv = L[i]
        uc, uv = U[i]
        assert np.all(lc < i) and np.all(uc > i)
        np.testing.assert_allclose(lv, W[i, lc], rtol=1e-13, atol=0)
        np.testing.assert_allclose(uv, W[i, uc], rtol=1e-13, atol=0)
        assert udiag[i] == pytest.approx(W[i, i], rel=1e-13)
    r = np.random.default_rng(seed).standard_normal(n)
    Lm = np.tril(W, -1) * (A.toarray() != 0) + np.eye(n)
    Um = np.triu(W) * (A.toarray() != 0)
    np.testing.assert_allclose(pilu_ref.apply((order, L, U, udiag), r), np.linalg.solve(Um, np.linalg.solve(Lm, r)), rtol=1e-10)


def _with_diagonal(A):
    """CSR of A whose pattern holds the diagonal even where it is 0 (as the assembled Stokes pressure block does)."""
    r, c = np.nonzero((A != 0) | np.eye(len(A), dtype=bool))
    S = sps.coo_matrix((A[r, c], (r, c)), shape=A.shape).tocsr()
    S.sort_indices()
    return S


def test_pilu0_in_natural_order_names_the_first_zero_pivot():
    # rows 0, 1 fine; row 2 has a zero diagonal and no earlier neighbour that fills it; row 4 also has one
    A = np.array([[2., 1, 0, 0, 0], [1, 3, 0, 0, 0], [0, 0, 0, 1, 0], [0, 0, 1, 4, 1], [0, 0, 0, 1, 0]])
    S = _with_diagonal(A)
    with pytest.raises(ZeroDivisionError, match="zero pivot in row 2"):
        pilu_ref.pilu0(S.indptr, S.indices, S.data, np.arange(5))
    P = _with_diagonal(A[[3, 0, 1, 2, 4]][:, [3, 0, 1, 2, 4]])     # row 3 first: it fills the two zero pivots
    _, _, _, udiag = pilu_ref.pilu0(P.indptr, P.indices, P.data, np.arange(5))
    assert udiag[3] == pytest.approx(-0.25) and udiag[4] == pytest.approx(-0.25)   # 0 - (1 / 4) * 1


def _csr(dense):
    S = sps.csr_matrix(np.asarray(dense, dtype=float))
    S.sort_indices()
    return S.indptr, S.indices


def test_depth_of_hand_counted_cases():
    assert _nilu_ref.depth(*_csr(np.eye(4)), 4) == (1, 1)                       # diagonal: one level each way
    tri = np.eye(5) + np.eye(5, k=1) + np.eye(5, k=-1)
    assert _nilu_ref.depth(*_csr(tri), 5) == (5, 5)                             # tridiagonal: a chain
    arrow = np.eye(5); arrow[4, :] = 1; arrow[:, 4] = 1
    assert _nilu_ref.depth(*_csr(arrow), 5) == (2, 2)                           # arrow: 0..3 independent, 4 after (before) them
    lower_only = np.eye(4); lower_only[3, 0] = lower_only[2, 1] = 1
    assert _nilu_ref.depth(*_csr(lower_only), 4) == (2, 1)                      # a pattern entry counts for its own row only
    # red-black 1-D Laplacian: evens 0, 2, 4, then odds 1, 3 (positions 3, 4) -- each odd needs two evens: two levels
    rb = np.zeros((5, 5)); perm = [0, 2, 4, 1, 3]; pos = {v: p for p, v in enumerate(perm)}
    for v in range(5):
        for w in (v - 1, v, v + 1):
            if 0 <= w < 5:
                rb[pos[v], pos[w]] = 1
    assert _nilu_ref.depth(*_csr(rb), 5) == (2, 2)
    # other ranks' columns (>= n) are dropped
    ip, ix = _csr(np.hstack([np.eye(3), np.ones((3, 2))]))
    assert _nilu_ref.depth(ip, ix, 3) == (1, 1)
