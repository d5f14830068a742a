"""TEST INFRASTRUCTURE ONLY -- textbook scalar ILU(0) (Saad, Iterative Methods for Sparse Linear Systems, alg. 10.4, IKJ variant) in a
given elimination order, NumPy.  It is the checker for csrc/pilu.cu: PETSc's default preconditioner for the reference's
snes_ksp_type = 'tfqmr' (NavierStokes/NavierStokesChannelFlow.py:282-291) is a point ILU(0) on the AIJ matrix of the mixed space; the
library factorises it in a multicolour order, and this file restates that factorisation for a CSR matrix in any numbering.

Rows are eliminated in the order (colour, row); within a colour no two rows share an entry, so that order does not change the
factor.  Only the first n = len(colour) rows and columns take part: other ranks' columns are dropped (block Jacobi over the ranks)."""
import numpy as np


def pilu0(indptr, indices, vals, colour):
    """Factorise.  Returns (order, L, U, udiag): L[i] / U[i] = (columns, values) of row i's entries eliminated before / after it
    (L with the multipliers a_ik / u_kk), udiag[i] = u_ii.  Raises ZeroDivisionError naming the row of a zero pivot."""
    colour = np.asarray(colour)
    n = len(colour)
    order = np.lexsort((np.arange(n), colour))
    rank = np.empty(n, dtype=np.int64)
    rank[order] = np.arange(n)
    pos = -np.ones(n, dtype=np.int64)                        # column -> slot in the row being factorised
    L, U = [None] * n, [None] * n
    udiag = np.zeros(n)
    for i in order:
        b, e = indptr[i], indptr[i + 1]
        keep = indices[b:e] < n
        cols = np.asarray(indices[b:e][keep], dtype=np.int64)
        w = np.array(vals[b:e][keep], dtype=np.float64)
        pos[cols] = np.arange(len(cols))
        rk = rank[cols]
        earlier = np.flatnonzero(rk < rank[i])
        for t in earlier[np.argsort(rk[earlier])]:           # k in elimination order
            k = cols[t]
            w[t] /= udiag[k]                                 # a_ik /= u_kk
            uc, uv = U[k]                                    # a_ij -= a_ik u_kj for the later j of row k that are in row i's pattern
            p = pos[uc]
            m = p >= 0
            w[p[m]] -= w[t] * uv[m]
        pos[cols] = -1
        d = np.flatnonzero(cols == i)
        udiag[i] = w[d[0]] if len(d) else 0.0
        if udiag[i] == 0.0 or not np.isfinite(udiag[i]):
            raise ZeroDivisionError(f"zero pivot in row {i}")
        L[i] = (cols[earlier], w[earlier])
        later = rk > rank[i]
        U[i] = (cols[later], w[later])
    return order, L, U, udiag


def apply(factor, r):
    """z = U^-1 L^-1 r (unit lower factor) on the first n entries of r."""
    order, L, U, udiag = factor
    z = np.array(r[: len(udiag)], dtype=np.float64)
    for i in order:
        c, v = L[i]
        z[i] -= v @ z[c]
    for i in order[::-1]:
        c, v = U[i]
        z[i] = (z[i] - v @ z[c]) / udiag[i]
    return z
