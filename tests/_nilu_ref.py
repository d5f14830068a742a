"""Dependency depth of ILU(0) in natural order, NumPy: the checker of NSAssembler.nilu_depth (csrc/nilu.cu, pc = 7).

Row i of the forward sweep needs the rows k < i of its pattern, row i of the backward sweep the rows j > i; only the first n rows and
columns take part (other ranks' columns are dropped).  The depth of a sweep is its number of levels: 1 + the longest chain of such
dependencies, i.e. the number of rows on the longest path of its DAG."""
import numpy as np


def depth(indptr, indices, n):
    """(levels of the forward sweep, levels of the backward sweep) of the owned block of a CSR matrix, eliminated in row order."""
    lo = np.zeros(n, dtype=np.int64)
    up = np.zeros(n, dtype=np.int64)
    for i in range(n):
        c = np.asarray(indices[indptr[i]:indptr[i + 1]])
        c = c[c < i]
        lo[i] = 1 + (lo[c].max() if len(c) else 0)
    for i in range(n - 1, -1, -1):
        c = np.asarray(indices[indptr[i]:indptr[i + 1]])
        c = c[(c > i) & (c < n)]
        up[i] = 1 + (up[c].max() if len(c) else 0)
    return int(lo.max()), int(up.max())
