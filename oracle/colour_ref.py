"""TEST INFRASTRUCTURE ONLY -- the Jones-Plassmann colouring of csrc/colour.cu restated in NumPy.  Both multicolour ILU(0)
preconditioners order their elimination by it (pc = 5 on the vertices of a vertex-blocked matrix, pc = 6 on the dofs with the
velocity class first); their exported colours must equal these exactly."""
import numpy as np


def hash32(x):
    x = np.asarray(x, dtype=np.uint32).copy()                # uint32 arithmetic wraps as on the device
    x ^= x >> np.uint32(16); x *= np.uint32(0x7feb352d); x ^= x >> np.uint32(15); x *= np.uint32(0x846ca68b); x ^= x >> np.uint32(16)
    return x


def colour(indptr, indices, n, shift=0, cls=None):
    """Colours of nodes 0..n-1.  Node e's neighbours are the columns j of CSR row e << shift, as j >> shift, other than e and below n.
    cls (0 / 1 per node): class 0 first, then class 1 from the first colour after class 0's, each class among its own neighbours."""
    indptr, indices = np.asarray(indptr), np.asarray(indices)
    cls = np.zeros(n, dtype=np.int64) if cls is None else np.asarray(cls, dtype=np.int64)
    nbrs = []
    for e in range(n):
        j = indices[indptr[e << shift]:indptr[(e << shift) + 1]].astype(np.int64) >> shift
        j = j[(j < n) & (j != e)]
        nbrs.append(j[cls[j] == cls[e]])
    h = hash32(np.arange(n)).astype(np.int64)
    col = np.full(n, -1, dtype=np.int64)
    base = 0
    for c in range(cls.max() + 1):
        while np.any(col[cls == c] < 0):
            prev = col.copy()                                # decisions on the colours at the start of the round
            for e in np.flatnonzero((cls == c) & (prev < 0)):
                j = nbrs[e]
                u = j[prev[j] < 0]
                if np.any((h[u] > h[e]) | ((h[u] == h[e]) & (u > e))):
                    continue                                 # an uncoloured neighbour goes first
                used = set(prev[j].tolist())
                k = base
                while k in used:
                    k += 1
                col[e] = k
        base = col.max() + 1
    return col
