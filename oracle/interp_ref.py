"""TEST INFRASTRUCTURE ONLY -- NumPy restatement of the point evaluation and non-matching interpolation of csrc/locate.cu
(nsgpu_eval / nsgpu_interpolate; dolfinx Function.eval / Function.interpolate_nonmatching in the reference).

Brute force over every cell, with the library's rules:
  1. inside: the lowest-numbered cell whose barycentric coordinates are all >= -tol           -> code c
  2. only if no cell passed and padding > 0: the cell at the smallest distance from p to the closed cell (ties to the lower
     cell number), accepted when that distance is <= padding; its polynomials are evaluated at p -> code -2 - c
  3. otherwise outside: value 0                                                                 -> code -1
Distances: tetrahedra = min over the faces of the point-to-triangle distance (plane distance when p projects inside the face,
else the nearest edge), triangles = min over the edges; an edge is taken with its end points in ascending node order.
Basis: mixed_element([P_k^gdim, P1]) in dolfinx layout -- P2 vertices first, then edges in basix order.
"""
import numpy as np

TET_EDGES = np.array([[2, 3], [1, 3], [1, 2], [0, 3], [0, 2], [0, 1]])
TRI_EDGES = np.array([[1, 2], [0, 2], [0, 1]])
TET_FACES = np.array([[1, 2, 3], [0, 2, 3], [0, 1, 3], [0, 1, 2]])


class Source:
    """A mixed function: mesh (x (n, 3), cells (nc, gdim + 1)), dofmap (caller numbering), velocity degree and dof values w."""

    def __init__(self, x, cells, dofmap=None, vdeg=1, w=None):
        self.x = np.asarray(x, dtype=np.float64)
        self.cells = np.asarray(cells, dtype=np.int64)
        self.gd = self.cells.shape[1] - 1
        self.dofmap = None if dofmap is None else np.asarray(dofmap, dtype=np.int64)
        self.vdeg = vdeg
        self.w = None if w is None else np.asarray(w, dtype=np.float64)
        gd = self.gd
        self.x0 = self.x[self.cells[:, 0], :gd]
        J = np.stack([self.x[self.cells[:, a + 1], :gd] - self.x0 for a in range(gd)], axis=2)   # J[c, i, a]
        self.K = np.linalg.inv(J)                                                               # K[c, a, i]

    def bary(self, p, cells=None):
        K, x0 = (self.K, self.x0) if cells is None else (self.K[cells], self.x0[cells])
        lam = np.einsum("cai,ci->ca", K, np.asarray(p, dtype=np.float64)[None, : self.gd] - x0)
        return np.concatenate([1.0 - lam.sum(axis=1, keepdims=True), lam], axis=1)

    def cell_dist(self, p):
        """distance from p to every closed cell (as the library computes it for points outside)"""
        p = np.asarray(p, dtype=np.float64)[: self.gd]
        if self.gd == 2:
            return np.sqrt(np.min([_seg_d2(self.x[:, :2], self.cells[:, i], self.cells[:, j], p) for i, j in TRI_EDGES], axis=0))
        return np.sqrt(np.min([_tri_d2(self.x, self.cells[:, f[0]], self.cells[:, f[1]], self.cells[:, f[2]], p) for f in TET_FACES], axis=0))

    def locate(self, p, tol=1e-12, padding=0.0):
        lam = self.bary(p)
        inside = np.flatnonzero((lam >= -tol).all(axis=1))
        if inside.size:
            return int(inside[0])
        if padding > 0.0:
            d = self.cell_dist(p)
            c = int(np.flatnonzero(d == d.min())[0])
            if d[c] <= padding:
                return -2 - c
        return -1

    def eval_cell(self, c, p):
        gd = self.gd
        lam = self.bary(p, np.array([c]))[0]
        if self.vdeg == 1:
            phi = lam
        else:
            edges = TET_EDGES if gd == 3 else TRI_EDGES
            phi = np.concatenate([lam * (2.0 * lam - 1.0), 4.0 * lam[edges[:, 0]] * lam[edges[:, 1]]])
        nvn = phi.size
        dm = self.dofmap[c]
        out = np.empty(gd + 1)
        for k in range(gd):
            out[k] = phi @ self.w[dm[gd * np.arange(nvn) + k]]
        out[gd] = lam @ self.w[dm[gd * nvn + np.arange(gd + 1)]]
        return out

    def eval(self, points, tol=1e-12, padding=0.0):
        points = np.asarray(points, dtype=np.float64).reshape(-1, 3)
        values = np.zeros((points.shape[0], self.gd + 1))
        codes = np.empty(points.shape[0], dtype=np.int64)
        for i, p in enumerate(points):
            codes[i] = code = self.locate(p, tol, padding)
            if code != -1:
                values[i] = self.eval_cell(code if code >= 0 else -2 - code, p)
        return values, codes


def nodes(x, cells, dofmap, vdeg):
    """Destination nodes, each once: (coordinates (m, 3), cell, local node) with the lowest (cell, local node) per node.  A node is
    named by its first velocity dof; local nodes are the vertices, then for P2 the edges in basix order."""
    x = np.asarray(x, dtype=np.float64)
    cells = np.asarray(cells, dtype=np.int64)
    dofmap = np.asarray(dofmap, dtype=np.int64)
    gd = cells.shape[1] - 1
    nvn = gd + 1 if vdeg == 1 else (10 if gd == 3 else 6)
    key = dofmap[:, gd * np.arange(nvn)]                              # (nc, nvn), c-major: the first occurrence is the lowest (c, node)
    _, first = np.unique(key.ravel(), return_index=True)
    c, node = first // nvn, first % nvn
    edges = TET_EDGES if gd == 3 else TRI_EDGES
    pts = np.empty((first.size, 3))
    v = node < gd + 1
    pts[v] = x[cells[c[v], node[v]]]
    e = edges[node[~v] - (gd + 1)]
    pts[~v] = 0.5 * (x[cells[c[~v], e[:, 0]]] + x[cells[c[~v], e[:, 1]]])
    if gd == 2:
        pts[:, 2] = 0.0
    return pts, c, node


def interpolate(src, x, cells, dofmap, vdeg, n_dofs, tol=1e-12, padding=0.0):
    """Function.interpolate_nonmatching of src onto the destination space: (w, n_extrapolated, n_outside)."""
    dofmap = np.asarray(dofmap, dtype=np.int64)
    gd = src.gd
    nvn = gd + 1 if vdeg == 1 else (10 if gd == 3 else 6)
    pts, c, node = nodes(x, cells, dofmap, vdeg)
    values, codes = src.eval(pts, tol, padding)
    w = np.zeros(n_dofs)
    for k in range(gd):
        w[dofmap[c, gd * node + k]] = values[:, k]
    v = node < gd + 1
    w[dofmap[c[v], gd * nvn + node[v]]] = values[v, gd]
    return w, int((codes <= -2).sum()), int((codes == -1).sum())


def _canonical(ia, ib):
    return np.minimum(ia, ib), np.maximum(ia, ib)


def _seg_d2(x, ia, ib, p):
    ia, ib = _canonical(ia, ib)
    a, b = x[ia], x[ib]
    ab, ap = b - a, p[None, :] - a
    den = (ab * ab).sum(axis=1)
    t = np.where(den > 0.0, (ap * ab).sum(axis=1) / np.where(den > 0.0, den, 1.0), 0.0)
    q = np.where((t <= 0.0)[:, None], a, np.where((t >= 1.0)[:, None], b, a + t[:, None] * ab))
    return ((p[None, :] - q) ** 2).sum(axis=1)


def _tri_d2(x, ia, ib, ic, p):
    a, b, c = x[ia], x[ib], x[ic]
    n = np.cross(b - a, c - a)
    nn = (n * n).sum(axis=1)
    s0 = (np.cross(b - a, p - a) * n).sum(axis=1)
    s1 = (np.cross(c - b, p - b) * n).sum(axis=1)
    s2 = (np.cross(a - c, p - c) * n).sum(axis=1)
    proj = (nn > 0.0) & (s0 >= 0.0) & (s1 >= 0.0) & (s2 >= 0.0)
    dn = ((p - a) * n).sum(axis=1)
    plane = dn * dn / np.where(nn > 0.0, nn, 1.0)
    edge = np.minimum(_seg_d2(x, ia, ib, p), np.minimum(_seg_d2(x, ib, ic, p), _seg_d2(x, ic, ia, p)))
    return np.where(proj, plane, edge)
