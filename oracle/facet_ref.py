"""TEST INFRASTRUCTURE ONLY -- NumPy restatement of the boundary functionals of csrc/boundary.cu (nsgpu_facet_integrals /
nsgpu_reaction; dolfinx ds(subdomain_data=facet_tags) integrals and the reaction forces of the reference's drag / lift checks).

Facet integrals: per tag [area, int u.n, int p n, int (grad u) n, int (grad u)^T n], (grad u)_ij = du_i/dx_j.  The facet's normal
and measure come from its own vertices (cross product / segment length, oriented away from the opposite vertex), and the rule is
a different exact one than the library's: the interior 3-point rule (2/3, 1/6, 1/6) on triangle facets and 3-point Gauss on
segments -- both exact for the integrands at vdeg <= 2, so the two agree to rounding.  Only pairs of owned cells are integrated.

Reaction: the velocity dofs in the closure of the tagged facets (vertices, plus edges for P2; a dof on two tags counts for both),
summed per component over an unconstrained residual vector (OracleBackend.unconstrained_residual in tests/_pins.py).
"""
import numpy as np

TET_EDGES = np.array([[2, 3], [1, 3], [1, 2], [0, 3], [0, 2], [0, 1]])
TRI_EDGES = np.array([[1, 2], [0, 2], [0, 1]])


def _nodes(gd, vdeg):
    return gd + 1 if vdeg == 1 else (10 if gd == 3 else 6)


def _basis(lam, gl, gd, vdeg):
    """velocity basis values (f, nvn) and gradients (f, nvn, gd) at barycentric points lam (f, gd + 1); gl: (f, gd + 1, gd)"""
    if vdeg == 1:
        return lam, gl
    E = TET_EDGES if gd == 3 else TRI_EDGES
    N = np.concatenate([lam * (2 * lam - 1), 4 * lam[:, E[:, 0]] * lam[:, E[:, 1]]], axis=1)
    dV = (4 * lam - 1)[:, :, None] * gl
    dE = 4 * (lam[:, E[:, 0], None] * gl[:, E[:, 1]] + lam[:, E[:, 1], None] * gl[:, E[:, 0]])
    return N, np.concatenate([dV, dE], axis=1)


def facet_integrals(x, cells, dofmap, vdeg, w, fcell, flf, ftag, n_tags=None, n_cells_owned=None):
    """(n_tags, 2 + 3 gdim) rows; w and dofmap in the same numbering."""
    x = np.asarray(x, dtype=np.float64)
    cells = np.asarray(cells, dtype=np.int64)
    dofmap = np.asarray(dofmap, dtype=np.int64)
    w = np.asarray(w, dtype=np.float64)
    gd = cells.shape[1] - 1
    fcell, flf, ftag = (np.asarray(a, dtype=np.int64).ravel() for a in (fcell, flf, ftag))
    n_tags = int(ftag.max()) + 1 if n_tags is None else n_tags
    out = np.zeros((n_tags, 2 + 3 * gd))
    own = fcell < (len(cells) if n_cells_owned is None else n_cells_owned)
    c, lf, tg = fcell[own], flf[own], ftag[own]
    if not len(c):
        return out
    X = x[cells[c], :gd]                                                   # (f, gd + 1, gd)
    J = np.stack([X[:, a + 1] - X[:, 0] for a in range(gd)], axis=2)       # J[f, i, a]
    K = np.linalg.inv(J)                                                   # K[f, a, i] = d lam_{a+1} / dx_i
    gl = np.concatenate([-K.sum(axis=1, keepdims=True), K], axis=1)        # (f, gd + 1, gd)
    fv = np.array([[a for a in range(gd + 1) if a != i] for i in range(gd + 1)])[lf]   # facet vertices (f, gd)
    P = np.take_along_axis(X, fv[:, :, None], axis=1)                      # (f, gd, gd)
    opp = X[np.arange(len(c)), lf]
    if gd == 3:
        nv = np.cross(P[:, 1] - P[:, 0], P[:, 2] - P[:, 0])
        area = 0.5 * np.linalg.norm(nv, axis=1)
        pts, wts = [(2 / 3, 1 / 6, 1 / 6), (1 / 6, 2 / 3, 1 / 6), (1 / 6, 1 / 6, 2 / 3)], [1 / 3] * 3
    else:
        t = P[:, 1] - P[:, 0]
        nv = np.stack([t[:, 1], -t[:, 0]], axis=1)
        area = np.linalg.norm(t, axis=1)
        g = np.sqrt(3 / 5)
        pts = [((1 + s) / 2, (1 - s) / 2) for s in (-g, 0.0, g)]
        wts = [5 / 18, 8 / 18, 5 / 18]
    n = nv / np.linalg.norm(nv, axis=1, keepdims=True)
    n = np.where(((P[:, 0] - opp) * n).sum(axis=1, keepdims=True) < 0, -n, n)   # away from the opposite vertex
    nvn = _nodes(gd, vdeg)
    wc = w[dofmap[c]]
    U = wc[:, : gd * nvn].reshape(-1, nvn, gd)                            # (f, node, comp)
    Pn = wc[:, gd * nvn:]
    rows = np.zeros((len(c), 2 + 3 * gd))
    for q, wq in zip(pts, wts):
        lam = np.zeros((len(c), gd + 1))
        np.put_along_axis(lam, fv, np.broadcast_to(np.array(q), (len(c), gd)), axis=1)
        N, dN = _basis(lam, gl, gd, vdeg)
        u = np.einsum("fn,fnk->fk", N, U)
        gu = np.einsum("fnk,fnj->fkj", U, dN)                              # gu[f, i, j] = du_i / dx_j
        p = (lam * Pn).sum(axis=1)
        W = (wq * area)[:, None]
        rows[:, 0] += W[:, 0]
        rows[:, 1] += W[:, 0] * (u * n).sum(axis=1)
        rows[:, 2:2 + gd] += W * p[:, None] * n
        rows[:, 2 + gd:2 + 2 * gd] += W * np.einsum("fij,fj->fi", gu, n)
        rows[:, 2 + 2 * gd:] += W * np.einsum("fji,fj->fi", gu, n)
    np.add.at(out, tg, rows)
    return out


def tagged_velocity_dofs(cells, dofmap, vdeg, fcell, flf, ftag, n_tags=None):
    """per tag: (dofs, components) of the velocity dofs in the closure of its facets (all pairs, owned or ghost cells)"""
    cells = np.asarray(cells)
    dofmap = np.asarray(dofmap, dtype=np.int64)
    gd = cells.shape[1] - 1
    fcell, flf, ftag = (np.asarray(a, dtype=np.int64).ravel() for a in (fcell, flf, ftag))
    n_tags = int(ftag.max()) + 1 if n_tags is None else n_tags
    E = TET_EDGES if gd == 3 else TRI_EDGES
    on = [[a for a in range(gd + 1) if a != i] + ([gd + 1 + e for e in range(len(E)) if i not in E[e]] if vdeg == 2 else [])
          for i in range(gd + 1)]
    out = []
    for t in range(n_tags):
        sel = ftag == t
        d = [dofmap[fcell[sel][lf == flf[sel]][:, None], gd * np.array(on[lf])[None, :] + k].ravel()
             for lf in range(gd + 1) for k in range(gd)]
        comp = [np.full(d[lf * gd + k].size, k) for lf in range(gd + 1) for k in range(gd)]
        dofs, first = np.unique(np.concatenate(d), return_index=True)
        out.append((dofs, np.concatenate(comp)[first]))
    return out


def reaction(R, cells, dofmap, vdeg, fcell, flf, ftag, n_tags=None):
    """(n_tags, gdim): the residual R (unconstrained, same numbering as dofmap) summed over each tag's velocity dofs per component"""
    gd = np.asarray(cells).shape[1] - 1
    R = np.asarray(R, dtype=np.float64)
    lists = tagged_velocity_dofs(cells, dofmap, vdeg, fcell, flf, ftag, n_tags)
    out = np.zeros((len(lists), gd))
    for t, (dofs, comp) in enumerate(lists):
        for k in range(gd):
            out[t, k] = R[dofs[comp == k]].sum()
    return out
