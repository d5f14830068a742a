"""The NumPy restatement of the boundary functionals (oracle/facet_ref.py) against closed forms and the DFG 2D-1 reference constants,
and gmsh_io.facet_integration_domain (the (cell, local facet, tag) triples of ds(subdomain_data=facet_tags)).  CPU only."""
import numpy as np
import pytest

import _pins as P
from oracle import facet_ref as R
from stabilized_navier_stokes_flow_fenicsx_b200 import gmsh_io as G
from stabilized_navier_stokes_flow_fenicsx_b200 import mesh as M

DUCT_BOX = (np.array([0.0, -0.5, -0.5]), np.array([4.0, 0.5, 0.5]))
RECT_BOX = (np.array([0.0, 0.0]), np.array([1.0, 1.0]))


def box_of(m):
    return DUCT_BOX if m.gdim == 3 else RECT_BOX


def face_tagged(m):
    """every exterior facet with the tag of its box face: 2 * axis + (0 at the low side, 1 at the high side)"""
    lo, hi = box_of(m)
    bf = G.boundary_facets(m)
    cen = m.x[bf][:, :, : m.gdim].mean(axis=1)
    tags = np.full(len(bf), -1, dtype=np.int32)
    for a in range(m.gdim):
        tags[np.abs(cen[:, a] - lo[a]) < 1e-12] = 2 * a
        tags[np.abs(cen[:, a] - hi[a]) < 1e-12] = 2 * a + 1
    assert (tags >= 0).all()
    return (bf,) + G.facet_integration_domain(m, bf, tags)


class Field:
    """u_i = a_i + B_ij x_j (+ Q_ijk x_j x_k for vdeg 2), p = p0 + g . x with seeded coefficients"""

    def __init__(self, gd, vdeg, seed=7):
        rng = np.random.default_rng(seed)
        self.gd, self.a, self.B = gd, rng.uniform(-1, 1, gd), rng.uniform(-1, 1, (gd, gd))
        self.Q = rng.uniform(-1, 1, (gd, gd, gd)) if vdeg == 2 else np.zeros((gd, gd, gd))
        self.p0, self.g = rng.uniform(-1, 1), rng.uniform(-1, 1, gd)

    def u(self, x):
        return self.a + x @ self.B.T + np.einsum("ijk,...j,...k->...i", self.Q, x, x)

    def grad(self, x):
        return self.B + np.einsum("ijk,...k->...ij", self.Q + self.Q.transpose(0, 2, 1), x)

    def p(self, x):
        return self.p0 + x @ self.g

    def state(self, sp):
        X = sp.dof_x[:, : self.gd]
        vals = np.concatenate([self.u(X), self.p(X)[:, None]], axis=1)
        return vals[np.arange(sp.n_dofs), sp.dof_comp]


def closed_form_rows(f, box):
    """exact rows [area, u.n, p n, (grad u) n, (grad u)^T n] of every box face (tensor 3-point Gauss, exact for degree <= 5)"""
    lo, hi = box
    gd = len(lo)
    s, wt = np.polynomial.legendre.leggauss(3)
    rows = np.zeros((2 * gd, 2 + 3 * gd))
    for a in range(gd):
        other = [b for b in range(gd) if b != a]
        grids = np.meshgrid(*[0.5 * (lo[b] + hi[b]) + 0.5 * (hi[b] - lo[b]) * s for b in other], indexing="ij")
        wq = np.prod(np.meshgrid(*[0.5 * (hi[b] - lo[b]) * wt for b in other], indexing="ij"), axis=0)
        for side, xa, sign in ((0, lo[a], -1.0), (1, hi[a], 1.0)):
            x = np.zeros(grids[0].shape + (gd,))
            x[..., a] = xa
            for k, b in enumerate(other):
                x[..., b] = grids[k]
            n = np.zeros(gd); n[a] = sign
            u, gu, p = f.u(x), f.grad(x), f.p(x)
            W = wq[..., None]
            r = rows[2 * a + side]
            r[0] = wq.sum()
            r[1] = (wq * (u @ n)).sum()
            r[2:2 + gd] = (W * p[..., None] * n).reshape(-1, gd).sum(axis=0)
            r[2 + gd:2 + 2 * gd] = (W * (gu @ n)).reshape(-1, gd).sum(axis=0)
            r[2 + 2 * gd:] = (W * np.einsum("...ji,j->...i", gu, n)).reshape(-1, gd).sum(axis=0)
    return rows


MESHES = {"duct": lambda: M.duct_mesh(3, 7), "rect": lambda: M.create_rectangle_tris(7, 5)}


@pytest.mark.parametrize("vdeg", [1, 2])
@pytest.mark.parametrize("mesh", list(MESHES))
def test_restatement_reproduces_closed_form_face_integrals(mesh, vdeg):
    m = MESHES[mesh]()
    sp = M.mixed_space(m, vdeg)
    f = Field(m.gdim, vdeg)
    _, fc, fl, ft = face_tagged(m)
    got = R.facet_integrals(m.x, m.cells, sp.dofmap, vdeg, f.state(sp), fc, fl, ft)
    ref = closed_form_rows(f, box_of(m))
    assert np.abs(got - ref).max() <= 1e-13 * np.abs(ref).max(), np.abs(got - ref).max()


def test_restatement_gives_the_dfg_2d_1_drag_and_lift(oracle):
    """the table of the boundary-functional design note: sigma-form within 2.5 % / 1 %, reaction within the existing pin"""
    m, sp, bcs, obstacle = P.dfg_problem()
    be = P.OracleBackend(oracle, m, sp, bcs)
    r = P.dfg_solve(be, sp, bcs, obstacle)
    n_cyl = m.meta["n_cyl"]
    bf = G.boundary_facets(m)
    cyl = bf[(bf < n_cyl).all(axis=1)]
    fc, fl, ft = G.facet_integration_domain(m, cyl, np.zeros(len(cyl), dtype=np.int32))
    scale = 2.0 / (0.1 * 0.2 ** 2)
    nu = 1e-3
    rows = R.facet_integrals(m.x, m.cells, sp.dofmap, 1, r["w"], fc, fl, ft)[0]
    force = -(nu * (rows[4:6] + rows[6:8]) - rows[2:4])
    cd, cl = scale * force
    assert abs(rows[0] - 2 * np.pi * 0.05) < 1e-3                           # the polygon's perimeter
    assert abs(cd / P.DFG_CD - 1.0) < 0.025 and abs(cl / P.DFG_CL - 1.0) < 0.01, (cd, cl)
    Ru = be.unconstrained_residual(dict(flavour=1, nu=nu), r["w"])
    react = R.reaction(Ru, m.cells, sp.dofmap, 1, fc, fl, ft)[0]
    dofs, _ = R.tagged_velocity_dofs(m.cells, sp.dofmap, 1, fc, fl, ft)[0]
    assert np.array_equal(dofs, np.sort(obstacle))                         # topological selection = the geometric one
    assert np.allclose(-scale * react, [r["cd"], r["cl"]], rtol=1e-12, atol=0)
    assert abs(-scale * react[0] / P.DFG_CD - 1.0) < 0.01 and abs(-scale * react[1] / P.DFG_CL - 1.0) < 0.05


@pytest.mark.parametrize("mesh", list(MESHES))
def test_facet_integration_domain_round_trips_through_msh(tmp_path, mesh):
    m = MESHES[mesh]()
    bf, fc, fl, ft = face_tagged(m)
    loc = ((1, 2, 3), (0, 2, 3), (0, 1, 3), (0, 1, 2)) if m.gdim == 3 else ((1, 2), (0, 2), (0, 1))
    faces = np.array([m.cells[c, loc[l]] for c, l in zip(fc, fl)])
    assert np.array_equal(np.sort(faces, axis=1), np.sort(bf, axis=1))    # local facet i is the facet opposite vertex i
    path = tmp_path / "m.msh"
    G.write_msh(path, m, bf, ft + 1)
    m2, _, f2, ft2, _ = G.read_msh(path)
    c2, l2, t2 = G.facet_integration_domain(m2, f2, ft2 - 1)
    assert np.array_equal(m2.cells, m.cells)
    key = lambda c, l, t: sorted(zip(c.tolist(), l.tolist(), t.tolist()))   # noqa: E731
    assert key(c2, l2, t2) == key(fc, fl, ft)


def test_facet_integration_domain_rejects_interior_and_unknown_facets():
    m = M.duct_mesh(2, 3)
    bf = G.boundary_facets(m)
    faces = [np.sort(m.cells[0, f]) for f in ((1, 2, 3), (0, 2, 3), (0, 1, 3), (0, 1, 2))]
    interior = next(f for f in faces if not (bf == f).all(axis=1).any())
    with pytest.raises(ValueError, match="two cells"):
        G.facet_integration_domain(m, np.vstack([bf[:3], interior]), np.zeros(4, dtype=np.int32))
    with pytest.raises(ValueError, match="no cell"):
        G.facet_integration_domain(m, np.array([[0, 1, m.n_vertices - 1]]), np.zeros(1, dtype=np.int32))
