"""The NumPy restatement of point evaluation / non-matching interpolation (oracle/interp_ref.py) that the GPU tests compare against:
polynomial reproduction, the lower cell on a shared face, and the extrapolation rule outside the mesh."""
import numpy as np
import pytest

from oracle import interp_ref as R
from stabilized_navier_stokes_flow_fenicsx_b200 import mesh as M


def poly_state(sp):
    """velocity of degree vdeg and linear pressure, sampled at the dof nodes"""
    X, c, gd = sp.dof_x, sp.dof_comp, sp.mesh.gdim
    x, y, z = X[:, 0], X[:, 1], X[:, 2]
    lin = [1.0 + 2.0 * x - y + 0.5 * z, -0.5 + x + 3.0 * y - z, 0.25 - x + y + 2.0 * z]
    quad = [lin[0] + x * y - 2.0 * z * z, lin[1] + x * x - y * z, lin[2] + 3.0 * x * z - y * y]
    vel = quad if sp.vdeg == 2 else lin
    return np.select([c == k for k in range(gd)] + [c == gd], vel[:gd] + [2.0 - x + 0.3 * y + 0.7 * z])


def poly_at(points, gd, vdeg):
    x, y, z = points[:, 0], points[:, 1], points[:, 2] if gd == 3 else 0.0 * points[:, 0]
    lin = [1.0 + 2.0 * x - y + 0.5 * z, -0.5 + x + 3.0 * y - z, 0.25 - x + y + 2.0 * z]
    quad = [lin[0] + x * y - 2.0 * z * z, lin[1] + x * x - y * z, lin[2] + 3.0 * x * z - y * y]
    vel = quad if vdeg == 2 else lin
    return np.column_stack(vel[:gd] + [2.0 - x + 0.3 * y + 0.7 * z])


@pytest.mark.parametrize("gd,vdeg", [(3, 1), (3, 2), (2, 1), (2, 2)])
def test_restatement_reproduces_global_polynomials(gd, vdeg):
    m = M.duct_mesh(2, 4) if gd == 3 else M.create_rectangle_tris(4, 5)
    sp = M.mixed_space(m, vdeg)
    src = R.Source(m.x, m.cells, sp.dofmap, vdeg, poly_state(sp))
    rng = np.random.default_rng(0)
    lo, hi = m.x.min(axis=0), m.x.max(axis=0)
    pts = lo + (hi - lo) * rng.uniform(0.0, 1.0, size=(60, 3))
    vals, codes = src.eval(pts)
    assert np.all(codes >= 0)
    assert np.abs(vals - poly_at(pts, gd, vdeg)).max() < 1e-12
    # interpolation onto a non-nested mesh of the same domain, P1 -> P2 allowed
    md = M.duct_mesh(3, 5) if gd == 3 else M.create_rectangle_tris(3, 7)
    spd = M.mixed_space(md, 2)
    w, ne, no = R.interpolate(src, md.x, md.cells, spd.dofmap, 2, spd.n_dofs)
    assert ne == 0 and no == 0
    exact = poly_at(spd.dof_x, gd, vdeg)[np.arange(spd.n_dofs), spd.dof_comp]
    assert np.abs(w - exact).max() < 1e-12


def test_point_on_a_shared_face_goes_to_the_lower_cell():
    m = M.duct_mesh(1, 1)
    src = R.Source(m.x, m.cells)
    cells = m.cells.astype(np.int64)
    found = 0
    for a in range(len(cells)):
        for b in range(a + 1, len(cells)):
            shared = np.intersect1d(cells[a], cells[b])
            if shared.size != 3:
                continue
            p = m.x[shared].mean(axis=0)
            assert (src.bary(p, np.array([a, b])) >= -1e-12).all()   # both cells hold the centroid of their common face
            assert src.locate(p) == a
            found += 1
    assert found >= 5
    # a vertex shared by every cell of the box
    assert src.locate(m.x[m.cells[0, 0]]) == 0


def test_outside_points_take_the_nearest_cell_within_padding():
    m = M.create_rectangle_tris(1, 1)             # cell 0 = (v0, v1, v3), cell 1 = (v0, v2, v3) on the unit square
    src = R.Source(m.x, m.cells)
    assert src.locate(np.array([1.5, 0.25, 0.0]), padding=1.0) == -2 - 0      # beyond the edge x = 1 of cell 0
    assert src.locate(np.array([-0.5, 0.75, 0.0]), padding=1.0) == -2 - 1     # beyond the edge x = 0 of cell 1
    assert src.locate(np.array([1.5, 1.5, 0.0]), padding=1.0) == -2 - 0       # the corner v3 is in both: the lower cell
    assert src.locate(np.array([1.5, 0.25, 0.0]), padding=0.4) == -1          # distance 0.5 > padding
    assert src.locate(np.array([1.5, 0.25, 0.0]), padding=0.5) == -2 - 0      # distance == padding is accepted
    assert src.locate(np.array([1.5, 0.25, 0.0])) == -1                        # padding 0: outside
    d = src.cell_dist(np.array([1.5, 2.0, 0.0]))
    assert np.allclose(d, [np.hypot(0.5, 1.0), np.hypot(0.5, 1.0)])
    # tetrahedra: distance to a face, to an edge and to a vertex of the unit cube
    mt = M.create_box_tets((1, 1, 1))
    st = R.Source(mt.x, mt.cells)
    assert np.isclose(st.cell_dist(np.array([0.5, 0.5, 1.25])).min(), 0.25)
    assert np.isclose(st.cell_dist(np.array([1.3, 0.5, 1.4])).min(), 0.5)
    assert np.isclose(st.cell_dist(np.array([1.2, 1.2, 1.2])).min(), np.sqrt(3 * 0.04))
    code = st.locate(np.array([1.2, 1.2, 1.2]), padding=0.5)
    assert code == -2 - 0                                                    # every tet holds the v0-v7 diagonal end v7
    # an extrapolated value is the nearest cell's polynomial at the point
    sp = M.mixed_space(m, 1)
    w = poly_state(sp)
    src = R.Source(m.x, m.cells, sp.dofmap, 1, w)
    vals, codes = src.eval(np.array([[1.5, 0.25, 0.0], [3.0, 0.25, 0.0]]), padding=1.0)
    assert list(codes) == [-2, -1]
    assert np.allclose(vals[0], poly_at(np.array([[1.5, 0.25, 0.0]]), 2, 1)[0]) and np.all(vals[1] == 0.0)
