"""The properties the kernel-path tests (test_kernel_paths_gpu.py) rely on, checked on the CPU: the meshes reach the topology
branches they are there for, orientations are mixed, the UGN state spans both LSIC branches."""
import numpy as np
import pytest

import _meshes as MS
from stabilized_navier_stokes_flow_fenicsx_b200 import mesh as M


def test_delaunay_tets_reach_the_gather_overflow_and_the_incidence_fetch():
    m = MS.delaunay_tets(14, seed=3)
    e = MS.edge_cell_counts(m.cells)
    v = MS.vertex_cell_counts(m.cells)
    assert e.max() > 8 and (e > 8).sum() > 100             # p1tet_ws: gather lists longer than the 8 inline entries
    assert (v > 3 * MS.NENT[(3, 2)]).sum() > 50             # rowown P2 tets: incidences beyond 3 NENT come from memory
    assert v.max() <= 63                                    # ... and the factorised P1-P1 plan still applies
    vol = MS.signed_measure(m)
    assert np.abs(vol).min() > 0 and (vol < 0).any() and (vol > 0).any()
    assert np.isclose(np.abs(vol).sum() / 6, 1.0)           # the cells tile the unit cube


def test_delaunay_tris_tile_the_square():
    m = MS.delaunay_tris(40, seed=0)
    a = MS.signed_measure(m)
    assert np.abs(a).min() > 0 and np.isclose(np.abs(a).sum() / 2, 1.0)
    assert MS.vertex_cell_counts(m.cells).max() > 3 * MS.NENT[(2, 1)]


def test_fan_mesh_has_a_vertex_in_more_than_63_cells():
    m = MS.fan_tets(40)
    v = MS.vertex_cell_counts(m.cells)
    assert v[0] == 2 * 40 - 4 and v.max() > 63
    vol = MS.signed_measure(m)
    assert np.abs(vol).min() > 0 and np.isclose(np.abs(vol).sum() / 6, 4.0 ** 3)
    bcs = MS.box_bcs(M.mixed_space(m, 1), lo=-2.0, hi=2.0)
    assert all(len(d) for d, _ in bcs)


@pytest.mark.parametrize("gd", [2, 3])
def test_structured_meshes_are_flipped_and_jittered(gd):
    m = MS.structured(gd, 3 if gd == 3 else 6, seed=1)
    vol = MS.signed_measure(m)
    assert 0.2 < (vol < 0).mean() < 0.5 and np.abs(vol).min() > 0
    assert np.isclose(np.abs(vol).sum(), 2.0 if gd == 2 else 6.0)
    assert len(np.unique(np.round(np.abs(vol), 12))) > 10   # not just the few shapes of the undisturbed lattice


@pytest.mark.parametrize("gd", [2, 3])
def test_flipped_p2_edge_dofs_follow_the_vertex_order(gd):
    """mixed_space after the flip: each local edge dof sits at the midpoint of the local vertices the edge is made of."""
    m = MS.structured(gd, 2, seed=3)
    sp = M.mixed_space(m, 2)
    edges = M.TET_EDGES if gd == 3 else M.TRI_EDGES
    for e, (a, b) in enumerate(edges):
        mid = 0.5 * (m.x[m.cells[:, a]] + m.x[m.cells[:, b]])
        np.testing.assert_array_equal(sp.dof_x[sp.dofmap[:, gd * (gd + 1 + e)]], mid)


@pytest.mark.parametrize("gd,vd", [(2, 1), (2, 2), (3, 1), (3, 2)])
def test_reynolds_split_state_spans_both_lsic_branches(gd, vd):
    sp = M.mixed_space(MS.structured(gd, 3 if gd == 3 else 6, seed=10 * gd + vd), vd)
    nu = 0.01
    re = MS.cell_reynolds(sp, MS.reynolds_split_state(sp, nu), nu)
    assert (re <= 3).mean() >= 0.1 and (re > 3).mean() >= 0.1


@pytest.mark.parametrize("gd,vd", [(2, 1), (2, 2), (3, 1), (3, 2)])
def test_centroid_speed_of_a_linear_field_is_exact(gd, vd):
    sp = M.mixed_space(MS.structured(gd, 2, seed=0), vd)
    w = np.where(sp.dof_comp < gd, 1.0 + sp.dof_x[:, 0] + 2 * sp.dof_x[:, 1], 0.0)
    c = sp.mesh.x[sp.mesh.cells].mean(axis=1)
    want = np.sqrt(gd) * (1.0 + c[:, 0] + 2 * c[:, 1])
    np.testing.assert_allclose(MS.centroid_speed(sp, w), want, rtol=1e-13)


@pytest.mark.parametrize("gd,vd", [(2, 1), (2, 2), (3, 1), (3, 2)])
def test_coop_boundary_sub_meshes(gd, vd):
    cpb = MS.coop_cells_per_block(gd, vd)
    assert cpb == 256 // MS.ndofs_cell(gd, vd)
    for d in (-1, 0, 1):
        m = MS.take_cells(MS.structured(gd, 4 if gd == 3 else 8, seed=4), 3 * cpb + d)
        assert m.n_cells == 3 * cpb + d and m.cells.max() == m.n_vertices - 1
        assert len(np.unique(m.cells)) == m.n_vertices


def test_boundary_sets_hold_rim_dofs_twice_and_whole_cells():
    sp = M.mixed_space(MS.structured(3, 3, seed=0), 2)
    bcs = MS.box_bcs(sp)
    mult = np.zeros(sp.n_dofs, dtype=int)
    for d, _ in bcs:
        np.add.at(mult, d, 1)
    assert mult.max() == 2
    cb = MS.cell_bcs(sp, seed=1)
    assert (sp.dof_comp[cb[0][0]] == 3).any() and np.isin(cb[1][0], cb[0][0]).all()
    w = MS.dirichlet_only_state(sp, bcs)
    assert np.count_nonzero(w) > 0 and np.all(w[np.setdiff1d(np.arange(sp.n_dofs), np.concatenate([d for d, _ in bcs]))] == 0)
