"""Boundary functionals on the device (csrc/boundary.cu: nsgpu_set_facets / nsgpu_facet_integrals / nsgpu_reaction) against closed
forms, the NumPy restatement (oracle/facet_ref.py), the host reaction of the DFG 2D-1 pin and the host residual."""
import ctypes

import numpy as np
import pytest

import _pins as P
from oracle import facet_ref as R
from stabilized_navier_stokes_flow_fenicsx_b200 import distributed as D
from stabilized_navier_stokes_flow_fenicsx_b200 import gmsh_io as G
from stabilized_navier_stokes_flow_fenicsx_b200 import mesh as M
from stabilized_navier_stokes_flow_fenicsx_b200._lib import NsgpuError
from stabilized_navier_stokes_flow_fenicsx_b200.assembler import NSAssembler
from test_facet_ref import Field, box_of, closed_form_rows, face_tagged
from test_interpolate_gpu import jittered_square

pytestmark = pytest.mark.gpu

EINVAL = -1
MESHES = {"duct": lambda: M.duct_mesh(3, 7), "rect": lambda: M.create_rectangle_tris(7, 5)}


def asm_with_facets(m, sp, dofmap=None, **kw):
    asm = NSAssembler(m.x, m.cells, sp.dofmap if dofmap is None else dofmap, vdeg=sp.vdeg, **kw)
    _, fc, fl, ft = face_tagged(m)
    assert asm.set_facets(fc, fl, ft) == 2 * m.gdim
    return asm, (fc, fl, ft)


def rel(a, b):
    return np.abs(a - b).max() / np.abs(b).max()


@pytest.mark.parametrize("vdeg", [1, 2])
@pytest.mark.parametrize("mesh", list(MESHES))
def test_facet_integrals_match_closed_forms(mesh, vdeg):
    m = MESHES[mesh]()
    sp = M.mixed_space(m, vdeg)
    f = Field(m.gdim, vdeg)
    asm, _ = asm_with_facets(m, sp)
    got = asm.facet_integrals(f.state(sp))
    ref = closed_form_rows(f, box_of(m))
    assert got.shape == (2 * m.gdim, 2 + 3 * m.gdim)
    assert rel(got, ref) <= 1e-12, rel(got, ref)
    asm.close()


@pytest.mark.parametrize("case", ["duct_p1", "duct_p2", "delaunay_p1", "delaunay_p2", "duct_p1_permuted"])
def test_facet_integrals_match_the_restatement(case):
    m = jittered_square(9, 3) if case.startswith("delaunay") else M.duct_mesh(3, 6)
    sp = M.mixed_space(m, 2 if "p2" in case else 1)
    w = np.random.default_rng(17).standard_normal(sp.n_dofs)
    _, fc, fl, ft = face_tagged(m)
    ref = R.facet_integrals(m.x, m.cells, sp.dofmap, sp.vdeg, w, fc, fl, ft)
    if case.endswith("permuted"):               # scattered caller numbering: the library renumbers internally
        perm = np.random.default_rng(5).permutation(sp.n_dofs).astype(np.int32)
        asm, _ = asm_with_facets(m, sp, dofmap=perm[sp.dofmap])
        wp = np.empty_like(w); wp[perm] = w
        got = asm.facet_integrals(wp)
    else:
        asm, _ = asm_with_facets(m, sp)
        got = asm.facet_integrals(w)
    assert rel(got, ref) <= 1e-13, rel(got, ref)
    asm.close()


@pytest.mark.parametrize("vdeg", [1, 2])
def test_outlet_and_inlet_flux_equal_the_plane_flux(vdeg):
    m = M.duct_mesh(4, 8)
    sp = M.mixed_space(m, vdeg)
    w = M.duct_state(sp)
    asm, _ = asm_with_facets(m, sp)
    rows = asm.facet_integrals(w)
    out, a_out = P.plane_flux(m, sp, w, 4.0)
    inl, a_in = P.plane_flux(m, sp, w, 0.0)
    assert abs(rows[1, 1] - out) <= 1e-12 * abs(out) and abs(rows[0, 1] + inl) <= 1e-12 * abs(inl)
    assert abs(rows[1, 0] - a_out) <= 1e-12 and abs(rows[0, 0] - a_in) <= 1e-12
    asm.close()


REACTION_CASES = {
    "gmetric_p1_duct": (lambda: M.duct_mesh(3, 6), 1, dict(flavour=0, nu=0.1)),
    "gmetric_p2_duct": (lambda: M.duct_mesh(3, 6), 2, dict(flavour=0, nu=0.1)),
    "stokes_p2_duct": (lambda: M.duct_mesh(3, 6), 2, dict(flavour=2, nu=1.0, alpha=1.0, sp=-1.0, beta=0.0)),
    "ugn_p1_cavity": (lambda: M.create_rectangle_tris(8, 8), 1, dict(flavour=1, nu=0.01)),
}


@pytest.mark.parametrize("case", list(REACTION_CASES))
def test_reaction_equals_the_host_sum_of_the_unconstrained_residual(case, oracle):
    mk, vdeg, fk = REACTION_CASES[case]
    m = mk()
    sp = M.mixed_space(m, vdeg)
    w = M.duct_state(sp) if m.gdim == 3 else M.cavity_state(sp)
    asm, (fc, fl, ft) = asm_with_facets(m, sp)
    asm.set_form(**fk)
    got = asm.reaction(w)
    asm.set_bcs([])
    asm.create_matrix(fetch=False)                              # the residual assembly needs the pattern; the reaction does not
    Rg = asm.residual(w)
    lists = R.tagged_velocity_dofs(m.cells, sp.dofmap, vdeg, fc, fl, ft)
    host = np.array([[Rg[d[c == k]].sum() for k in range(m.gdim)] for d, c in lists])
    mag = np.array([[np.abs(Rg[d[c == k]]).sum() for k in range(m.gdim)] for d, c in lists])
    assert (np.abs(got - host) <= 1e-12 * mag).all(), np.abs(got - host).max()
    form = oracle.Form(gdim=m.gdim, vdeg=vdeg, **fk)
    Ro = oracle.assemble_residual(form, m.x, m.cells, sp.dofmap, w, None, None)
    ref = R.reaction(Ro, m.cells, sp.dofmap, vdeg, fc, fl, ft)
    assert (np.abs(got - ref) <= 1e-12 * mag).all(), np.abs(got - ref).max()
    asm.close()


def test_dfg_2d_1_drag_and_lift_on_the_device():
    m, sp, bcs, obstacle = P.dfg_problem()
    be = P.GpuBackend(m, sp, bcs)
    r = P.dfg_solve(be, sp, bcs, obstacle)
    bf = G.boundary_facets(m)
    cyl = bf[(bf < m.meta["n_cyl"]).all(axis=1)]              # the first n_cyl vertices are the cylinder's
    fc, fl, ft = G.facet_integration_domain(m, cyl, np.zeros(len(cyl), dtype=np.int32))
    asm = be.asm
    assert asm.set_facets(fc, fl, ft) == 1
    scale, nu = 2.0 / (0.1 * 0.2 ** 2), 1e-3
    cd, cl = -scale * asm.reaction(r["w"])[0]
    assert abs(cd - r["cd"]) <= 1e-10 * abs(r["cd"]) and abs(cl - r["cl"]) <= 1e-10 * abs(r["cl"]), (cd, cl, r["cd"], r["cl"])
    assert abs(cd / P.DFG_CD - 1.0) < 0.01 and abs(cl / P.DFG_CL - 1.0) < 0.05
    rows = asm.facet_integrals(r["w"])[0]
    sd, sl = -scale * (nu * (rows[4:6] + rows[6:8]) - rows[2:4])
    print(f"DFG 2D-1 on the device: reaction Cd {cd:.6f} Cl {cl:.6f}; sigma-form Cd {sd:.6f} Cl {sl:.6f}")
    assert abs(sd / P.DFG_CD - 1.0) < 0.025 and abs(sl / P.DFG_CL - 1.0) < 0.01
    be.close()


def _box_face_facets(m, box):
    """exterior facets of a (partial) mesh that lie on a face of the global box, tagged as in face_tagged"""
    lo, hi = box
    bf = G.boundary_facets(m)
    cen = m.x[bf][:, :, : m.gdim].mean(axis=1)
    tags = np.full(len(bf), -1, dtype=np.int32)
    for a in range(m.gdim):
        tags[np.abs(cen[:, a] - lo[a]) < 1e-12] = 2 * a
        tags[np.abs(cen[:, a] - hi[a]) < 1e-12] = 2 * a + 1
    keep = tags >= 0
    return G.facet_integration_domain(m, bf[keep], tags[keep])


def test_partitions_add_up_and_ghost_cells_are_skipped():
    nc, nl = 3, 8
    m = M.duct_mesh(nc, nl)
    sp = M.mixed_space(m, 1)
    w = M.duct_state(sp)
    whole, _ = asm_with_facets(m, sp)
    whole.set_form(flavour=0, nu=0.1)
    ref_i, ref_r = whole.facet_integrals(w), whole.reaction(w)
    whole.close()
    # two x-slab partitions (distributed.duct_partition) as single-rank contexts without a communicator
    tot_i, tot_r = np.zeros_like(ref_i), np.zeros_like(ref_r)
    for rank in range(2):
        part = D.duct_partition(nc, nl, rank, 2)
        pm = M.Mesh(3, part.x, part.cells)
        asm = NSAssembler(part.x, part.cells, part.dofmap, vdeg=1, n_dofs_owned=part.n_owned, n_dofs_ghost=part.n_ghost,
                          n_cells_owned=part.n_cells_owned)
        asm.set_form(flavour=0, nu=0.1)
        assert asm.set_facets(*_box_face_facets(pm, box_of(m))) == 6
        tot_i += asm.facet_integrals(part.w); tot_r += asm.reaction(part.w)
        asm.close()
    assert rel(tot_i, ref_i) <= 1e-13 and rel(tot_r, ref_r) <= 1e-13, (rel(tot_i, ref_i), rel(tot_r, ref_r))
    # the same mesh twice, each context owning one half of the cells and holding the other half as ghost cells (all pairs passed)
    half = m.n_cells // 2
    tot_i, tot_r = np.zeros_like(ref_i), np.zeros_like(ref_r)
    for order in (np.arange(m.n_cells), np.roll(np.arange(m.n_cells), -half)):
        mo = M.Mesh(3, m.x, m.cells[order])
        asm = NSAssembler(m.x, mo.cells, sp.dofmap[order], vdeg=1, n_cells_owned=half if order[0] == 0 else m.n_cells - half)
        asm.set_form(flavour=0, nu=0.1)
        asm.set_facets(*_box_face_facets(mo, box_of(m)))
        tot_i += asm.facet_integrals(w); tot_r += asm.reaction(w)
        asm.close()
    assert rel(tot_i, ref_i) <= 1e-13 and rel(tot_r, ref_r) <= 1e-13, (rel(tot_i, ref_i), rel(tot_r, ref_r))


def test_determinism_device_variants_and_status_codes():
    m = M.duct_mesh(3, 6)
    sp = M.mixed_space(m, 2)
    w = M.duct_state(sp)
    asm, (fc, fl, ft) = asm_with_facets(m, sp)
    asm.set_form(flavour=0, nu=0.1)
    a1, r1 = asm.facet_integrals(w), asm.reaction(w)
    a2, r2 = asm.facet_integrals(w), asm.reaction(w)
    assert np.array_equal(a1, a2) and np.array_equal(r1, r2)
    w_dev, ai_dev, re_dev = asm.dev_alloc(8 * sp.n_dofs), asm.dev_alloc(8 * a1.size), asm.dev_alloc(8 * r1.size)
    asm.h2d(w_dev, w)
    asm.facet_integrals_dev(w_dev, ai_dev)
    asm.reaction_dev(w_dev, re_dev)
    asm.sync()
    ad, rd = np.empty_like(a1), np.empty_like(r1)
    asm.d2h(ad, ai_dev); asm.d2h(rd, re_dev)
    assert np.array_equal(ad, a1) and np.array_equal(rd, r1)
    for p in (w_dev, ai_dev, re_dev):
        asm.dev_free(p)
    lib, ctx = asm.lib, asm.ctx
    n = len(fc)
    good = [np.ascontiguousarray(a, dtype=np.int32) for a in (fc, fl, ft)]

    def call(c, l, t, count=n):
        arrs = [a.ctypes.data_as(ctypes.c_void_p) if a is not None else None for a in (c, l, t)]
        return lib.nsgpu_set_facets(ctx, count, *arrs, None)

    def bad(k, v):
        a = [x.copy() for x in good]
        a[k][n // 2] = v
        return a

    cases = [(None, good[1], good[2]), (good[0], None, good[2]), (good[0], good[1], None),
             bad(0, -1), bad(0, m.n_cells), bad(1, -1), bad(1, 4), bad(2, -1), bad(2, 64)]
    for c, l, t in cases:
        assert call(c, l, t) == EINVAL
        assert np.array_equal(asm.facet_integrals(w), a1) and np.array_equal(asm.reaction(w), r1)
    assert call(*good) == 0 and np.array_equal(asm.facet_integrals(w), a1)
    # before set_mesh / set_space, and a functional before set_facets
    fresh = ctypes.c_void_p()
    assert lib.nsgpu_create(ctypes.byref(fresh), 0) == 0
    assert lib.nsgpu_set_facets(fresh, n, *[a.ctypes.data_as(ctypes.c_void_p) for a in good], None) == EINVAL
    lib.nsgpu_destroy(fresh)
    other = NSAssembler(m.x, m.cells, sp.dofmap, vdeg=2)
    with pytest.raises(NsgpuError, match="set_facets first"):
        other.facet_integrals(w)
    other.close()
    asm.close()
