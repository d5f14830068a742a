"""Every assembly kernel path against the CPU oracle (oracle/oracle.py), on a B200 (-m gpu).

Each case selects its path explicitly (options kernel, rowown, rowown_lean, ws, pipe, stream_host), asserts
``last_kernel_name()`` after every call so that a silent fallback fails, poisons the values with NaN before every Jacobian
pass (the row-owner and factorised kernels skip the zero-fill and must write every entry), and checks the four entry points
(``jacobian``, ``residual``, ``jacobian_residual``, ``jacobian_residual_dev`` with want_J 1 and 0) and ``mult``.  Patterns
are compared bit for bit, values to 1e-12 relative to the largest magnitude of the compared array.

Coverage of the (element, form) x path matrix (section A on jittered structured meshes with a third of the cells flipped,
states s1-s3 and, for UGN, s4; section B on Delaunay meshes).  Stokes runs twice: with PSPG (sp = 1, beta > 0) and
unstabilised (sp = -1, beta = 0).  "rowown" on G-metric tets is the lean block formulation (rowown_lean = 1), "rowown_lean0"
the unsplit entity blocks.

| pair              | generic_row | generic_coop       | rowown            | rowown_lean0      | p1tet_ws / pipe / tiles |
|-------------------|-------------|--------------------|-------------------|-------------------|-------------------------|
| P1 tri G-metric   | A, B        | A, B               | A, B (a)          | n/s (b)           | n/s (c)                 |
| P2 tri G-metric   | A, B        | A, B               | A, B (a)          | n/s (b)           | n/s (c)                 |
| P1 tri UGN        | A, B        | A, B               | A, B              | n/s (b)           | n/s (c)                 |
| P2 tri UGN        | A, B        | A, B               | A, B              | n/s (b)           | n/s (c)                 |
| P1 tri Stokes x2  | A, B        | A, B               | A, B              | n/s (b)           | n/s (c)                 |
| P2 tri Stokes x2  | A, B        | A, B               | A, B              | n/s (b)           | n/s (c)                 |
| P1 tet G-metric   | A, B        | fan mesh (d)       | fan mesh (d)      | fan mesh (d)      | A, B (+ streamed, F)    |
| P2 tet G-metric   | A, B        | A, B               | A, B              | A, B              | n/s (c)                 |
| P1 tet UGN        | A, B        | A, B               | A, B              | n/s (b)           | n/s (c)                 |
| P2 tet UGN        | A, B        | A, B               | A, B              | n/s (b)           | n/s (c)                 |
| P1 tet Stokes x2  | A, B        | A, B               | A, B              | n/s (b)           | n/s (c)                 |
| P2 tet Stokes x2  | A, B        | A, B               | A, B              | n/s (b)           | n/s (c)                 |

A = ``test_path_matrix``, B = ``test_unstructured_mesh``, fan mesh = ``test_fan_vertex_refuses_the_p1_plan``, F =
``test_stream_chunks_are_bitwise_identical``; n/s = not selectable:
(a) the lean formulation is compiled for tetrahedra only, so on triangles rowown_lean has no effect and "rowown" is the
    unsplit formulation;
(b) rowown_lean only switches the G-metric form on tetrahedra;
(c) the factorised kernels exist for the G-metric form on P1-P1 tetrahedra only (kernel = 2 raises EUNSUPPORTED elsewhere);
(d) while the factorised plan exists AUTO takes it, so generic_coop and rowown run on P1 G-metric tets only when the plan is
    refused (a vertex in more than 63 cells).
Further sections: C multi-round row-owner grids, D edge sizes and fallbacks, E Dirichlet sets changed on a live context,
F options (spmv_blocks x spmv_wide, stream_chunks)."""
import functools

import numpy as np
import pytest

import _meshes as MS
from stabilized_navier_stokes_flow_fenicsx_b200 import mesh as M
from stabilized_navier_stokes_flow_fenicsx_b200._lib import NsgpuError
from stabilized_navier_stokes_flow_fenicsx_b200.assembler import NSAssembler

pytestmark = pytest.mark.gpu
RTOL = 1e-12

FORMS = {
    "gmetric": dict(flavour=0, nu=0.05),
    "ugn": dict(flavour=1, nu=0.01),
    "stokes_pspg": dict(flavour=2, nu=1.0, alpha=1.0, sp=1.0, beta=0.2),
    "stokes_plain": dict(flavour=2, nu=1.0, alpha=1.0, sp=-1.0, beta=0.0),
}
ELEMENTS = [(2, 1), (2, 2), (3, 1), (3, 2)]
_BASE = dict(kernel=0, rowown=1, rowown_lean=1, ws=1, pipe=1, stream_host=0)
PATHS = {
    "generic_row": (dict(kernel=1), "generic_row"),
    "generic_coop": (dict(rowown=0), "generic_coop"),
    "rowown": (dict(rowown=2), "rowown"),
    "rowown_lean0": (dict(rowown=2, rowown_lean=0), "rowown"),
    "p1tet_ws": (dict(kernel=2), "p1tet_ws"),
    "p1tet_pipe": (dict(kernel=2, ws=0), "p1tet_pipe"),
    "p1tet_tiles": (dict(kernel=2, ws=0, pipe=0), "p1tet_tiles"),
}


def selectable(gd, vd, form, path):
    fast_pair = gd == 3 and vd == 1 and form == "gmetric"
    if path.startswith("p1tet_"):
        return fast_pair
    if path in ("generic_coop", "rowown"):
        return not fast_pair
    if path == "rowown_lean0":
        return gd == 3 and vd == 2 and form == "gmetric"
    return True


MATRIX = [(gd, vd, f, p) for gd, vd in ELEMENTS for f in FORMS for p in PATHS if selectable(gd, vd, f, p)]
MATRIX_IDS = [f"{'tri' if gd == 2 else 'tet'}-P{vd}-{f}-{p}" for gd, vd, f, p in MATRIX]


# ------------------------------------------------------------------------------------------------- helpers
def _close(got, want, what):
    assert np.isfinite(got).all(), f"{what}: {np.count_nonzero(~np.isfinite(got))} non-finite entries"
    err = np.abs(got - want).max() if len(want) else 0.0
    assert err <= RTOL * np.abs(want).max(), f"{what}: max abs err {err:.3e}, max |ref| {np.abs(want).max():.3e}"


class Ref:
    """The oracle's pattern, Jacobian and residual (assemble_vector + apply_lifting + set_bc) of one space."""

    def __init__(self, oracle, m, sp, big=False):
        self.oracle, self.m, self.sp = oracle, m, sp
        build = oracle.build_pattern_c if big else oracle.build_pattern
        self.indptr, self.indices = build(sp.dofmap, sp.n_dofs)

    def __call__(self, w, bcs, fk):
        o = self.oracle
        form = o.Form(gdim=self.m.gdim, vdeg=self.sp.vdeg, **fk)
        if bcs:
            marker, value, mult = o.bc_arrays(self.sp.n_dofs, [b[0] for b in bcs], [b[1] for b in bcs])
        else:
            marker = value = mult = None
        vals = o.assemble_jacobian(form, self.m.x, self.m.cells, self.sp.dofmap, w, self.indptr, self.indices, marker, mult)
        F = o.assemble_residual(form, self.m.x, self.m.cells, self.sp.dofmap, w, marker, value)
        if bcs:
            o.set_bc(F, [b[0] for b in bcs], [b[1] for b in bcs], w)
        return vals, F


def _assembler(m, sp, bcs, fk, opts):
    asm = NSAssembler(m.x, m.cells, sp.dofmap, vdeg=sp.vdeg)
    asm.set_form(**fk)
    if bcs is not None:
        asm.set_bcs(bcs)
    for k, v in {**_BASE, **opts}.items():
        asm.set_option(k, v)
    return asm


def _check_pattern(asm, ref):
    gp, gi = asm.create_matrix()
    np.testing.assert_array_equal(gp, ref.indptr)
    np.testing.assert_array_equal(gi, ref.indices)


def check_entry_points(asm, ref, w, bcs, fk, expect, tag=""):
    """jacobian, residual, jacobian_residual, jacobian_residual_dev (want_J 1 and 0) and mult against the oracle."""
    vals, F = ref(w, bcs, fk)
    n = ref.sp.n_dofs
    nan = np.full(asm.nnz, np.nan)

    def name(what):
        assert asm.last_kernel_name() == expect, f"{tag} {what}: ran {asm.last_kernel_name()!r}, selected {expect!r}"

    asm.set_values(nan)
    gv = asm.jacobian(w); name("jacobian")
    _close(gv, vals, f"{tag} jacobian")
    gF = asm.residual(w); name("residual")
    _close(gF[:n], F, f"{tag} residual")
    asm.set_values(nan)
    gv, gF = asm.jacobian_residual(w); name("jacobian_residual")
    _close(gv, vals, f"{tag} jacobian_residual J")
    _close(gF[:n], F, f"{tag} jacobian_residual F")
    nb = 8 * asm.n_cols
    x_dev, F_dev = asm.dev_alloc(nb), asm.dev_alloc(nb)
    try:
        Fh = np.full(asm.n_cols, np.nan)
        asm.h2d(x_dev, w); asm.h2d(F_dev, Fh)
        asm.set_values(nan)
        asm.jacobian_residual_dev(x_dev, True, F_dev); asm.sync(); name("jacobian_residual_dev(want_J=1)")
        asm.d2h(Fh, F_dev)
        _close(asm.get_values(), vals, f"{tag} dev J")
        _close(Fh[:n], F, f"{tag} dev F (want_J=1)")
        Fh[:] = np.nan; asm.h2d(F_dev, Fh)
        asm.jacobian_residual_dev(x_dev, False, F_dev); asm.sync(); name("jacobian_residual_dev(want_J=0)")
        asm.d2h(Fh, F_dev)
        _close(Fh[:n], F, f"{tag} dev F (want_J=0)")
    finally:
        asm.dev_free(x_dev); asm.dev_free(F_dev)
    xv = np.random.default_rng(1).standard_normal(n)
    _close(asm.mult(xv), ref.oracle.spmv(ref.indptr, ref.indices, vals, xv), f"{tag} mult")
    return vals, F


# ------------------------------------------------------------------------------------------------- A: element x form x path
@pytest.mark.parametrize("gd,vd,form,path", MATRIX, ids=MATRIX_IDS)
def test_path_matrix(oracle, gd, vd, form, path):
    """All 12 (element, form) pairs (Stokes twice) on every path that can be selected for them, on a jittered structured mesh with
    a third of the cells flipped, at the states s1 (smooth + noise), s2 (off the Dirichlet values: lifting active), s3 (zero except
    on the Dirichlet dofs: UGN's |u| = 0 branch, G-metric's tau without a velocity term) and, for UGN, s4 (cell Reynolds numbers
    on both sides of 3)."""
    m = MS.structured(gd, 3 if gd == 3 else 6, seed=10 * gd + vd)
    assert (MS.signed_measure(m) < 0).mean() > 0.2
    sp = M.mixed_space(m, vd)
    bcs = MS.box_bcs(sp)
    fk = FORMS[form]
    opts, expect = PATHS[path]
    ref = Ref(oracle, m, sp)
    asm = _assembler(m, sp, bcs, fk, opts)
    _check_pattern(asm, ref)
    s1 = MS.smooth_state(sp, seed=gd + vd)
    states = {"s1": s1, "s2": s1 + 0.01 * np.random.default_rng(7).standard_normal(sp.n_dofs), "s3": MS.dirichlet_only_state(sp, bcs)}
    if form == "ugn":
        s4 = MS.reynolds_split_state(sp, fk["nu"])
        re = MS.cell_reynolds(sp, s4, fk["nu"])
        assert (re <= 3).mean() >= 0.1 and (re > 3).mean() >= 0.1
        states["s4"] = s4
    for s, w in states.items():
        check_entry_points(asm, ref, w, bcs, fk, expect, tag=s)
    asm.close()


# ------------------------------------------------------------------------------------------------- B: unstructured meshes
@functools.lru_cache(maxsize=None)
def _delaunay(gd):
    return MS.delaunay_tets(14, seed=3) if gd == 3 else MS.delaunay_tris(40, seed=0)


@pytest.mark.parametrize("gd,vd,form,path", MATRIX, ids=MATRIX_IDS)
def test_unstructured_mesh(oracle, gd, vd, form, path):
    """The matrix of A on Delaunay meshes of jittered lattices: edges in more than 8 cells (the warp-specialised kernel's gather-list
    overflow) and, for P2 tets, vertices in more than 30 cells (the row-owner kernel fetches incidences beyond 3 NENT from memory)."""
    m = _delaunay(gd)
    if gd == 3:
        assert MS.edge_cell_counts(m.cells).max() > 8
        assert MS.vertex_cell_counts(m.cells).max() > 3 * MS.NENT[(3, 2)]
    sp = M.mixed_space(m, vd)
    bcs = MS.box_bcs(sp)
    fk = FORMS[form]
    opts, expect = PATHS[path]
    ref = Ref(oracle, m, sp)
    asm = _assembler(m, sp, bcs, fk, opts)
    _check_pattern(asm, ref)
    w = MS.smooth_state(sp, seed=5) + 0.01 * np.random.default_rng(8).standard_normal(sp.n_dofs)
    check_entry_points(asm, ref, w, bcs, fk, expect, tag="delaunay")
    if path == "p1tet_ws":                              # the streamed host-vector path of the same kernel
        asm.set_option("stream_host", 1)
        vals, F = ref(w, bcs, fk)
        asm.set_values(np.full(asm.nnz, np.nan))
        gv, gF = asm.jacobian_residual(w)
        assert asm.last_kernel_name() == "p1tet_ws (streamed host vectors)"
        _close(gv, vals, "streamed J"); _close(gF, F, "streamed F")
    asm.close()


# ------------------------------------------------------------------------------------------------- C: multi-round row-owner grids
def _n_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.mark.parametrize("gd,vd,form", [(2, 1, "ugn"), (2, 2, "ugn"), (3, 1, "ugn"), (3, 2, "gmetric")],
                         ids=["tri-P1-ugn", "tri-P2-ugn", "tet-P1-ugn", "tet-P2-gmetric"])
def test_rowown_grid_stride_rounds(oracle, gd, vd, form):
    """k_rowown caps its grid at 16 n_sms CTAs of at most 4 (32 // NENT) entity groups and prefetches the next round's entity
    header: size the mesh so that every entity class needs at least two grid-stride rounds, and compare every entry."""
    g_max = 4 * (32 // MS.NENT[(gd, vd)])
    need = 16 * _n_sms() * g_max
    if gd == 2:
        n = int(np.ceil(np.sqrt(need))) + 1
        m = MS.flip_cells(M.create_rectangle_tris(n, n), seed=2)[0]
    else:
        n = int(np.ceil(need ** (1.0 / 3))) + (0 if vd == 2 else 1)
        m = MS.flip_cells(M.create_box_tets((n, n, n)), seed=2)[0]
    sp = M.mixed_space(m, vd)
    nv, ne = MS.n_entities(sp)
    assert nv > need and (vd == 1 or ne > need), (nv, ne, need)
    bcs = MS.box_bcs(sp)
    fk = FORMS[form]
    ref = Ref(oracle, m, sp, big=True)
    asm = _assembler(m, sp, bcs, fk, dict(rowown=2))
    _check_pattern(asm, ref)
    w = MS.smooth_state(sp, seed=3) + 0.01 * np.random.default_rng(9).standard_normal(sp.n_dofs)
    vals, F = ref(w, bcs, fk)
    asm.set_values(np.full(asm.nnz, np.nan))
    gv, gF = asm.jacobian_residual(w)
    assert asm.last_kernel_name() == "rowown"
    _close(gv, vals, "J"); _close(gF, F, "F")
    gF = asm.residual(w)
    assert asm.last_kernel_name() == "rowown"
    _close(gF, F, "residual-only F")
    asm.close()


# ------------------------------------------------------------------------------------------------- D: edge sizes and fallbacks
def _tiny_bcs(sp):
    """The velocity of vertex 0 (0.2, 0.3[, 0.4]) and the pressure of the last vertex (0.1)."""
    gd = sp.mesh.gdim
    v0 = np.flatnonzero((np.abs(sp.dof_x - sp.mesh.x[0]).sum(1) == 0) & (sp.dof_comp < gd)).astype(np.int32)
    pl = np.flatnonzero((np.abs(sp.dof_x - sp.mesh.x[-1]).sum(1) == 0) & (sp.dof_comp == gd)).astype(np.int32)
    return [(v0, 0.2 + 0.1 * sp.dof_comp[v0]), (pl, np.full(len(pl), 0.1))]


TINY = [(gd, vd, f, p, k) for gd, vd, f, p in MATRIX if f in ("gmetric", "ugn") for k in ("1cell", "2cells", "box")]
TINY_IDS = [f"{'tri' if gd == 2 else 'tet'}-P{vd}-{f}-{p}-{k}" for gd, vd, f, p, k in TINY]


@pytest.mark.parametrize("gd,vd,form,path,kind", TINY, ids=TINY_IDS)
def test_tiny_meshes(oracle, gd, vd, form, path, kind):
    """1 cell, 2 cells sharing a facet (the second flipped), 1 box (6 tets / 2 triangles), on every path."""
    m = MS.single_cells(gd, 1 if kind == "1cell" else 2) if kind != "box" else (
        M.create_box_tets((1, 1, 1)) if gd == 3 else M.create_rectangle_tris(1, 1))
    sp = M.mixed_space(m, vd)
    bcs = _tiny_bcs(sp)
    fk = FORMS[form]
    opts, expect = PATHS[path]
    ref = Ref(oracle, m, sp)
    asm = _assembler(m, sp, bcs, fk, opts)
    _check_pattern(asm, ref)
    w = MS.smooth_state(sp, seed=1, noise=0.05)
    check_entry_points(asm, ref, w, bcs, fk, expect, tag=kind)
    asm.close()


COOP = [(gd, vd, d) for gd, vd in ELEMENTS for d in (-1, 0, 1)]


@pytest.mark.parametrize("gd,vd,delta", COOP, ids=[f"{'tri' if gd == 2 else 'tet'}-P{vd}-3CPB{d:+d}" for gd, vd, d in COOP])
def test_coop_block_boundaries(oracle, gd, vd, delta):
    """generic_coop with 3 CPB - 1, 3 CPB and 3 CPB + 1 cells (CPB = 256 // ND cells per CTA): the last CTA is one cell short,
    exactly full, or holds a single cell."""
    n_cells = 3 * MS.coop_cells_per_block(gd, vd) + delta
    m = MS.take_cells(MS.structured(gd, 4 if gd == 3 else 8, seed=4), n_cells)
    assert m.n_cells == n_cells
    sp = M.mixed_space(m, vd)
    bcs = _tiny_bcs(sp)
    fk = FORMS["ugn"]
    ref = Ref(oracle, m, sp)
    asm = _assembler(m, sp, bcs, fk, PATHS["generic_coop"][0])
    _check_pattern(asm, ref)
    check_entry_points(asm, ref, MS.smooth_state(sp, seed=2, noise=0.05), bcs, fk, "generic_coop")
    asm.close()


def test_fan_vertex_refuses_the_p1_plan(oracle):
    """A vertex in more than 63 cells: the factorised P1-P1 plan is refused.  AUTO runs generic_coop, kernel = 2 raises
    EUNSUPPORTED and leaves the context usable, rowown = 2 runs the lean row-owner blocks (and rowown_lean = 0 the unsplit ones),
    MatMult runs the CSR kernel."""
    m = MS.fan_tets(40)
    assert MS.vertex_cell_counts(m.cells).max() > 63
    sp = M.mixed_space(m, 1)
    bcs = MS.box_bcs(sp, lo=-2.0, hi=2.0)
    fk = FORMS["gmetric"]
    ref = Ref(oracle, m, sp)
    w = MS.smooth_state(sp, seed=6, noise=0.05)
    asm = _assembler(m, sp, bcs, fk, {})
    _check_pattern(asm, ref)
    check_entry_points(asm, ref, w, bcs, fk, "generic_coop", tag="auto")
    assert asm.last_spmv_name() == "spmv_csr"
    asm.set_option("kernel", 2)
    with pytest.raises(NsgpuError) as e:
        asm.jacobian_residual(w)
    assert "(-3)" in str(e.value)                        # NSGPU_EUNSUPPORTED
    with pytest.raises(NsgpuError):
        asm.residual(w)
    asm.set_option("kernel", 0)
    check_entry_points(asm, ref, w, bcs, fk, "generic_coop", tag="after the refusal")
    asm.set_option("rowown", 2)
    check_entry_points(asm, ref, w, bcs, fk, "rowown", tag="rowown lean")
    asm.set_option("rowown_lean", 0)
    check_entry_points(asm, ref, w, bcs, fk, "rowown", tag="rowown unsplit")
    asm.set_option("kernel", 1)
    check_entry_points(asm, ref, w, bcs, fk, "generic_row", tag="generic_row")
    assert asm.last_spmv_name() == "spmv_csr"
    asm.close()


# ------------------------------------------------------------------------------------------------- E: Dirichlet sets on a live context
FAMILIES = [(3, 1, "gmetric", "p1tet_ws"), (3, 1, "gmetric", "p1tet_pipe"), (3, 1, "gmetric", "p1tet_tiles"),
            (3, 2, "gmetric", "rowown"), (3, 2, "gmetric", "rowown_lean0"), (2, 2, "ugn", "rowown"), (3, 1, "stokes_pspg", "rowown"),
            (2, 1, "ugn", "generic_coop"), (3, 2, "stokes_plain", "generic_coop"), (3, 1, "ugn", "generic_row"), (2, 2, "gmetric", "generic_row")]


@pytest.mark.parametrize("gd,vd,form,path", FAMILIES, ids=[f"{'tri' if gd == 2 else 'tet'}-P{vd}-{f}-{p}" for gd, vd, f, p in FAMILIES])
def test_bc_sets_on_a_live_context(oracle, gd, vd, form, path):
    """reference BCs -> no BCs -> whole cells constrained (velocity and pressure dofs, some held twice) -> reference BCs, on one
    context; J and F against the oracle after every change, BC diagonals of dofs held by two objects equal to 2."""
    m = MS.structured(gd, 3 if gd == 3 else 6, seed=20 + gd + vd)
    sp = M.mixed_space(m, vd)
    fk = FORMS[form]
    opts, expect = PATHS[path]
    ref = Ref(oracle, m, sp)
    w = MS.smooth_state(sp, seed=4) + 0.01 * np.random.default_rng(3).standard_normal(sp.n_dofs)
    asm = _assembler(m, sp, MS.box_bcs(sp), fk, opts)
    _check_pattern(asm, ref)
    for step, bcs in enumerate([MS.box_bcs(sp), [], MS.cell_bcs(sp, seed=gd + vd), MS.box_bcs(sp)]):
        if step:
            asm.set_bcs(bcs)
        vals, _ = check_entry_points(asm, ref, w, bcs, fk, expect, tag=f"BC step {step}")
        if bcs:
            _, _, mult = oracle.bc_arrays(sp.n_dofs, [b[0] for b in bcs], [b[1] for b in bcs])
            twice = np.flatnonzero(mult == 2)
            assert len(twice)
            diag = np.array([vals[ref.indptr[r] + np.searchsorted(ref.indices[ref.indptr[r]:ref.indptr[r + 1]], r)] for r in twice])
            gv = asm.get_values()
            gdiag = np.array([gv[ref.indptr[r] + np.searchsorted(ref.indices[ref.indptr[r]:ref.indptr[r + 1]], r)] for r in twice])
            assert (diag == 2.0).all() and (gdiag == 2.0).all()
    asm.close()


# ------------------------------------------------------------------------------------------------- F: options
def test_spmv_blocks_and_width(oracle):
    """spmv_blocks 4 / 5 / 6 x spmv_wide 0 / 1 of the vertex-blocked MatMult: each against the oracle, all within 1e-14 of each other."""
    m = M.duct_mesh(6, 16); sp = M.mixed_space(m, 1)
    bcs, fk = M.duct_bcs(sp), dict(flavour=0, nu=0.1)
    ref = Ref(oracle, m, sp)
    w = M.duct_state(sp) + 0.01 * np.random.default_rng(2).standard_normal(sp.n_dofs)
    vals, _ = ref(w, bcs, fk)
    asm = _assembler(m, sp, bcs, fk, {})
    _check_pattern(asm, ref)
    asm.jacobian_residual(w, fetch_vals=False)
    xv = np.random.default_rng(6).standard_normal(sp.n_dofs)
    yo = oracle.spmv(ref.indptr, ref.indices, vals, xv)
    ys = []
    for blocks in (4, 5, 6):
        for wide in (0, 1):
            asm.set_option("spmv_blocks", blocks); asm.set_option("spmv_wide", wide)
            y = asm.mult(xv)
            assert asm.last_spmv_name() == "spmv_block4"
            _close(y, yo, f"spmv_blocks={blocks} spmv_wide={wide}")
            ys.append(y)
    for y in ys[1:]:
        assert np.abs(y - ys[0]).max() <= 1e-14 * np.abs(ys[0]).max()
    asm.close()


@pytest.mark.parametrize("kind", ["duct", "delaunay"])
def test_stream_chunks_are_bitwise_identical(oracle, kind):
    """The streamed host path cut into 1, 2, 3, 7 and 64 chunks gives exactly what the plain copy-assemble-copy path gives."""
    if kind == "duct":
        m = M.duct_mesh(10, 32); sp = M.mixed_space(m, 1); bcs = M.duct_bcs(sp)
        w = M.duct_state(sp) + 0.01 * np.random.default_rng(1).standard_normal(sp.n_dofs)
    else:
        m = _delaunay(3); sp = M.mixed_space(m, 1); bcs = MS.box_bcs(sp)
        w = MS.smooth_state(sp, seed=2) + 0.01 * np.random.default_rng(1).standard_normal(sp.n_dofs)
    fk = dict(flavour=0, nu=0.05)
    ref = Ref(oracle, m, sp)
    vals, F = ref(w, bcs, fk)
    asm = _assembler(m, sp, bcs, fk, dict(kernel=2))
    asm.create_matrix(fetch=False)
    v0, F0 = asm.jacobian_residual(w)
    expect = asm.last_kernel_name()
    assert expect in ("p1tet_ws", "p1tet_pipe")
    _close(v0, vals, "J"); _close(F0, F, "F")
    asm.set_option("stream_host", 1)
    for chunks in (1, 2, 3, 7, 64):
        asm.set_option("stream_chunks", chunks)
        asm.set_values(np.full(asm.nnz, np.nan))
        v, Fs = asm.jacobian_residual(w)
        assert asm.last_kernel_name() == expect + " (streamed host vectors)", (chunks, asm.last_kernel_name())
        np.testing.assert_array_equal(v, v0)
        np.testing.assert_array_equal(Fs, F0)
    asm.close()
