"""Pins for the CPU oracle (oracle/ns_oracle.c).  The reference has no tests and its arithmetic lives in
un-vendored packages, so the pins are: (1) golden element tensors from an independent symbolic
evaluation of the forms as written in the reference (oracle/symbolic_ref.py), (2) finite differences,
(3) patch tests, (4) structural identities, (5) the sparsity set-union definition."""
import os

import numpy as np
import pytest

from stabilized_navier_stokes_flow_fenicsx_b200 import mesh as M

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "element_golden.npz")


def _golden_cases():
    d = np.load(GOLDEN)
    return sorted({k.split("/")[0] for k in d.files})


@pytest.mark.parametrize("name", _golden_cases())
def test_element_matches_symbolic_golden(oracle, name):
    d = np.load(GOLDEN)
    flavour, gdim, vdeg = (int(v) for v in d[name + "/meta"])
    nu, Ci, alpha, sp, beta = d[name + "/params"]
    form = oracle.Form(flavour, gdim, vdeg, nu, Ci, alpha, sp, beta)
    Ae, be = oracle.element(form, d[name + "/x"], d[name + "/w"])
    # tolerance: 1e-12 relative to the largest entry of the tensor (north-star assembly tolerance)
    assert np.abs(be - d[name + "/be"]).max() <= 1e-12 * np.abs(d[name + "/be"]).max()
    assert np.abs(Ae - d[name + "/Ae"]).max() <= 1e-12 * np.abs(d[name + "/Ae"]).max()


FORMS = [
    ("gmetric_p1_tet", dict(flavour=0, gdim=3, vdeg=1, nu=0.1)),
    ("gmetric_p2_tet", dict(flavour=0, gdim=3, vdeg=2, nu=0.02)),
    ("ugn_p1_tri", dict(flavour=1, gdim=2, vdeg=1, nu=0.01)),
    ("ugn_p2_tri", dict(flavour=1, gdim=2, vdeg=2, nu=0.01)),
    ("ugn_p1_tet", dict(flavour=1, gdim=3, vdeg=1, nu=0.01)),
    ("gmetric_p1_tri", dict(flavour=0, gdim=2, vdeg=1, nu=0.05)),
    ("gmetric_p2_tri", dict(flavour=0, gdim=2, vdeg=2, nu=0.05)),
    ("ugn_p2_tet", dict(flavour=1, gdim=3, vdeg=2, nu=0.01)),
] + [(f"stokes_{v}_p{k}_{c}", dict(flavour=2, gdim=g, vdeg=k, nu=1.0, alpha=a, sp=s, beta=b))
     for v, a, s, b in (("pspg", 1.0, 1.0, 0.2), ("plain", 0.7, -1.0, 0.0)) for k in (1, 2) for c, g in (("tri", 2), ("tet", 3))]


def _rand_cell(rng, gd, scale=0.1):
    ref = np.vstack([np.zeros(gd), np.eye(gd)])
    x = np.zeros((gd + 1, 3))
    x[:, :gd] = (ref + 0.2 * rng.standard_normal((gd + 1, gd))) * scale
    return x


@pytest.mark.parametrize("name,kw", FORMS)
def test_jacobian_is_derivative_of_residual(oracle, name, kw):
    """SURVEY 8c pin (2): || J d - (F(w+eps d) - F(w-eps d)) / 2 eps || / || J d || < 1e-7."""
    rng = np.random.default_rng(7)
    form = oracle.Form(**kw)
    nd = form.ndofs_cell
    for _ in range(5):
        x = _rand_cell(rng, form.gdim)
        w = rng.standard_normal(nd)
        d = rng.standard_normal(nd)
        Ae, _ = oracle.element(form, x, w)
        eps = 1e-6
        _, bp = oracle.element(form, x, w + eps * d, want_A=False)
        _, bm = oracle.element(form, x, w - eps * d, want_A=False)
        fd = (bp - bm) / (2 * eps)
        assert np.linalg.norm(Ae @ d - fd) / np.linalg.norm(Ae @ d) < 1e-7


def test_stokes_is_linear_and_block_structured(oracle):
    rng = np.random.default_rng(3)
    form = oracle.Form(flavour=2, gdim=3, vdeg=1, nu=1.0, alpha=1.0, sp=1.0, beta=0.2)
    x = _rand_cell(rng, 3)
    w = rng.standard_normal(16)
    Ae, be = oracle.element(form, x, w)
    np.testing.assert_allclose(Ae @ w, be, rtol=0, atol=1e-14 * np.abs(Ae).max() * 16)
    Avv, Avp, Apv, App = Ae[:12, :12], Ae[:12, 12:], Ae[12:, :12], Ae[12:, 12:]
    np.testing.assert_allclose(Avv, Avv.T, atol=1e-15)          # grad u : grad v symmetric
    np.testing.assert_allclose(Avp, -Apv.T, atol=1e-15)         # -p div v  vs  + q div u
    np.testing.assert_allclose(App, App.T, atol=1e-15)
    # P2-P1 duct flavour has the opposite pressure sign (DuctStokesFlow.py:191) and no PSPG block
    form = oracle.Form(flavour=2, gdim=3, vdeg=2, nu=1.0, alpha=1.0, sp=-1.0, beta=0.0)
    Ae, _ = oracle.element(form, x, rng.standard_normal(34))
    np.testing.assert_allclose(Ae[:30, 30:], -Ae[30:, :30].T, atol=1e-15)
    assert np.abs(Ae[30:, 30:]).max() == 0.0


def test_patch_constant_state_has_zero_interior_residual(oracle):
    """SURVEY 8c pin (3): u = const, p = const  =>  residual rows of interior dofs vanish."""
    mesh = M.create_box_tets((3, 3, 3))
    sp = M.mixed_space(mesh, 1)
    w = np.zeros(sp.n_dofs)
    w[sp.dof_comp == 0], w[sp.dof_comp == 1], w[sp.dof_comp == 2], w[sp.dof_comp == 3] = 0.7, -0.3, 0.2, 1.9
    form = oracle.Form(flavour=0, gdim=3, vdeg=1, nu=0.1)
    b = oracle.assemble_residual(form, mesh.x, mesh.cells, sp.dofmap, w)
    X = sp.dof_x
    interior = np.all((X > 1e-9) & (X < 1 - 1e-9), axis=1)
    assert interior.sum() == 8 * 4
    assert np.abs(b[interior]).max() < 1e-14
    assert np.abs(b[~interior]).max() > 1e-3                   # boundary rows see -p n and u.n


def test_pattern_is_sorted_unique_union(oracle):
    mesh = M.create_box_tets((2, 3, 2))
    sp = M.mixed_space(mesh, 1)
    indptr, indices = oracle.build_pattern(sp.dofmap, sp.n_dofs)
    want = [set() for _ in range(sp.n_dofs)]
    for row in sp.dofmap:
        for i in row:
            want[i].update(int(j) for j in row)
    for r in range(sp.n_dofs):
        got = indices[indptr[r]:indptr[r + 1]]
        assert list(got) == sorted(want[r])


def test_structured_duct_sizes_match_survey(oracle):
    """SURVEY Appendix A.6: 10x10x40 -> 24 000 cells, 4 961 vertices, 19 844 dofs, 1 063 696 nnz."""
    mesh = M.duct_mesh(10, 40)
    sp = M.mixed_space(mesh, 1)
    indptr, indices = oracle.build_pattern(sp.dofmap, sp.n_dofs)
    assert (mesh.n_cells, mesh.n_vertices, sp.n_dofs, len(indices)) == (24000, 4961, 19844, 1063696)
    # all tets positively sized and filling the duct volume 4 x 1 x 1
    X = mesh.x[mesh.cells]
    vol = np.abs(np.linalg.det(X[:, 1:] - X[:, :1])) / 6
    assert abs(vol.sum() - 4.0) < 1e-12 and vol.min() > 0


def test_global_assembly_bc_semantics(oracle):
    """assemble_matrix zeroes BC rows/cols and puts the BC-object multiplicity on the diagonal;
    lifting adds A[:,bc](g - x); set_bc writes x - g  (NavierStokesChannelFlow.py:64-67,74)."""
    mesh = M.duct_mesh(2, 3)
    sp = M.mixed_space(mesh, 1)
    bcs = M.duct_bcs(sp)
    w = M.duct_state(sp)
    form = oracle.Form(flavour=0, gdim=3, vdeg=1, nu=0.1)
    marker, value, mult = oracle.bc_arrays(sp.n_dofs, [b[0] for b in bcs], [b[1] for b in bcs])
    assert mult.max() == 2                                      # wall/inlet rim dofs are held twice
    indptr, indices = oracle.build_pattern(sp.dofmap, sp.n_dofs)
    vals = oracle.assemble_jacobian(form, mesh.x, mesh.cells, sp.dofmap, w, indptr, indices, marker, mult)
    vals0 = oracle.assemble_jacobian(form, mesh.x, mesh.cells, sp.dofmap, w, indptr, indices)
    import scipy.sparse as sps
    A = sps.csr_matrix((vals, indices, indptr), shape=(sp.n_dofs,) * 2)
    A0 = sps.csr_matrix((vals0, indices, indptr), shape=(sp.n_dofs,) * 2)
    bc = np.nonzero(marker)[0]
    D = A[bc][:, bc].toarray()
    np.testing.assert_array_equal(D, np.diag(mult[bc].astype(float)))
    free = np.nonzero(marker == 0)[0]
    assert abs(A[bc][:, free]).max() == 0 and abs(A[free][:, bc]).max() == 0
    np.testing.assert_allclose(A[free][:, free].toarray(), A0[free][:, free].toarray(), rtol=0, atol=1e-15)  # summation order (OpenMP)
    # residual: lifting uses the un-zeroed Jacobian
    b_nolift = oracle.assemble_residual(form, mesh.x, mesh.cells, sp.dofmap, w, lifting=False)
    b = oracle.assemble_residual(form, mesh.x, mesh.cells, sp.dofmap, w, marker, value)
    delta = np.zeros(sp.n_dofs)
    delta[bc] = value[bc] - w[bc]
    np.testing.assert_allclose(b, b_nolift + A0 @ delta, rtol=0, atol=1e-13 * np.abs(b).max())
    oracle.set_bc(b, [x[0] for x in bcs], [x[1] for x in bcs], w)
    np.testing.assert_allclose(b[bc], w[bc] - value[bc], rtol=0, atol=0)
    # SpMV restatement against scipy
    xv = np.random.default_rng(0).standard_normal(sp.n_dofs)
    np.testing.assert_allclose(oracle.spmv(indptr, indices, vals, xv), A @ xv, rtol=0, atol=1e-13)


def test_ugn_zero_velocity_cell_is_finite(oracle):
    """SURVEY A.4 NaN hazard: d|u| is defined as 0 where |u| = 0."""
    form = oracle.Form(flavour=1, gdim=2, vdeg=1, nu=0.01)
    x = np.array([[0, 0, 0], [0.1, 0, 0], [0, 0.1, 0]], dtype=float)
    w = np.zeros(9)
    w[6:] = [0.3, -0.2, 0.5]
    Ae, be = oracle.element(form, x, w)
    assert np.isfinite(Ae).all() and np.isfinite(be).all()


def test_oracle_reproduces_the_dfg_2d_1_reference_values(oracle):
    """A pin that comes from the reference side (SURVEY 8c): DFG_2D_Validation.py:202-203 holds Cd = 5.57953523384 and
    Cl = 0.010618948146 for the UGN-stabilised P1-P1 solve of the 2D-1 benchmark.  The oracle's UGN form + dolfinx-semantics
    assembly, driven by Newton on a 5 462-cell triangulation of the same domain, must land on them."""
    import _pins as P
    m, sp, bcs, obstacle = P.dfg_problem()
    r = P.dfg_solve(P.OracleBackend(oracle, m, sp, bcs), sp, bcs, obstacle)
    assert r["newton"][-1][1] < 1e-8, r["newton"]
    assert abs(r["cd"] / P.DFG_CD - 1.0) < 0.01, r["cd"]
    assert abs(r["cl"] / P.DFG_CL - 1.0) < 0.05, r["cl"]
    assert abs(r["dp"] / P.DFG_DP - 1.0) < 0.04, r["dp"]
