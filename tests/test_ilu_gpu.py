"""Multicolour block ILU(0) preconditioner of the device-resident TFQMR (csrc/ilu.cu, pc = 5): the colouring against its NumPy
restatement (oracle/colour_ref.py), the factorisation against a NumPy restatement of block ILU(0) in the same elimination order
(oracle/ilu_ref.py), and the solve against a sparse LU."""
import numpy as np
import pytest
import scipy.sparse as sps
import scipy.sparse.linalg as spla
from scipy.spatial import Delaunay

from oracle import colour_ref, ilu_ref
from stabilized_navier_stokes_flow_fenicsx_b200 import mesh as M
from stabilized_navier_stokes_flow_fenicsx_b200.assembler import NSAssembler

pytestmark = pytest.mark.gpu


def _setup(n_cross, n_long, nu=0.1):
    m = M.duct_mesh(n_cross, n_long); sp = M.mixed_space(m, 1)
    asm = NSAssembler(m.x, m.cells, sp.dofmap, vdeg=1, options={"renumber": 0})    # vertex-blocked already: internal order = caller's
    asm.set_form(flavour=0, nu=nu); asm.set_bcs(M.duct_bcs(sp))
    indptr, indices = asm.create_matrix()
    vals = asm.jacobian(M.duct_state(sp))
    return m, sp, asm, indptr, indices, vals


def test_ilu_application_matches_the_block_ilu0_restatement():
    m, sp, asm, indptr, indices, vals = _setup(4, 10)
    rng = np.random.default_rng(3)
    r = rng.standard_normal(sp.n_dofs)
    z = asm.ilu_apply(r)
    colour, nc = asm.ilu_colours()
    assert 4 <= nc <= 20 and colour.min() == 0 and colour.max() == nc - 1
    # a proper colouring of the vertex graph of the matrix
    A = sps.csr_matrix((vals, indices, indptr), shape=(sp.n_dofs, sp.n_dofs))
    G = sps.coo_matrix((np.ones(A.nnz), (A.tocoo().row // 4, A.tocoo().col // 4))).tocsr().tocoo()
    off = G.row != G.col
    assert np.all(colour[G.row[off]] != colour[G.col[off]])
    assert np.array_equal(colour, colour_ref.colour(indptr, indices, sp.n_dofs // 4, shift=2))
    blocks, dinv, order, rank = ilu_ref.block_ilu0(indptr, indices, vals, colour)
    zr = ilu_ref.apply(blocks, dinv, order, rank, r)
    assert np.abs(z - zr).max() <= 1e-10 * np.abs(zr).max()
    # and it is a preconditioner: M^-1 A is much closer to the identity than the block-Jacobi one
    x = rng.standard_normal(sp.n_dofs)
    e_ilu = np.linalg.norm(asm.ilu_apply(A @ x, refactor=False) - x) / np.linalg.norm(x)
    assert e_ilu < 0.9
    z2 = asm.ilu_apply(r)                       # same colouring, same factors: bitwise reproducible
    assert np.array_equal(z, z2)
    asm.close()


def _delaunay_setup():
    """P1-P1 on a Delaunay tetrahedralisation of a 7x7x7 lattice with jittered interior points, velocity fixed on the boundary: block
    rows longer than 16, which the sixteen-lane factorisation kernel does not take."""
    g = np.linspace(0.0, 1.0, 7)
    x = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    inner = np.all((x > 0) & (x < 1), axis=1)
    x[inner] += np.random.default_rng(2).uniform(-0.04, 0.04, (inner.sum(), 3))
    tets = Delaunay(x).simplices
    p = x[tets]
    vol = np.abs(np.einsum("ij,ij->i", np.cross(p[:, 1] - p[:, 0], p[:, 2] - p[:, 0]), p[:, 3] - p[:, 0]))
    m = M.Mesh(3, x, np.ascontiguousarray(tets[vol > 1e-12], dtype=np.int32))     # drop the flat slivers on the faces of the cube
    sp = M.mixed_space(m, 1)
    bnd = np.flatnonzero(np.any((sp.dof_x == 0.0) | (sp.dof_x == 1.0), axis=1) & (sp.dof_comp < 3)).astype(np.int32)
    asm = NSAssembler(m.x, m.cells, sp.dofmap, vdeg=1, options={"renumber": 0})
    asm.set_form(flavour=0, nu=0.1); asm.set_bcs([(bnd, np.zeros(len(bnd)))])
    indptr, indices = asm.create_matrix()
    w = 0.1 * np.random.default_rng(4).standard_normal(sp.n_dofs)
    w[bnd] = 0.0
    vals = asm.jacobian(w)
    return sp, asm, indptr, indices, vals


def test_ilu_application_with_block_rows_longer_than_16():
    sp, asm, indptr, indices, vals = _delaunay_setup()
    assert (np.diff(indptr)[::4] // 4).max() > 16          # blocks in the longest block row
    r = np.random.default_rng(3).standard_normal(sp.n_dofs)
    z = asm.ilu_apply(r)
    colour, nc = asm.ilu_colours()
    assert np.array_equal(colour, colour_ref.colour(indptr, indices, sp.n_dofs // 4, shift=2))
    blocks, dinv, order, rank = ilu_ref.block_ilu0(indptr, indices, vals, colour)
    zr = ilu_ref.apply(blocks, dinv, order, rank, r)
    assert np.abs(z - zr).max() <= 1e-10 * np.abs(zr).max()
    assert np.array_equal(z, asm.ilu_apply(r))
    asm.close()


def test_tfqmr_with_ilu_converges_in_fewer_iterations_than_block_jacobi():
    m, sp, asm, indptr, indices, vals = _setup(8, 24)
    rng = np.random.default_rng(5)
    b = rng.standard_normal(sp.n_dofs)
    A = sps.csr_matrix((vals, indices, indptr), shape=(sp.n_dofs, sp.n_dofs)).tocsc()
    x_ref = spla.spsolve(A, b)
    x4, i4 = asm.tfqmr(b, rtol=1e-10, max_it=4000, pc=4)
    x5, i5 = asm.tfqmr(b, rtol=1e-10, max_it=4000, pc=5)
    assert np.abs(x4 - x_ref).max() <= 1e-6 * np.abs(x_ref).max()
    assert np.abs(x5 - x_ref).max() <= 1e-6 * np.abs(x_ref).max()
    assert i5["rnorm"] <= 1e-9 * np.linalg.norm(b)
    assert i5["its"] < 0.6 * i4["its"], (i4, i5)
    asm.close()


def test_ilu_needs_the_vertex_blocked_layout():
    m = M.create_rectangle_tris(8, 8); sp = M.mixed_space(m, 1)
    asm = NSAssembler(m.x, m.cells, sp.dofmap, vdeg=1)
    asm.set_form(flavour=1, nu=0.01); asm.set_bcs(M.cavity_bcs(sp))
    asm.create_matrix(fetch=False)
    asm.jacobian(M.cavity_state(sp), fetch=False)
    from stabilized_navier_stokes_flow_fenicsx_b200._lib import NsgpuError
    with pytest.raises(NsgpuError):
        asm.tfqmr(np.ones(sp.n_dofs), pc=5)
    asm.close()
