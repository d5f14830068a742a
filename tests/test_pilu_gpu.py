"""Multicolour point ILU(0) preconditioner of the device-resident TFQMR (csrc/pilu.cu, pc = 6) on the spaces pc = 5 does not cover:
the factorisation against the NumPy restatement of ILU(0) in the exported elimination order (oracle/pilu_ref.py), the solves
against a sparse LU, the reference pins solved on the device, the zero-pivot status, and the two-rank solve."""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sps
import scipy.sparse.linalg as spla

import _pins as P
from oracle import colour_ref, pilu_ref
from stabilized_navier_stokes_flow_fenicsx_b200 import mesh as M
from stabilized_navier_stokes_flow_fenicsx_b200._lib import NsgpuError
from stabilized_navier_stokes_flow_fenicsx_b200.assembler import NSAssembler

pytestmark = pytest.mark.gpu

CASES = ["cavity_ugn_p1", "duct_gmetric_p2", "duct_stokes_p2_beta0", "duct_gmetric_p1_scattered"]


def _dirichlet_state(n, bcs):
    w = np.zeros(n)
    for d, v in bcs:
        w[d] = v
    return w


def _case(name, options=None):
    """(assembler, CSR pattern + values in the caller's numbering, right-hand side, pressure flag per dof) of a Newton-step system."""
    if name == "cavity_ugn_p1":
        m = M.create_rectangle_tris(24, 24); sp = M.mixed_space(m, 1)
        bcs, w, fk = M.cavity_bcs(sp), M.cavity_state(sp), dict(flavour=1, nu=0.01)
        dofmap, is_p = sp.dofmap, sp.dof_comp == 2
    elif name == "duct_gmetric_p2":
        m = M.duct_mesh(3, 8); sp = M.mixed_space(m, 2)
        bcs, w, fk = M.duct_bcs(sp), M.duct_state(sp), dict(flavour=0, nu=0.02)
        dofmap, is_p = sp.dofmap, sp.dof_comp == 3
    elif name == "duct_stokes_p2_beta0":                               # StokesFlow/DuctStokesFlow.py:188-192: zero pressure diagonal
        m = M.duct_mesh(4, 12); sp = M.mixed_space(m, 2)
        bcs = P.uniform_inlet_duct_bcs(sp)
        w, fk = _dirichlet_state(sp.n_dofs, bcs), dict(flavour=2, nu=1.0, alpha=1.0, sp=-1.0, beta=0.0)
        dofmap, is_p = sp.dofmap, sp.dof_comp == 3
    else:                                                              # dofs of a vertex scattered: the library renumbers internally
        m = M.duct_mesh(4, 10); sp = M.mixed_space(m, 1)
        perm = np.random.default_rng(3).permutation(sp.n_dofs).astype(np.int32)
        dofmap = perm[sp.dofmap]
        bcs = [(perm[d], v) for d, v in M.duct_bcs(sp)]
        w = np.empty(sp.n_dofs); w[perm] = M.duct_state(sp)
        is_p = np.empty(sp.n_dofs, dtype=bool); is_p[perm] = sp.dof_comp == 3
        fk = dict(flavour=0, nu=0.1)
    asm = NSAssembler(m.x, m.cells, dofmap, vdeg=sp.vdeg, options=options)
    asm.set_form(**fk); asm.set_bcs(bcs)
    indptr, indices = asm.create_matrix()
    vals, F = asm.jacobian_residual(w)
    return asm, indptr, indices, vals, F[: sp.n_dofs], is_p


@pytest.mark.parametrize("name", CASES)
def test_pilu_application_matches_the_ilu0_restatement(name):
    asm, indptr, indices, vals, F, is_p = _case(name)
    n = asm.n_owned
    r = np.random.default_rng(7).standard_normal(n)
    z = asm.pilu_apply(r)
    colour, nc, nvc = asm.pilu_colours()
    print(f"{name}: {n} dofs, {nc} colours ({nvc} velocity)")
    assert nc <= 1024 and colour.min() == 0 and colour.max() == nc - 1
    # a proper colouring of the pattern graph, velocity colours below every pressure colour
    rows = np.repeat(np.arange(n), np.diff(indptr[: n + 1]))
    cols = indices[: indptr[n]]
    off = (cols < n) & (cols != rows)
    assert np.all(colour[rows[off]] != colour[cols[off]])
    assert colour[~is_p].max() == nvc - 1 and colour[is_p].min() == nvc
    zr = pilu_ref.apply(pilu_ref.pilu0(indptr, indices, vals, colour), r)
    assert np.abs(z - zr).max() <= 1e-10 * np.abs(zr).max(), np.abs(z - zr).max() / np.abs(zr).max()
    assert np.array_equal(z, asm.pilu_apply(r))                       # same colouring, same factor: bitwise reproducible
    assert np.array_equal(z, asm.pilu_apply(r, refactor=False))
    asm.close()


@pytest.mark.parametrize("name", CASES[:3])
def test_pilu_colours_match_the_colouring_restatement(name):
    asm, indptr, indices, vals, F, is_p = _case(name, options={"renumber": 0})     # internal numbering = the caller's
    colour, nc, nvc = asm.pilu_colours()
    ref = colour_ref.colour(indptr, indices, asm.n_owned, cls=is_p)
    assert np.array_equal(colour, ref)
    assert nc == ref.max() + 1 and nvc == ref[~is_p].max() + 1
    asm.close()


@pytest.mark.parametrize("name", CASES)
def test_tfqmr_with_point_ilu_matches_the_direct_solve(name):
    asm, indptr, indices, vals, b, is_p = _case(name)
    n = asm.n_owned
    A = sps.csr_matrix((vals, indices, indptr), shape=(n, n)).tocsc()
    x_ref = spla.spsolve(A, b)
    x6, i6 = asm.tfqmr(b, rtol=1e-10, max_it=5000, pc=6)
    x1, i1 = asm.tfqmr(b, rtol=1e-10, max_it=5000, pc=1)
    print(f"{name}: TFQMR iterations to rtol 1e-10: pc = 6 {i6['its']}, pc = 1 {i1['its']} (rnorm {i1['rnorm']:.2e} / ||b|| {np.linalg.norm(b):.2e})")
    assert i6["rnorm"] <= 1e-9 * np.linalg.norm(b), i6
    assert np.linalg.norm(x6 - x_ref) <= 1e-8 * np.linalg.norm(x_ref), i6
    if name in ("cavity_ugn_p1", "duct_gmetric_p2"):
        assert i6["its"] < 0.5 * i1["its"], (i6, i1)
    if name == "duct_stokes_p2_beta0":                                 # Jacobi has no pressure diagonal to invert here
        converged1 = i1["rnorm"] <= 1e-9 * np.linalg.norm(b) and np.linalg.norm(x1 - x_ref) <= 1e-8 * np.linalg.norm(x_ref)
        assert not converged1 or i1["its"] > 2 * i6["its"], (i6, i1)
    asm.close()


def test_zero_pivot_is_reported_and_the_context_recovers():
    asm, indptr, indices, vals, b, is_p = _case("duct_gmetric_p1_scattered")
    n = asm.n_owned
    asm.set_values(np.zeros(asm.nnz))
    with pytest.raises(NsgpuError, match=r"zero pivot in row \d+"):
        asm.tfqmr(b, pc=6)
    with pytest.raises(NsgpuError, match="zero pivot"):
        asm.pilu_apply(b)
    b_dev, x_dev = asm.dev_alloc(8 * n), asm.dev_alloc(8 * asm.n_cols)
    asm.h2d(b_dev, b); asm.h2d(x_dev, np.ones(asm.n_cols))
    with pytest.raises(NsgpuError, match="zero pivot"):
        asm.tfqmr_dev(b_dev, x_dev, pc=6)
    xo = np.empty(asm.n_cols)
    asm.d2h(xo, x_dev)
    assert np.all(np.isfinite(xo))                                     # nothing of the failed factor reached the output
    asm.set_values(vals)
    x, info = asm.tfqmr(b, rtol=1e-10, max_it=5000, pc=6)
    x_ref = spla.spsolve(sps.csr_matrix((vals, indices, indptr), shape=(n, n)).tocsc(), b)
    assert np.linalg.norm(x - x_ref) <= 1e-8 * np.linalg.norm(x_ref), info
    asm.dev_free(b_dev); asm.dev_free(x_dev)
    asm.close()


def test_dfg_2d_1_on_the_device_with_point_ilu():
    """DFG_2D_Validation.py end to end through newton_dev(pc = 6): the Stokes guess of _pins.dfg_solve, then the UGN Newton solve,
    every linear solve by TFQMR + point ILU(0) on the device (no host LU); drag, lift and pressure drop as tests/test_reference_pins.py."""
    m, sp, bcs, obstacle = P.dfg_problem()
    nu = 1e-3
    asm = NSAssembler(m.x, m.cells, sp.dofmap, vdeg=1)
    asm.set_bcs(bcs)
    asm.create_matrix(fetch=False)
    w = _dirichlet_state(sp.n_dofs, bcs)
    w_dev = asm.dev_alloc(8 * asm.n_cols)
    asm.h2d(w_dev, w)
    asm.set_form(flavour=2, nu=nu, alpha=nu, sp=1.0, beta=0.2 / nu)
    h_st = asm.newton_dev(w_dev, rtol=1e-10, atol=1e-12, max_it=3, ksp_rtol=1e-10, ksp_max_it=5000, pc=6, linesearch="basic")
    asm.set_form(flavour=1, nu=nu)
    h_ns = asm.newton_dev(w_dev, rtol=1e-10, atol=1e-10, max_it=30, ksp_rtol=1e-10, ksp_max_it=5000, pc=6)
    asm.d2h(w, w_dev)
    asm.dev_free(w_dev)
    print("stokes", h_st, "\nnewton", h_ns)
    assert h_ns[-1]["fnorm"] <= max(1e-10, 1e-10 * h_ns[0]["fnorm"]), h_ns
    asm.set_bcs([])
    R = asm.residual(w)
    asm.close()
    fx = -R[obstacle[sp.dof_comp[obstacle] == 0]].sum()
    fy = -R[obstacle[sp.dof_comp[obstacle] == 1]].sum()
    scale = 2.0 / (0.1 * 0.2 ** 2)
    from scipy.spatial import cKDTree
    pv = np.flatnonzero(sp.dof_comp == 2)
    tree = cKDTree(sp.dof_x[pv][:, :2])
    dp = w[pv[tree.query([0.15, 0.2])[1]]] - w[pv[tree.query([0.25, 0.2])[1]]]
    cd, cl = scale * fx, scale * fy
    print(f"Cd {cd:.5f} Cl {cl:.6f} dp {dp:.5f}")
    assert abs(cd / P.DFG_CD - 1.0) < 0.01, cd
    assert abs(cl / P.DFG_CL - 1.0) < 0.05, cl
    assert abs(dp / P.DFG_DP - 1.0) < 0.04, dp


def test_duct_stokes_known_output_with_point_ilu():
    """StokesFlow/DuctStokesFlow.py's known output (tests/test_reference_pins.py) with the unstabilised Taylor-Hood operator solved by
    TFQMR + point ILU(0) on the device instead of a sparse LU: centreline / mean velocity at the outlet 2.0962."""
    m = M.duct_mesh(6, 24); sp = M.mixed_space(m, 2)
    bcs = P.uniform_inlet_duct_bcs(sp)
    asm = NSAssembler(m.x, m.cells, sp.dofmap, vdeg=2)
    asm.set_form(flavour=2, nu=1.0, alpha=1.0, sp=-1.0, beta=0.0)
    asm.set_bcs(bcs)
    asm.create_matrix(fetch=False)
    w = _dirichlet_state(sp.n_dofs, bcs)
    _, F = asm.jacobian_residual(w, fetch_vals=False)
    dx, info = asm.tfqmr(F, rtol=1e-10, max_it=5000, pc=6)
    asm.close()
    print("duct stokes", info)
    assert info["rnorm"] <= 1e-9 * np.linalg.norm(F), info
    w = w - dx
    outflux, area_o = P.plane_flux(m, sp, w, 4.0)
    X, c = sp.dof_x, sp.dof_comp
    ctr = np.flatnonzero((c == 0) & (np.abs(X[:, 0] - 4.0) < 1e-12) & (np.abs(X[:, 1]) < 1e-12) & (np.abs(X[:, 2]) < 1e-12))
    ratio = w[ctr[0]] / (outflux / area_o)
    assert abs(ratio - P.DUCT_RATIO) < 5e-3, ratio


def test_two_gpu_point_ilu_solve():
    """Block Jacobi over two ranks with point ILU(0) per rank (needs >= 2 GPUs; skipped on the single-GPU tier):
    tests/multigpu_pilu_check.py under torchrun."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29617", os.path.join(root, "tests", "multigpu_pilu_check.py")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
