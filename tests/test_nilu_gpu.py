"""Point ILU(0) in the caller's order of the dofs (csrc/nilu.cu, pc = 7), PETSc's default preconditioner as PETSc eliminates it:
the application against the NumPy ILU(0) in natural order (oracle/pilu_ref.pilu0 with colour = arange(n)), the sweep depths against
tests/_nilu_ref.py, the zero-pivot row, the solves against a sparse LU and the reference pins, determinism, alternation with pc = 6,
and the two-rank solve."""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sps
import scipy.sparse.linalg as spla

import _meshes
import _nilu_ref
import _pins as P
from oracle import pilu_ref
from stabilized_navier_stokes_flow_fenicsx_b200 import mesh as M
from stabilized_navier_stokes_flow_fenicsx_b200._lib import NsgpuError
from stabilized_navier_stokes_flow_fenicsx_b200.assembler import NSAssembler

pytestmark = pytest.mark.gpu

CASES = ["cavity_ugn_p1", "duct_gmetric_p2", "duct_stokes_p2_beta0", "duct_gmetric_p1_scattered", "delaunay_tets_ugn_p1"]


def _dirichlet_state(n, bcs):
    w = np.zeros(n)
    for d, v in bcs:
        w[d] = v
    return w


def _renumbered(sp, bcs, w, new_of_old):
    """dofmap, bcs, state and pressure flags of a space under the caller's numbering new = new_of_old[old]."""
    dofmap = new_of_old[sp.dofmap].astype(np.int32)
    bcs = [(new_of_old[d].astype(np.int32), v) for d, v in bcs]
    w2 = np.empty(sp.n_dofs); w2[new_of_old] = w
    is_p = np.empty(sp.n_dofs, dtype=bool); is_p[new_of_old] = sp.dof_comp == sp.mesh.gdim
    return dofmap, bcs, w2, is_p


def _case(name, new_of_old=None):
    """(assembler, CSR pattern + values in the caller's numbering, right-hand side, caller numbering of the vertex-blocked dofs) of a
    Newton-step system.  new_of_old renumbers the space's dofs."""
    if name == "cavity_ugn_p1":
        m = M.create_rectangle_tris(24, 24); sp = M.mixed_space(m, 1)
        bcs, w, fk = M.cavity_bcs(sp), M.cavity_state(sp), dict(flavour=1, nu=0.01)
    elif name == "duct_gmetric_p2":
        m = M.duct_mesh(3, 8); sp = M.mixed_space(m, 2)
        bcs, w, fk = M.duct_bcs(sp), M.duct_state(sp), dict(flavour=0, nu=0.02)
    elif name == "duct_stokes_p2_beta0":                               # StokesFlow/DuctStokesFlow.py:188-192: zero pressure diagonal
        m = M.duct_mesh(4, 12); sp = M.mixed_space(m, 2)
        bcs = P.uniform_inlet_duct_bcs(sp)
        w, fk = _dirichlet_state(sp.n_dofs, bcs), dict(flavour=2, nu=1.0, alpha=1.0, sp=-1.0, beta=0.0)
    elif name == "duct_gmetric_p1_scattered":                          # dofs of a vertex scattered: the library renumbers internally
        m = M.duct_mesh(4, 10); sp = M.mixed_space(m, 1)
        bcs, w, fk = M.duct_bcs(sp), M.duct_state(sp), dict(flavour=0, nu=0.1)
        if new_of_old is None:
            new_of_old = np.random.default_rng(3).permutation(sp.n_dofs).astype(np.int32)
    else:                                                              # unstructured tetrahedra
        m = _meshes.delaunay_tets(8); sp = M.mixed_space(m, 1)
        bcs, w, fk = _meshes.box_bcs(sp), _meshes.smooth_state(sp), dict(flavour=1, nu=0.05)
    if new_of_old is None:
        new_of_old = np.arange(sp.n_dofs, dtype=np.int32)
    dofmap, bcs, w, _ = _renumbered(sp, bcs, w, new_of_old)
    asm = NSAssembler(m.x, m.cells, dofmap, vdeg=sp.vdeg)
    asm.set_form(**fk); asm.set_bcs(bcs)
    indptr, indices = asm.create_matrix()
    vals, F = asm.jacobian_residual(w)
    return asm, indptr, indices, vals, F[: sp.n_dofs], new_of_old


def _natural(indptr, indices, vals, n):
    """ILU(0) restatement in the caller's order, or the row of its zero pivot"""
    try:
        return pilu_ref.pilu0(indptr, indices, vals, np.arange(n)), None
    except ZeroDivisionError as e:
        return None, int(str(e).split()[-1])


@pytest.mark.parametrize("name", CASES)
def test_nilu_application_matches_ilu0_in_natural_order(name):
    asm, indptr, indices, vals, F, new_of_old = _case(name)
    n = asm.n_owned
    r = np.random.default_rng(7).standard_normal(n)
    fac, bad = _natural(indptr, indices, vals, n)
    if fac is None:                                                   # natural order meets a zero pivot: the same row on the device
        with pytest.raises(NsgpuError, match=rf"zero pivot in row {bad}\b"):
            asm.nilu_apply(r)
        asm.close()
        return
    z = asm.nilu_apply(r)
    zr = pilu_ref.apply(fac, r)
    err = np.abs(z - zr).max() / np.abs(zr).max()
    print(f"{name}: {n} dofs, rel err {err:.2e}")
    assert err <= 1e-10, err
    if name == "duct_gmetric_p1_scattered":                           # the order follows the caller, not the internal vertex blocks
        blocked = np.argsort(new_of_old)                              # rank of caller dof c in the vertex-blocked numbering
        zb = pilu_ref.apply(pilu_ref.pilu0(indptr, indices, vals, blocked), r)
        assert np.abs(z - zb).max() > 1e-6 * np.abs(zb).max()
    asm.close()


@pytest.mark.parametrize("name", CASES)
def test_nilu_depth_matches_the_numpy_count(name):
    asm, indptr, indices, vals, F, _ = _case(name)
    d = asm.nilu_depth()
    ref = _nilu_ref.depth(indptr, indices, asm.n_owned)
    print(f"{name}: {asm.n_owned} dofs, depth {d}")
    assert d == ref
    asm.close()


def _stokes_numbering(pressure_first_dof):
    """Taylor-Hood Stokes duct numbered velocity dofs first, then pressure dofs; with pressure_first_dof, the pressure dof of that
    index is moved to just before the first of its velocity neighbours, which then all come after it: its pivot is a zero diagonal."""
    m = M.duct_mesh(4, 12); sp = M.mixed_space(m, 2)
    is_p = sp.dof_comp == 3
    order = np.concatenate([np.flatnonzero(~is_p), np.flatnonzero(is_p)])
    if pressure_first_dof is not None:
        p = np.flatnonzero(is_p)[pressure_first_dof]
        nbr = np.unique(sp.dofmap[np.any(sp.dofmap == p, axis=1)])
        order = order[order != p]
        at = np.flatnonzero(np.isin(order, nbr[~is_p[nbr]]))[0]
        order = np.insert(order, at, p)
    new_of_old = np.empty(sp.n_dofs, dtype=np.int32)
    new_of_old[order] = np.arange(sp.n_dofs)
    return new_of_old, (None if pressure_first_dof is None else int(new_of_old[p]))


def test_zero_pivot_row_matches_the_restatement():
    new_of_old, moved = _stokes_numbering(pressure_first_dof=40)
    asm, indptr, indices, vals, b, _ = _case("duct_stokes_p2_beta0", new_of_old)
    fac, bad = _natural(indptr, indices, vals, asm.n_owned)
    print(f"moved pressure dof at {moved}, restatement breaks down at row {bad}")
    assert fac is None and bad <= moved
    with pytest.raises(NsgpuError, match=rf"zero pivot in row {bad}\b"):
        asm.tfqmr(b, pc=7)
    with pytest.raises(NsgpuError, match=rf"zero pivot in row {bad}\b"):
        asm.nilu_apply(b)
    asm.close()
    # pressure dofs last: every pressure pivot carries its Schur term; both factorise, and the solve converges
    asm, indptr, indices, vals, b, _ = _case("duct_stokes_p2_beta0", _stokes_numbering(None)[0])
    n = asm.n_owned
    fac, bad = _natural(indptr, indices, vals, n)
    assert fac is not None
    r = np.random.default_rng(5).standard_normal(n)
    zr = pilu_ref.apply(fac, r)
    assert np.abs(asm.nilu_apply(r) - zr).max() <= 1e-10 * np.abs(zr).max()
    x, info = asm.tfqmr(b, rtol=1e-10, max_it=5000, pc=7)
    x_ref = spla.spsolve(sps.csr_matrix((vals, indices, indptr), shape=(n, n)).tocsc(), b)
    assert np.linalg.norm(x - x_ref) <= 1e-8 * np.linalg.norm(x_ref), info
    asm.close()


@pytest.mark.parametrize("name", [c for c in CASES if c != "duct_stokes_p2_beta0"])
def test_tfqmr_with_natural_order_ilu_matches_the_direct_solve(name):
    asm, indptr, indices, vals, b, _ = _case(name)
    n = asm.n_owned
    x_ref = spla.spsolve(sps.csr_matrix((vals, indices, indptr), shape=(n, n)).tocsc(), b)
    x7, i7 = asm.tfqmr(b, rtol=1e-10, max_it=5000, pc=7)
    x6, i6 = asm.tfqmr(b, rtol=1e-10, max_it=5000, pc=6)
    print(f"{name}: TFQMR iterations to rtol 1e-10: pc = 7 {i7['its']}, pc = 6 {i6['its']}")
    assert i7["rnorm"] <= 1e-9 * np.linalg.norm(b), i7
    assert np.linalg.norm(x7 - x_ref) <= 1e-8 * np.linalg.norm(x_ref), i7
    asm.close()


def test_determinism_and_alternation_with_pc6():
    name = "duct_gmetric_p1_scattered"
    asm, indptr, indices, vals, b, _ = _case(name)
    r = np.random.default_rng(11).standard_normal(asm.n_owned)
    zs = [asm.nilu_apply(r) for _ in range(5)]                       # five factorise-and-apply rounds
    assert all(np.array_equal(zs[0], z) for z in zs[1:])
    assert np.array_equal(zs[0], asm.nilu_apply(r, refactor=False))
    got = []
    for pc in (6, 7, 6, 7):
        got.append(asm.tfqmr(b, rtol=1e-10, max_it=5000, pc=pc))
    asm.close()
    for pc in (6, 7):
        fresh, _, _, _, bf, _ = _case(name)
        xf, inf = fresh.tfqmr(bf, rtol=1e-10, max_it=5000, pc=pc)
        fresh.close()
        for x, info in got[(pc == 7)::2]:
            assert np.array_equal(x, xf) and info["its"] == inf["its"], (pc, info, inf)


def test_dfg_2d_1_on_the_device_with_natural_order_ilu():
    """DFG_2D_Validation.py end to end through newton_dev(pc = 7): the Stokes guess, then the UGN Newton solve, every linear solve by
    TFQMR + ILU(0) in the caller's order on the device; drag, lift and pressure drop as tests/test_reference_pins.py."""
    m, sp, bcs, obstacle = P.dfg_problem()
    nu = 1e-3
    asm = NSAssembler(m.x, m.cells, sp.dofmap, vdeg=1)
    asm.set_bcs(bcs)
    asm.create_matrix(fetch=False)
    w = _dirichlet_state(sp.n_dofs, bcs)
    w_dev = asm.dev_alloc(8 * asm.n_cols)
    asm.h2d(w_dev, w)
    asm.set_form(flavour=2, nu=nu, alpha=nu, sp=1.0, beta=0.2 / nu)
    h_st = asm.newton_dev(w_dev, rtol=1e-10, atol=1e-12, max_it=3, ksp_rtol=1e-10, ksp_max_it=5000, pc=7, linesearch="basic")
    asm.set_form(flavour=1, nu=nu)
    h_ns = asm.newton_dev(w_dev, rtol=1e-10, atol=1e-10, max_it=30, ksp_rtol=1e-10, ksp_max_it=5000, pc=7)
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


def test_two_gpu_natural_order_ilu_solve():
    """Block Jacobi over two ranks with ILU(0) of each rank's block in its local order (needs >= 2 GPUs; skipped on the single-GPU
    tier): tests/multigpu_nilu_check.py under torchrun."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29619", os.path.join(root, "tests", "multigpu_nilu_check.py")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
