"""Point evaluation and non-matching interpolation on the device (csrc/locate.cu: nsgpu_eval / nsgpu_interpolate) against exact
polynomials and the NumPy restatement (oracle/interp_ref.py), and the coarse-to-fine start of the DFG 2D-1 Newton solve."""
import ctypes

import numpy as np
import pytest
from scipy.spatial import Delaunay

import _pins as P
from oracle import interp_ref as R
from stabilized_navier_stokes_flow_fenicsx_b200 import mesh as M
from stabilized_navier_stokes_flow_fenicsx_b200._lib import NsgpuError
from stabilized_navier_stokes_flow_fenicsx_b200.assembler import NSAssembler
from test_interpolate_ref import poly_at, poly_state

pytestmark = pytest.mark.gpu


def jittered_square(n, seed):
    """Delaunay triangulation of a jittered n x n lattice of the unit square (boundary points stay on the boundary)"""
    g = np.linspace(0.0, 1.0, n + 1)
    X, Y = np.meshgrid(g, g, indexing="ij")
    pts = np.column_stack((X.ravel(), Y.ravel()))
    inner = (pts > 0.0).all(axis=1) & (pts < 1.0).all(axis=1)
    pts[inner] += np.random.default_rng(seed).uniform(-0.3, 0.3, size=(inner.sum(), 2)) / n
    T = Delaunay(pts).simplices.astype(np.int32)
    x = np.zeros((len(pts), 3)); x[:, :2] = pts
    return M.Mesh(2, x, T)


def asm_of(m, sp, **kw):
    return NSAssembler(m.x, m.cells, sp.dofmap, vdeg=sp.vdeg, **kw)


def ref_source(m, sp, w):
    return R.Source(m.x, m.cells, sp.dofmap, sp.vdeg, w)


CASES = {
    "tet_p1_to_p1": (lambda: M.duct_mesh(3, 8), 1, lambda: M.duct_mesh(4, 11), 1),
    "tet_p1_to_p2": (lambda: M.duct_mesh(3, 8), 1, lambda: M.duct_mesh(4, 11), 2),
    "tet_p2_to_p2": (lambda: M.duct_mesh(3, 8), 2, lambda: M.duct_mesh(4, 11), 2),
    "tri_p1_to_p1": (lambda: M.create_rectangle_tris(9, 7), 1, lambda: jittered_square(12, 1), 1),
    "tri_p2_to_p2": (lambda: jittered_square(8, 2), 2, lambda: M.create_rectangle_tris(11, 13), 2),
}


@pytest.mark.parametrize("name", list(CASES))
def test_interpolation_reproduces_polynomials_on_non_nested_meshes(name):
    ms, vs, md, vd = CASES[name]
    ms, md = ms(), md()
    sps_, spd = M.mixed_space(ms, vs), M.mixed_space(md, vd)
    src, dst = asm_of(ms, sps_), asm_of(md, spd)
    w, info = dst.interpolate_nonmatching(src, poly_state(sps_))
    exact = poly_at(spd.dof_x, md.gdim, vs)[np.arange(spd.n_dofs), spd.dof_comp]
    err = np.abs(w - exact).max() / np.abs(exact).max()
    print(f"{name}: {spd.n_dofs} destination dofs, max rel err {err:.2e}, {info}")
    assert info == {"n_extrapolated": 0, "n_outside": 0}
    assert err <= 1e-12
    src.close(); dst.close()


def _strictly_inside(ref, pts, codes, margin=1e-9):
    """points whose cell holds them with every barycentric coordinate > margin (no other cell contains them)"""
    ok = codes >= 0
    out = np.zeros(len(pts), dtype=bool)
    for i in np.flatnonzero(ok):
        out[i] = ref.bary(pts[i], np.array([codes[i]]))[0].min() > margin
    return out


@pytest.mark.parametrize("kind", ["duct_p2", "cavity_p1"])
def test_eval_and_interpolation_of_a_general_field_match_the_restatement(kind):
    if kind == "duct_p2":
        ms = M.duct_mesh(3, 8); sp = M.mixed_space(ms, 2); w = M.duct_state(sp)
        md = M.duct_mesh(4, 11); spd = M.mixed_space(md, 1)
        lo, hi = np.array([-0.1, -0.6, -0.6]), np.array([4.1, 0.6, 0.6])
    else:
        ms = M.create_rectangle_tris(10, 10); sp = M.mixed_space(ms, 1); w = M.cavity_state(sp)
        md = jittered_square(9, 4); spd = M.mixed_space(md, 2)
        lo, hi = np.array([-0.05, -0.05, 0.0]), np.array([1.05, 1.05, 0.0])
    src, dst = asm_of(ms, sp), asm_of(md, spd)
    ref = ref_source(ms, sp, w)
    scale = np.abs(w).max()
    pts = lo + (hi - lo) * np.random.default_rng(11).uniform(0.0, 1.0, size=(600, 3))
    vals, cells = src.eval(w, pts)
    rvals, rcodes = ref.eval(pts)
    assert (cells == -1).sum() > 10 and (cells >= 0).sum() > 300
    assert np.abs(vals - rvals).max() / scale <= 1e-12
    strict = _strictly_inside(ref, pts, rcodes)
    assert strict.sum() > 300 and np.array_equal(cells[strict], rcodes[strict])
    assert np.array_equal(cells == -1, rcodes == -1)
    wd, info = dst.interpolate_nonmatching(src, w)
    rw, ne, no = R.interpolate(ref, md.x, md.cells, spd.dofmap, spd.vdeg, spd.n_dofs)
    assert info == {"n_extrapolated": ne, "n_outside": no} == {"n_extrapolated": 0, "n_outside": 0}
    assert np.abs(wd - rw).max() / scale <= 1e-12
    src.close(); dst.close()


def test_dof_numbering_does_not_change_the_result():
    ms, md = M.duct_mesh(3, 8), M.duct_mesh(4, 11)
    sps_, spd = M.mixed_space(ms, 1), M.mixed_space(md, 1)
    w = M.duct_state(sps_)
    src, dst = asm_of(ms, sps_), asm_of(md, spd)
    base, _ = dst.interpolate_nonmatching(src, w)
    ps = np.random.default_rng(5).permutation(sps_.n_dofs).astype(np.int32)
    pd = np.random.default_rng(6).permutation(spd.n_dofs).astype(np.int32)
    src_p = NSAssembler(ms.x, ms.cells, ps[sps_.dofmap], vdeg=1)     # scattered numbering: renumbered inside the library
    dst_p = NSAssembler(md.x, md.cells, pd[spd.dofmap], vdeg=1)
    wp = np.empty_like(w); wp[ps] = w
    got, _ = dst_p.interpolate_nonmatching(src_p, wp)
    assert np.array_equal(got[pd], base)
    vals, cells = src.eval(w, spd.dof_x[:200])
    vals_p, cells_p = src_p.eval(wp, spd.dof_x[:200])
    assert np.array_equal(vals, vals_p) and np.array_equal(cells, cells_p)
    # device-pointer variant, asynchronous on the destination's stream
    ws_dev, wd_dev, cnt_dev = src_p.dev_alloc(8 * sps_.n_dofs), dst_p.dev_alloc(8 * spd.n_dofs), dst_p.dev_alloc(16)
    src_p.h2d(ws_dev, wp)
    dst_p.interpolate_nonmatching_dev(src_p, ws_dev, wd_dev, counts_dev=cnt_dev)
    out, cnt = np.empty(spd.n_dofs), np.empty(2, dtype=np.int64)
    dst_p.d2h(out, wd_dev); dst_p.d2h(cnt, cnt_dev)
    assert np.array_equal(out, got) and list(cnt) == [0, 0]
    n = 200
    p_dev, v_dev, c_dev = src_p.dev_alloc(24 * n), src_p.dev_alloc(32 * n), src_p.dev_alloc(4 * n)
    src_p.h2d(p_dev, np.ascontiguousarray(spd.dof_x[:n]))
    src_p.eval_dev(ws_dev, n, p_dev, v_dev, c_dev)
    vd, cd = np.empty((n, 4)), np.empty(n, dtype=np.int32)
    src_p.d2h(vd, v_dev); src_p.d2h(cd, c_dev)
    assert np.array_equal(vd, vals) and np.array_equal(cd, cells)
    for p in (ws_dev, p_dev, v_dev, c_dev):
        src_p.dev_free(p)
    dst_p.dev_free(wd_dev); dst_p.dev_free(cnt_dev)
    for a in (src, dst, src_p, dst_p):
        a.close()


def test_points_outside_the_source_are_zero_or_extrapolated():
    ms = M.duct_mesh(3, 8); sp = M.mixed_space(ms, 1); w = M.duct_state(sp)
    md = M.create_box_tets((13, 5, 5), p0=(-1e-3, -0.501, -0.501), p1=(4.001, 0.501, 0.501)); spd = M.mixed_space(md, 1)
    src, dst = asm_of(ms, sp), asm_of(md, spd)
    ref = ref_source(ms, sp, w)
    X = md.x
    layer = (X[:, 0] < 0.0) | (X[:, 0] > 4.0) | (np.abs(X[:, 1]) > 0.5) | (np.abs(X[:, 2]) > 0.5)
    scale = np.abs(w).max()
    wd, info = dst.interpolate_nonmatching(src, w)
    assert info == {"n_extrapolated": 0, "n_outside": int(layer.sum())}
    assert np.all(wd[np.isin(np.arange(spd.n_dofs) // 4, np.flatnonzero(layer))] == 0.0)
    rw, ne, no = R.interpolate(ref, md.x, md.cells, spd.dofmap, 1, spd.n_dofs)
    assert (ne, no) == (0, int(layer.sum())) and np.abs(wd - rw).max() / scale <= 1e-12
    vals, cells = src.eval(w, X)
    assert np.array_equal(cells == -1, layer) and np.all(vals[layer] == 0.0)
    wd2, info2 = dst.interpolate_nonmatching(src, w, padding=2e-3)
    assert info2 == {"n_extrapolated": int(layer.sum()), "n_outside": 0}
    rw2, ne2, no2 = R.interpolate(ref, md.x, md.cells, spd.dofmap, 1, spd.n_dofs, padding=2e-3)
    assert (ne2, no2) == (int(layer.sum()), 0)
    assert np.abs(wd2 - rw2).max() / scale <= 1e-12
    vals2, cells2 = src.eval(w, X, padding=2e-3)
    _, rcodes2 = ref.eval(X, padding=2e-3)
    assert np.all(cells2[layer] <= -2) and np.array_equal(cells2[layer], rcodes2[layer])
    src.close(); dst.close()


def test_bad_arguments_return_status_codes_and_leave_the_context_usable():
    ms = M.duct_mesh(2, 4); sp = M.mixed_space(ms, 1); w = M.duct_state(sp)
    mt = M.create_rectangle_tris(4, 4); spt = M.mixed_space(mt, 1)
    src, tri = asm_of(ms, sp), asm_of(mt, spt)
    lib = src.lib
    pts = np.ascontiguousarray(ms.x[:5])
    vals = np.empty((5, 4)); cells = np.empty(5, dtype=np.int32)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    assert lib.nsgpu_eval(src.ctx, None, 5, p(pts), 1e-12, 0.0, p(vals), p(cells)) == -1
    assert lib.nsgpu_eval(src.ctx, p(w), 5, None, 1e-12, 0.0, p(vals), p(cells)) == -1
    assert lib.nsgpu_eval(src.ctx, p(w), 5, p(pts), -1e-12, 0.0, p(vals), p(cells)) == -1
    assert lib.nsgpu_eval(src.ctx, p(w), 5, p(pts), 1e-12, -1.0, p(vals), p(cells)) == -1
    wt = np.empty(spt.n_dofs)
    assert lib.nsgpu_interpolate(src.ctx, p(w), tri.ctx, p(wt), 1e-12, 0.0, None, None) == -1          # gdim mismatch
    assert b"gdim" in lib.nsgpu_last_error(tri.ctx)
    assert lib.nsgpu_interpolate(src.ctx, None, src.ctx, p(w), 1e-12, 0.0, None, None) == -1
    assert lib.nsgpu_interpolate(src.ctx, p(w), src.ctx, p(np.empty_like(w)), -1.0, 0.0, None, None) == -1
    with pytest.raises(NsgpuError, match="non-negative"):
        src.eval(w, pts, tol=-1.0)
    vals, cells = src.eval(w, pts)                                   # still usable: the vertices are in the mesh
    assert np.all(cells >= 0)
    ref = ref_source(ms, sp, w)
    assert np.abs(vals - ref.eval(pts)[0]).max() <= 1e-12 * np.abs(w).max()
    src.close(); tri.close()


def _dirichlet_state(n, bcs):
    w = np.zeros(n)
    for d, v in bcs:
        w[d] = v
    return w


def _ns_solve(asm, w, bcs, nu, stokes):
    """newton_dev(pc = 6) on w (host, in/out): optionally the Stokes guess of _pins.dfg_solve first, then the UGN Navier-Stokes solve"""
    w_dev = asm.dev_alloc(8 * asm.n_cols)
    asm.h2d(w_dev, w)
    h_st = []
    if stokes:
        asm.set_form(flavour=2, nu=nu, alpha=nu, sp=1.0, beta=0.2 / nu)
        h_st = asm.newton_dev(w_dev, rtol=1e-10, atol=1e-12, max_it=3, ksp_rtol=1e-10, ksp_max_it=5000, pc=6, linesearch="basic")
    asm.set_form(flavour=1, nu=nu)
    h_ns = asm.newton_dev(w_dev, rtol=1e-10, atol=1e-10, max_it=30, ksp_rtol=1e-10, ksp_max_it=5000, pc=6)
    asm.d2h(w, w_dev)
    asm.dev_free(w_dev)
    return h_st, h_ns


def _its(h):
    return len(h) - 1, sum(e.get("ksp_its", 0) for e in h)


def test_dfg_2d_1_fine_newton_started_from_the_interpolated_coarse_solution():
    """NavierStokesChannelFlow.py's solve_NS_flow pattern on DFG 2D-1: solve on a coarse mesh, interpolate_nonmatching onto the fine
    mesh, Newton on the fine mesh from the interpolant (off the Dirichlet values: lifting on the first iterate); drag, lift and the
    pressure drop uh.eval'd at (0.15, 0.2) and (0.25, 0.2) as DFG_2D_Validation.py reports it."""
    nu = 1e-3
    mc = M.dfg_cylinder_mesh(h_far=0.04, n_cyl=48); spc = M.mixed_space(mc, 1); bcs_c, _ = M.dfg_bcs(spc)
    coarse = asm_of(mc, spc)
    coarse.set_bcs(bcs_c); coarse.create_matrix(fetch=False)
    wc = _dirichlet_state(spc.n_dofs, bcs_c)
    _, hc = _ns_solve(coarse, wc, bcs_c, nu, stokes=True)
    assert hc[-1]["fnorm"] <= max(1e-10, 1e-10 * hc[0]["fnorm"]), hc

    m, sp, bcs, obstacle = P.dfg_problem()
    fine = asm_of(m, sp)
    w0, info = fine.interpolate_nonmatching(coarse, wc, padding=1e-3)
    coarse.close()
    print("interpolation", info)
    assert info["n_outside"] == 0
    fine.set_bcs(bcs); fine.create_matrix(fetch=False)
    w = w0.copy()
    _, h_int = _ns_solve(fine, w, bcs, nu, stokes=False)
    assert h_int[-1]["fnorm"] <= max(1e-10, 1e-10 * h_int[0]["fnorm"]), h_int

    ws = _dirichlet_state(sp.n_dofs, bcs)                            # the Stokes-start run of test_dfg_2d_1_on_the_device_with_point_ilu
    h_st, h_ns = _ns_solve(fine, ws, bcs, nu, stokes=True)
    print(f"fine mesh Newton / Krylov iterations: from the interpolated coarse solution {_its(h_int)}, "
          f"from the Stokes guess {_its(h_ns)} (+ Stokes {_its(h_st)})")

    (vals, cells) = fine.eval(w, np.array([[0.15, 0.2, 0.0], [0.25, 0.2, 0.0]]))
    assert np.all(cells >= 0)
    dp = vals[0, 2] - vals[1, 2]
    fine.set_bcs([])
    Rv = fine.residual(w)
    fine.close()
    scale = 2.0 / (0.1 * 0.2 ** 2)
    cd = scale * -Rv[obstacle[sp.dof_comp[obstacle] == 0]].sum()
    cl = scale * -Rv[obstacle[sp.dof_comp[obstacle] == 1]].sum()
    print(f"Cd {cd:.5f} Cl {cl:.6f} dp {dp:.5f}")
    assert abs(cd / P.DFG_CD - 1.0) < 0.01, cd
    assert abs(cl / P.DFG_CL - 1.0) < 0.05, cl
    assert abs(dp / P.DFG_DP - 1.0) < 0.04, dp
