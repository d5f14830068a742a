"""Launched by torchrun (one rank per GPU): point evaluation and non-matching interpolation on a communicator, against the
multi-rank restatement (tests/_interp_dist_ref.eval_distributed) and the serial device calls on the unpartitioned meshes; the
status agreement of bad calls; the coarse-to-fine Newton start on the duct.  Exit code 0 = every check passed."""
import ctypes
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from oracle import interp_ref as R  # noqa: E402
from _interp_dist_ref import eval_distributed  # noqa: E402
from stabilized_navier_stokes_flow_fenicsx_b200 import distributed as D  # noqa: E402
from stabilized_navier_stokes_flow_fenicsx_b200 import mesh as M  # noqa: E402
from stabilized_navier_stokes_flow_fenicsx_b200.assembler import NSAssembler  # noqa: E402
import _meshes  # noqa: E402

DEV = int(os.environ.get("LOCAL_RANK", 0))
EINVAL = -1


def log(comm, msg):
    print(f"rank {comm.rank}/{comm.size}: {msg}", flush=True)


def dist_asm(part, comm, vdeg, bcs=True):
    """a context on the rank's partition with its own communicator, pattern and halo plan"""
    asm = NSAssembler(part.x, part.cells, part.dofmap, vdeg=vdeg, n_dofs_owned=part.n_owned, n_dofs_ghost=part.n_ghost,
                      n_cells_owned=part.n_cells_owned, device=DEV)
    asm.set_form(flavour=0, nu=0.1)
    if bcs and part.bcs:
        asm.set_bcs(part.bcs)
    D.attach(asm, part, comm)
    D.finish_pattern_exchange(asm, part, comm)
    return asm


def serial_asm(mesh, sp):
    return NSAssembler(mesh.x, mesh.cells, sp.dofmap, vdeg=sp.vdeg, device=DEV)


def slab_ranks(mesh, size, axis):
    c = mesh.x[mesh.cells, axis].mean(axis=1)
    lo, hi = mesh.x[:, axis].min(), mesh.x[:, axis].max()
    return np.minimum(((c - lo) / (hi - lo) * size).astype(np.int64), size - 1)


def check_eval(comm):
    rank, size = comm.rank, comm.size
    n_cross, n_long, pad = 6, 12, 0.05
    parts = [D.duct_partition(n_cross, n_long, r, size) for r in range(size)]
    part = parts[rank]
    src = [R.Source(p.x, p.cells, p.dofmap, 1, p.w) for p in parts]
    asm = dist_asm(part, comm, 1)
    rng = np.random.default_rng(100 + rank)
    if rank == 1:
        pts = np.zeros((0, 3))                                           # this rank asks about nothing
    else:
        cuts = 4.0 * np.array([k0 for k0, _ in D.slab_ranges(n_long, size)] + [n_long]) / n_long
        inner = np.column_stack([rng.uniform(0, 4, 300), rng.uniform(-0.5, 0.5, (300, 2))])
        iface = np.column_stack([rng.choice(cuts, 60), rng.uniform(-0.5, 0.5, (60, 2))])
        band = np.column_stack([rng.uniform(0, 4, 60), np.full(60, 0.5 + 0.5 * pad), rng.uniform(-0.45, 0.45, 60)])
        ends = np.column_stack([np.full(30, -0.5 * pad), rng.uniform(-0.45, 0.45, (30, 2))])
        out = np.column_stack([rng.uniform(0, 4, 30), np.full(30, 0.5 + 3 * pad), rng.uniform(-0.5, 0.5, 30)])
        pts = np.concatenate([inner, iface, band, ends, out])
    values, cells = asm.eval(part.w, pts, tol=1e-12, padding=pad)
    ask = [np.zeros((0, 3))] * size
    ask[rank] = pts
    ref_v, ref_c, _ = eval_distributed(src, ask, tol=1e-12, padding=pad)[rank]
    np.testing.assert_array_equal(cells, ref_c)
    np.testing.assert_allclose(values, ref_v, rtol=0, atol=1e-12)
    # inside points against the serial device eval of the whole duct
    m = M.duct_mesh(n_cross, n_long); sp = M.mixed_space(m, 1)
    w = M.duct_state(sp, noise=0.0) + 1e-3 * np.random.default_rng(1234).standard_normal(sp.n_dofs)
    ser = serial_asm(m, sp)
    sv, sc = ser.eval(w, pts, tol=1e-12, padding=pad)
    inside = cells >= 0
    np.testing.assert_array_equal(sc >= 0, inside)
    np.testing.assert_allclose(values[inside], sv[inside], rtol=0, atol=1e-12)
    n_cls = [int((cells >= 0).sum()), int((cells <= -2).sum()), int((cells == -1).sum())]
    tot = [comm.sum(v) for v in n_cls]
    log(comm, f"eval: {len(pts)} points, inside / extrapolated / outside {n_cls} (all ranks {tot}), matches the restatement and serial")
    ser.close()
    return asm, part


def interp_case(comm, name, src_mesh, src_sp, dst_mesh, dst_sp, src_rank, dst_rank, w_src_serial, padding):
    """distributed interpolate vs the serial one; src_mesh / dst_mesh are the partitions themselves when src_rank is None (the
    duct's duct_partition), else partition_cells cuts the meshes by src_rank / dst_rank.  Returns (src asm, dst asm)."""
    rank, size = comm.rank, comm.size
    if src_rank is None:
        ps, pd = src_mesh, dst_mesh
        dst_serial_dof = pd.local_to_global
    else:
        ps = D.partition_cells(src_mesh, src_sp, src_rank, rank, size, w=w_src_serial)
        pd = D.partition_cells(dst_mesh, dst_sp, dst_rank, rank, size)
        dst_serial_dof = pd.meta["serial_dof"]
    a_src = dist_asm(ps, comm, src_sp.vdeg, bcs=False)
    a_dst = dist_asm(pd, comm, dst_sp.vdeg, bcs=False)
    w1, info1 = a_dst.interpolate_nonmatching(a_src, ps.w, tol=1e-12, padding=padding)
    w2, info2 = a_dst.interpolate_nonmatching(a_src, ps.w, tol=1e-12, padding=padding)
    assert np.array_equal(w1.view(np.int64), w2.view(np.int64)) and info1 == info2, f"{name}: two calls differ"
    s_src, s_dst = serial_asm(src_sp.mesh, src_sp), serial_asm(dst_sp.mesh, dst_sp)
    w_ref, info_ref = s_dst.interpolate_nonmatching(s_src, w_src_serial, tol=1e-12, padding=padding)
    s_src.close(); s_dst.close()
    err = np.abs(w1 - w_ref[dst_serial_dof]).max()
    assert err <= 1e-12, f"{name}: max |w - serial| = {err:.3e}"
    assert info1 == info_ref, f"{name}: counts {info1} != serial {info_ref}"
    # ghost entries are bitwise the owners' values
    import torch.distributed as dist
    own = {int(g): float(v) for g, v in zip(pd.local_to_global[:pd.n_owned], w1[:pd.n_owned])}
    allown = [None] * size
    dist.all_gather_object(allown, own)
    for k in range(pd.n_owned, pd.n_owned + pd.n_ghost):
        g, o = int(pd.local_to_global[k]), int(pd.ghost_owner[k - pd.n_owned])
        assert allown[o][g] == w1[k], f"{name}: ghost {k} differs from its owner's value"
    log(comm, f"interpolate {name}: {pd.n_owned} owned + {pd.n_ghost} ghost dofs, max err {err:.1e} vs serial, counts {info1}, "
              f"ghosts bitwise, two calls bitwise")
    return a_src, a_dst


def check_interpolate(comm):
    size = comm.size
    # P1 -> P1 duct slabs whose cuts do not line up
    cs, cf = (4, 9), (6, 16)
    ms, mf = M.duct_mesh(*cs), M.duct_mesh(*cf)
    ss, sf = M.mixed_space(ms, 1), M.mixed_space(mf, 1)
    ws = M.duct_state(ss, noise=0.0) + 1e-3 * np.random.default_rng(1234).standard_normal(ss.n_dofs)
    ps, pf = D.duct_partition(*cs, comm.rank, size), D.duct_partition(*cf, comm.rank, size)
    np.testing.assert_allclose(ps.w, ws[ps.local_to_global], rtol=0, atol=1e-14)
    a, b = interp_case(comm, "P1->P1 duct", ps, ss, pf, sf, None, None, ws, 0.0)
    a.close(); b.close()
    # P1 -> P2 tetrahedra: Delaunay source cut along x, structured destination cut along y
    ms = _meshes.delaunay_tets(8); ss = M.mixed_space(ms, 1)
    md = M.create_box_tets((4, 4, 4)); sd = M.mixed_space(md, 2)
    ws = _meshes.smooth_state(ss)
    a, b = interp_case(comm, "P1->P2 tets", ms, ss, md, sd, slab_ranks(ms, size, 0), slab_ranks(md, size, 1), ws, 1e-3)
    a.close(); b.close()
    # P1 -> P1 triangles
    ms = _meshes.delaunay_tris(14); ss = M.mixed_space(ms, 1)
    md = M.create_rectangle_tris(9, 9); sd = M.mixed_space(md, 1)
    ws = _meshes.smooth_state(ss)
    a, b = interp_case(comm, "P1->P1 triangles", ms, ss, md, sd, slab_ranks(ms, size, 1), slab_ranks(md, size, 0), ws, 1e-3)
    a.close(); b.close()


def check_status(comm, asm, part):
    """bad calls: every rank returns the same code without hanging; a correct call succeeds afterwards"""
    lib = asm.lib
    w = np.ascontiguousarray(part.w)
    wp = w.ctypes.data_as(ctypes.c_void_p)
    out = np.zeros(part.n_owned + part.n_ghost)
    op = out.ctypes.data_as(ctypes.c_void_p)
    # source and destination with different nranks: a one-rank source
    single = NSAssembler(part.x, part.cells, part.dofmap, vdeg=1, device=DEV)
    rc = lib.nsgpu_interpolate(single.ctx, wp, asm.ctx, op, 1e-12, 0.0, None, None)
    assert rc == EINVAL, f"mismatched nranks: rc {rc}"
    # a NULL array on rank 0 only
    rc = lib.nsgpu_interpolate(asm.ctx, None if comm.rank == 0 else wp, asm.ctx, op, 1e-12, 0.0, None, None)
    assert rc == EINVAL, f"NULL w_src on rank 0: rc {rc}"
    pts = np.array([[1.0, 0.0, 0.0]])
    vals = np.zeros((1, 4))
    rc = lib.nsgpu_eval(asm.ctx, wp, 1, pts.ctypes.data_as(ctypes.c_void_p), 1e-12, 0.0,
                        None if comm.rank == comm.size - 1 else vals.ctypes.data_as(ctypes.c_void_p), None)
    assert rc == EINVAL, f"NULL values on the last rank: rc {rc}"
    # the context stays usable
    w2, info = asm.interpolate_nonmatching(asm, w)
    n = part.n_owned + part.n_ghost
    assert np.abs(w2[:n] - w[:n]).max() <= 1e-12 and info == {"n_extrapolated": 0, "n_outside": 0}
    v, c = asm.eval(w, pts)
    assert c[0] >= -1
    single.close()
    log(comm, "status: mismatched nranks and one-rank NULL arrays give EINVAL on every rank; the next call succeeds")


def check_newton(comm):
    """coarse duct solved by newton_dev, interpolated onto the fine duct, newton_dev from there (counts recorded, not asserted)"""
    rank, size = comm.rank, comm.size
    runs = []
    ws = None
    for n_cross, n_long in ((4, 12), (8, 24)):
        part = D.duct_partition(n_cross, n_long, rank, size)
        asm = dist_asm(part, comm, 1)
        w_dev = asm.dev_alloc(8 * asm.n_cols)
        if ws is None:
            w0 = part.w.copy()
        else:
            a_src, w_src = ws
            w0, info = asm.interpolate_nonmatching(a_src, w_src)
            for dofs, vals in part.bcs:
                w0[dofs] = vals
        w = np.zeros(asm.n_cols)
        w[: len(w0)] = w0
        asm.h2d(w_dev, w)
        hist = asm.newton_dev(w_dev, rtol=1e-8, atol=1e-10, max_it=30, ksp_rtol=1e-8, ksp_max_it=5000, pc=6)
        asm.d2h(w, w_dev)
        asm.dev_free(w_dev)
        conv = hist[-1]["fnorm"] <= max(1e-10, 1e-8 * hist[0]["fnorm"])
        its = len(hist) - 1
        ksp = sum(h.get("ksp_its", 0) for h in hist)
        runs.append((n_cross, n_long, its, ksp, conv, hist[0]["fnorm"], hist[-1]["fnorm"]))
        if ws is not None:
            ws[0].close()
        ws = (asm, w[: part.n_owned + part.n_ghost].copy())
    ws[0].close()
    for n_cross, n_long, its, ksp, conv, f0, f1 in runs:
        log(comm, f"newton_dev duct {n_cross}x{n_long}: {its} Newton / {ksp} TFQMR iterations, |F| {f0:.2e} -> {f1:.2e}, converged {conv}")
    assert runs[-1][4], "the fine Newton solve from the interpolated coarse solution did not converge"


def main():
    import torch
    comm = D.Comm.from_env()
    name = torch.cuda.get_device_name(DEV)
    log(comm, f"device {name}")
    asm, part = check_eval(comm)
    check_interpolate(comm)
    check_status(comm, asm, part)
    asm.close()
    check_newton(comm)
    log(comm, "all checks passed")
    comm.close()


if __name__ == "__main__":
    main()
