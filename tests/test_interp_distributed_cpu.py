"""CPU tests of the multi-rank point ownership restatement (tests/_interp_dist_ref.eval_distributed) against the serial
Source.eval, and of distributed.partition_cells: its plans reproduce the serial oracle J and F for P2-P1 tetrahedra and P1 triangles (gloo, 2 and 3
ranks, the same plan test test_distributed_cpu.py runs on duct_partition)."""
import os
import sys

import numpy as np
import pytest
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from oracle import interp_ref as R  # noqa: E402
from _interp_dist_ref import eval_distributed  # noqa: E402
from stabilized_navier_stokes_flow_fenicsx_b200 import distributed as D  # noqa: E402
from stabilized_navier_stokes_flow_fenicsx_b200 import mesh as M  # noqa: E402
import _meshes  # noqa: E402


def slab_ranks(mesh, size, axis=0):
    """cell -> rank by the centroid along one axis, in ``size`` slabs of equal width"""
    c = mesh.x[mesh.cells, axis].mean(axis=1)
    lo, hi = mesh.x[:, axis].min(), mesh.x[:, axis].max()
    return np.minimum(((c - lo) / (hi - lo) * size).astype(np.int64), size - 1)


def sources(mesh, sp, w, cell_rank, size):
    parts = [D.partition_cells(mesh, sp, cell_rank, r, size, w=w) for r in range(size)]
    return parts, [R.Source(p.x, p.cells, p.dofmap, sp.vdeg, p.w) for p in parts]


def classes(codes):
    return np.where(codes >= 0, 1, np.where(codes == -1, 0, 2))


MESHES = {
    "duct": lambda: M.mixed_space(M.duct_mesh(3, 8), 1),
    "delaunay_tets": lambda: M.mixed_space(_meshes.delaunay_tets(6), 2),
    "triangles": lambda: M.mixed_space(_meshes.delaunay_tris(12), 1),
}


@pytest.mark.parametrize("kind", sorted(MESHES))
@pytest.mark.parametrize("size", [2, 3])
def test_eval_distributed_matches_serial(kind, size):
    sp = MESHES[kind]()
    mesh = sp.mesh
    gd = mesh.gdim
    w = _meshes.smooth_state(sp)
    serial = R.Source(mesh.x, mesh.cells, sp.dofmap, sp.vdeg, w)
    _, src = sources(mesh, sp, w, slab_ranks(mesh, size, axis=1 if kind == "triangles" else 0), size)
    lo, hi = mesh.x.min(axis=0), mesh.x.max(axis=0)
    rng = np.random.default_rng(7 + size)
    pad = 0.05 * (hi - lo).max()
    pts = []
    for q in range(size):
        if q == 1:
            pts.append(np.zeros((0, 3)))          # a rank that asks about nothing
            continue
        p = lo - 2 * pad + (hi - lo + 4 * pad) * rng.random((40, 3))      # inside, in the padding band and outside
        v = mesh.x[rng.choice(mesh.n_vertices, 8, replace=False)]          # vertices: many on the rank interfaces
        p = np.concatenate([p, v])
        if gd == 2:
            p[:, 2] = 0.0
        pts.append(p)
    res = eval_distributed(src, pts, tol=1e-12, padding=pad)
    n_cls = np.zeros(3, dtype=np.int64)
    n_ref = np.zeros(3, dtype=np.int64)
    for q in range(size):
        values, codes, owner = res[q]
        assert values.shape == (len(pts[q]), gd + 1) and codes.shape == (len(pts[q]),)
        ref_v, ref_c = serial.eval(pts[q], tol=1e-12, padding=pad)
        np.testing.assert_array_equal(classes(codes), classes(ref_c))
        inside = codes >= 0
        np.testing.assert_allclose(values[inside], ref_v[inside], rtol=0, atol=1e-13)
        # local first: a point inside one of the asking rank's own cells never resolves elsewhere
        own = np.array([src[q].locate(p, 1e-12) >= 0 for p in pts[q]], dtype=bool)
        assert (owner[own] == q).all()
        n_cls += np.bincount(classes(codes), minlength=3)
        n_ref += np.bincount(classes(ref_c), minlength=3)
    assert (n_cls == n_ref).all()
    assert n_cls[1] > 0 and n_cls[0] > 0 and n_cls[2] > 0


def test_eval_distributed_interface_and_padding_ties():
    mesh = M.create_rectangle_tris(4, 4)
    sp = M.mixed_space(mesh, 1)
    w = _meshes.smooth_state(sp, noise=0.0)
    _, src = sources(mesh, sp, w, slab_ranks(mesh, 2), 2)
    # interface x = 0.5: inside on both ranks, each asking rank keeps its own cell; the P1 field is continuous there
    p = np.array([[0.5, 0.3, 0.0], [0.5, 0.5, 0.0]])
    r0, r1 = eval_distributed(src, [p, p], tol=1e-12)
    assert (r0[2] == 0).all() and (r1[2] == 1).all() and (r0[1] >= 0).all() and (r1[1] >= 0).all()
    np.testing.assert_allclose(r0[0], r1[0], rtol=0, atol=1e-14)
    # below the interface vertex (0.5, 0): the same distance to cells of both ranks -> the lower rank, from either side
    t = np.array([[0.5, -0.1, 0.0]])
    assert src[0].cell_dist(t[0]).min() == src[1].cell_dist(t[0]).min()
    for q in (0, 1):
        pts = [np.zeros((0, 3)), np.zeros((0, 3))]
        pts[q] = t
        v, c, o = eval_distributed(src, pts, tol=1e-12, padding=0.2)[q]
        assert o[0] == 0 and c[0] <= -2
    # beyond the padding: outside, value 0
    v, c, o = eval_distributed(src, [np.array([[0.5, -0.3, 0.0]]), np.zeros((0, 3))], tol=1e-12, padding=0.2)[0]
    assert c[0] == -1 and o[0] == -1 and (v == 0).all()


# ------------------------------------------------------------------------------------------------ partition_cells plans
def _plan_worker(rank, size, port, kind, errs):
    try:
        import torch  # noqa: F401
        os.environ.update(RANK=str(rank), WORLD_SIZE=str(size), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        import scipy.sparse as sps
        from oracle import oracle
        from test_distributed_cpu import OracleProvider, _exchange_values
        comm = D.Comm.from_env("gloo")
        if kind == "p2tet":
            mesh = M.create_box_tets((3, 3, 3)); vdeg = 2
        else:
            mesh = _meshes.delaunay_tris(9); vdeg = 1
        sp = M.mixed_space(mesh, vdeg)
        gd = mesh.gdim
        w, bcs = _meshes.smooth_state(sp), _meshes.box_bcs(sp)
        part = D.partition_cells(mesh, sp, slab_ranks(mesh, size), rank, size, w=w, bcs=bcs)
        prov = OracleProvider(part)
        plans = D.build_plans(part, comm, prov, gdim=gd, vdeg=vdeg)
        n_owned, n_dofs = part.n_owned, part.n_owned + part.n_ghost
        form = oracle.Form(0, gd, vdeg, 0.1)
        marker, value, mult = oracle.bc_arrays(sp.n_dofs, [b[0] for b in bcs], [b[1] for b in bcs])
        gp, gi = oracle.build_pattern(sp.dofmap, sp.n_dofs)
        gv = oracle.assemble_jacobian(form, mesh.x, mesh.cells, sp.dofmap, w, gp, gi, marker, mult)
        gF = oracle.assemble_residual(form, mesh.x, mesh.cells, sp.dofmap, w, marker, value)
        oracle.set_bc(gF, [b[0] for b in bcs], [b[1] for b in bcs], w)
        A = sps.csr_matrix((gv, gi, gp), shape=(sp.n_dofs,) * 2)
        s_of_local = part.meta["serial_dof"]
        np.testing.assert_array_equal(part.w, w[s_of_local])
        assert (np.diff(part.local_to_global[:n_owned]) == 1).all() and part.local_to_global[0] == part.global_offset
        # forward halo (dofmap ghosts and column ghosts): serial dof of a column ghost through the owners' answers
        neigh, sptr, sidx, rptr, ridx = plans.halo
        xloc = np.zeros(plans.n_cols)
        xloc[:n_owned] = w[s_of_local[:n_owned]]
        xloc[ridx] = _exchange_values(comm, neigh, sptr, xloc[sidx], rptr)
        sloc = np.zeros(plans.n_cols)
        sloc[:n_owned] = s_of_local[:n_owned]
        sloc[ridx] = _exchange_values(comm, neigh, sptr, sloc[sidx], rptr)
        serial_col = sloc.astype(np.int64)
        np.testing.assert_array_equal(serial_col[:n_dofs], s_of_local)
        np.testing.assert_array_equal(xloc, w[serial_col])
        # J: owned cells, ghost rows to their owners, BC diagonal on owned rows; compared row by row with the serial matrix
        lmarker, lvalue, lmult = oracle.bc_arrays(n_dofs, [b[0] for b in part.bcs], [b[1] for b in part.bcs])
        lv = oracle.assemble_jacobian(form, part.x, part.cells, part.dofmap, xloc[:n_dofs], prov.indptr, prov.indices, lmarker, None,
                                      n_owned=n_owned, n_cells_owned=part.n_cells_owned)
        rn, sp_ptr, sp_pos, rp_ptr, rp_pos = plans.rows
        np.add.at(lv, rp_pos, _exchange_values(comm, rn, sp_ptr, lv[sp_pos], rp_ptr))
        for d in np.nonzero(lmult[:n_owned] > 0)[0]:
            seg = prov.indices[prov.indptr[d]:prov.indptr[d + 1]]
            lv[prov.indptr[d] + np.searchsorted(seg, d)] += lmult[d]
        for r in range(n_owned):
            seg = slice(prov.indptr[r], prov.indptr[r + 1])
            scols = serial_col[prov.indices[seg]]
            ref = A.getrow(int(s_of_local[r]))
            order = np.argsort(scols)
            np.testing.assert_array_equal(scols[order], ref.indices)
            np.testing.assert_allclose(lv[seg][order], ref.data, rtol=0, atol=1e-13 * np.abs(gv).max())
        # F: reverse halo-add, set_bc on owned dofs
        lF = oracle.assemble_residual(form, part.x, part.cells, part.dofmap, xloc[:n_dofs], lmarker, lvalue, n_cells_owned=part.n_cells_owned)
        lFx = np.zeros(plans.n_cols); lFx[:n_dofs] = lF
        np.add.at(lFx, sidx, _exchange_values(comm, neigh, rptr, lFx[ridx], sptr))
        oracle.set_bc(lFx, [b[0] for b in part.bcs], [b[1] for b in part.bcs], xloc, n_owned=n_owned)
        np.testing.assert_allclose(lFx[:n_owned], gF[s_of_local[:n_owned]], rtol=0, atol=1e-13 * np.abs(gF).max())
        comm.close()
    except Exception:
        import traceback
        errs.put((rank, traceback.format_exc()))


@pytest.mark.parametrize("kind", ["p2tet", "p1tri"])
@pytest.mark.parametrize("size", [2, 3])
def test_partition_cells_plans_reproduce_serial_assembly(kind, size):
    from oracle import oracle
    oracle.build()
    ctx = mp.get_context("spawn")
    errs = ctx.Queue()
    port = 31500 + (os.getpid() % 2000) + 10 * size + (kind == "p1tri")
    procs = [ctx.Process(target=_plan_worker, args=(r, size, port, kind, errs)) for r in range(size)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=240)
    msgs = []
    while not errs.empty():
        msgs.append(errs.get())
    for p in procs:
        if p.is_alive():
            p.terminate()
            msgs.append((-1, "worker hung"))
    assert not msgs, "\n".join(f"rank {r}:\n{m}" for r, m in msgs)
    assert all(p.exitcode == 0 for p in procs)


def test_partition_cells_layout():
    sp = M.mixed_space(M.create_box_tets((2, 2, 3)), 2)
    cr = slab_ranks(sp.mesh, 3, axis=2)
    parts = [D.partition_cells(sp.mesh, sp, cr, r, 3) for r in range(3)]
    assert sum(p.n_owned for p in parts) == sp.n_dofs
    assert [p.global_offset for p in parts] == [0, parts[0].n_owned, parts[0].n_owned + parts[1].n_owned]
    for p in parts:
        owner_of_global = np.searchsorted([q.global_offset for q in parts], p.ghost_global, side="right") - 1
        np.testing.assert_array_equal(owner_of_global, p.ghost_owner)
        assert (p.ghost_owner < p.rank).all()          # the lowest rank among a dof's cells owns it
