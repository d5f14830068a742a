"""Cell-partitioned multi-GPU plumbing (host side): x-slab partition of the synthetic duct in dolfinx
owned+ghost layout, vector halo plans, ghost-row (J.assemble) plans, and the thin communicator wrapper.

One process per GPU.  ``torch.distributed`` (NCCL on the GPU box, gloo in the CPU tests) is used only for
the set-up exchanges and for barriers / max-over-ranks timing; the per-iteration halo traffic runs inside
libnsgpu.so over its own NCCL communicator (csrc/halo.cu).

Mirrors: ``x.ghostUpdate(INSERT, FORWARD)``, ``F.ghostUpdate(ADD, REVERSE)``, ``J.assemble()``
(NavierStokes/NavierStokesChannelFlow.py:57-60, :66, :75) and dolfinx ``SparsityPattern.finalize``.
"""
import os
from dataclasses import dataclass, field

import numpy as np

from . import mesh as M


# ------------------------------------------------------------------------------------------------ comm
class Comm:
    """Minimal communicator facade: single process, or torch.distributed (nccl / gloo)."""

    def __init__(self, rank=0, size=1, dist=None, device=None):
        self.rank, self.size, self.dist, self.device = rank, size, dist, device

    @staticmethod
    def single():
        return Comm()

    @staticmethod
    def from_env(backend=None):
        import torch
        import torch.distributed as dist
        rank, size = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
        local = int(os.environ.get("LOCAL_RANK", rank))
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        device = None
        if backend == "nccl":
            torch.cuda.set_device(local)
            device = torch.device("cuda", local)
        if not dist.is_initialized():
            dist.init_process_group(backend=backend, rank=rank, world_size=size)
        return Comm(rank, size, dist, device)

    @staticmethod
    def from_mpi4py(comm, local_rank=None):
        """The communicator a dolfinx script already has (``mesh.comm`` / ``MPI.COMM_WORLD``,
        NavierStokes/NavierStokesChannelFlow.py:99-101, launched by ``mpirun -n 6``): same facade as the torchrun one, over
        mpi4py.  The NCCL unique id of the library's own communicator travels through ``bcast_bytes``."""
        return MpiComm(comm, local_rank)

    def _t(self, arr):
        import torch
        t = torch.from_numpy(np.ascontiguousarray(arr))
        return t.to(self.device) if self.device is not None else t

    def barrier(self):
        if self.size > 1:
            self.dist.barrier()

    def _reduce(self, v, op):
        if self.size == 1:
            return v
        import torch
        t = torch.tensor([float(v)], dtype=torch.float64, device=self.device)
        self.dist.all_reduce(t, op=op)
        return float(t.item())

    def max(self, v):
        return self._reduce(v, self.dist.ReduceOp.MAX) if self.size > 1 else v

    def sum(self, v):
        if self.size == 1:
            return v
        import torch
        t = torch.tensor([int(v)], dtype=torch.int64, device=self.device)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return int(t.item())

    def bcast_bytes(self, data, n, root=0):
        """Broadcast n bytes (bytes object on root, ignored elsewhere)."""
        if self.size == 1:
            return data
        import torch
        buf = np.frombuffer(data, dtype=np.uint8).copy() if self.rank == root else np.zeros(n, dtype=np.uint8)
        t = self._t(buf)
        self.dist.broadcast(t, src=root)
        return t.cpu().numpy().tobytes()

    def exchange(self, send):
        """Sparse all-to-all of int64 arrays: ``send`` maps peer rank -> array; returns peer -> array."""
        if self.size == 1:
            return {}
        import torch
        counts = np.zeros(self.size, dtype=np.int64)
        for p, a in send.items():
            counts[p] = len(a)
        all_counts = [torch.zeros(self.size, dtype=torch.int64, device=self.device) for _ in range(self.size)]
        self.dist.all_gather(all_counts, self._t(counts))
        all_counts = np.stack([c.cpu().numpy() for c in all_counts])      # [src][dst]
        out = {}
        # pairwise ordered send/recv (works on both nccl and gloo)
        for src in range(self.size):
            for dst in range(self.size):
                n = int(all_counts[src, dst])
                if n == 0 or src == dst:
                    continue
                if self.rank == src:
                    self.dist.send(self._t(np.asarray(send[dst], dtype=np.int64)), dst=dst)
                elif self.rank == dst:
                    t = torch.zeros(n, dtype=torch.int64, device=self.device)
                    self.dist.recv(t, src=src)
                    out[src] = t.cpu().numpy()
        return out

    def close(self):
        if self.size > 1 and self.dist.is_initialized():
            self.dist.barrier()
            self.dist.destroy_process_group()


class MpiComm(Comm):
    """Comm facade over an mpi4py communicator (anything with Get_rank / Get_size / Barrier / allreduce / bcast / alltoall)."""

    def __init__(self, comm, local_rank=None):
        super().__init__(comm.Get_rank(), comm.Get_size(), None, None)
        self.comm = comm
        self.local_rank = self.rank if local_rank is None else local_rank

    def barrier(self):
        if self.size > 1:
            self.comm.Barrier()

    def max(self, v):
        return v if self.size == 1 else max(self.comm.allgather(float(v)))

    def sum(self, v):
        return v if self.size == 1 else int(sum(self.comm.allgather(int(v))))

    def bcast_bytes(self, data, n, root=0):
        return data if self.size == 1 else self.comm.bcast(data if self.rank == root else None, root=root)

    def exchange(self, send):
        if self.size == 1:
            return {}
        out = self.comm.alltoall([np.asarray(send[p], dtype=np.int64) if p in send else None for p in range(self.size)])
        return {p: np.asarray(a, dtype=np.int64) for p, a in enumerate(out) if a is not None and p != self.rank and len(a)}

    def close(self):
        self.barrier()


# ------------------------------------------------------------------------------------------------ partition
@dataclass
class Partition:
    """Rank-local arrays in dolfinx layout (owned dofs/cells first, ghosts after)."""
    rank: int
    size: int
    x: np.ndarray
    cells: np.ndarray
    dofmap: np.ndarray
    n_cells_owned: int
    n_owned: int
    n_ghost: int
    global_offset: int                 # first global dof owned by this rank
    ghost_global: np.ndarray           # (n_ghost,) global dof index of each ghost
    ghost_owner: np.ndarray            # (n_ghost,) owning rank
    local_to_global: np.ndarray        # (n_owned + n_ghost,)
    w: np.ndarray                      # state, local layout
    bcs: list
    meta: dict = field(default_factory=dict)

    def owned_nnz(self, asm):
        """nnz held in rows this rank owns (for whole-job nnz bookkeeping)."""
        return asm.owned_nnz()


def slab_ranges(n_long, size):
    """Balanced contiguous box-layer ranges along the duct axis."""
    base, rem = divmod(n_long, size)
    starts = [r * base + min(r, rem) for r in range(size + 1)]
    return [(starts[r], starts[r + 1]) for r in range(size)]


def duct_partition(n_cross, n_long, rank, size, length=4.0, seed=1234, noise=1e-3):
    """x-slab partition of the structured duct (SURVEY 8e).  Shared interface planes are owned by the lower
    rank; there are no ghost cells (GhostMode.none, as for gmsh-imported meshes)."""
    k0, k1 = slab_ranges(n_long, size)[rank]
    nl = k1 - k0
    if nl <= 0:
        raise ValueError("more ranks than box layers")
    plane = (n_cross + 1) ** 2
    x0 = length * k0 / n_long
    local = M.create_box_tets((n_cross, n_cross, nl), p0=(x0, -0.5, -0.5), p1=(length * k1 / n_long, 0.5, 0.5), axes=(1, 2, 0))
    # local vertex v = plane index (k - k0) * plane + in-plane index; plane k0 is a ghost plane for rank > 0
    nvl = local.n_vertices
    if rank == 0:
        perm = np.arange(nvl, dtype=np.int64)                 # all owned
        n_owned_v = nvl
    else:
        perm = np.concatenate([np.arange(plane, nvl), np.arange(plane)])   # new order: owned planes, then ghost plane
        n_owned_v = nvl - plane
    inv = np.empty(nvl, dtype=np.int64)
    inv[perm] = np.arange(nvl)
    xl = local.x[perm]
    cells = inv[local.cells].astype(np.int32)
    mloc = M.Mesh(3, xl, cells, local.shape, dict(local.meta, kind="duct_slab"))
    sp = M.mixed_space(mloc, 1)
    # global vertex ids (same numbering as the unpartitioned duct_mesh)
    gv = (k0 * plane + perm).astype(np.int64)
    l2g = (4 * gv[:, None] + np.arange(4)[None, :]).ravel()
    n_owned, n_ghost = 4 * n_owned_v, 4 * (nvl - n_owned_v)
    global_offset = 0 if rank == 0 else 4 * (k0 + 1) * plane
    ghost_global = l2g[n_owned:]
    ghost_owner = np.full(n_ghost, rank - 1, dtype=np.int32)
    # state: analytic part from coordinates, noise indexed by global dof so that every partition sees the same field
    w = M.duct_state(sp, seed=seed, noise=0.0)
    if noise:
        ntot = 4 * plane * (n_long + 1)
        w = w + noise * np.random.default_rng(seed).standard_normal(ntot)[l2g]
    bcs = M.duct_bcs(sp, length=length)
    return Partition(rank, size, xl, cells, sp.dofmap, mloc.n_cells, n_owned, n_ghost, global_offset, ghost_global, ghost_owner,
                     l2g, w, bcs, {"k0": k0, "k1": k1, "plane": plane})


def partition_cells(mesh, space, cell_rank, rank, size, w=None, bcs=None):
    """Partition of any mesh and mixed space (tets or triangles, P1-P1 or P2-P1) by a given cell -> rank map, in the layout of
    ``duct_partition``: the owned cells are those with ``cell_rank == rank`` (no ghost cells), each dof is owned by the lowest rank
    among the cells that contain it, global dofs are numbered contiguously by rank (ascending serial dof within a rank), and
    locally the owned dofs come first, then the ghosts, each in global order.  ``w`` (serial numbering) and ``bcs`` (list of
    (dofs, values) in serial numbering) are mapped to the local numbering; ``meta["serial_dof"]`` is the serial dof of every local
    dof."""
    cell_rank = np.asarray(cell_rank, dtype=np.int64)
    if cell_rank.shape != (mesh.n_cells,) or cell_rank.min() < 0 or cell_rank.max() >= size:
        raise ValueError("cell_rank must give a rank in [0, size) for every cell")
    dm = np.asarray(space.dofmap, dtype=np.int64)
    owner = np.full(space.n_dofs, size, dtype=np.int64)
    np.minimum.at(owner, dm, np.broadcast_to(cell_rank[:, None], dm.shape))
    serial_of_global = np.argsort(owner, kind="stable")                 # global dof -> serial dof
    global_of_serial = np.empty(space.n_dofs, dtype=np.int64)
    global_of_serial[serial_of_global] = np.arange(space.n_dofs)
    global_offset = int((owner < rank).sum())
    own_cells = np.nonzero(cell_rank == rank)[0]
    if own_cells.size == 0:
        raise ValueError(f"rank {rank} owns no cell")
    local_serial = np.unique(dm[own_cells])
    mine = owner[local_serial] == rank
    owned, ghost = local_serial[mine], local_serial[~mine]
    owned = owned[np.argsort(global_of_serial[owned])]
    ghost = ghost[np.argsort(global_of_serial[ghost])]
    serial_dof = np.concatenate([owned, ghost])
    local_of_serial = np.full(space.n_dofs, -1, dtype=np.int64)
    local_of_serial[serial_dof] = np.arange(len(serial_dof))
    verts = np.unique(mesh.cells[own_cells])
    local_vertex = np.full(mesh.n_vertices, -1, dtype=np.int64)
    local_vertex[verts] = np.arange(len(verts))
    cells = local_vertex[mesh.cells[own_cells]].astype(np.int32)
    dofmap = local_of_serial[dm[own_cells]].astype(np.int32)
    l2g = global_of_serial[serial_dof]
    n_owned, n_ghost = len(owned), len(ghost)
    w_local = None if w is None else np.asarray(w, dtype=np.float64)[serial_dof]
    bcs_local = []
    for dofs, vals in (bcs or []):
        ld = local_of_serial[np.asarray(dofs, dtype=np.int64)]
        keep = ld >= 0
        bcs_local.append((ld[keep].astype(np.int32), np.asarray(vals, dtype=np.float64)[keep]))
    return Partition(rank, size, mesh.x[verts], cells, dofmap, len(own_cells), n_owned, n_ghost, global_offset, l2g[n_owned:],
                     owner[ghost].astype(np.int32), l2g, w_local, bcs_local, {"serial_dof": serial_dof, "cells": own_cells})


# ------------------------------------------------------------------------------------------------ plans
def entity_tables(dofmap, gdim, vdeg, n_dofs):
    """leader / slot / size of every local dof: dofs on one mesh entity (vertex: gdim velocity components +
    pressure; P2 edge: gdim components) share their cell incidence -- same grouping as csrc/pattern.cu."""
    nv = gdim + 1
    ne = 0 if vdeg == 1 else (6 if gdim == 3 else 3)
    poff = gdim * (nv + ne)
    leader = np.arange(n_dofs, dtype=np.int64)
    slot = np.zeros(n_dofs, dtype=np.int64)
    size = np.ones(n_dofs, dtype=np.int64)
    dm = np.asarray(dofmap, dtype=np.int64)
    for n in range(nv):
        lead = dm[:, gdim * n]
        for c in range(gdim):
            d = dm[:, gdim * n + c]
            leader[d], slot[d], size[d] = lead, c, gdim + 1
        d = dm[:, poff + n]
        leader[d], slot[d], size[d] = lead, gdim, gdim + 1
    for e in range(ne):
        lead = dm[:, gdim * (nv + e)]
        for c in range(gdim):
            d = dm[:, gdim * (nv + e) + c]
            leader[d], slot[d], size[d] = lead, c, gdim
    return leader, slot, size


@dataclass
class Plans:
    n_cols: int
    col_ghost_global: np.ndarray        # global index of the column ghosts appended after the dofmap ghosts
    col_ghost_owner: np.ndarray
    halo: tuple                         # (neigh, send_ptr, send_idx, recv_ptr, recv_idx)
    rows: tuple                         # (neigh, send_ptr, send_pos, recv_ptr, recv_pos)
    extra: tuple                        # (extra_rows, extra_cols, colx_leader, colx_slot, colx_size)


def _group(ranks):
    """stable grouping: returns {rank: index array} in ascending rank order."""
    out = {}
    for r in np.unique(ranks):
        out[int(r)] = np.nonzero(ranks == r)[0]
    return out


def build_plans(part, comm, provider, gdim=3, vdeg=1):
    """Everything dolfinx / PETSc set up behind ``create_matrix`` and ``Mat.assemble`` on more than one rank:
    the extra pattern entries owners receive for their rows (SparsityPattern.finalize), the column ghosts
    those entries introduce, the vector halo lists and the ghost-row value-exchange lists.

    ``provider`` builds patterns and returns rows of them: the GPU assembler in production, an oracle-backed
    stand-in in the CPU tests.  All index exchange goes through ``comm.exchange`` (sparse all-to-all)."""
    rank = comm.rank
    n_owned, n_ghost = part.n_owned, part.n_ghost
    n_dofs = n_owned + n_ghost
    l2g = np.asarray(part.local_to_global, dtype=np.int64)
    off = part.global_offset
    leader, slot, size = entity_tables(part.dofmap, gdim, vdeg, n_dofs)
    owner_local = np.concatenate([np.full(n_owned, rank, dtype=np.int64), np.asarray(part.ghost_owner, dtype=np.int64)])

    # 1. preliminary pattern from the owned cells; ship the ghost rows' entries to the row owners
    provider.build_pattern()
    grow_local = np.arange(n_owned, n_dofs, dtype=np.int32)
    _, gptr, gidx = provider.get_rows(grow_local)
    counts = np.diff(gptr)
    ent_row = np.repeat(grow_local.astype(np.int64), counts)
    ent_col = gidx.astype(np.int64)
    row_owner = owner_local[ent_row]
    send = {}
    order_by_owner = _group(row_owner)
    for o, sel in order_by_owner.items():
        c = ent_col[sel]
        send[o] = np.stack([l2g[ent_row[sel]], l2g[c], owner_local[c], l2g[leader[c]], slot[c], size[c]], 1).ravel()
    recv = comm.exchange(send)

    # 2. owners: map received entries to local (row, col); unknown columns become new column ghosts
    srcs = sorted(recv)
    msgs = [recv[r].reshape(-1, 6) for r in srcs]
    lens = [len(m) for m in msgs]
    m = np.concatenate(msgs) if msgs else np.zeros((0, 6), dtype=np.int64)
    lrow = m[:, 0] - off
    assert ((lrow >= 0) & (lrow < n_owned)).all(), "received a row this rank does not own"
    gcol = m[:, 1]
    lcol = np.empty(len(gcol), dtype=np.int64)
    mine = (gcol >= off) & (gcol < off + n_owned)
    lcol[mine] = gcol[mine] - off
    gg = np.asarray(part.ghost_global, dtype=np.int64)
    gorder = np.argsort(gg, kind="stable")
    gsorted = gg[gorder]
    nm = np.nonzero(~mine)[0]
    ug, first, inv = np.unique(gcol[nm], return_index=True, return_inverse=True)
    pos = np.searchsorted(gsorted, ug)
    known = (pos < len(gsorted)) & (gsorted[np.minimum(pos, max(len(gsorted) - 1, 0))] == ug) if len(gsorted) else np.zeros(len(ug), bool)
    ul = np.empty(len(ug), dtype=np.int64)
    ul[known] = n_owned + gorder[pos[known]]
    nx = int((~known).sum())
    ul[~known] = n_dofs + np.arange(nx)
    lcol[nm] = ul[inv]
    meta = m[nm[first[~known]]]                                  # first occurrence describes the new column ghost
    new_global = ug[~known]
    new_owner, new_gleader, new_slot, new_size = meta[:, 2], meta[:, 3], meta[:, 4], meta[:, 5]
    lead_pos = np.searchsorted(new_global, new_gleader)
    assert nx == 0 or (new_global[np.minimum(lead_pos, nx - 1)] == new_gleader).all(), "entity of a new column ghost arrived incomplete"
    colx_leader = (n_dofs + lead_pos).astype(np.int32)
    recv_entries, o0 = {}, 0
    for r, n in zip(srcs, lens):
        recv_entries[r] = (lrow[o0:o0 + n], lcol[o0:o0 + n])
        o0 += n
    extra = (lrow.astype(np.int32), lcol.astype(np.int32), colx_leader, new_slot.astype(np.int32), new_size.astype(np.int32))

    # 3. final pattern
    provider.build_pattern(*extra)
    n_cols = n_dofs + nx

    # 4. vector halo over dofmap ghosts + column ghosts
    ghost_global = np.concatenate([gg, new_global])
    ghost_owner = np.concatenate([np.asarray(part.ghost_owner, dtype=np.int64), new_owner])
    req_groups = _group(ghost_owner) if len(ghost_owner) else {}
    requests = {o: ghost_global[sel] for o, sel in req_groups.items()}
    asked = comm.exchange(requests)                       # what other ranks need from me
    neigh = sorted(set(req_groups) | set(asked))
    send_ptr, send_idx, recv_ptr, recv_idx = [0], [], [0], []
    for o in neigh:
        si = (asked[o] - off) if o in asked else np.zeros(0, np.int64)
        assert ((si >= 0) & (si < n_owned)).all(), "asked for a dof this rank does not own"
        ri = (n_owned + req_groups[o]) if o in req_groups else np.zeros(0, np.int64)
        send_idx.append(si); recv_idx.append(ri)
        send_ptr.append(send_ptr[-1] + len(si)); recv_ptr.append(recv_ptr[-1] + len(ri))
    cat = lambda a, dt: (np.concatenate(a).astype(dt) if a else np.zeros(0, dt))
    halo = (np.array(neigh, dtype=np.int32), np.array(send_ptr, dtype=np.int64), cat(send_idx, np.int32),
            np.array(recv_ptr, dtype=np.int64), cat(recv_idx, np.int32))

    # 5. ghost-row value exchange: senders' positions (final pattern, same entry order as step 1) and
    #    receivers' positions of the matching (row, col)
    gstart, gptr2, gidx2 = provider.get_rows(grow_local)
    assert np.array_equal(gptr2, gptr) and np.array_equal(gidx2, gidx), "ghost rows changed between the two pattern builds"
    ent_pos = np.repeat(gstart, counts) + (np.arange(len(ent_row)) - np.repeat(gptr[:-1], counts))
    rneigh = sorted(set(order_by_owner) | set(recv_entries))
    sp_ptr, sp_pos, rp_ptr, rp_pos = [0], [], [0], []
    for o in rneigh:
        spos = ent_pos[order_by_owner[o]] if o in order_by_owner else np.zeros(0, np.int64)
        if o in recv_entries:
            lrow, lcol = recv_entries[o]
            urows, inv = np.unique(lrow, return_inverse=True)
            ustart, uptr, uidx = provider.get_rows(urows.astype(np.int32))
            # vectorised search: rows are sorted by column, so (row-rank, column) keys are globally sorted
            ncol_key = int(max(int(uidx.max()) if len(uidx) else 0, int(lcol.max()) if len(lcol) else 0)) + 1
            row_of = np.repeat(np.arange(len(urows), dtype=np.int64), np.diff(uptr))
            keys = row_of * ncol_key + uidx.astype(np.int64)
            want = inv.astype(np.int64) * ncol_key + lcol
            j = np.searchsorted(keys, want)
            assert (j < len(keys)).all() and (keys[np.minimum(j, len(keys) - 1)] == want).all(), "received entry missing from the final pattern"
            rpos = ustart[inv] + (j - uptr[inv])
        else:
            rpos = np.zeros(0, np.int64)
        sp_pos.append(spos); rp_pos.append(rpos)
        sp_ptr.append(sp_ptr[-1] + len(spos)); rp_ptr.append(rp_ptr[-1] + len(rpos))
    rows = (np.array(rneigh, dtype=np.int32), np.array(sp_ptr, dtype=np.int64), cat(sp_pos, np.int64),
            np.array(rp_ptr, dtype=np.int64), cat(rp_pos, np.int64))
    return Plans(n_cols, new_global, new_owner, halo, rows, extra)


def attach(asm, part, comm):
    """Create the library's NCCL communicator (unique id broadcast over the host communicator)."""
    if comm.size == 1:
        return
    uid = asm.comm_unique_id() if comm.rank == 0 else None
    uid = comm.bcast_bytes(uid, 128, root=0)
    asm.comm_init(comm.rank, comm.size, uid)


def finish_pattern_exchange(asm, part, comm):
    """Build the final pattern and install the halo / ghost-row plans on the assembler."""
    if comm.size == 1:
        asm.create_matrix(fetch=False)
        return None
    plans = build_plans(part, comm, asm, gdim=asm.gdim, vdeg=asm.vdeg)
    asm.set_halo(*plans.halo)
    asm.set_row_exchange(*plans.rows)
    return plans
