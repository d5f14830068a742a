"""Launched by torchrun (one rank per GPU): ILU(0) of each rank's diagonal block in the rank's local dof order (pc = 7, block Jacobi
over the ranks) on the slab-partitioned P1-P1 duct.  Each rank's application is held against oracle/pilu_ref.pilu0 of its owned block
with colour = arange(n_owned), and the KSPTFQMR solve against a serial direct solve.  Exit code 0 = both within tolerance."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import scipy.sparse as sps
    import scipy.sparse.linalg as spla

    from oracle import oracle, pilu_ref
    from stabilized_navier_stokes_flow_fenicsx_b200 import _lib
    from stabilized_navier_stokes_flow_fenicsx_b200 import distributed as D
    from stabilized_navier_stokes_flow_fenicsx_b200 import mesh as M
    from stabilized_navier_stokes_flow_fenicsx_b200.assembler import NSAssembler
    n_cross, n_long = 6, 20
    comm = D.Comm.from_env()
    rank, size = comm.rank, comm.size
    part = D.duct_partition(n_cross, n_long, rank, size)
    asm = NSAssembler(part.x, part.cells, part.dofmap, vdeg=1, n_dofs_owned=part.n_owned, n_dofs_ghost=part.n_ghost,
                      n_cells_owned=part.n_cells_owned, device=int(os.environ.get("LOCAL_RANK", 0)))
    asm.set_form(flavour=0, nu=0.1)
    asm.set_bcs(part.bcs)
    D.attach(asm, part, comm)
    D.finish_pattern_exchange(asm, part, comm)
    n_owned = part.n_owned
    # serial oracle: Jacobian and residual of the same state, direct solve
    m = M.duct_mesh(n_cross, n_long); sp = M.mixed_space(m, 1)
    w, bcs = M.duct_state(sp), M.duct_bcs(sp)
    marker, value, mult = oracle.bc_arrays(sp.n_dofs, [b[0] for b in bcs], [b[1] for b in bcs])
    gp, gi = oracle.build_pattern(sp.dofmap, sp.n_dofs)
    form = oracle.Form(0, 3, 1, 0.1)
    gv = oracle.assemble_jacobian(form, m.x, m.cells, sp.dofmap, w, gp, gi, marker, mult)
    gF = oracle.assemble_residual(form, m.x, m.cells, sp.dofmap, w, marker, value)
    oracle.set_bc(gF, [b[0] for b in bcs], [b[1] for b in bcs], w)
    x_ref = spla.spsolve(sps.csr_matrix((gv, gi, gp), shape=(sp.n_dofs,) * 2).tocsc(), gF)
    l2g = part.local_to_global
    vals, F = asm.jacobian_residual(part.w.copy())
    indptr = np.empty(asm.n_dofs + 1, dtype=np.int64)
    indices = np.empty(asm.nnz, dtype=np.int32)
    _lib.check(asm.ctx, asm.lib.nsgpu_get_pattern(asm.ctx, indptr.ctypes.data, indices.ctypes.data), "get_pattern")
    # the rank's preconditioner: ILU(0) of its owned block (other ranks' columns dropped) in its local order
    r = np.random.default_rng(100 + rank).standard_normal(n_owned)
    z = asm.nilu_apply(r)
    zr = pilu_ref.apply(pilu_ref.pilu0(indptr, indices, vals, np.arange(n_owned)), r)
    perr = np.abs(z - zr).max() / np.abs(zr).max()
    assert perr <= 1e-10, f"rank {rank}: application differs from the block restatement by {perr}"
    x7, info7 = asm.tfqmr(F[:n_owned], rtol=1e-12, max_it=4000, pc=7)
    err = np.abs(x7 - x_ref[l2g[:n_owned]]).max()
    assert err <= 1e-8 * np.abs(x_ref).max(), f"rank {rank}: TFQMR + natural-order ILU err {err} {info7}"
    print(f"rank {rank}/{size}: application rel err {perr:.2e}, TFQMR + ILU(0) in local order err {err:.2e} in {info7['its']} its, "
          f"depth {asm.nilu_depth()}, n_owned {n_owned}", flush=True)
    asm.close()
    comm.close()


if __name__ == "__main__":
    main()
