"""Launched by torchrun (one rank per GPU): KSPTFQMR with the multicolour point ILU(0) of each rank's diagonal block (pc = 6, block
Jacobi over the ranks) on the slab-partitioned P1-P1 duct, against a serial direct solve.  Exit code 0 = within 1e-8."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import scipy.sparse as sps
    import scipy.sparse.linalg as spla

    from oracle import oracle
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
    _, F = asm.jacobian_residual(part.w.copy())
    colour, nc, nvc = asm.pilu_colours()
    x6, info6 = asm.tfqmr(F[:n_owned], rtol=1e-12, max_it=4000, pc=6)
    x1, info1 = asm.tfqmr(F[:n_owned], rtol=1e-12, max_it=4000, pc=1)
    err = np.abs(x6 - x_ref[l2g[:n_owned]]).max()
    assert err <= 1e-8 * np.abs(x_ref).max(), f"rank {rank}: TFQMR + point ILU err {err} {info6}"
    print(f"rank {rank}/{size}: TFQMR + point ILU(0) err {err:.2e} in {info6['its']} its (Jacobi: {info1['its']}), "
          f"{nc} colours ({nvc} velocity), n_owned {n_owned}", flush=True)
    asm.close()
    comm.close()


if __name__ == "__main__":
    main()
