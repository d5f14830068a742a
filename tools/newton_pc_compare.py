"""Device-resident Newton solve of the duct (Re = 10, SNES settings of NavierStokesChannelFlow.py:286-291) with the two
preconditioners of the device TFQMR, by default 4x4 vertex-block Jacobi (pc = 4) and multicolour block ILU(0) (pc = 5).
Prints one JSON line per preconditioner: Newton steps, Krylov iterations, wall time.
Usage: newton_pc_compare.py n_cross n_long [pc,pc,...] [ksp_max_it]"""
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stabilized_navier_stokes_flow_fenicsx_b200 import mesh as M
from stabilized_navier_stokes_flow_fenicsx_b200.assembler import NSAssembler

n_cross, n_long = (int(sys.argv[1]), int(sys.argv[2])) if len(sys.argv) > 2 else (32, 128)
m = M.duct_mesh(n_cross, n_long); sp = M.mixed_space(m, 1)
bcs = M.duct_bcs(sp)
marker = np.zeros(sp.n_dofs, dtype=bool); value = np.zeros(sp.n_dofs)
for d, v in bcs:
    marker[d] = True; value[d] = v
w0 = np.where(marker, value, 0.0)
pcs = tuple(int(p) for p in sys.argv[3].split(",")) if len(sys.argv) > 3 else (4, 5)
ksp_max_it = int(sys.argv[4]) if len(sys.argv) > 4 else 20000
names = {4: "4x4 vertex-block Jacobi", 5: "multicolour block ILU(0)", 6: "multicolour point ILU(0)", 7: "point ILU(0) in the caller's order"}
sols = {}
for pc in pcs:
    asm = NSAssembler(m.x, m.cells, sp.dofmap, vdeg=1)
    asm.set_form(flavour=0, nu=0.1); asm.set_bcs(bcs)
    asm.create_matrix(fetch=False)
    w_dev = asm.dev_alloc(8 * asm.n_cols)
    asm.h2d(w_dev, w0)
    asm.sync()
    t0 = time.perf_counter()
    hist = asm.newton_dev(w_dev, pc=pc, ksp_max_it=ksp_max_it)
    asm.sync()
    dt = time.perf_counter() - t0
    w = np.empty(asm.n_cols); asm.d2h(w, w_dev)
    sols[pc] = w[: sp.n_dofs].copy()
    its = [h.get("ksp_its", 0) for h in hist]
    print(json.dumps({"pc": names[pc], "cells": m.n_cells, "dofs": sp.n_dofs,
                      "newton_steps": len(hist) - 1, "fnorm": [h["fnorm"] for h in hist], "krylov_iterations": its, "krylov_total": int(sum(its)),
                      "seconds": dt, "colours": asm.ilu_colours()[1] if pc == 5 else None}), flush=True)
    asm.close()
a, b = sols[pcs[0]], sols[pcs[-1]]
print(json.dumps({"solution_difference_max": float(np.abs(a - b).max()), "solution_max": float(np.abs(a).max())}))
