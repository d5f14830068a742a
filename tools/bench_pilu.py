"""Cost of the multicolour point ILU(0) preconditioner (pc = 6) on one GPU, on a Newton-step system J dx = F of two sizes a user runs:
the P2-P1 G-metric duct 40 x 40 x 80 (768 k cells, the flavour / viscosity of bench.py's other_paths.p2p1_gmetric) and a UGN P1-P1
lid-driven cavity of 4.2 M triangles.  Prints one JSON line per matrix (and writes them to --out):

  colours             number of colours (velocity colours) of the elimination order
  spmv_ms             one CSR SpMV of the same matrix (kernel time, CUDA events)
  iter_ms_pc6/pc0     marginal TFQMR iteration (17-iteration solve minus 2-iteration solve, / 15), pc = 6 and no preconditioner
  apply_ms            one application z = U^-1 L^-1 r: (iter_ms_pc6 - iter_ms_pc0) / 2 (two applications per iteration)
  factor_ms           factorisation: (0-iteration solve with pc = 6) - (the same with pc = 0) - 2 applications
  its_pc6 / its_pc1   TFQMR iterations to rtol 1e-8 (capped at --max-it) with pc = 6 and with point Jacobi

Every time is a median of three, after a warm-up of every call, on the context's stream (nsgpu_timer_start / _stop).  The card's
name and power limit are read in the same run and printed with the numbers."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from stabilized_navier_stokes_flow_fenicsx_b200 import mesh as M  # noqa: E402
from stabilized_navier_stokes_flow_fenicsx_b200.assembler import NSAssembler  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip() or "nvidia-smi unavailable"


def timed(asm, fn, reps=3):
    fn()                                                   # warm-up of this exact call
    ts = []
    for _ in range(reps):
        asm.timer_start()
        fn()
        ts.append(asm.timer_stop())
    return float(np.median(ts))


def measure(name, m, sp, bcs, w, fk, max_it):
    asm = NSAssembler(m.x, m.cells, sp.dofmap, vdeg=sp.vdeg)
    asm.set_form(**fk); asm.set_bcs(bcs)
    asm.create_matrix(fetch=False)
    n, nc_all = asm.n_owned, asm.n_cols
    x_dev, b_dev, y_dev = asm.dev_alloc(8 * nc_all), asm.dev_alloc(8 * nc_all), asm.dev_alloc(8 * nc_all)
    asm.h2d(x_dev, w)
    asm.jacobian_residual_dev(x_dev, True, b_dev)              # J and F of the state: the Newton-step system
    asm.sync()
    nnz_owned = asm.owned_nnz()
    _, nc, nvc = asm.pilu_colours()
    asm.spmv_dev(x_dev, y_dev)
    ks = []
    for _ in range(5):
        asm.spmv_dev(x_dev, y_dev)
        ks.append(asm.last_kernel_ms())
    spmv_ms = float(np.median(ks))

    def solve(pc, its, rtol=0.0):
        return lambda: asm.tfqmr_dev(b_dev, y_dev, rtol=rtol, max_it=its, pc=pc)
    t = {(pc, its): timed(asm, solve(pc, its)) for pc in (0, 6) for its in (0, 2, 17)}
    it6 = (t[(6, 17)] - t[(6, 2)]) / 15
    it0 = (t[(0, 17)] - t[(0, 2)]) / 15
    apply_ms = (it6 - it0) / 2
    factor_ms = t[(6, 0)] - t[(0, 0)] - 2 * apply_ms
    i6 = asm.tfqmr_dev(b_dev, y_dev, rtol=1e-8, max_it=max_it, pc=6)
    i1 = asm.tfqmr_dev(b_dev, y_dev, rtol=1e-8, max_it=max_it, pc=1)
    bn = asm.norm_dev(b_dev)
    launches = 2 * nc - 1
    out = {"case": name, "cells": int(m.n_cells), "dofs": int(n), "nnz_owned": int(nnz_owned), "colours": nc, "velocity_colours": nvc,
           "spmv_ms": spmv_ms, "apply_ms": apply_ms, "apply_over_spmv": apply_ms / spmv_ms, "apply_launches": launches,
           "apply_us_per_launch": 1e3 * apply_ms / launches, "factor_ms": factor_ms, "iter_ms_pc6": it6, "iter_ms_pc0": it0,
           "its_pc6": i6["its"], "rel_rnorm_pc6": i6["rnorm"] / bn, "its_pc1": i1["its"], "rel_rnorm_pc1": i1["rnorm"] / bn, "max_it": max_it,
           "solve_ms": {f"pc{pc}_its{k}": v for (pc, k), v in t.items()}}
    for p in (x_dev, b_dev, y_dev):
        asm.dev_free(p)
    asm.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--max-it", type=int, default=5000, help="iteration cap of the rtol 1e-8 solves")
    ap.add_argument("--small", action="store_true", help="tiny meshes (a rehearsal of the script, not a measurement)")
    args = ap.parse_args()
    gpu = card()
    lines = []
    nd = (4, 8) if args.small else (40, 80)
    m = M.duct_mesh(*nd)
    sp = M.mixed_space(m, 2)
    lines.append(measure(f"duct_p2p1_gmetric_{nd[0]}x{nd[0]}x{nd[1]}", m, sp, M.duct_bcs(sp), M.duct_state(sp), dict(flavour=0, nu=1.0 / 50), args.max_it))
    nx = 24 if args.small else 1450
    m = M.create_rectangle_tris(nx, nx)
    sp = M.mixed_space(m, 1)
    lines.append(measure(f"cavity_ugn_p1p1_{nx}x{nx}", m, sp, M.cavity_bcs(sp), M.cavity_state(sp), dict(flavour=1, nu=0.01), args.max_it))
    with open(args.out, "w") if args.out else open(os.devnull, "w") as f:
        for d in lines:
            d["gpu"] = gpu
            s = json.dumps(d)
            print(s, flush=True)
            f.write(s + "\n")


if __name__ == "__main__":
    main()
