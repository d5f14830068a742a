"""Point ILU(0) in the caller's order (pc = 7) beside the multicolour point ILU(0) (pc = 6) on one GPU, on a Newton-step system
J dx = F of three sizes a user runs: the P1-P1 duct M (50 x 50 x 200, 3.0 M cells), the P2-P1 G-metric duct 40 x 40 x 80 and the UGN
P1-P1 lid-driven cavity 1450^2.  One JSON line per matrix and preconditioner (written to --out as well):

  plan_ms             first factorisation minus a later one: the plan (colouring for pc = 6, ranks for pc = 7, packed layout)
  factor_ms           factorisation: (0-iteration solve with pc) - (the same with pc = 0) - 2 applications
  apply_ms            one application z = U^-1 L^-1 r: marginal TFQMR iteration with pc minus that with pc = 0, / 2 (two applications
                      per iteration; CUDA events around solves of many applications; the packed factor of every case is larger than
                      the 126 MB L2)
  spmv_ms             one CSR SpMV of the same matrix, for scale
  depth_lower/upper   levels of the forward / backward dependency DAG of pc = 7 (rows on the longest path)
  its, rel_rnorm      TFQMR to rtol 1e-8, at most --max-it iterations and about --budget-s seconds of solving (the cap is reported)

Every time is on the context's stream (nsgpu_timer_start / _stop), after a warm-up of the same call.  The card's name and power
limit are read in the same run and printed with the numbers."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from stabilized_navier_stokes_flow_fenicsx_b200 import mesh as M  # noqa: E402
from stabilized_navier_stokes_flow_fenicsx_b200.assembler import NSAssembler  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip() or "nvidia-smi unavailable"


def timed(asm, fn):
    asm.timer_start()
    fn()
    return asm.timer_stop()


def measure(name, m, sp, bcs, w, fk, max_it, budget_s):
    asm = NSAssembler(m.x, m.cells, sp.dofmap, vdeg=sp.vdeg)
    asm.set_form(**fk); asm.set_bcs(bcs)
    asm.create_matrix(fetch=False)
    n, nc_all = asm.n_owned, asm.n_cols
    x_dev, b_dev, y_dev = asm.dev_alloc(8 * nc_all), asm.dev_alloc(8 * nc_all), asm.dev_alloc(8 * nc_all)
    asm.h2d(x_dev, w)
    asm.jacobian_residual_dev(x_dev, True, b_dev)              # J and F of the state: the Newton-step system
    asm.sync()
    nnz_owned = asm.owned_nnz()
    asm.spmv_dev(x_dev, y_dev)
    ks = []
    for _ in range(5):
        asm.spmv_dev(x_dev, y_dev)
        ks.append(asm.last_kernel_ms())
    spmv_ms = float(np.median(ks))
    bn = asm.norm_dev(b_dev)

    def solve(pc, its, rtol=0.0):
        return lambda: asm.tfqmr_dev(b_dev, y_dev, rtol=rtol, max_it=its, pc=pc)
    t00 = [timed(asm, solve(0, 0)) for _ in range(2)][-1]
    t0 = {k: [timed(asm, solve(0, k)) for _ in range(2)][-1] for k in (1, 11)}
    it0 = (t0[11] - t0[1]) / 10
    out = []
    for pc in (6, 7):
        first = timed(asm, solve(pc, 0))                       # plan + factorisation
        f0 = timed(asm, solve(pc, 0))
        t1 = timed(asm, solve(pc, 1))
        k = int(max(2, min(20, 2000.0 / max(t1 - f0, 1e-3))))  # about two seconds of iterations
        tk = timed(asm, solve(pc, 1 + k))
        itp = (tk - t1) / k
        apply_ms = (itp - it0) / 2
        factor_ms = f0 - t00 - 2 * apply_ms
        cap = int(min(max_it, max(10, budget_s * 1e3 / itp)))
        t = time.perf_counter()
        info = asm.tfqmr_dev(b_dev, y_dev, rtol=1e-8, max_it=cap, pc=pc)
        solve_s = time.perf_counter() - t
        d = {"case": name, "pc": pc, "cells": int(m.n_cells), "dofs": int(n), "nnz_owned": int(nnz_owned), "spmv_ms": spmv_ms,
             "plan_ms": first - f0, "factor_ms": factor_ms, "apply_ms": apply_ms, "apply_over_spmv": apply_ms / spmv_ms,
             "iter_ms": itp, "iter_ms_pc0": it0, "timed_iterations": k, "its": info["its"], "rel_rnorm": info["rnorm"] / bn,
             "converged": bool(info["rnorm"] <= 1e-8 * bn * 1.0001 or info["its"] < cap), "its_cap": cap, "solve_s": solve_s}
        if pc == 6:
            _, nc, nvc = asm.pilu_colours()
            d.update(colours=nc, velocity_colours=nvc)
        else:
            d["depth_lower"], d["depth_upper"] = asm.nilu_depth()
        print(json.dumps(d), flush=True)
        out.append(d)
    for p in (x_dev, b_dev, y_dev):
        asm.dev_free(p)
    asm.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--max-it", type=int, default=5000, help="iteration cap of the rtol 1e-8 solves")
    ap.add_argument("--budget-s", type=float, default=60.0, help="about this many seconds per rtol 1e-8 solve (lowers the cap)")
    ap.add_argument("--cases", default="duct_M,duct_p2,cavity", help="comma list of duct_M, duct_p2, cavity")
    ap.add_argument("--small", action="store_true", help="tiny meshes (a rehearsal of the script, not a measurement)")
    args = ap.parse_args()
    gpu = card()
    lines = []
    for c in args.cases.split(","):
        if c == "duct_M":
            nd = (6, 12) if args.small else (50, 200)
            m = M.duct_mesh(*nd); sp = M.mixed_space(m, 1)
            lines += measure(f"duct_p1p1_gmetric_{nd[0]}x{nd[0]}x{nd[1]}", m, sp, M.duct_bcs(sp), M.duct_state(sp), dict(flavour=0, nu=0.1),
                             args.max_it, args.budget_s)
        elif c == "duct_p2":
            nd = (4, 8) if args.small else (40, 80)
            m = M.duct_mesh(*nd); sp = M.mixed_space(m, 2)
            lines += measure(f"duct_p2p1_gmetric_{nd[0]}x{nd[0]}x{nd[1]}", m, sp, M.duct_bcs(sp), M.duct_state(sp), dict(flavour=0, nu=1.0 / 50),
                             args.max_it, args.budget_s)
        elif c == "cavity":
            nx = 24 if args.small else 1450
            m = M.create_rectangle_tris(nx, nx); sp = M.mixed_space(m, 1)
            lines += measure(f"cavity_ugn_p1p1_{nx}x{nx}", m, sp, M.cavity_bcs(sp), M.cavity_state(sp), dict(flavour=1, nu=0.01),
                             args.max_it, args.budget_s)
    with open(args.out, "w") if args.out else open(os.devnull, "w") as f:
        for d in lines:
            d["gpu"] = gpu
            f.write(json.dumps(d) + "\n")
    print(json.dumps({"gpu": gpu}), flush=True)


if __name__ == "__main__":
    main()
