"""Non-matching interpolation throughput (csrc/locate.cu, nsgpu_interpolate_dev): the 50x50x200 P1-P1 duct (3.0 M cells) onto the
128x128x512 P1-P1 duct (L: 8.5 M nodes, 34.1 M dofs) and onto a 40x40x80 P2-P1 duct.  Contexts with mesh and space only (no
pattern).  Times: the one-off locator build of the source (first nsgpu_eval on one point, host clock around the synchronous call),
then nsgpu_interpolate_dev with CUDA events on the destination's stream, median of 10 calls after 2 warm-up calls.  Prints one JSON
line per workload and appends them to the file --out names (profiles/r5_interpolate.jsonl holds the committed run)."""
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


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout
        name, power = [s.strip() for s in out.splitlines()[0].split(",")]
        return name, power
    except Exception as e:  # the numbers are still device-timed; the card is then unknown
        return f"unknown ({e})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--src", default="50,200")
    ap.add_argument("--dst", action="append", help="n_cross,n_long,vdeg (default: 128,512,1 and 40,80,2)")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", help="append the JSON lines to this file")
    a = ap.parse_args()
    dsts = a.dst or ["128,512,1", "40,80,2"]
    name, power = gpu_info()
    nc_s, nl_s = (int(v) for v in a.src.split(","))
    ms = M.duct_mesh(nc_s, nl_s)
    sps_ = M.mixed_space(ms, 1)
    w = M.duct_state(sps_)
    src = NSAssembler(ms.x, ms.cells, sps_.dofmap, vdeg=1)
    ws_dev = src.dev_alloc(8 * sps_.n_dofs)
    src.h2d(ws_dev, w)
    one = np.array([[1.0, 0.0, 0.0]])
    t0 = time.perf_counter()
    src.eval(w, one)                                                   # builds the locator
    t_build = time.perf_counter() - t0
    t0 = time.perf_counter()
    src.eval(w, one)
    t_eval1 = time.perf_counter() - t0
    rows = []
    for spec in dsts:
        nc, nl, vd = (int(v) for v in spec.split(","))
        md = M.duct_mesh(nc, nl)
        spd = M.mixed_space(md, vd)
        n_nodes = md.n_vertices + (0 if vd == 1 else len(spd.edges))
        dst = NSAssembler(md.x, md.cells, spd.dofmap, vdeg=vd)
        wd_dev = dst.dev_alloc(8 * spd.n_dofs)
        cnt_dev = dst.dev_alloc(16)
        for _ in range(2):
            dst.interpolate_nonmatching_dev(src, ws_dev, wd_dev, counts_dev=cnt_dev)
        dst.sync()
        ms_list = []
        for _ in range(a.reps):
            dst.timer_start()
            dst.interpolate_nonmatching_dev(src, ws_dev, wd_dev, counts_dev=cnt_dev)
            ms_list.append(dst.timer_stop())
        cnt = np.empty(2, dtype=np.int64)
        dst.d2h(cnt, cnt_dev)
        # spot check against the field: the duct state is smooth, so the interpolant is close to it at the nodes
        wd = np.empty(spd.n_dofs)
        dst.d2h(wd, wd_dev)
        exact = M.duct_state(spd, noise=0.0)
        med = float(np.median(ms_list))
        row = {"what": "nsgpu_interpolate_dev, duct P1-P1 onto duct", "gpu": name, "power_limit": power,
               "src": {"n_cross": nc_s, "n_long": nl_s, "vdeg": 1, "cells": int(ms.n_cells), "dofs": int(sps_.n_dofs)},
               "dst": {"n_cross": nc, "n_long": nl, "vdeg": vd, "cells": int(md.n_cells), "nodes": int(n_nodes), "dofs": int(spd.n_dofs)},
               "ms_median": med, "ms_min": float(min(ms_list)), "ms_max": float(max(ms_list)), "reps": a.reps,
               "nodes_per_s": n_nodes / (med * 1e-3), "dofs_per_s": spd.n_dofs / (med * 1e-3),
               "locator_build_s": t_build, "eval_one_point_s": t_eval1,
               "n_extrapolated": int(cnt[0]), "n_outside": int(cnt[1]),
               "max_abs_diff_vs_noise_free_state": float(np.abs(wd - exact).max())}
        print(json.dumps(row), flush=True)
        rows.append(row)
        dst.dev_free(wd_dev); dst.dev_free(cnt_dev)
        dst.close()
        del md, spd, exact, wd
    src.dev_free(ws_dev)
    src.close()
    if a.out:
        with open(a.out, "a") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
