"""Boundary-functional throughput (csrc/boundary.cu): nsgpu_facet_integrals_dev with every exterior facet of the P1-P1 duct tagged by
box face (6 tags), and nsgpu_reaction_dev of the G-metric form over the four side walls (one tag), on M (50x50x200, 3.0 M cells) and L
(128x128x512, 50.3 M cells).  Times: nsgpu_set_facets (host clock around the synchronous call), then each _dev call with CUDA events
on the context's stream, median of 10 calls after 2 warm-up calls.  Prints one JSON line per workload and appends them to the file
--out names (profiles/r6_boundary.jsonl holds the committed run)."""
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

TET_FACETS = np.array([[1, 2, 3], [0, 2, 3], [0, 1, 3], [0, 1, 2]])


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout
        name, power = [s.strip() for s in out.splitlines()[0].split(",")]
        return name, power
    except Exception as e:  # the numbers are still device-timed; the card is then unknown
        return f"unknown ({e})", "unknown"


def duct_exterior_facets(m, n_cross, n_long, length):
    """(cell, local facet, tag) of every exterior facet of duct_mesh, tag = 2 * axis + side (x: 0 / 1, y: 2 / 3, z: 4 / 5).  Only the
    cells of the boxes on the boundary are examined (cells are box-major, 6 per box, duct axis slowest)."""
    b = np.arange(m.n_cells // 6)
    i0, i1, i2 = b % n_cross, (b // n_cross) % n_cross, b // (n_cross * n_cross)
    edge = (i0 == 0) | (i0 == n_cross - 1) | (i1 == 0) | (i1 == n_cross - 1) | (i2 == 0) | (i2 == n_long - 1)
    cand = (6 * b[edge][:, None] + np.arange(6)[None, :]).ravel()
    lo, hi = np.array([0.0, -0.5, -0.5]), np.array([length, 0.5, 0.5])
    out = []
    for lf in range(4):
        X = m.x[m.cells[cand][:, TET_FACETS[lf]]]                       # (k, 3 vertices, 3)
        for a in range(3):
            for side, v in ((0, lo[a]), (1, hi[a])):
                on = (np.abs(X[:, :, a] - v) < 1e-12).all(axis=1)
                out.append(np.stack([cand[on], np.full(on.sum(), lf), np.full(on.sum(), 2 * a + side)], axis=1))
    return np.concatenate(out).astype(np.int32).T


def timed(asm, fn, reps):
    for _ in range(2):
        fn()
    asm.sync()
    ms = []
    for _ in range(reps):
        asm.timer_start()
        fn()
        ms.append(asm.timer_stop())
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mesh", action="append", help="n_cross,n_long (default: 50,200 and 128,512)")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", help="append the JSON lines to this file")
    a = ap.parse_args()
    name, power = gpu_info()
    rows = []
    for spec in a.mesh or ["50,200", "128,512"]:
        nc, nl = (int(v) for v in spec.split(","))
        m = M.duct_mesh(nc, nl)
        sp = M.mixed_space(m, 1)
        w = M.duct_state(sp)
        fc, fl, ft = duct_exterior_facets(m, nc, nl, 4.0)
        asm = NSAssembler(m.x, m.cells, sp.dofmap, vdeg=1)
        asm.set_form(flavour=0, nu=0.1)
        w_dev, out_dev = asm.dev_alloc(8 * sp.n_dofs), asm.dev_alloc(8 * 6 * 11)
        asm.h2d(w_dev, w)
        t0 = time.perf_counter()
        n_tags = asm.set_facets(fc, fl, ft)
        t_set_faces = time.perf_counter() - t0
        ms_int = timed(asm, lambda: asm.facet_integrals_dev(w_dev, out_dev), a.reps)
        integ = np.empty((n_tags, 11))
        asm.d2h(integ, out_dev)
        walls = ft >= 2
        t0 = time.perf_counter()
        asm.set_facets(fc[walls], fl[walls], np.zeros(walls.sum(), dtype=np.int32))
        t_set_walls = time.perf_counter() - t0
        ms_rea = timed(asm, lambda: asm.reaction_dev(w_dev, out_dev), a.reps)
        react = np.empty(3)
        asm.d2h(react, out_dev)
        row = {"what": "boundary functionals, duct P1-P1", "gpu": name, "power_limit": power,
               "mesh": {"n_cross": nc, "n_long": nl, "cells": int(m.n_cells), "dofs": int(sp.n_dofs)},
               "exterior_facets": int(len(fc)), "wall_facets": int(walls.sum()),
               "facet_integrals_ms_median": float(np.median(ms_int)), "facet_integrals_ms_min": float(min(ms_int)),
               "facet_integrals_ms_max": float(max(ms_int)),
               "reaction_ms_median": float(np.median(ms_rea)), "reaction_ms_min": float(min(ms_rea)), "reaction_ms_max": float(max(ms_rea)),
               "reps": a.reps, "set_facets_faces_s": t_set_faces, "set_facets_walls_s": t_set_walls,
               "areas": integ[:, 0].tolist(), "inlet_flux": float(integ[0, 1]), "outlet_flux": float(integ[1, 1]),
               "wall_reaction": react.tolist()}
        print(json.dumps(row), flush=True)
        rows.append(row)
        asm.dev_free(w_dev); asm.dev_free(out_dev)
        asm.close()
        del m, sp, w
    if a.out:
        with open(a.out, "a") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
