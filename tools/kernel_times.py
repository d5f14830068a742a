"""Device time per kernel of the P1-P1 assembly on bench.py's duct, one GPU, from torch.profiler (CUPTI kernel records).

  python tools/kernel_times.py [--workload L|M|S] [--steps K] [--label TEXT] [--out FILE]

Builds the workload exactly as bench.py does, warms up, then profiles K fused Jacobian + residual assemblies and K
residual-only assemblies.  Appends one JSON line to FILE (and prints it): the card's name, power limit and maximum SM
clock, the free-text label (say, which code was measured), the library's own CUDA-event time of the assembly kernel (`last_kernel_ms`, mean over the K steps), and per pass
every kernel the profiler saw with its launch count and mean device time.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import CI, NU, WORKLOADS  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = (s.strip() for s in q.stdout.strip().split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="L", choices=sorted(WORKLOADS))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--label", default="")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile
    from stabilized_navier_stokes_flow_fenicsx_b200.assembler import NSAssembler
    from stabilized_navier_stokes_flow_fenicsx_b200 import distributed as D

    n_cross, n_long = WORKLOADS[args.workload]
    comm = D.Comm.single()
    part = D.duct_partition(n_cross, n_long, 0, 1)
    asm = NSAssembler(part.x, part.cells, part.dofmap, vdeg=1, n_dofs_owned=part.n_owned, n_dofs_ghost=part.n_ghost,
                      n_cells_owned=part.n_cells_owned, device=0)
    asm.set_form(flavour=0, nu=NU, Ci=CI)
    asm.set_bcs(part.bcs)
    D.attach(asm, part, comm)
    D.finish_pattern_exchange(asm, part, comm)
    nbytes = 8 * asm.n_cols
    x_dev, F_dev = asm.dev_alloc(nbytes), asm.dev_alloc(nbytes)
    w = np.zeros(asm.n_cols)
    w[: asm.n_dofs] = part.w
    asm.h2d(x_dev, w)

    line = {"tool": "tools/kernel_times.py", "label": args.label, "workload": args.workload, "cells": part.n_cells_owned, "steps": args.steps,
            "card": card(), "passes": {}}
    for name, want_j in (("jacobian_residual", True), ("residual", False)):
        for _ in range(args.warmup):
            asm.jacobian_residual_dev(x_dev, want_j, F_dev)
        asm.sync()
        events_ms = []
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.steps):
                asm.jacobian_residual_dev(x_dev, want_j, F_dev)
                events_ms.append(asm.last_kernel_ms())
            asm.sync()
            torch.cuda.synchronize()
        kernels = []
        for e in prof.key_averages():
            if e.device_time_total <= 0:
                continue
            kernels.append({"kernel": e.key, "launches": e.count, "mean_ms": e.device_time_total / e.count / 1e3,
                            "total_ms": e.device_time_total / 1e3})
        kernels.sort(key=lambda k: -k["total_ms"])
        line["passes"][name] = {"assembly_kernel": asm.last_kernel_name(), "event_ms_mean": float(np.mean(events_ms)),
                                "event_ms_min": float(np.min(events_ms)), "event_ms_max": float(np.max(events_ms)),
                                "kernels": kernels}
    asm.close()
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "a") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
