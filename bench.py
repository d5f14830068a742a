#!/usr/bin/env python
"""bench.py -- NS Jacobian+residual assembly throughput (Mcells/s) and HBM-roofline fraction on B200.

A "step" is one pass of the hot path over the whole synthetic structured-tet duct: zero J and F,
fused Jacobian + residual assembly (incl. lifting, BC rows/cols, BC diagonal, set_bc), i.e. what
NonlinearPDE_SNESProblem.J + .F do at one Newton iterate (NavierStokes/NavierStokesChannelFlow.py:51-75).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload L|M|S] [--impl ours|reference] [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU); the duct is cut into x-slabs (strong scaling: the total
mesh is fixed).  One JSON line is printed by rank 0.  See DESIGN.md "Measurement" for the byte model.
--dump-outputs DIR (1 GPU) writes what the last timed step computed to DIR/*.npy (see dump_outputs).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {  # n_cross, n_long  (BASELINE.md section 3)
    "S": (10, 40),       # 24 000 cells  (mesh length 0.1, domain length 4)
    "M": (50, 200),      # 3.0 M cells
    "L": (128, 512),     # 50.33 M cells -- the configuration the metric is quoted on
}
NU, CI = 0.1, 36.0
# dram__bytes_read.sum + dram__bytes_write.sum of the assembly kernel, one launch, from the committed ncu --set full capture
# (default kernel options, 1 GPU): 6.03 GB read + 16.46 GB written, against 21.0 GB algorithmic (the pipelined kernel reads
# one vertex list per tile instead of eight indices per incidence, which removed ~9 GB of index traffic).
# Keyed by (workload, kernel name): the figures are only quoted when the run used that kernel on that workload on 1 GPU.
NCU_PROFILE = {
    ("L", "p1tet_pipe"): {"traffic": 22.49e9, "flop_per_cell": 5426, "source": "profiles/r1c_ncu_full_L_p1tet_pipe.txt"},
    # round 2, warp-specialised kernel: dram 8.12 GB read + 16.47 GB written (the per-tile blobs add ~2 GB of reads); executed
    # fp64 thread instructions 2 * 104.92 G DFMA + 42.93 G DMUL + 38.44 G DADD (source page of the capture)
    ("L", "p1tet_ws"): {"traffic": 24.58e9, "flop_per_cell": 5786, "source": "profiles/r2_ncu_full_L_p1tet_ws.txt"},
}
# executed fp64 work of the row-owner kernels per cell when no capture of the exact kernel is on file: 2*DFMA + DADD + DMUL thread
# instructions, 4 incidences per cell (the algebra is the same code in every variant; DESIGN.md 4.3 derives the count)
FLOP_PER_CELL_MODEL = 5786


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def algorithmic_bytes(nc, nv, ndof, nnz, nodes_per_cell=4, ndofs_cell=16):
    """Compulsory traffic (SURVEY 8d / BASELINE.md 3): every input read once, every output written once."""
    jf = 8 * nnz + 4 * nc * (nodes_per_cell + ndofs_cell) + 24 * nv + 16 * ndof
    f = 4 * nc * (nodes_per_cell + ndofs_cell) + 24 * nv + 16 * ndof
    spmv = 12 * nnz + 8 * (ndof + 1) + 8 * ndof + 8 * ndof
    return jf, f, spmv


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) >= 7 and r[3 + k].lower().startswith("active") for r in self.rows)]
        pw = [float(r[2]) for r in self.rows if len(r) >= 7 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": reasons}


# ------------------------------------------------------------------------------------------- reference arm
CPU_SAMPLE_LAYERS = {"L": 6, "M": 40, "S": 40}   # box layers of the duct in the CPU sample: L 589 824 cells, M 600 000, S the whole mesh


def cpu_sample_run(steps, warmup, workload):
    """Oracle (CPU restatement of the reference algorithm, OpenMP over ALL host cores) on a bounded slab of the same duct:
    same cross-section and box size as the GPU workload, fewer box layers along the axis.  The sample and the thread count
    do not depend on the number of GPUs or on what the launcher exported (torchrun sets OMP_NUM_THREADS=1)."""
    from oracle import oracle
    from stabilized_navier_stokes_flow_fenicsx_b200 import mesh as M
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    oracle.set_num_threads(cores)
    cores = oracle.num_threads()
    n_cross, n_long_full = WORKLOADS[workload]
    n_long = min(CPU_SAMPLE_LAYERS[workload], n_long_full)
    length = 4.0 * n_long / n_long_full
    m = M.duct_mesh(n_cross, n_long, length=length)
    sp = M.mixed_space(m, 1)
    w, bcs = M.duct_state(sp), M.duct_bcs(sp, length=length)
    marker, value, mult = oracle.bc_arrays(sp.n_dofs, [b[0] for b in bcs], [b[1] for b in bcs])
    indptr, indices = oracle.build_pattern_c(sp.dofmap, sp.n_dofs)          # create_matrix(): untimed, like the GPU arm's set-up
    form = oracle.Form(0, 3, 1, NU, CI)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        oracle.assemble_jacobian(form, m.x, m.cells, sp.dofmap, w, indptr, indices, marker, mult)
        F = oracle.assemble_residual(form, m.x, m.cells, sp.dofmap, w, marker, value)
        oracle.set_bc(F, [b[0] for b in bcs], [b[1] for b in bcs], w)
        t = time.perf_counter() - t0
        if it >= warmup:
            times.append(t)
    ms = 1e3 * float(np.mean(times))
    return {"value": m.n_cells / (ms * 1e-3) / 1e6, "unit": "Mcells/s", "cores": cores, "kind": "port",
            "sample": f"{n_cross}x{n_cross}x{n_long} box slab of the duct ({m.n_cells} cells), oracle J+F incl. CSR insertion by row search, "
                      f"OpenMP {cores} threads, {len(times)} step(s) after {warmup} warm-up; restated CPU baseline -- not dolfinx (not installable)",
            "ms_per_step": ms, "cells": m.n_cells}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_cross, n_long = WORKLOADS[args.workload]
    r = cpu_sample_run(args.steps, args.warmup, args.workload)
    line = {"impl": "reference", "metric": "NS Jacobian+residual assembly throughput", "value": r["value"], "unit": "Mcells/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"structured-tet duct {args.workload} ({n_cross}x{n_cross}x{n_long} boxes, P1-P1 G-metric, nu={NU}); bounded sample: {r['sample']}"},
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": "Mcells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------- our arm
DUMP_MAX_ENTRIES = 1 << 21      # per dumped array: 16 MB of float64


def dump_outputs(asm, F_dev, out_dir):
    """Write what one step hands its caller to out_dir as float64 .npy files: residual.npy, the residual F of the owned rows,
    and jacobian_values.npy, the CSR values of J in the caller's row order.  An output longer than DUMP_MAX_ENTRIES is cut to
    a fixed sample: F at seeded positions, J as whole rows in seeded blocks of 256 consecutive rows.  The bench's inputs are
    seeded as well, so two builds of the project can be compared entry for entry."""
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(7)
    n = asm.n_owned
    F = np.empty(n)
    asm.d2h(F, F_dev)
    if n > DUMP_MAX_ENTRIES:
        F = F[np.sort(rng.choice(n, DUMP_MAX_ENTRIES, replace=False))]
    vals_dev = asm.values_dev()
    if asm.nnz <= DUMP_MAX_ENTRIES:
        J = asm.get_value_range(0, asm.nnz, vals_dev)
    else:
        block = 256
        n_blocks = max(1, DUMP_MAX_ENTRIES * n // asm.nnz // block)          # about DUMP_MAX_ENTRIES values in all
        first = block * np.sort(rng.choice(n // block, n_blocks, replace=False))
        start, ptr, _ = asm.get_rows(np.concatenate([first, first + block - 1]))
        last = np.arange(n_blocks) + n_blocks                                # positions of the blocks' last rows
        end = start[last] + ptr[last + 1] - ptr[last]
        J = np.concatenate([asm.get_value_range(b, e - b, vals_dev) for b, e in zip(start[:n_blocks], end)])
    np.save(os.path.join(out_dir, "residual.npy"), F)
    np.save(os.path.join(out_dir, "jacobian_values.npy"), J)


def run_ours(args):
    from stabilized_navier_stokes_flow_fenicsx_b200 import mesh as M
    from stabilized_navier_stokes_flow_fenicsx_b200.assembler import NSAssembler
    from stabilized_navier_stokes_flow_fenicsx_b200 import distributed as D

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs needs a one-GPU run: every rank holds only its slab of the outputs")
    comm = D.Comm.from_env() if world > 1 else D.Comm.single()
    n_cross, n_long = WORKLOADS[args.workload]

    t_setup = time.perf_counter()
    part = D.duct_partition(n_cross, n_long, rank, world)          # rank-local slab in dolfinx layout
    asm = NSAssembler(part.x, part.cells, part.dofmap, vdeg=1, n_dofs_owned=part.n_owned, n_dofs_ghost=part.n_ghost,
                      n_cells_owned=part.n_cells_owned, device=local_rank)
    asm.set_form(flavour=0, nu=NU, Ci=CI)
    asm.set_bcs(part.bcs)
    if args.kernel is not None:
        asm.set_option("kernel", args.kernel)
    if args.ws is not None:
        asm.set_option("ws", args.ws)
    if os.environ.get("NSGPU_OVERLAP") is not None:                 # experiment switch: 0 = serial exchanges after the kernel
        asm.set_option("overlap", int(os.environ["NSGPU_OVERLAP"]))
    if os.environ.get("NSGPU_SM_RESERVE") is not None:
        asm.set_option("sm_reserve", int(os.environ["NSGPU_SM_RESERVE"]))
    if args.pipe is not None:
        asm.set_option("pipe", args.pipe)
    D.attach(asm, part, comm)                                       # the library's own NCCL communicator
    D.finish_pattern_exchange(asm, part, comm)                      # pattern (+ SparsityPattern.finalize exchange), halo / ghost-row plans
    setup_s = time.perf_counter() - t_setup

    nbytes = 8 * asm.n_cols                                         # owned + ghost + column-ghost entries
    x_dev, F_dev, y_dev = asm.dev_alloc(nbytes), asm.dev_alloc(nbytes), asm.dev_alloc(nbytes)
    w_local = np.zeros(asm.n_cols)
    w_local[: asm.n_dofs] = part.w
    asm.h2d(x_dev, w_local)

    def step():
        asm.jacobian_residual_dev(x_dev, True, F_dev)

    launches0 = None
    for _ in range(args.warmup):
        step()
    asm.sync()
    comm.barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = asm.launch_count()
    kernel_ms = []
    asm.timer_start()
    for _ in range(args.steps):
        step()
        if args.per_step_sync:
            kernel_ms.append(asm.last_kernel_ms())
    total_ms = asm.timer_stop()
    asm.sync()
    comm.barrier()
    launches = asm.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = comm.max(total_ms / args.steps)
    if args.dump_outputs:
        dump_outputs(asm, F_dev, args.dump_outputs)

    # dominant kernel alone (CUDA events on the library's stream around the assembly kernel), timed live
    kms = []
    for _ in range(min(args.steps, 10)):
        step()
        kms.append(asm.last_kernel_ms())
    kernel_ms_avg = comm.max(float(np.mean(kms)))
    kname = asm.last_kernel_name()                                   # the variant the timed steps ran

    # residual only, SpMV
    f_ms = []
    for _ in range(3 + min(args.steps, 10)):
        asm.jacobian_residual_dev(x_dev, False, F_dev)
        f_ms.append(asm.last_kernel_ms())
    f_ms = comm.max(float(np.mean(f_ms[3:])))
    j_ms = []
    for _ in range(3 + min(args.steps, 10)):
        asm.jacobian_residual_dev(x_dev, True, None)            # Jacobian only (SURVEY 8d asks for J-only, F-only, fused, SpMV)
        j_ms.append(asm.last_kernel_ms())
    j_ms = comm.max(float(np.mean(j_ms[3:])))
    s_ms = []
    for _ in range(3 + min(args.steps, 10)):
        asm.spmv_dev(x_dev, y_dev)
        s_ms.append(asm.last_kernel_ms())
    s_ms = comm.max(float(np.mean(s_ms[3:])))

    # end to end through the public host API: pinned x -> H2D -> J+F (J stays resident for MatMult) -> D2H F
    xh = asm.pinned_empty(asm.n_dofs)
    Fh = asm.pinned_empty(asm.n_dofs)
    xh[:] = part.w
    e2e_steps = max(2, min(args.steps, 5))
    asm.jacobian_residual(xh, F_out=Fh, fetch_vals=False)
    comm.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        asm.jacobian_residual(xh, F_out=Fh, fetch_vals=False)
    e2e_ms = comm.max(1e3 * (time.perf_counter() - t0) / e2e_steps)
    # partition-independent checksums of one assembly (all ranks' owned rows): ||F||_2 and ||J||_F
    asm.jacobian_residual_dev(x_dev, True, F_dev)
    f_checksum = asm.norm_dev(F_dev)
    j_checksum = asm.values_norm()
    fp64_peak = asm.fp64_peak()                                      # live DFMA micro-benchmark on this GPU

    # AIJ mode: the CSR values come back to (pinned) host memory as well -- what createAIJWithArrays / MatUpdateMPIAIJWithArrays needs
    e2e_aij_ms = None
    if not args.no_aij:
        try:
            vh = asm.pinned_empty(asm.nnz)
            asm.jacobian_residual(xh, vals_out=vh, F_out=Fh)
            comm.barrier()
            t0 = time.perf_counter()
            asm.jacobian_residual(xh, vals_out=vh, F_out=Fh)
            e2e_aij_ms = comm.max(1e3 * (time.perf_counter() - t0))
        except Exception as ex:                                      # pinned allocation of 8 * nnz bytes can fail on a small host
            e2e_aij_ms = None
            aij_note = str(ex)

    # what one Newton iterate costs through the SNES callbacks (F then J at the same state, host vectors), with the
    # residual call assembling the Jacobian in the same pass (option fuse_fj) -- and the Krylov iteration on the resident J
    asm.set_option("fuse_fj", 1)
    asm.residual(xh, out=Fh); asm.jacobian(xh, fetch=False)
    comm.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        asm.residual(xh, out=Fh)
        asm.jacobian(xh, fetch=False)
    snes_ms = comm.max(1e3 * (time.perf_counter() - t0) / e2e_steps)
    asm.set_option("fuse_fj", 0)
    asm.jacobian_residual_dev(x_dev, True, F_dev)
    asm.tfqmr_dev(F_dev, y_dev, rtol=0.0, max_it=1, pc=4)          # allocate work vectors
    tk = []
    for k_its in (2, 17):                                          # marginal cost of an iteration: (t(17) - t(2)) / 15
        asm.sync(); comm.barrier()
        t0 = time.perf_counter()
        kinfo = asm.tfqmr_dev(F_dev, y_dev, rtol=0.0, max_it=k_its, pc=4)
        tk.append((kinfo["its"], comm.max(1e3 * (time.perf_counter() - t0))))
    tfqmr_ms = (tk[1][1] - tk[0][1]) / max(tk[1][0] - tk[0][0], 1)
    tfqmr_solve_overhead_ms = tk[0][1] - tk[0][0] * tfqmr_ms       # set-up product, preconditioner extraction, true-residual check
    tfqmr_ilu = None
    if not args.no_extras:
        try:                                                       # the same with the multicolour block ILU(0) (pc = 5)
            tq = []
            asm.tfqmr_dev(F_dev, y_dev, rtol=0.0, max_it=1, pc=5)   # one-off colouring / plan of the ILU outside the timed solves
            for k_its in (3, 33):                                  # 30 iterations apart: the factorisation time of a solve varies by tens of ms
                asm.sync(); comm.barrier()
                t0 = time.perf_counter()
                ki = asm.tfqmr_dev(F_dev, y_dev, rtol=0.0, max_it=k_its, pc=5)
                tq.append((ki["its"], comm.max(1e3 * (time.perf_counter() - t0))))
            ms_it = (tq[1][1] - tq[0][1]) / max(tq[1][0] - tq[0][0], 1)
            tfqmr_ilu = {"ms_per_iteration": ms_it, "per_solve_overhead_ms": tq[0][1] - tq[0][0] * ms_it, "colours": asm.ilu_colours()[1],
                         "what": "pc = 5: multicolour 4x4-block ILU(0), block Jacobi over the ranks; the per-solve overhead holds the factorisation"}
        except Exception as e:                                     # noqa: BLE001 -- reported, not fatal
            tfqmr_ilu = {"error": str(e)[:200]}
    other = other_paths() if (world == 1 and not args.no_extras) else None

    nc_total = 6 * n_cross * n_cross * n_long
    nv_total = (n_cross + 1) ** 2 * (n_long + 1)
    ndof_total = 4 * nv_total
    nnz_total = comm.sum(part.owned_nnz(asm))
    b_jf, b_f, b_spmv = algorithmic_bytes(nc_total, nv_total, ndof_total, nnz_total)
    hbm, how = peaks()
    hbm_total = hbm * world

    prof = NCU_PROFILE.get((args.workload, kname)) if world == 1 else None
    flop_per_cell = prof["flop_per_cell"] if prof else FLOP_PER_CELL_MODEL
    if rank == 0:
        value = nc_total / (ms_per_step * 1e-3) / 1e6
        achieved = b_jf / (kernel_ms_avg * 1e-3) / 1e9
        line = {
            "metric": "NS Jacobian+residual assembly throughput", "value": value, "unit": "Mcells/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"structured-tet duct {args.workload}: {n_cross}x{n_cross}x{n_long} boxes x 6 tets = {nc_total} cells, "
                                   f"{ndof_total} dofs, nnz {nnz_total}; P1-P1 G-metric SUPG/PSPG/LSIC, nu={NU}, Ci={CI}; "
                                   f"BCs wall/inlet/outlet; x-slab partition over {world} GPU(s)",
                       "l2": "inputs larger than L2 (no flush needed)" if b_jf / world > 4 * 126e6 else "working set near L2 size: latency-bound case",
                       "kernel": kname, "setup_s": round(setup_s, 2)},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_total, "unit": "GB/s", "frac": achieved / hbm_total,
                         "traffic": prof["traffic"] if prof else None,
                         "traffic_source": (prof["source"] + " (same kernel, same workload, 1 GPU)") if prof else None,
                         "peak_source": how, "kernel_ms": kernel_ms_avg, "algorithmic_bytes": b_jf,
                         "note": "the J kernel's binding ceiling is the fp64 pipe, not HBM (SURVEY 8d, DESIGN.md 4.3): see the fp64 block"},
            "fp64": {"flop_per_cell_executed": flop_per_cell, "achieved_TFLOP/s": flop_per_cell * nc_total / (kernel_ms_avg * 1e-3) / 1e12,
                     "peak_TFLOP/s": fp64_peak * world, "frac": flop_per_cell * nc_total / (kernel_ms_avg * 1e-3) / 1e12 / (fp64_peak * world),
                     "peak_source": "DFMA micro-benchmark run live in this process (nsgpu_fp64_peak)",
                     "flop_source": (prof["source"] if prof else "instruction-count model of the row-owner algebra (DESIGN.md 4.3); no ncu capture of this kernel/workload on file")},
            "residual_only": {"ms": f_ms, "Mcells/s": nc_total / (f_ms * 1e-3) / 1e6, "GB/s": b_f / (f_ms * 1e-3) / 1e9,
                              "frac": b_f / (f_ms * 1e-3) / 1e9 / hbm_total},
            "jacobian_only": {"ms": j_ms, "Mcells/s": nc_total / (j_ms * 1e-3) / 1e6},
            "spmv": {"ms": s_ms, "GB/s": b_spmv / (s_ms * 1e-3) / 1e9, "frac": b_spmv / (s_ms * 1e-3) / 1e9 / hbm_total,
                     "GFLOP/s": 2 * nnz_total / (s_ms * 1e-3) / 1e9,
                     "note": "GB/s uses the CSR byte model of BASELINE.md (12 B/nnz + vectors); the vertex-blocked kernel reads one column "
                             "index per 4x4 block, so the bytes it actually moves are ~8.8 B/nnz",
                     "moved_GB/s": (8.0 * nnz_total + 8.0 * nnz_total / 16 + 56.0 * ndof_total / 4 + 16.0 * ndof_total) / (s_ms * 1e-3) / 1e9},
            "e2e": {"value": nc_total / (e2e_ms * 1e-3) / 1e6, "unit": "Mcells/s", "h2d_bytes_per_step": 8 * ndof_total,
                    "d2h_bytes_per_step": 8 * ndof_total, "ms_per_step": e2e_ms,
                    "what": "NSAssembler.jacobian_residual(x_host_pinned) -> F_host; J stays device-resident for MatMult (MatShell mode)"},
            "e2e_aij": {"ms_per_step": e2e_aij_ms, "Mcells/s": (nc_total / (e2e_aij_ms * 1e-3) / 1e6) if e2e_aij_ms else None,
                        "d2h_bytes_per_step": 8 * ndof_total + 8 * nnz_total,
                        "what": "same call with the CSR values copied to pinned host memory too (AIJ mode: PCIe-bound)"},
            "checksums": {"F_l2": f_checksum, "J_frobenius": j_checksum,
                          "what": "norms over all ranks' owned rows after one assembly: equal (to rounding) at every GPU count"},
            "snes_iterate": {"ms": snes_ms, "what": "NonlinearPDE_SNESProblem-style callback pair per Newton iterate: nsgpu_residual(x_host) -> F_host "
                                                      "then nsgpu_jacobian(x_host) (J stays resident), option fuse_fj: the residual pass assembles J, the Jacobian "
                                                      "call recognises the state on the device and reuses it"},
            "tfqmr": {"ms_per_iteration": tfqmr_ms, "iterations_timed": tk[1][0] - tk[0][0], "pc": "4x4 vertex-block Jacobi",
                      "per_solve_overhead_ms": tfqmr_solve_overhead_ms,
                      "what": "device-resident KSPTFQMR iteration on the resident Jacobian: 2 MatMult + fused vector updates / reductions "
                              "(marginal cost: the difference of a 17- and a 2-iteration solve); per_solve_overhead_ms = preconditioner extraction, "
                              "the set-up product and the true-residual check of one solve"},
            "tfqmr_ilu": tfqmr_ilu,
            "other_paths": other,
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        if world == 1 and not args.no_cpu_baseline:
            r = cpu_sample_run(1, 1, args.workload)
            line["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
        print(json.dumps(line), flush=True)
    for p in (x_dev, F_dev, y_dev):
        asm.dev_free(p)
    asm.close()
    comm.close()


def other_paths():
    """The other hot-path rows of SURVEY section 8 on small fixed inputs (1 GPU): the second element pair and the streamline tracer."""
    from stabilized_navier_stokes_flow_fenicsx_b200 import mesh as M
    from stabilized_navier_stokes_flow_fenicsx_b200 import streamtrace as ST
    from stabilized_navier_stokes_flow_fenicsx_b200.assembler import NSAssembler
    out = {}
    m = M.duct_mesh(24, 48); sp = M.mixed_space(m, 2)
    a2 = NSAssembler(m.x, m.cells, sp.dofmap, vdeg=2)
    a2.set_form(flavour=0, nu=1.0 / 50); a2.set_bcs(M.duct_bcs(sp))
    a2.create_matrix(fetch=False)
    xd, Fd = a2.dev_alloc(8 * a2.n_cols), a2.dev_alloc(8 * a2.n_cols)
    a2.h2d(xd, M.duct_state(sp))
    ts = []
    for it in range(8):
        a2.jacobian_residual_dev(xd, True, Fd)
        if it >= 3:
            ts.append(a2.last_kernel_ms())
    ms = float(np.median(ts))
    out["p2p1_gmetric"] = {"cells": m.n_cells, "nnz": int(a2.nnz), "kernel": a2.last_kernel_name(), "jf_ms": ms, "Mcells/s": m.n_cells / ms / 1e3,
                           "what": "fused J+F on P2-P1 Taylor-Hood tets (BASELINE config 4 pair), atomics-free row-owner kernel"}
    a2.close()
    m = M.duct_mesh(10, 40)
    y, z = m.x[:, 1], m.x[:, 2]
    prof = (1 - 4 * y * y) * (1 - 4 * z * z)
    u = np.column_stack((1.5 * prof + 0.02, -0.6 * z * prof, 0.6 * y * prof))
    tr = ST.StreamTracer(m.x, m.cells, u)
    rng = np.random.default_rng(5)
    seeds = np.hstack((np.full((40000, 1), 0.3), rng.uniform(-0.3, 0.3, size=(40000, 2))))
    tr.trace(seeds[:256])
    t0 = time.perf_counter()
    end, status, tf, ns = tr.trace(seeds)
    dt = time.perf_counter() - t0
    out["streamtrace"] = {"seeds": 40000, "cells": m.n_cells, "ms_host_to_host": 1e3 * dt, "kernel_ms": tr.last_kernel_ms(), "seeds_per_s": 40000 / dt,
                          "accepted_steps": int(ns.sum()), "reached_x_3.7": int((status == 1).sum()),
                          "what": "streamtrace.py's 40 000 seeds (RK45, rtol 1e-3, max_step 0.125, events) in one nsgpu_trace_run call"}
    tr.close()
    return out


def asm_kernel_name(asm):
    return asm.last_kernel_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("NSGPU_WORKLOAD", "L"), choices=sorted(WORKLOADS))
    ap.add_argument("--kernel", type=int, default=None, help="0 auto, 1 generic, 2 fast")
    ap.add_argument("--ws", type=int, default=None, help="0: do not use the warp-specialised variant of the factorised kernel")
    ap.add_argument("--pipe", type=int, default=None, help="0: do not use the software-pipelined variant either (plain tile kernel)")
    ap.add_argument("--per-step-sync", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the small P2-P1 / streamline-tracer measurements (other_paths)")
    ap.add_argument("--no-aij", action="store_true", help="skip the AIJ-mode end-to-end step (values to pinned host memory)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the residual and Jacobian values of the last timed step to DIR/*.npy (1 GPU; sampled above 2^21 entries)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
