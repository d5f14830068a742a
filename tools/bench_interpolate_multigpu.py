"""Non-matching interpolation on several GPUs (csrc/locate.cu, nsgpu_interpolate_dev on a communicator), run under torchrun with one
rank per GPU: the 50x50x200 P1-P1 duct (M) onto the 128x128x512 P1-P1 duct (L), both x-slab partitioned (duct_partition), the same
workload as tools/bench_interpolate.py on one GPU.  The cuts of the two meshes do not line up, so the destination nodes between a
rank's source cut and its destination cut are evaluated by the neighbouring rank.  Times: CUDA events on the destination's stream
around nsgpu_interpolate_dev, median of 10 calls after 2 warm-up calls, max over the ranks.  Prints one JSON line (rank 0) and
appends it to the file --out names."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from stabilized_navier_stokes_flow_fenicsx_b200 import distributed as D  # noqa: E402
from stabilized_navier_stokes_flow_fenicsx_b200.assembler import NSAssembler  # noqa: E402


def gpu_info(dev):
    out = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, timeout=30).stdout
    name, power = [s.strip() for s in out.splitlines()[0].split(",")]
    return name, power


def context(part, comm, dev):
    asm = NSAssembler(part.x, part.cells, part.dofmap, vdeg=1, n_dofs_owned=part.n_owned, n_dofs_ghost=part.n_ghost,
                      n_cells_owned=part.n_cells_owned, device=dev)
    asm.set_form(flavour=0, nu=0.1)
    D.attach(asm, part, comm)
    D.finish_pattern_exchange(asm, part, comm)      # the destination's halo plan refreshes its ghost entries
    return asm


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--src", default="50,200")
    ap.add_argument("--dst", default="128,512")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", help="append the JSON line to this file (rank 0)")
    a = ap.parse_args()
    comm = D.Comm.from_env()
    rank, size = comm.rank, comm.size
    dev = int(os.environ.get("LOCAL_RANK", rank))
    name, power = gpu_info(dev)
    nc_s, nl_s = (int(v) for v in a.src.split(","))
    nc_d, nl_d = (int(v) for v in a.dst.split(","))
    ps, pd = D.duct_partition(nc_s, nl_s, rank, size), D.duct_partition(nc_d, nl_d, rank, size)
    src, dst = context(ps, comm, dev), context(pd, comm, dev)
    ws_dev, wd_dev, cnt_dev = src.dev_alloc(8 * src.n_cols), dst.dev_alloc(8 * dst.n_cols), dst.dev_alloc(16)
    src.h2d(ws_dev, ps.w)
    # owned destination nodes outside this rank's source slab: the points this rank sends to other ranks (one rank each, the
    # neighbour whose slab holds them; a node on a source cut is inside a local cell and stays here)
    k0, k1 = D.slab_ranges(nl_s, size)[rank]
    x0, x1 = 4.0 * k0 / nl_s, 4.0 * k1 / nl_s
    xo = pd.x[: pd.n_owned // 4, 0]
    sent = int(((xo < x0 - 1e-12) | (xo > x1 + 1e-12)).sum())
    times = []
    for it in range(2 + a.reps):
        comm.barrier()
        dst.timer_start()                              # CUDA events on the destination's stream
        dst.interpolate_nonmatching_dev(src, ws_dev, wd_dev, counts_dev=cnt_dev)
        if it >= 2:
            times.append(dst.timer_stop())
        else:
            dst.timer_stop()
    cnt = np.empty(2, dtype=np.int64)
    dst.d2h(cnt, cnt_dev)
    med = float(np.median(times))
    ms_max = comm.max(med)
    sent_all = [0] * size
    import torch.distributed as dist
    dist.all_gather_object(sent_all, sent)
    row = {"workload": f"interpolate_dev M {nc_s}x{nc_s}x{nl_s} P1-P1 -> L {nc_d}x{nc_d}x{nl_d} P1-P1, x-slabs", "ranks": size,
           "ms_median_max_over_ranks": round(ms_max, 3), "ms_median_rank0": round(med, 3), "dst_nodes": (nc_d + 1) ** 2 * (nl_d + 1),
           "points_sent_per_rank": sent_all, "n_extrapolated": int(cnt[0]), "n_outside": int(cnt[1]), "reps": a.reps, "warmup": 2,
           "gpu": name, "power_limit": power}
    if rank == 0:
        print(json.dumps(row), flush=True)
        if a.out:
            with open(a.out, "a") as f:
                f.write(json.dumps(row) + "\n")
    src.close(); dst.close()
    comm.close()


if __name__ == "__main__":
    main()
