"""TEST INFRASTRUCTURE ONLY -- NumPy restatement of point evaluation on a communicator (nsgpu_eval / nsgpu_interpolate over several
ranks, csrc/locate.cu; dolfinx determine_point_ownership), on top of the one-rank restatement oracle/interp_ref.Source built over each
rank's owned cells."""
import numpy as np


def eval_distributed(sources, points_per_rank, tol=1e-12, padding=0.0):
    """nsgpu_eval on a communicator: ``sources[r]`` is rank r's Source over its owned cells (local cell numbering), each rank asks
    about its own points.  Per point of rank q:
      1. inside an owned cell of q (lowest such cell)                                          -> code c (q's numbering)
      2. else inside on the lowest other rank r that has one (its lowest such cell)             -> code c (r's numbering)
      3. else, padding > 0: the smallest point-to-cell distance over every rank's owned cells, ties to the lower rank, then the
         lower cell, accepted when <= padding; that cell's polynomials at p                   -> code -2 - c
      4. otherwise value 0                                                                      -> code -1
    Returns per rank (values (n, gdim + 1), codes (n,), resolving rank (n,), -1 outside)."""
    out = []
    for q, pts in enumerate(points_per_rank):
        pts = np.asarray(pts, dtype=np.float64).reshape(-1, 3)
        values = np.zeros((pts.shape[0], sources[q].gd + 1))
        codes = np.full(pts.shape[0], -1, dtype=np.int64)
        owner = np.full(pts.shape[0], -1, dtype=np.int64)
        order = [q] + [r for r in range(len(sources)) if r != q]
        for i, p in enumerate(pts):
            for r in order:
                c = sources[r].locate(p, tol, 0.0)
                if c >= 0:
                    codes[i], owner[i] = c, r
                    values[i] = sources[r].eval_cell(c, p)
                    break
            else:
                if padding > 0.0:
                    best = None
                    for r in range(len(sources)):
                        d = sources[r].cell_dist(p)
                        c = int(np.flatnonzero(d == d.min())[0])
                        if d[c] <= padding and (best is None or d[c] < best[0]):
                            best = (d[c], r, c)
                    if best is not None:
                        _, r, c = best
                        codes[i], owner[i] = -2 - c, r
                        values[i] = sources[r].eval_cell(c, p)
        out.append((values, codes, owner))
    return out
