"""Mesh, state and boundary-condition builders of the kernel-path tests (tests/test_kernel_paths_gpu.py, tests/test_meshes.py).

Everything is generated from a seed.  The meshes live in the unit square / cube (the fan mesh in [-2, 2]^3) with the boundary
vertices exactly on the faces, so boundary dofs are found by comparing coordinates with 0 and 1."""
import numpy as np
from scipy.spatial import Delaunay

from stabilized_navier_stokes_flow_fenicsx_b200 import mesh as M

# entities per cell of the row-owner kernel (rowown.cu): vertices + P2 edges
NENT = {(2, 1): 3, (2, 2): 6, (3, 1): 4, (3, 2): 10}


def ndofs_cell(gdim, vdeg):
    nvn = gdim + 1 if vdeg == 1 else (6 if gdim == 2 else 10)
    return gdim * nvn + gdim + 1


def coop_cells_per_block(gdim, vdeg):
    """Cells per CTA of the cooperative generic kernel (CoopCfg in assemble.cu: 256 // ND)."""
    return 256 // ndofs_cell(gdim, vdeg)


def _compact(gdim, x, cells, meta=None):
    used = np.unique(cells)
    remap = -np.ones(len(x), dtype=np.int64)
    remap[used] = np.arange(len(used))
    xx = np.zeros((len(used), 3))
    xx[:, :x.shape[1]] = x[used]
    return M.Mesh(gdim, xx, np.ascontiguousarray(remap[cells], dtype=np.int32), (), dict(meta or {}))


def signed_measure(mesh):
    """Signed area / volume (times 2 / 6) of every cell: negative for the cells whose vertex order is flipped."""
    p = mesh.x[mesh.cells][:, :, :mesh.gdim]
    d = p[:, 1:] - p[:, :1]
    return np.linalg.det(d)


def flip_cells(mesh, frac=1.0 / 3, seed=0):
    """Swap the first two vertices of a fraction of the cells (negative Jacobians).  Call before ``mixed_space`` so the P2 edge
    dofs follow the new local vertex order.  Returns a new mesh and the flipped-cell mask."""
    cells = mesh.cells.copy()
    flip = np.random.default_rng(seed).random(len(cells)) < frac
    cells[flip, 0], cells[flip, 1] = cells[flip, 1].copy(), cells[flip, 0].copy()
    return M.Mesh(mesh.gdim, mesh.x.copy(), cells, mesh.shape, dict(mesh.meta)), flip


def jitter_interior(mesh, amount, seed=0):
    """Move the interior vertices of a unit square / cube mesh by up to ``amount`` (absolute) in every direction."""
    x = mesh.x.copy()
    gd = mesh.gdim
    inner = np.all((x[:, :gd] > 1e-12) & (x[:, :gd] < 1 - 1e-12), axis=1)
    x[inner, :gd] += np.random.default_rng(seed).uniform(-amount, amount, (inner.sum(), gd))
    return M.Mesh(gd, x, mesh.cells.copy(), mesh.shape, dict(mesh.meta))


def structured(gdim, n, seed=0):
    """Unit square (n x n squares, 2 triangles each) or cube (n x n x n boxes, 6 tets each), interior vertices jittered by
    15 % of the spacing and a third of the cells flipped."""
    m = M.create_rectangle_tris(n, n) if gdim == 2 else M.create_box_tets((n, n, n))
    m = jitter_interior(m, 0.15 / n, seed)
    return flip_cells(m, seed=seed + 1)[0]


def delaunay_tets(n=12, seed=3, jitter=0.25):
    """Delaunay tetrahedralisation of an n^3 lattice of the unit cube with interior points jittered by up to ``jitter`` of the
    spacing; the flat slivers Delaunay leaves on the cube faces are dropped.  Mixed orientation (scipy's order)."""
    g = np.linspace(0.0, 1.0, n)
    x = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    inner = np.all((x > 0) & (x < 1), axis=1)
    h = 1.0 / (n - 1)
    x[inner] += np.random.default_rng(seed).uniform(-jitter * h, jitter * h, (inner.sum(), 3))
    t = Delaunay(x).simplices
    p = x[t]
    vol = np.einsum("ij,ij->i", np.cross(p[:, 1] - p[:, 0], p[:, 2] - p[:, 0]), p[:, 3] - p[:, 0])
    return _compact(3, x, t[np.abs(vol) > 1e-9 * h ** 3], {"kind": "delaunay_tets"})


def delaunay_tris(n=40, seed=0):
    """Delaunay triangulation of the unit square: n points per side on the boundary, (n - 2)^2 uniformly random interior points
    (vertices in up to ~12 cells, more than a jittered lattice gives)."""
    g = np.linspace(0.0, 1.0, n)
    z, o = np.zeros(n - 2), np.ones(n - 2)
    bnd = np.concatenate([np.stack([g, 0 * g], 1), np.stack([g, 0 * g + 1], 1), np.stack([z, g[1:-1]], 1), np.stack([o, g[1:-1]], 1)])
    x = np.concatenate([bnd, np.random.default_rng(seed).uniform(0.01, 0.99, ((n - 2) ** 2, 2))])
    h = 1.0 / (n - 1)
    t = Delaunay(x).simplices
    p = x[t]
    area = (p[:, 1, 0] - p[:, 0, 0]) * (p[:, 2, 1] - p[:, 0, 1]) - (p[:, 1, 1] - p[:, 0, 1]) * (p[:, 2, 0] - p[:, 0, 0])
    return _compact(2, x, t[np.abs(area) > 1e-9 * h ** 2], {"kind": "delaunay_tris"})


def fan_tets(n_sphere=40):
    """A vertex in more than 63 cells: Delaunay of the origin, ``n_sphere`` points on the sphere of radius 1/2 around it (Fibonacci
    spiral) and the corners and face centres of the cube [-2, 2]^3.  The origin's cells are the cones over the sphere points' hull
    triangles: 2 n_sphere - 4 of them."""
    k = np.arange(n_sphere) + 0.5
    phi = np.arccos(1 - 2 * k / n_sphere)
    th = np.pi * (1 + 5 ** 0.5) * k
    sph = 0.5 * np.stack([np.cos(th) * np.sin(phi), np.sin(th) * np.sin(phi), np.cos(phi)], 1)
    corners = 2.0 * np.array([[i, j, l] for i in (-1, 1) for j in (-1, 1) for l in (-1, 1)], dtype=float)
    faces = 2.0 * np.concatenate([np.eye(3), -np.eye(3)])
    x = np.concatenate([np.zeros((1, 3)), sph, corners, faces])
    t = Delaunay(x).simplices
    p = x[t]
    vol = np.einsum("ij,ij->i", np.cross(p[:, 1] - p[:, 0], p[:, 2] - p[:, 0]), p[:, 3] - p[:, 0])
    return _compact(3, x, t[np.abs(vol) > 1e-12], {"kind": "fan", "lo": -2.0, "hi": 2.0})


def take_cells(mesh, n, seed=0):
    """A connected-ish sub-mesh of exactly n cells (the first n in lexicographic order of their centroids), vertices compacted."""
    c = mesh.x[mesh.cells].mean(axis=1)
    order = np.lexsort(c.T[::-1])
    return _compact(mesh.gdim, mesh.x, mesh.cells[np.sort(order[:n])], dict(mesh.meta))


def single_cells(gdim, n):
    """1 reference-like cell, or 2 cells sharing a facet (the second one flipped)."""
    if gdim == 2:
        x = np.array([[0.0, 0, 0], [1.0, 0.1, 0], [0.2, 0.9, 0], [1.1, 1.0, 0]])
        cells = np.array([[0, 1, 2], [1, 2, 3]][:n], dtype=np.int32)
    else:
        x = np.array([[0.0, 0, 0], [1.0, 0.1, 0], [0.2, 0.9, 0.1], [0.1, 0.2, 1.0], [0.9, 0.8, 0.9]])
        cells = np.array([[0, 1, 2, 3], [2, 1, 3, 4]][:n], dtype=np.int32)
    return _compact(gdim, x, cells)


# ------------------------------------------------------------------------------------------------- degrees
def edge_cell_counts(cells):
    """Cells around every edge (tets: 6 edges per cell; triangles: 3)."""
    k = cells.shape[1]
    pairs = np.array([[a, b] for a in range(k) for b in range(a + 1, k)])
    e = np.sort(cells[:, pairs].reshape(-1, 2).astype(np.int64), axis=1)
    _, cnt = np.unique(e[:, 0] * (int(cells.max()) + 1) + e[:, 1], return_counts=True)
    return cnt


def vertex_cell_counts(cells):
    return np.bincount(cells.ravel(), minlength=int(cells.max()) + 1)


def n_entities(space):
    """(vertices, P2 edges) of a space: the two entity classes of the row-owner kernel."""
    return space.mesh.n_vertices, 0 if space.edges is None else len(space.edges)


# ------------------------------------------------------------------------------------------------- states / BCs
def box_bcs(space, lo=0.0, hi=1.0, tol=1e-12):
    """[walls, inlet, outlet pressure] on the box [lo, hi]^gdim: no-slip on the faces normal to axes 1.., a non-zero inflow on
    x = lo (every velocity component; its rim dofs are held by the wall object too, diagonal 2) and p = 0.3 on x = hi."""
    X, c = space.dof_x, space.dof_comp
    gd = space.mesh.gdim
    vel = c < gd
    s = (X - lo) / (hi - lo)
    on_wall = np.zeros(len(X), dtype=bool)
    for a in range(1, gd):
        on_wall |= (np.abs(s[:, a]) < tol) | (np.abs(s[:, a] - 1) < tol)
    wall = np.flatnonzero(vel & on_wall)
    inlet = np.flatnonzero(vel & (np.abs(s[:, 0]) < tol))
    prof = np.prod([4 * s[inlet, a] * (1 - s[inlet, a]) for a in range(1, gd)], axis=0)
    g_in = np.where(c[inlet] == 0, prof, 0.1 * prof * (1 + c[inlet]))
    outlet = np.flatnonzero((c == gd) & (np.abs(s[:, 0] - 1) < tol))
    return [(wall.astype(np.int32), np.zeros(len(wall))), (inlet.astype(np.int32), g_in),
            (outlet.astype(np.int32), np.full(len(outlet), 0.3))]


def cell_bcs(space, frac=0.1, seed=0):
    """Whole cells constrained: every dof (velocity and pressure) of a random tenth of the cells in one object with random values,
    and a second object that holds a random half of those dofs again (diagonal 2)."""
    rng = np.random.default_rng(seed)
    cells = rng.random(space.dofmap.shape[0]) < frac
    dofs = np.unique(space.dofmap[cells]).astype(np.int32)
    again = np.sort(rng.choice(dofs, len(dofs) // 2, replace=False)).astype(np.int32)
    return [(dofs, rng.standard_normal(len(dofs))), (again, rng.standard_normal(len(again)))]


def smooth_state(space, seed=1234, noise=1e-3, scale=1.0):
    """(s1) smooth field + noise: u_c = scale (0.6 + 0.4 sin(2 x + c) cos(3 y + z)), p = 1 - x."""
    X, c = space.dof_x, space.dof_comp
    gd = space.mesh.gdim
    x, y, z = X[:, 0], X[:, 1], X[:, 2]
    w = np.where(c < gd, scale * (0.6 + 0.4 * np.sin(2 * x + c) * np.cos(3 * y + z)), 1.0 - x)
    return w + noise * np.random.default_rng(seed).standard_normal(space.n_dofs)


def dirichlet_only_state(space, bcs):
    """(s3) the reference's initial guess: zero except on the Dirichlet dofs, which carry their values (last object wins)."""
    w = np.zeros(space.n_dofs)
    for d, v in bcs:
        w[np.asarray(d)] = v
    return w


def centroid_speed(space, w):
    """|u| at every cell centroid (P1: mean of the vertex values; P2: weights lam (2 lam - 1) at the vertices, 4 lam_i lam_j at
    the edges)."""
    gd = space.mesh.gdim
    nv = gd + 1
    dm = space.dofmap
    if space.vdeg == 1:
        wt = np.full(nv, 1.0 / nv)
    else:
        lam = 1.0 / nv
        wt = np.concatenate([np.full(nv, lam * (2 * lam - 1)), np.full(3 if gd == 2 else 6, 4 * lam * lam)])
    u = np.stack([(w[dm[:, gd * np.arange(len(wt)) + c]] * wt).sum(axis=1) for c in range(gd)], 1)
    return np.linalg.norm(u, axis=1)


def cell_diameter(mesh):
    p = mesh.x[mesh.cells]
    k = p.shape[1]
    return np.max([np.linalg.norm(p[:, a] - p[:, b], axis=1) for a in range(k) for b in range(a + 1, k)], axis=0)


def cell_reynolds(space, w, nu):
    """UGN's ReU = |u| h / (2 nu) at the cell centroids (h = cell diameter)."""
    return centroid_speed(space, w) * cell_diameter(space.mesh) / (2 * nu)


def reynolds_split_state(space, nu, seed=1234):
    """(s4) the smooth state with the velocity scaled so that the median cell Reynolds number is 3: UGN's LSIC parameter takes
    both of its branches (ReU <= 3 and ReU > 3)."""
    w = smooth_state(space, seed)
    re = cell_reynolds(space, w, nu)
    k = 3.0 / np.median(re)
    return np.where(space.dof_comp < space.mesh.gdim, k * w, w)
