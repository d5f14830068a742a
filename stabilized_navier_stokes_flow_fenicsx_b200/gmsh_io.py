"""Standalone ingestion of the gmsh meshes the reference drivers write (SURVEY 8f rank 3).

``image2gmsh3D.py:523-525`` writes ``ChannelMesh.msh`` (MSH 4.1 ASCII, gmsh's default) with the physical groups
inlet_1 = 1, inlet_2 = 2, outlet = 3, wall = 4 on surfaces and "fluid" on the volume (``:435-440``); the drivers read it
back through ``gmshio.model_to_mesh`` (``NavierStokesChannelFlow.py:107-116``) and locate the Dirichlet dofs with
``locate_dofs_topological(..., ft.find(marker))`` (``:127-147``).  This module does the same without gmsh or dolfinx:

* ``read_msh`` -- nodes, the cells of the highest dimension that carry a physical group, and the tagged facets;
* ``facet_dofs`` -- the dofs of a mixed P_k^d x P1 space on the facets of a marker (vertices, plus edges for P2): what
  ``locate_dofs_topological`` returns for that sub-space;
* ``write_msh`` -- the inverse (used by the tests, and to hand a synthetic duct to the reference scripts).

The dof numbering produced by ``mesh.mixed_space`` on a mesh read here is vertex-blocked in gmsh node order, not dolfinx's
reordered one -- the assembler renumbers internally anyway (csrc/renumber.cu), and results are numbering-independent up to
the permutation."""
import numpy as np

from .mesh import Mesh, TET_EDGES, TRI_EDGES

_NODES_PER = {1: 2, 2: 3, 4: 4, 15: 1}          # gmsh element type -> nodes (line, triangle, tetrahedron, point)
_DIM_OF = {15: 0, 1: 1, 2: 2, 4: 3}
_TYPE_OF_DIM = {0: 15, 1: 1, 2: 2, 3: 4}


def _sections(text):
    out, name, buf = {}, None, []
    for line in text.splitlines():
        s = line.strip()
        if s.startswith("$End"):
            out[name] = buf
            name, buf = None, []
        elif s.startswith("$"):
            name, buf = s[1:], []
        elif name is not None:
            buf.append(s)
    return out


def read_msh(path):
    """Returns (Mesh, cell_tags, facets, facet_tags, names): cells of the top dimension in file order (first-order
    simplices), the physical tag of each cell, the tagged facets as vertex tuples with their physical tags, and the
    physical-group names {(dim, tag): name}."""
    sec = _sections(open(path).read())
    ver = sec["MeshFormat"][0].split()
    if not ver[0].startswith("4") or ver[1] != "0":
        raise ValueError(f"{path}: need MSH 4.x ASCII (got version {ver[0]}, binary flag {ver[1]})")
    names = {}
    for line in sec.get("PhysicalNames", [])[1:]:
        d, t, nm = line.split(maxsplit=2)
        names[(int(d), int(t))] = nm.strip('"')
    # entity -> physical tags
    phys = {0: {}, 1: {}, 2: {}, 3: {}}
    ent = sec["Entities"]
    npts, ncur, nsur, nvol = (int(v) for v in ent[0].split())
    k = 1
    for _ in range(npts):
        f = ent[k].split(); k += 1
        nph = int(f[4])
        phys[0][int(f[0])] = [int(v) for v in f[5:5 + nph]]
    for dim, cnt in ((1, ncur), (2, nsur), (3, nvol)):
        for _ in range(cnt):
            f = ent[k].split(); k += 1
            nph = int(f[7])
            phys[dim][int(f[0])] = [int(v) for v in f[8:8 + nph]]
    # nodes
    nd = sec["Nodes"]
    nblocks, nnodes = (int(v) for v in nd[0].split()[:2])
    tags, xyz = np.empty(nnodes, dtype=np.int64), np.empty((nnodes, 3))
    k, at = 1, 0
    for _ in range(nblocks):
        nb = int(nd[k].split()[3]); k += 1
        tags[at:at + nb] = [int(v) for v in nd[k:k + nb]]; k += nb
        xyz[at:at + nb] = [[float(v) for v in ln.split()[:3]] for ln in nd[k:k + nb]]; k += nb
        at += nb
    order = np.argsort(tags, kind="stable")
    tags, xyz = tags[order], xyz[order]
    # elements
    el = sec["Elements"]
    nblocks = int(el[0].split()[0])
    by_dim = {0: [], 1: [], 2: [], 3: []}
    k = 1
    for _ in range(nblocks):
        edim, etag, etype, nb = (int(v) for v in el[k].split()); k += 1
        if etype not in _NODES_PER:
            raise ValueError(f"{path}: element type {etype} is not a first-order simplex")
        conn = np.array([[int(v) for v in ln.split()[1:1 + _NODES_PER[etype]]] for ln in el[k:k + nb]], dtype=np.int64).reshape(nb, _NODES_PER[etype])
        k += nb
        for p in phys[edim].get(etag, []):
            by_dim[edim].append((p, conn))
    tdim = max(d for d in by_dim if by_dim[d])
    cells = np.concatenate([c for _, c in by_dim[tdim]])
    cell_tags = np.concatenate([np.full(len(c), p, dtype=np.int32) for p, c in by_dim[tdim]])
    facets = np.concatenate([c for _, c in by_dim[tdim - 1]]) if by_dim[tdim - 1] else np.zeros((0, tdim), dtype=np.int64)
    facet_tags = np.concatenate([np.full(len(c), p, dtype=np.int32) for p, c in by_dim[tdim - 1]]) if by_dim[tdim - 1] else np.zeros(0, np.int32)
    # node tags -> contiguous vertex ids (only the nodes the cells use, like model_to_mesh)
    used = np.unique(cells)
    vid = -np.ones(int(tags.max()) + 1, dtype=np.int64)
    vid[used] = np.arange(len(used))
    x = xyz[np.searchsorted(tags, used)]
    m = Mesh(tdim, np.ascontiguousarray(x), vid[cells].astype(np.int32), (), {"kind": "gmsh", "path": str(path)})
    return m, cell_tags, vid[facets].astype(np.int32), facet_tags, names


def write_msh(path, mesh, facets, facet_tags, names=None, cell_tag=1):
    """MSH 4.1 ASCII with one entity per physical group (what a reader needs; no CAD topology)."""
    tdim = mesh.gdim
    groups = sorted(set(int(t) for t in facet_tags))
    names = dict(names or {})
    with open(path, "w") as f:
        f.write("$MeshFormat\n4.1 0 8\n$EndMeshFormat\n")
        f.write(f"$PhysicalNames\n{len(groups) + 1}\n")
        for g in groups:
            f.write(f'{tdim - 1} {g} "{names.get((tdim - 1, g), "group%d" % g)}"\n')
        f.write(f'{tdim} {cell_tag} "{names.get((tdim, cell_tag), "fluid")}"\n$EndPhysicalNames\n')
        lo, hi = mesh.x.min(axis=0), mesh.x.max(axis=0)
        box = " ".join(repr(float(v)) for v in (*lo, *hi))
        ns, nv = (len(groups), 1) if tdim == 3 else (1, 0)
        nc = len(groups) if tdim == 2 else 0
        f.write(f"$Entities\n0 {nc} {ns} {nv}\n")
        for g in groups:
            f.write(f"{g} {box} 1 {g} 0\n")
        f.write(f"1 {box} 1 {cell_tag} 0\n$EndEntities\n")
        n = mesh.n_vertices
        f.write(f"$Nodes\n1 {n} 1 {n}\n{tdim} 1 0 {n}\n")
        f.write("\n".join(str(i + 1) for i in range(n)) + "\n")
        f.write("\n".join(" ".join(repr(float(v)) for v in p) for p in mesh.x) + "\n$EndNodes\n")
        ne = len(facets) + mesh.n_cells
        f.write(f"$Elements\n{len(groups) + 1} {ne} 1 {ne}\n")
        eid = 1
        for g in groups:
            sel = facets[np.asarray(facet_tags) == g]
            f.write(f"{tdim - 1} {g} {_TYPE_OF_DIM[tdim - 1]} {len(sel)}\n")
            for row in sel:
                f.write(f"{eid} " + " ".join(str(int(v) + 1) for v in row) + "\n"); eid += 1
        f.write(f"{tdim} 1 {_TYPE_OF_DIM[tdim]} {mesh.n_cells}\n")
        for row in mesh.cells:
            f.write(f"{eid} " + " ".join(str(int(v) + 1) for v in row) + "\n"); eid += 1
        f.write("$EndElements\n")


def boundary_facets(mesh):
    """Facets (vertex tuples, sorted) that belong to exactly one cell."""
    loc = ((1, 2, 3), (0, 2, 3), (0, 1, 3), (0, 1, 2)) if mesh.gdim == 3 else ((1, 2), (0, 2), (0, 1))
    allf = np.sort(np.concatenate([mesh.cells[:, f] for f in loc]).astype(np.int64), axis=1)
    uniq, cnt = np.unique(allf, axis=0, return_counts=True)
    return uniq[cnt == 1].astype(np.int32)


def facet_integration_domain(mesh, facets, facet_tags):
    """The (cell, local facet, tag) triples of ``ds(subdomain_data=facet_tags)`` for the tagged facets of ``read_msh`` /
    ``boundary_facets`` (what dolfinx's compute_integration_domains gives; local facet i is the facet opposite vertex i).
    Raises ValueError for a facet that belongs to no cell or to two cells (an interior facet)."""
    gd = mesh.gdim
    loc = ((1, 2, 3), (0, 2, 3), (0, 1, 3), (0, 1, 2)) if gd == 3 else ((1, 2), (0, 2), (0, 1))
    nc = mesh.n_cells
    allf = np.sort(np.concatenate([mesh.cells[:, f] for f in loc]).astype(np.int64), axis=1)
    owner = np.arange(len(loc) * nc, dtype=np.int64)                        # row k: cell k % nc, local facet k // nc
    order = np.lexsort(allf.T[::-1])
    allf, owner = allf[order], owner[order]
    want = np.sort(np.asarray(facets, dtype=np.int64).reshape(-1, gd), axis=1)
    tags = np.asarray(facet_tags, dtype=np.int32).ravel()
    if len(tags) != len(want):
        raise ValueError("facets and facet_tags differ in length")
    nv = max(int(mesh.n_vertices), 1)
    both = np.concatenate([allf, want])
    k = both[:, 0] * nv + both[:, 1]                                       # vertex pairs, then triples through the pair's rank
    if gd == 3:
        k = np.unique(k, return_inverse=True)[1].ravel().astype(np.int64) * nv + both[:, 2]
    ka, kw = k[: len(allf)], k[len(allf):]
    lo, hi = np.searchsorted(ka, kw, "left"), np.searchsorted(ka, kw, "right")
    cnt = hi - lo
    if (cnt == 0).any():
        raise ValueError(f"facet {want[np.flatnonzero(cnt == 0)[0]].tolist()} belongs to no cell")
    if (cnt > 1).any():
        raise ValueError(f"facet {want[np.flatnonzero(cnt > 1)[0]].tolist()} is shared by two cells (interior facet)")
    k = owner[lo]
    return (k % nc).astype(np.int32), (k // nc).astype(np.int32), tags.copy()


def facet_dofs(space, facets, facet_tags, marker, sub="velocity"):
    """locate_dofs_topological((W.sub(i), V), tdim - 1, ft.find(marker)) for the mixed space of mesh.mixed_space:
    velocity -> all components on the vertices (and, for P2, the edges) of the marked facets; pressure -> the vertices."""
    gd = space.mesh.gdim
    bs = gd + 1
    sel = np.asarray(facets)[np.asarray(facet_tags) == marker].astype(np.int64)
    verts = np.unique(sel)
    if sub == "pressure":
        return (bs * verts + gd).astype(np.int32)
    dofs = [(bs * verts[:, None] + np.arange(gd)[None, :]).ravel()]
    if space.vdeg == 2 and len(sel):
        nv = space.mesh.n_vertices
        key = np.minimum(space.edges[:, 0], space.edges[:, 1]).astype(np.int64) * nv + np.maximum(space.edges[:, 0], space.edges[:, 1])
        order = np.argsort(key)
        pairs = ((0, 1), (1, 2), (0, 2)) if gd == 3 else ((0, 1),)
        ek = np.unique(np.concatenate([np.minimum(sel[:, i], sel[:, j]) * nv + np.maximum(sel[:, i], sel[:, j]) for i, j in pairs]))
        e = order[np.searchsorted(key[order], ek)]
        dofs.append((bs * nv + gd * e[:, None] + np.arange(gd)[None, :]).ravel())
    return np.sort(np.concatenate(dofs)).astype(np.int32)
