"""NumPy restatement of the isosurface rules of csrc/isosurface.cu (include/knerf.h, "mesh export"): marching
tetrahedra on the Kuhn split, vertices in (grid point, delta) order, triangles in (cell, tet, triangle) order.  Test
infrastructure: the GPU tests compare the kernel with it index for index, the CPU tests check its topology and
geometry on analytic fields.  Written independently of the kernel: the triangles come from a table of the 16 inside
patterns of each tet, built once from the orientation rule."""
from __future__ import annotations

import numpy as np

DELTAS = np.array([(1, 0, 0), (0, 1, 0), (0, 0, 1), (1, 1, 0), (1, 0, 1), (0, 1, 1), (1, 1, 1)], dtype=np.int64)
PERMS = [(0, 1, 2), (0, 2, 1), (1, 0, 2), (1, 2, 0), (2, 0, 1), (2, 1, 0)]
_DELTA_INDEX = {tuple(d): i for i, d in enumerate(DELTAS.tolist())}


def tet_corners(tet: int) -> np.ndarray:
    a, b, _ = PERMS[tet]
    c = np.zeros((4, 3), np.int64)
    c[1, a] = 1
    c[2, a] = c[2, b] = 1
    c[3] = 1
    return c


def _oriented(corners, tri, inside):
    """tri: 3 edges (pairs of tet corners); keep the order if the normal of the midpoint triangle points from the inside
    corners' centroid to the outside ones', else swap the last two"""
    mid = np.array([corners[a] + corners[b] for a, b in tri])           # doubled midpoints
    normal = np.cross(mid[1] - mid[0], mid[2] - mid[0])
    ins = [v for v in range(4) if inside[v]]
    outs = [v for v in range(4) if not inside[v]]
    direction = corners[outs].mean(0) - corners[ins].mean(0)
    dot = float(normal @ direction)
    assert dot != 0.0
    return tri if dot > 0 else [tri[0], tri[2], tri[1]]


def _table():
    """table[tet][pattern] = list of triangles, each 3 edges (lower corner, upper corner); pattern bit v = corner v in"""
    table = []
    for tet in range(6):
        corners = tet_corners(tet)
        rows = []
        for pat in range(16):
            inside = [(pat >> v) & 1 == 1 for v in range(4)]
            ins = [v for v in range(4) if inside[v]]
            outs = [v for v in range(4) if not inside[v]]
            if len(ins) == 1:
                tris = [[(ins[0], o) for o in outs]]
            elif len(ins) == 3:
                tris = [[(i, outs[0]) for i in ins]]
            elif len(ins) == 2:
                (a, b), (c, d) = ins, outs
                tris = [[(a, c), (a, d), (b, d)], [(a, c), (b, d), (b, c)]]
            else:
                tris = []
            rows.append([[tuple(sorted(e)) for e in _oriented(corners, t, inside)] for t in tris])
        table.append(rows)
    return table


TABLE = _table()


def _gradient(f: np.ndarray, spacing) -> np.ndarray:
    """central differences, one-sided on the faces, fp32, in field units per world unit: [nx,ny,nz,3]"""
    g = np.zeros(f.shape + (3,), np.float32)
    for ax in range(3):
        h = np.float32(spacing[ax])
        fm = np.moveaxis(f, ax, 0)
        gm = np.moveaxis(g[..., ax], ax, 0)
        gm[1:-1] = (fm[2:] - fm[:-2]) / (np.float32(2) * h)
        gm[0] = (fm[1] - fm[0]) / h
        gm[-1] = (fm[-1] - fm[-2]) / h
    return g


def isosurface(field, iso: float, origin=(0.0, 0.0, 0.0), spacing=(1.0, 1.0, 1.0)):
    """field [nx,ny,nz] -> (vertices [V,3] fp32, normals [V,3] fp32, triangles [T,3] int64)"""
    f = np.ascontiguousarray(field, dtype=np.float32)
    nx, ny, nz = f.shape
    iso = np.float32(iso)
    origin = np.asarray(origin, np.float32)
    spacing = np.asarray(spacing, np.float32)
    inside = f > iso
    cross = np.zeros((nx, ny, nz, 7), bool)
    for d, (dx, dy, dz) in enumerate(DELTAS):
        cross[:nx - dx, :ny - dy, :nz - dz, d] = inside[:nx - dx, :ny - dy, :nz - dz] != inside[dx:, dy:, dz:]
    flat = cross.reshape(-1, 7)
    vid = np.cumsum(flat.reshape(-1)).reshape(flat.shape) - 1            # vertex index of every crossing (p, d)
    pts, ds = np.nonzero(flat)                                           # (point, delta) order
    p = np.stack(np.unravel_index(pts, (nx, ny, nz)), -1)
    dl = DELTAS[ds]
    q = p + dl
    fp = f[p[:, 0], p[:, 1], p[:, 2]]
    fq = f[q[:, 0], q[:, 1], q[:, 2]]
    t = (iso - fp) / (fq - fp)
    pos = origin + spacing * (p.astype(np.float32) + t[:, None] * dl.astype(np.float32))
    g = _gradient(f, spacing)
    gp, gq = g[p[:, 0], p[:, 1], p[:, 2]], g[q[:, 0], q[:, 1], q[:, 2]]
    n = gp + t[:, None] * (gq - gp)
    length = np.sqrt((n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1]) + n[:, 2] * n[:, 2])
    safe = np.where(length > 0, length, np.float32(1))
    normals = np.where(length[:, None] > 0, -(n / safe[:, None]), np.float32(0)).astype(np.float32)

    # triangles: every (tet, pattern) for all cells at once, then sorted by (cell, tet, triangle)
    ci, cj, ck = np.meshgrid(np.arange(nx - 1), np.arange(ny - 1), np.arange(nz - 1), indexing="ij")
    cells = np.stack([ci.reshape(-1), cj.reshape(-1), ck.reshape(-1)], -1)
    cell_lin = (cells[:, 0] * ny + cells[:, 1]) * nz + cells[:, 2]
    keys, tris = [], []
    for tet in range(6):
        corners = tet_corners(tet)
        pat = np.zeros(len(cells), np.int64)
        for v in range(4):
            c = cells + corners[v]
            pat |= inside[c[:, 0], c[:, 1], c[:, 2]].astype(np.int64) << v
        for pv in range(16):
            sel = np.nonzero(pat == pv)[0]
            if len(sel) == 0:
                continue
            for s, tri in enumerate(TABLE[tet][pv]):
                idx = []
                for lo, hi in tri:
                    base = cells[sel] + corners[lo]
                    d = _DELTA_INDEX[tuple((corners[hi] - corners[lo]).tolist())]
                    qlin = (base[:, 0] * ny + base[:, 1]) * nz + base[:, 2]
                    assert flat[qlin, d].all()
                    idx.append(vid[qlin, d])
                tris.append(np.stack(idx, -1))
                keys.append(cell_lin[sel] * 12 + tet * 2 + s)
    if tris:
        keys, tris = np.concatenate(keys), np.concatenate(tris)
        tris = tris[np.argsort(keys, kind="stable")]
    else:
        tris = np.zeros((0, 3), np.int64)
    return pos.astype(np.float32), normals, tris.astype(np.int64)


def edge_manifold(tris: np.ndarray) -> bool:
    """every undirected edge in exactly two triangles, used once in each direction (closed, consistently oriented)"""
    directed = np.concatenate([tris[:, [0, 1]], tris[:, [1, 2]], tris[:, [2, 0]]])
    u = np.unique(directed, axis=0)
    if len(u) != len(directed):
        return False
    rev = {tuple(e) for e in u.tolist()}
    return all((b, a) in rev for a, b in u.tolist())


def euler_characteristic(n_vertices: int, tris: np.ndarray) -> int:
    edges = np.sort(np.concatenate([tris[:, [0, 1]], tris[:, [1, 2]], tris[:, [2, 0]]]), axis=1)
    return int(n_vertices - len(np.unique(edges, axis=0)) + len(tris))


def signed_volume(vertices: np.ndarray, tris: np.ndarray) -> float:
    """divergence theorem: sum of v0 . (v1 x v2) / 6 (positive for outward-facing triangles)"""
    v = vertices.astype(np.float64)
    a, b, c = v[tris[:, 0]], v[tris[:, 1]], v[tris[:, 2]]
    return float(np.einsum("ij,ij->i", a, np.cross(b, c)).sum() / 6.0)


def face_normals(vertices: np.ndarray, tris: np.ndarray) -> np.ndarray:
    v = vertices.astype(np.float64)
    return np.cross(v[tris[:, 1]] - v[tris[:, 0]], v[tris[:, 2]] - v[tris[:, 0]])


def grid(n, lo, hi):
    """(coordinates [nx,ny,nz,3] fp32, origin, spacing) of an n^3 lattice on [lo, hi]^3, points as the kernel places
    them (origin + spacing * index)"""
    ns = (n,) * 3 if np.isscalar(n) else tuple(n)
    lo3, hi3 = np.broadcast_to(np.float32(lo), 3), np.broadcast_to(np.float32(hi), 3)
    spacing = ((hi3 - lo3) / (np.asarray(ns, np.float32) - 1)).astype(np.float32)
    axes = [lo3[a] + spacing[a] * np.arange(ns[a], dtype=np.float32) for a in range(3)]
    xyz = np.stack(np.meshgrid(*axes, indexing="ij"), -1).astype(np.float32)
    return xyz, lo3.astype(np.float32), spacing

