"""TEST INFRASTRUCTURE — topology and geometry checks on triangle meshes (numpy), shared by the marching-cubes tests."""
from __future__ import annotations

import numpy as np


def directed_edges(tris):
    t = np.asarray(tris, np.int64)
    return np.concatenate([t[:, [0, 1]], t[:, [1, 2]], t[:, [2, 0]]])


def edge_keys(e, nv):
    return e[:, 0] * nv + e[:, 1]


def unpaired_half_edges(tris, nv):
    """Directed edges (i, j) without a twin (j, i); asserts no directed edge occurs twice."""
    e = directed_edges(tris)
    key = edge_keys(e, nv)
    assert np.unique(key).size == key.size, "a directed edge occurs twice"
    twin = np.isin(edge_keys(e[:, ::-1], nv), key)
    return e[~twin]


def assert_closed(tris, nv):
    """Every directed edge has exactly one twin and every vertex is referenced."""
    assert unpaired_half_edges(tris, nv).shape[0] == 0
    assert np.unique(np.asarray(tris)).size == nv


def euler_characteristic(tris, nv):
    e = directed_edges(tris)
    und = np.unique(np.sort(e, axis=1), axis=0)
    return nv - und.shape[0] + len(tris)


def face_normals(verts, tris):
    p = np.asarray(verts, np.float64)[np.asarray(tris)]
    return np.cross(p[:, 1] - p[:, 0], p[:, 2] - p[:, 0])


def volume(verts, tris):
    """Signed enclosed volume by the divergence theorem (positive for outward winding)."""
    p = np.asarray(verts, np.float64)[np.asarray(tris)]
    return float(np.einsum("ij,ij->i", p[:, 0], np.cross(p[:, 1], p[:, 2])).sum() / 6.0)


def area(verts, tris):
    return float(0.5 * np.linalg.norm(face_normals(verts, tris), axis=1).sum())


def vertex_edges(values, iso):
    """The lattice edge of every vertex by the numbering contract of fi_marching_cubes: (node coords (V, 3) as x y z,
    axis (V,)), ordered by the lower node's linear index, then axis."""
    a = np.asarray(values, np.float32)
    out = (a - np.float32(iso)) >= 0
    crossed = np.zeros(a.shape + (3,), bool)
    crossed[:, :, :-1, 0] = out[:, :, :-1] != out[:, :, 1:]
    crossed[:, :-1, :, 1] = out[:, :-1, :] != out[:, 1:, :]
    crossed[:-1, :, :, 2] = out[:-1, :, :] != out[1:, :, :]
    z, y, x, ax = np.nonzero(crossed)  # C order: z, y, x, axis = linear node index, then axis
    return np.stack([x, y, z], axis=1), ax


def contract_vertices(values, iso):
    """Vertex positions by the contract's fp32 expression float(coord_lo) + a / (a - b) (numpy float32, no FMA)."""
    a = np.asarray(values, np.float32)
    node, ax = vertex_edges(a, iso)
    hi = node.copy()
    hi[np.arange(len(ax)), ax] += 1
    lo_v = a[node[:, 2], node[:, 1], node[:, 0]] - np.float32(iso)
    hi_v = a[hi[:, 2], hi[:, 1], hi[:, 0]] - np.float32(iso)
    p = node.astype(np.float32)
    p[np.arange(len(ax)), ax] += lo_v / (lo_v - hi_v)
    return p


def face_contour(verts, tris, values, iso, axis, coord):
    """Unpaired half-edges whose two vertices sit on lattice edges of the plane `axis` = coord, as float32 rows
    (u0, w0, u1, w1) in the plane's coordinates (u, w = the two other axes, increasing)."""
    v = np.asarray(verts, np.float32)
    node, ax = vertex_edges(values, iso)
    in_plane = (ax != axis) & (node[:, axis] == coord)
    e = unpaired_half_edges(tris, len(v))
    e = e[in_plane[e[:, 0]] & in_plane[e[:, 1]]]
    u, w = [b for b in range(3) if b != axis]
    return np.stack([v[e[:, 0], u], v[e[:, 0], w], v[e[:, 1], u], v[e[:, 1], w]], axis=1)


def face_plane(values, axis, coord):
    """The (height, width) = (w, u) 2D field of lattice plane `axis` = coord of a (nz, ny, nx) array."""
    a = np.asarray(values)
    if axis == 0:
        return a[:, :, coord]          # (z, y): u = y, w = z
    if axis == 1:
        return a[:, coord, :]          # (z, x): u = x, w = z
    return a[coord, :, :]              # (y, x): u = x, w = y


def same_segments(got, want):
    """Equal as multisets of bit patterns (the 2D list is in cell order, the mesh's in triangle order)."""
    g = np.ascontiguousarray(got, np.float32).view(np.uint32).reshape(-1, 4)
    w = np.ascontiguousarray(want, np.float32).view(np.uint32).reshape(-1, 4)
    if g.shape != w.shape:
        return False
    return np.array_equal(g[np.lexsort(g.T[::-1])], w[np.lexsort(w.T[::-1])])


def reversed_segments(s):
    s = np.asarray(s)
    return s[:, [2, 3, 0, 1]]


# which orientation the mesh's boundary on each lattice face has relative to fi_marching_squares of that plane:
# the face normal pointing out of the lattice, crossed with the 2D plane's (u, w, u x w) frame
FACE_DIRECTION = {(0, "min"): "same", (0, "max"): "reversed", (1, "min"): "reversed", (1, "max"): "same",
                  (2, "min"): "same", (2, "max"): "reversed"}


def smooth_field(shape, seed, pad=True, scale=4.0):
    """Random smooth field: sum of a few Gaussian bumps minus a level; with pad the border nodes are set positive
    (outside) so the surface does not touch the lattice faces."""
    rng = np.random.default_rng(seed)
    nz, ny, nx = shape
    z, y, x = np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")
    f = np.zeros(shape, np.float64)
    for _ in range(6):
        c = rng.uniform(0, 1, 3) * np.array(shape)
        s = rng.uniform(0.15, 0.35) * min(shape)
        f += np.exp(-(((z - c[0]) ** 2 + (y - c[1]) ** 2 + (x - c[2]) ** 2) / (2 * s * s)))
    f = scale * (0.6 - f / f.max())
    if pad:
        f[0], f[-1], f[:, 0], f[:, -1], f[:, :, 0], f[:, :, -1] = 1, 1, 1, 1, 1, 1
    return f.astype(np.float32)
