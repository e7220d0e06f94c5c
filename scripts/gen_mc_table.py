"""Writes field_interpolation_b200/csrc/mc_table.cuh: the marching-cubes case table of fi_marching_cubes.

    python scripts/gen_mc_table.py            # rewrite the header
    python scripts/gen_mc_table.py --check    # exit 1 when the committed header differs

The table is derived, not typed in.  For each of the 256 corner configurations of a cell (bit c set when corner
c = x + 2y + 4z is "outside", value - iso >= 0):
  1. every cube face gets the marching-squares segments of its four corners.  A face with alternating corners cuts
     off the corner whose two in-plane coordinates are both 0 and the one where both are 1, the resolution
     emilib::marching_squares uses for its configs 6 and 9 (csrc/isosurface.cu).  A face is resolved from its own
     corners only, so the two cells that share it put the same segments on it and the mesh has no cracks;
  2. each segment is directed so that, seen from outside the cell, the outside corners lie to its left
     (outward face normal N, direction d: N x d points to the outside side);
  3. the directed segments are chained into loops (every crossed edge starts one segment and ends one);
  4. each loop is fan-triangulated, which winds (P1 - P0) x (P2 - P0) toward the outside.  The fan starts at the
     first edge of the loop (loops start at their lowest edge) none of whose diagonals lies in a cube face, so every
     mesh edge that two cells share is a face segment and the mesh is a closed 2-manifold away from the lattice border.

Edge e = 4 * axis + k runs along `axis` from the corner whose other two coordinates are (k & 1, k >> 1), taken in
increasing axis order.
"""
from __future__ import annotations

import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "..", "field_interpolation_b200", "csrc", "mc_table.cuh")


def corner_coords(c):
    return (c & 1, (c >> 1) & 1, (c >> 2) & 1)


def corner_index(p):
    return p[0] + 2 * p[1] + 4 * p[2]


def other_axes(axis):
    return [b for b in range(3) if b != axis]


def edge_id(axis, p):
    """The edge along `axis` through the cell point p (p[axis] ignored)."""
    u, w = other_axes(axis)
    return 4 * axis + p[u] + 2 * p[w]


def edge_lower_corner(e):
    axis, k = e >> 2, e & 3
    u, w = other_axes(axis)
    p = [0, 0, 0]
    p[u], p[w] = k & 1, k >> 1
    return corner_index(p)


def edge_crossed(config, e):
    lo = edge_lower_corner(e)
    hi = lo + (1 << (e >> 2))
    return ((config >> lo) & 1) != ((config >> hi) & 1)


def edge_midpoint(e):
    p = list(corner_coords(edge_lower_corner(e)))
    p[e >> 2] = 0.5
    return p


def sub(a, b):
    return [a[i] - b[i] for i in range(3)]


def cross(a, b):
    return [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]


def dot(a, b):
    return sum(a[i] * b[i] for i in range(3))


# emilib's pairing of the four face edges per 2D config (bit 1 = (0,0), 2 = (1,0), 4 = (0,1), 8 = (1,1) in the face's
# (u, w) coordinates); L, T, R, B = the w-edge at u = 0, the u-edge at w = 0, the w-edge at u = 1, the u-edge at w = 1.
L, T, R, B = range(4)
MS_PAIRS = [[], [(L, T)], [(T, R)], [(L, R)], [(B, L)], [(B, T)], [(T, L), (B, R)], [(B, R)],
            [(R, B)], [(L, T), (R, B)], [(T, B)], [(L, B)], [(R, L)], [(R, T)], [(T, L)], []]


def face_segments(config, axis, side):
    """Directed segments (from edge, to edge) that configuration `config` puts on the cell face axis = side."""
    u, w = other_axes(axis)

    def point(i, j):
        p = [0, 0, 0]
        p[axis], p[u], p[w] = side, i, j
        return p

    face_edge = {L: edge_id(w, point(0, 0)), T: edge_id(u, point(0, 0)), R: edge_id(w, point(1, 0)), B: edge_id(u, point(0, 1))}
    out = [(config >> corner_index(point(i, j))) & 1 for j in (0, 1) for i in (0, 1)]
    ms = out[0] | out[1] << 1 | out[2] << 2 | out[3] << 3
    normal = [0, 0, 0]
    normal[axis] = 1 if side else -1
    segs = []
    for a, b in MS_PAIRS[ms]:
        ea, eb = face_edge[a], face_edge[b]
        ma, mb = edge_midpoint(ea), edge_midpoint(eb)
        left = cross(normal, sub(mb, ma))
        # No face corner lies on the line through two edge midpoints.  The segment either cuts off one corner (the
        # only corner on its side; in a saddle the far side also holds the other cut-off corner) or splits the face
        # in two pairs; either way a corner on the smaller side touches the segment and decides.
        on_left = [dot(left, sub(point(i, j), ma)) > 0 for j in (0, 1) for i in (0, 1)]
        pick = on_left.index(True) if sum(on_left) <= 2 else on_left.index(False)
        if on_left[pick] != bool(out[pick]):
            ea, eb = eb, ea
        segs.append((ea, eb))
    return segs


def loops(config):
    nxt = {}
    for axis in range(3):
        for side in (0, 1):
            for a, b in face_segments(config, axis, side):
                assert a not in nxt, (config, a)
                nxt[a] = b
    crossed = [e for e in range(12) if edge_crossed(config, e)]
    assert sorted(nxt) == crossed and sorted(nxt.values()) == crossed, config
    out, used = [], set()
    for start in crossed:
        if start in used:
            continue
        loop, e = [], start
        while e not in used:
            used.add(e)
            loop.append(e)
            e = nxt[e]
        assert e == start, config
        out.append(loop)
    return out


def edge_faces(e):
    """The two cube faces (axis, side) that hold edge e."""
    p = corner_coords(edge_lower_corner(e))
    return {(a, p[a]) for a in other_axes(e >> 2)}


def triangles(config):
    tris = []
    for loop in loops(config):
        # Fan from the first edge of the loop whose diagonals all cross the cell's interior.  A diagonal between two
        # edges on one face would lie in that face, where the neighbouring cell may draw the same diagonal: the edge
        # would then be shared by four triangles.  Interior diagonals belong to this cell alone.
        k = len(loop)
        for s in range(k):
            apex = loop[s]
            if not any(edge_faces(apex) & edge_faces(loop[(s + j) % k]) for j in range(2, k - 1)):
                break
        else:
            raise AssertionError(f"config {config}: no fan apex for loop {loop}")
        rot = loop[s:] + loop[:s]
        for i in range(1, k - 1):
            tris.append((rot[0], rot[i], rot[i + 1]))
    return tris


def build_tables():
    return [triangles(c) for c in range(256)]


def render() -> str:
    tables = build_tables()
    max_tri = max(len(t) for t in tables)
    lines = [
        "// GENERATED by scripts/gen_mc_table.py -- do not edit.  Marching-cubes case table of fi_marching_cubes",
        "// (csrc/marching_cubes.cuh) and of its CPU port; the script's docstring states how each case is derived.",
        "// config: bit c set when corner c = x + 2y + 4z of the cell is outside (value - iso >= 0).",
        "// Edge e = 4 * axis + k runs along `axis` from the corner whose other two coordinates are (k & 1, k >> 1).",
        "#pragma once",
        "",
        "#include <cstdint>",
        "",
        "#if defined(__CUDACC__) || defined(FI_B200_EMU)",
        "#define FI_MC_TABLE __device__ const",
        "#else",
        "#define FI_MC_TABLE const",
        "#endif",
        "",
        "namespace fi_mc {",
        "",
        f"constexpr int kMaxTriangles = {max_tri};  // per cell",
        "",
        "// lower corner of each edge",
        "static FI_MC_TABLE uint8_t kEdgeCorner[12] = {" + ", ".join(str(edge_lower_corner(e)) for e in range(12)) + "};",
        "",
        "// triangles per configuration",
        "static FI_MC_TABLE uint8_t kTriCount[256] = {",
    ]
    for r in range(0, 256, 32):
        lines.append("\t" + ", ".join(str(len(tables[c])) for c in range(r, r + 32)) + ",")
    lines.append("};")
    lines.append("")
    lines.append("// edges of each triangle, (P1 - P0) x (P2 - P0) toward the outside; unused slots 0xff")
    lines.append(f"static FI_MC_TABLE uint8_t kTriEdges[256][{3 * max_tri}] = {{")
    for c in range(256):
        flat = [e for t in tables[c] for e in t] + [255] * (3 * (max_tri - len(tables[c])))
        lines.append("\t{" + ", ".join(str(e) for e in flat) + "},")
    lines.append("};")
    lines.append("")
    lines.append("}  // namespace fi_mc")
    lines.append("")
    return "\n".join(lines)


def main(argv):
    text = render()
    if "--check" in argv:
        with open(OUT) as f:
            same = f.read() == text
        print("mc_table.cuh is up to date" if same else "mc_table.cuh differs from the generator")
        return 0 if same else 1
    with open(OUT, "w") as f:
        f.write(text)
    print(os.path.normpath(OUT))
    return 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
