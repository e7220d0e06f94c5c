"""CPU: the marching-cubes case table (field_interpolation_b200/csrc/mc_table.cuh) and the CPU port of fi_marching_cubes
(tests/mc_port.cpp) — the generator reproduces the committed header, every case is a set of closed loops, cells that
share a face agree on it, the port's meshes are closed, consistently wound and carry the 2D contour on every lattice
face."""
import os
import re
import sys

import numpy as np
import pytest

import mesh_checks as M
from conftest import ROOT, bits
from mc_port import port as mc_port

sys.path.insert(0, os.path.join(ROOT, "scripts"))
import gen_mc_table as G  # noqa: E402

TABLES = G.build_tables()
MAX_TRIANGLES = int(re.search(r"kMaxTriangles = (\d+);", G.render()).group(1))


def test_generator_reproduces_committed_header():
    with open(G.OUT) as f:
        assert f.read() == G.render()


def _boundary(tris):
    """Directed edges of a cell's triangles (in edge ids) that have no twin inside the cell."""
    half = [(t[i], t[(i + 1) % 3]) for t in tris for i in range(3)]
    assert len(set(half)) == len(half)
    return [h for h in half if (h[1], h[0]) not in set(half)]


def test_every_crossed_edge_is_on_exactly_one_loop():
    for cfg in range(256):
        crossed = sorted(e for e in range(12) if G.edge_crossed(cfg, e))
        tris = TABLES[cfg]
        assert sorted({e for t in tris for e in t}) == crossed
        b = _boundary(tris)
        assert sorted(h[0] for h in b) == crossed and sorted(h[1] for h in b) == crossed, cfg
        assert sum(len(lp) for lp in G.loops(cfg)) == len(crossed)
        assert len(tris) <= MAX_TRIANGLES


def _face_of(e1, e2):
    """The cube face (axis, side) holding both edges, from their lower corners and axes."""
    p1, p2 = G.corner_coords(G.edge_lower_corner(e1)), G.corner_coords(G.edge_lower_corner(e2))
    for axis in range(3):
        if axis not in (e1 >> 2, e2 >> 2) and p1[axis] == p2[axis]:
            return axis, p1[axis]
    raise AssertionError((e1, e2))


def _face_edges(cfg, axis, side):
    """Boundary half-edges of case cfg on cube face (axis, side), each edge given by its in-face position."""
    out = set()
    for a, b in _boundary(TABLES[cfg]):
        if _face_of(a, b) == (axis, side):
            out.add((_in_face(a, axis), _in_face(b, axis)))
    return out


def _in_face(e, axis):
    p = list(G.corner_coords(G.edge_lower_corner(e)))
    p[axis] = None
    return e >> 2, tuple(p)


def test_boundary_half_edges_lie_on_cube_faces():
    for cfg in range(256):
        for a, b in _boundary(TABLES[cfg]):
            _face_of(a, b)


def test_cells_sharing_a_face_agree_on_it():
    """Cell A below and cell B above a face (along `axis`): when A's side-1 corners equal B's side-0 corners, both put
    the same segments on that face, with directions reversed."""
    for axis in range(3):
        bit = 1 << axis
        lower = [c for c in range(8) if not c & bit]
        for a in range(256):
            for b in range(0, 256, 7):  # a spread of partners; the face corners are what matters
                # make B's lower face equal A's upper face
                bb = b
                for c in lower:
                    bb = (bb & ~(1 << c)) | (((a >> (c | bit)) & 1) << c)
                up = _face_edges(a, axis, 1)
                down = _face_edges(bb, axis, 0)
                assert {(y, x) for x, y in up} == down, (axis, a, bb)


@pytest.mark.parametrize("seed", range(4))
def test_port_meshes_closed_on_random_smooth_fields(seed):
    f = M.smooth_field((20 + seed, 23, 18 + 2 * seed), seed)
    v, t = mc_port().marching_cubes(f, 0.0)
    assert len(t) > 0
    M.assert_closed(t, len(v))
    # the border is outside, so the mesh encloses the inside; wound toward the outside, its volume is positive
    assert M.volume(v, t) > 0


def test_port_faces_carry_the_2d_contour(port):
    rng = np.random.default_rng(5)
    f = rng.standard_normal((9, 11, 13)).astype(np.float32)
    f[rng.random(f.shape) < 0.1] = 0.0
    f[rng.random(f.shape) < 0.05] = -0.0
    for iso in (0.0, 0.3):
        v, t = mc_port().marching_cubes(f, iso)
        assert np.array_equal(bits(v), bits(M.contract_vertices(f, iso)))
        for axis, n in ((0, 13), (1, 11), (2, 9)):
            for which, coord in (("min", 0), ("max", n - 1)):
                got = M.face_contour(v, t, f, iso, axis, coord)
                want = port.iso_surface(M.face_plane(f, axis, coord), iso)
                assert len(want) > 0
                if M.FACE_DIRECTION[(axis, which)] == "reversed":
                    want = M.reversed_segments(want)
                assert M.same_segments(got, want), (axis, which, iso)
