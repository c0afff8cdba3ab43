"""CPU: the generated marching-cubes table (simplerecon_b200/csrc/gen_mc_table.py) — the committed
header is what the generator writes, and every configuration's triangles form a closed,
consistently oriented patch whose boundary on each cube face depends on that face alone."""
from collections import Counter

import numpy as np
import pytest

from oracle.mesh_oracle import G


def test_header_is_regenerated_byte_for_byte():
    assert G.HEADER.read_text() == G.render()


def _edge_pos(e):
    c0, c1 = G.edge_corners(e)
    return (np.array(G.corner_offset(c0)) + np.array(G.corner_offset(c1))) / 2.0


def _face_of(e0, e1):
    """The cube face containing both edges, as (axis, side), or None for an interior segment."""
    p, q = _edge_pos(e0), _edge_pos(e1)
    for a in range(3):
        for side in (0.0, 1.0):
            if p[a] == side and q[a] == side:
                return a, int(side)
    return None


@pytest.mark.parametrize("config", range(256))
def test_configuration_is_a_closed_oriented_patch(config):
    tris = G.TABLE[config]
    crossing = set(G.crossing_edges(config))
    used = {e for t in tris for e in t}
    assert used == crossing                                   # only crossing edges, and all of them
    directed = Counter((t[s], t[(s + 1) % 3]) for t in tris for s in range(3))
    assert max(directed.values(), default=1) == 1
    boundary = {}
    for (a, b) in directed:
        if (b, a) in directed:                                # inside the cell: once each way
            continue
        assert _face_of(a, b) is not None, (config, a, b)     # else on a cube face, once
        boundary.setdefault(_face_of(a, b), set()).add((a, b))
    # the boundary on each face is exactly the face's own segments, from its 4 corner signs
    for ring in G.faces():
        offs = np.array([G.corner_offset(c) for c in ring])
        a = int(np.flatnonzero((offs == offs[0]).all(0))[0])
        segs = set(G.face_segments(ring, config))
        assert boundary.get((a, int(offs[0][a])), set()) == segs, (config, ring)
        # ... and only those 4 signs: flipping a corner off the face leaves them unchanged
        for c in range(8):
            if c not in ring:
                assert set(G.face_segments(ring, config ^ (1 << c))) == segs


@pytest.mark.parametrize("config", range(1, 255))
def test_triangles_face_away_from_the_below_corners(config):
    """For a lone below (or above) corner the patch's normal points from below to above."""
    below = [c for c in range(8) if config >> c & 1]
    if len(below) not in (1, 7):
        return
    lone = below[0] if len(below) == 1 else next(c for c in range(8) if not config >> c & 1)
    sign = 1.0 if len(below) == 1 else -1.0
    for t in G.TABLE[config]:
        p = [_edge_pos(e) for e in t]
        n = np.cross(p[1] - p[0], p[2] - p[0])
        assert sign * np.dot(n, np.mean(p, 0) - np.array(G.corner_offset(lone))) > 0
