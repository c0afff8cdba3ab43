"""Generates ``srcv_mc_table.h``: the marching-cubes triangle table of ``srcv_mesh.cuh``.

    python simplerecon_b200/csrc/gen_mc_table.py          (rewrites the header next to this file)

The table is derived, not typed in, so that its one property that matters can be read off the
construction: two cells that share a face cut that face the same way, so the mesh has no cracks.

Numbering (a cell is the cube between voxels (i, j, k) and (i + 1, j + 1, k + 1)):

* corner ``c`` (0..7) sits at offset ``(c & 1, (c >> 1) & 1, (c >> 2) & 1)`` along (axis 0, 1, 2);
  bit ``c`` of a configuration is set iff that corner is *below* the level (value < 0);
* edge ``e`` (0..11) runs along axis ``a = e >> 2`` from the corner whose offset along ``a`` is 0;
  its two other offsets, in increasing axis order, are ``(e & 1, (e >> 1) & 1)``.  The voxel at
  that corner *owns* the edge's vertex;
* a triangle ``(e0, e1, e2)`` winds counter-clockwise seen from the side above the level, i.e.
  ``(p1 - p0) x (p2 - p0)`` points toward increasing values.

Construction of the entry of one configuration:

1. every cube face gets iso-segments from its own 4 corner signs only.  Walking the face's corners
   counter-clockwise as seen from outside the cube, a segment runs from the edge where the walk
   enters a run of below corners to the edge where it leaves it, so the below side lies to the
   segment's right.  On an ambiguous face (the two below corners diagonal) each below corner is cut
   off on its own: the two below corners are never connected;
2. every crossing edge lies on two faces and is the start of one segment and the end of another,
   so the segments link into closed loops;
3. each loop ``v0 v1 ... vn-1`` is fan-triangulated as ``(v0, vi, vi+1)``.

A face shared by two cells is seen from outside with opposite orientations, so it gets the same
segments, reversed: both cells put their boundary edges in the same places and the surface keeps
one orientation across the face.  (The classic published tables resolve ambiguous faces per cell
and can crack there.)  The loops come out in the order of their first face and edge, so the table
is deterministic.
"""
from __future__ import annotations

import sys
from pathlib import Path

HEADER = Path(__file__).resolve().parent / "srcv_mc_table.h"


def corner_offset(c: int):
    return (c & 1, (c >> 1) & 1, (c >> 2) & 1)


def corner_index(off) -> int:
    return off[0] | (off[1] << 1) | (off[2] << 2)


def edge_corners(e: int):
    """(start corner, end corner) of edge e: the end is one step further along the edge's axis."""
    a, r = e >> 2, e & 3
    others = [x for x in range(3) if x != a]
    off = [0, 0, 0]
    off[others[0]], off[others[1]] = r & 1, (r >> 1) & 1
    c0 = corner_index(off)
    off[a] = 1
    return c0, corner_index(off)


def edge_between(c0: int, c1: int) -> int:
    o0, o1 = corner_offset(c0), corner_offset(c1)
    diff = [x for x in range(3) if o0[x] != o1[x]]
    assert len(diff) == 1
    a = diff[0]
    others = [x for x in range(3) if x != a]
    return (a << 2) | o0[others[0]] | (o0[others[1]] << 1)


def faces():
    """The six cube faces as 4 corners, counter-clockwise seen from outside (right-handed about
    the outward normal)."""
    out = []
    for a in range(3):
        u, v = (a + 1) % 3, (a + 2) % 3          # (u, v, a) is a right-handed frame
        for side in (0, 1):
            ring = []
            for du, dv in ((0, 0), (1, 0), (1, 1), (0, 1)):
                off = [0, 0, 0]
                off[a], off[u], off[v] = side, du, dv
                ring.append(corner_index(off))
            out.append(ring if side == 1 else ring[::-1])   # outward normal is +a on side 1, -a on side 0
    return out


def face_segments(ring, below):
    """Directed iso-segments (start edge, end edge) of one face, from its 4 corner signs only."""
    b = [bool(below >> c & 1) for c in ring]
    n_below = sum(b)
    if n_below in (0, 4):
        return []
    segs = []
    if n_below == 2 and b[0] == b[2]:             # ambiguous: cut each below corner off on its own
        for i in range(4):
            if b[i]:
                segs.append((edge_between(ring[i - 1], ring[i]), edge_between(ring[i], ring[(i + 1) % 4])))
        return segs
    enter = [i for i in range(4) if not b[i - 1] and b[i]]
    leave = [i for i in range(4) if b[i] and not b[(i + 1) % 4]]
    assert len(enter) == len(leave) == 1
    i, j = enter[0], leave[0]
    return [(edge_between(ring[i - 1], ring[i]), edge_between(ring[j], ring[(j + 1) % 4]))]


def loops(config: int):
    nxt = {}
    for ring in faces():
        for s, t in face_segments(ring, config):
            assert s not in nxt
            nxt[s] = t
    out, seen = [], set()
    for s in nxt:                                 # dict order: first face, then segment order
        if s in seen:
            continue
        loop, e = [], s
        while e not in seen:
            seen.add(e)
            loop.append(e)
            e = nxt[e]
        assert e == s
        out.append(loop)
    return out


def triangles(config: int):
    tris = []
    for loop in loops(config):
        for i in range(1, len(loop) - 1):
            tris.append((loop[0], loop[i], loop[i + 1]))
    return tris


def crossing_edges(config: int):
    return [e for e in range(12) if (config >> edge_corners(e)[0] & 1) != (config >> edge_corners(e)[1] & 1)]


TABLE = [triangles(c) for c in range(256)]
MAX_TRIS = max(len(t) for t in TABLE)


def render() -> str:
    lines = [
        "// GENERATED by gen_mc_table.py -- do not edit; regenerate with",
        "//   python simplerecon_b200/csrc/gen_mc_table.py",
        "// Marching-cubes triangles per configuration of the 8 corner signs (bit c set = corner c",
        "// below the level).  Corner, edge and winding conventions: the generator's docstring.",
        "#pragma once",
        "",
        "namespace srcv {",
        "namespace mc {",
        "",
        f"constexpr int kMaxTris = {MAX_TRIS};",
        "",
        "// number of triangles of each configuration",
        "__device__ const unsigned char kTriCount[256] = {",
    ]
    for r in range(0, 256, 16):
        lines.append("    " + ", ".join(f"{len(TABLE[c])}" for c in range(r, r + 16)) + ",")
    lines += ["};", "", "// edges of each triangle, three per triangle, -1 after the last",
              f"__device__ const signed char kTriEdges[256][{3 * MAX_TRIS}] = {{"]
    for c in range(256):
        flat = [e for t in TABLE[c] for e in t]
        flat += [-1] * (3 * MAX_TRIS - len(flat))
        lines.append("    {" + ", ".join(str(e) for e in flat) + "},")
    lines += ["};", "", "}  // namespace mc", "}  // namespace srcv", ""]
    return "\n".join(lines)


if __name__ == "__main__":
    text = render()
    if len(sys.argv) > 1 and sys.argv[1] == "--check":
        sys.exit(0 if HEADER.read_text() == text else 1)
    HEADER.write_text(text)
    print(f"{HEADER}: {sum(len(t) for t in TABLE)} triangles, at most {MAX_TRIS} per cell")
