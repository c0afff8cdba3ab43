"""numpy restatement of the mesh-extraction output contract — TEST INFRASTRUCTURE.

Only tests/ and scripts/ import this.  It states what ``TSDF.extract_mesh`` (csrc/srcv_mesh.cuh)
returns, independently of how the kernels find it: vertex ids come from ``np.unique`` over int64
edge keys, not from row scans, and the triangles from the generated table of
``simplerecon_b200/csrc/gen_mc_table.py`` (imported from the generator, not parsed from the header).

Contract (level 0 on the values clamped to [-1, 1] in fp32; NaN clamps to -1 like fmin/fmax):
* a corner is below iff its value is < 0 (0 is above); (X-1)(Y-1)(Z-1) cells, no padding;
* one vertex per edge whose ends lie on different sides; on the edge from voxel a to b = a + e_axis,
  t = (0 - v_a) / (v_b - v_a) and the position is a with its axis coordinate replaced by a_axis + t;
* normal = normalize((1 - t) g(a) + t g(b)), g = numpy.gradient of the clamped values; sum of
  squares as (x*x + y*y) + z*z; a zero vector stays zero;
* dropped: a triangle with two vertices at equal fp32 positions (allow_degenerate=False), and with
  single_mesh every triangle that needs a vertex on an edge from exactly -1 to exactly +1;
* only referenced vertices are kept, ordered by owner voxel linear index then axis; faces ordered
  by cell linear index then table order.
Every operation is one fp32 numpy operation, in the order above.
"""
from __future__ import annotations

import importlib.util
from pathlib import Path

import numpy as np

_GEN = Path(__file__).resolve().parents[1] / "simplerecon_b200" / "csrc" / "gen_mc_table.py"


def _load_table():
    spec = importlib.util.spec_from_file_location("_srcv_gen_mc_table", _GEN)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


G = _load_table()
TRI_COUNT = np.array([len(t) for t in G.TABLE], dtype=np.int64)
TRI_EDGES = np.full((256, G.MAX_TRIS, 3), -1, dtype=np.int64)
for _c, _tris in enumerate(G.TABLE):
    for _t, _tri in enumerate(_tris):
        TRI_EDGES[_c, _t] = _tri
EDGE_C0 = np.array([G.edge_corners(e)[0] for e in range(12)], dtype=np.int64)
EDGE_C1 = np.array([G.edge_corners(e)[1] for e in range(12)], dtype=np.int64)
EDGE_AXIS = np.arange(12, dtype=np.int64) >> 2
CORNER_OFF = np.array([G.corner_offset(c) for c in range(8)], dtype=np.int64)   # (8, 3)


def clamp(values) -> np.ndarray:
    v = np.asarray(values).astype(np.float32)
    return np.fmin(np.fmax(v, np.float32(-1)), np.float32(1))


def _excluded(va, vb):
    return (va == -vb) & ((va == 1) | (va == -1))


def extract(values, single_mesh: bool = False):
    """(verts (V,3) float32, faces (F,3) int32, normals (V,3) float32) of the fp16 volume."""
    v = clamp(values)
    X, Y, Z = v.shape
    if min(X, Y, Z) < 2:
        raise ValueError("every dimension must be >= 2")
    n = np.array([X, Y, Z], dtype=np.int64)
    corners = [v[o[0]:X - 1 + o[0], o[1]:Y - 1 + o[1], o[2]:Z - 1 + o[2]] for o in CORNER_OFF]
    config = np.zeros((X - 1, Y - 1, Z - 1), dtype=np.int64)
    for c in range(8):
        config |= (corners[c] < 0).astype(np.int64) << c
    cell_lin = np.flatnonzero(TRI_COUNT[config] > 0)          # C order = cell linear index order
    ci, cj, ck = np.unravel_index(cell_lin, config.shape)
    cfg = config.reshape(-1)[cell_lin]
    cval = np.stack([c.reshape(-1)[cell_lin] for c in corners], 1)            # (C, 8)
    # one row per (cell, table triangle), cell-major
    nt = TRI_COUNT[cfg]
    cell = np.repeat(np.arange(len(cfg)), nt)
    tri = np.arange(len(cell)) - np.repeat(np.cumsum(nt) - nt, nt)
    edges = TRI_EDGES[cfg[cell], tri]                                          # (T, 3)
    c0, c1, ax = EDGE_C0[edges], EDGE_C1[edges], EDGE_AXIS[edges]
    va = np.take_along_axis(cval[cell], c0, 1)
    vb = np.take_along_axis(cval[cell], c1, 1)
    owner = np.stack([ci[cell], cj[cell], ck[cell]], -1)[:, None, :] + CORNER_OFF[c0]   # (T, 3, 3)
    t = (np.float32(0) - va) / (vb - va)
    pos = owner.astype(np.float32)
    sel = np.arange(3)[None, None, :] == ax[..., None]
    pos = np.where(sel, pos + t[..., None], pos)
    keep = np.ones(len(cell), dtype=bool)
    for s, u in ((0, 1), (1, 2), (0, 2)):
        keep &= ~np.all(pos[:, s] == pos[:, u], -1)
    if single_mesh:
        keep &= ~np.any(_excluded(va, vb), 1)
    owner, ax = owner[keep], ax[keep]
    key = ((owner[..., 0] * n[1] + owner[..., 1]) * n[2] + owner[..., 2]) * 3 + ax               # (F, 3) int64
    uniq, inv = np.unique(key.reshape(-1), return_inverse=True)
    faces = inv.reshape(-1, 3).astype(np.int32)
    verts, normals = vertices(v, uniq)
    return verts, faces, normals


def vertices(v: np.ndarray, keys: np.ndarray):
    """Positions and normals of the vertices with edge keys (owner linear index * 3 + axis)."""
    X, Y, Z = v.shape
    a = keys % 3
    i, j, k = np.unravel_index(keys // 3, (X, Y, Z))
    bi, bj, bk = i + (a == 0), j + (a == 1), k + (a == 2)
    va, vb = v[i, j, k], v[bi, bj, bk]
    t = (np.float32(0) - va) / (vb - va)
    pos = np.stack([i, j, k], 1).astype(np.float32)
    sel = np.arange(3)[None, :] == a[:, None]
    pos = np.where(sel, pos + t[:, None], pos)
    g = np.gradient(v)
    assert all(x.dtype == np.float32 for x in g)
    omt = np.float32(1) - t
    nrm = np.stack([omt * g[x][i, j, k] + t * g[x][bi, bj, bk] for x in range(3)], 1)
    l2 = (nrm[:, 0] * nrm[:, 0] + nrm[:, 1] * nrm[:, 1]) + nrm[:, 2] * nrm[:, 2]
    nz = l2 > 0
    nrm[nz] = nrm[nz] / np.sqrt(l2[nz])[:, None]
    return pos.astype(np.float32), nrm.astype(np.float32)


def level_in_range(values) -> bool:
    """skimage's check: level 0 inside [min, max] of the clamped volume."""
    v = clamp(values)
    return bool(v.min() <= 0 <= v.max())
