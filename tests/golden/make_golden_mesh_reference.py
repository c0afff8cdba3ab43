"""Records what the unmodified reference's mesh export does, for tests/test_mesh_vs_reference.py.

    python tests/golden/make_golden_mesh_reference.py   (needs a SimpleRecon checkout: $SIMPLERECON_REF)

Writes tests/golden/reference/tsdf_mesh.npz: what ``TSDF.to_mesh`` (tools/tsdf.py:125-157) hands
to scikit-image's ``measure.marching_cubes`` and to ``trimesh.Trimesh``, captured with recording
stand-ins for both (neither is installed, and neither is needed to pin the reference's side of
those calls); the dims and origin ``TSDF.from_mesh`` (:51-67) gives for a stand-in mesh; and the
signatures of ``to_mesh``, ``save`` and ``from_mesh``.  The inputs are stored with the outputs.
"""
from __future__ import annotations

import inspect
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from oracle.ref_import import load_reference_tsdf  # noqa: E402

OUT = Path(__file__).resolve().parent / "reference" / "tsdf_mesh.npz"


def record() -> dict:
    R = load_reference_tsdf()
    g = np.random.default_rng(7)
    voxel = 0.04
    origin = np.array([-1.2345, 0.5678, 2.3456], dtype=np.float32)
    bounds = {"xmin": origin[0], "xmax": origin[0] + 0.3, "ymin": origin[1], "ymax": origin[1] + 0.3,
              "zmin": origin[2], "zmax": origin[2] + 0.3}
    ref = R.TSDF.from_bounds(bounds, voxel_size=voxel)
    values = (g.standard_normal(tuple(ref.tsdf_values.shape)) * 1.5).astype(np.float16)   # beyond [-1, 1]
    ref.tsdf_values = torch.from_numpy(values)
    fixed_verts = (g.random((37, 3)) * 8).astype(np.float32)
    fixed_faces = g.integers(0, 37, (20, 3)).astype(np.int64)
    fixed_norms = g.standard_normal((37, 3)).astype(np.float32)
    calls, meshes = [], []

    def marching_cubes(volume, **kw):
        calls.append((volume, kw))
        return fixed_verts, fixed_faces, fixed_norms, np.zeros(37, np.float32)

    class Trimesh:
        def __init__(self, **kw):
            meshes.append(kw)

    R.module.measure.marching_cubes = marching_cubes
    R.module.trimesh.Trimesh = Trimesh
    out = {"values": values, "origin": origin, "voxel_size": np.array(voxel), "fixed_verts": fixed_verts}
    for single in (False, True):
        ref.to_mesh(export_single_mesh=single)
        vol, kw = calls[-1]
        out[f"single{int(single)}_volume"] = np.asarray(vol)
        out[f"single{int(single)}_kwargs"] = np.array(sorted(f"{k}={v!r}" for k, v in kw.items()))
        out[f"single{int(single)}_mesh_keys"] = np.array(sorted(meshes[-1]))
        out[f"single{int(single)}_world_verts"] = np.asarray(meshes[-1]["vertices"])
    ref.to_mesh(scale_to_world=False)
    out["unscaled_verts"] = np.asarray(meshes[-1]["vertices"])

    class Mesh:
        vertices = g.standard_normal((50, 3)) * 2.0 + np.array([0.3, -1.0, 4.0])

    m = R.TSDF.from_mesh(Mesh(), voxel_size=0.05)
    out.update(mesh_vertices=Mesh.vertices, from_mesh_dims=np.array(m.tsdf_values.shape),
               from_mesh_origin=m.origin.numpy().copy())
    out["signatures"] = np.array([" ".join([n] + list(inspect.signature(getattr(R.TSDF, n)).parameters))
                                  for n in ("to_mesh", "save", "from_mesh")])
    return out


if __name__ == "__main__":
    OUT.parent.mkdir(exist_ok=True)
    np.savez_compressed(OUT, **record())
    print(OUT, OUT.stat().st_size, "bytes")
