"""CPU: TSDF.to_mesh / save / from_mesh against what the reference's (tools/tsdf.py:51-67,
:125-168) were recorded doing with stand-ins for scikit-image and trimesh
(tests/golden/make_golden_mesh_reference.py), and the calls OurFuser (tools/fusers_helper.py:48-82)
makes, driven through the emulated kernels with a recording trimesh."""
import inspect
import sys
import types

import numpy as np
import pytest
import torch

from oracle import mesh_oracle as M
from oracle import tsdf_oracle as T
from simplerecon_b200 import tsdf as tsdf_mod
from simplerecon_b200.synthetic import make_tsdf_case
from tests.parity import load_reference_outputs
from tests.test_emu_mesh import emulated  # noqa: F401  (fixture)


@pytest.fixture()
def fake_trimesh(monkeypatch):
    rec = types.SimpleNamespace(meshes=[], exports=[])

    class Trimesh:
        def __init__(self, **kw):
            self.kw = kw
            rec.meshes.append(kw)

    def export_mesh(mesh, path, file_type=None, **kw):
        rec.exports.append((mesh, path, file_type))

    m = types.ModuleType("trimesh")
    m.Trimesh = Trimesh
    m.exchange = types.SimpleNamespace(export=types.SimpleNamespace(export_mesh=export_mesh))
    monkeypatch.setitem(sys.modules, "trimesh", m)
    return rec


def _golden():
    return {k: (v.numpy() if torch.is_tensor(v) else v) for k, v in load_reference_outputs("tsdf_mesh").items()}


def _ours(R):
    v = torch.from_numpy(R["values"])
    return tsdf_mod.TSDF(v, torch.zeros_like(v), float(R["voxel_size"]), torch.from_numpy(R["origin"]))


def test_signatures():
    R = _golden()
    for line in R["signatures"]:
        name, *ref_params = str(line).split()
        ours = inspect.signature(getattr(tsdf_mod.TSDF, name)).parameters
        assert list(ours)[:len(ref_params)] == ref_params, name
        assert all(p.default is not inspect.Parameter.empty for p in list(ours.values())[len(ref_params):])


def test_marching_cubes_input_and_arguments():
    """The reference clamps the fp32 copy to [-1, 1] and calls marching_cubes(level=0,
    allow_degenerate=False[, single_mesh=True]); the oracle's (and kernel's) input is the same array."""
    R = _golden()
    for single in (0, 1):
        assert np.array_equal(M.clamp(R["values"]).view(np.uint32), R[f"single{single}_volume"].view(np.uint32))
        kw = {"allow_degenerate=False", "level=0"} | ({"single_mesh=True"} if single else set())
        assert set(map(str, R[f"single{single}_kwargs"])) == kw
        assert set(map(str, R[f"single{single}_mesh_keys"])) == {"vertices", "faces", "normals"}


def test_world_scaling_is_bitwise(monkeypatch, fake_trimesh):
    R = _golden()
    vol = _ours(R)
    verts = torch.from_numpy(R["fixed_verts"])
    faces = torch.zeros((1, 3), dtype=torch.int32)
    monkeypatch.setattr(tsdf_mod.TSDF, "_extract", lambda self, single: (verts, faces, verts.clone(), True))
    for single in (0, 1):
        vol.to_mesh(export_single_mesh=bool(single))
        got = np.asarray(fake_trimesh.meshes[-1]["vertices"])
        assert got.dtype == np.float32
        assert np.array_equal(got.view(np.uint32), R[f"single{single}_world_verts"].view(np.uint32))
    vol.to_mesh(scale_to_world=False)
    assert np.array_equal(np.asarray(fake_trimesh.meshes[-1]["vertices"]), R["unscaled_verts"])


def test_from_mesh_bounds():
    R = _golden()
    mesh = types.SimpleNamespace(vertices=R["mesh_vertices"])
    vol = tsdf_mod.TSDF.from_mesh(mesh, voxel_size=0.05, device="cpu")
    assert list(vol.tsdf_values.shape) == list(R["from_mesh_dims"])
    assert torch.equal(vol.origin.half(), torch.from_numpy(R["from_mesh_origin"]))


def test_our_fuser_calls_through_the_swap(emulated, fake_trimesh, tmp_path):  # noqa: F811
    """OurFuser with a ground-truth mesh: TSDF.from_mesh, fuse, then export_mesh / get_mesh, which
    call tsdf.to_mesh(export_single_mesh=True) and trimesh.exchange.export.export_mesh."""
    c = make_tsdf_case(seed=2, frames=2, voxel_size=0.12, height=48, width=64)
    b = c["bounds"]
    gt = types.SimpleNamespace(vertices=np.array([[b["xmin"], b["ymin"], b["zmin"]],
                                                  [b["xmax"], b["ymax"], b["zmax"]]]) + np.array([0.36, 0.36, 0.36]) * [[1], [-1]])
    tsdf_pred = tsdf_mod.TSDF.from_mesh(gt, voxel_size=0.12, device="cpu")
    fuser = tsdf_mod.TSDFFuser(tsdf_pred, max_depth=3.0)
    fuser.integrate_depth(depth_b1hw=c["depth"].half(), cam_T_world_T_b44=c["cam_T_world"].half(), K_b44=c["K"].half())
    import trimesh
    trimesh.exchange.export.export_mesh(fuser.tsdf.to_mesh(export_single_mesh=True), str(tmp_path / "m.ply"))
    mesh = fuser.tsdf.to_mesh(export_single_mesh=True)
    assert fake_trimesh.exports[-1][0].kw is fake_trimesh.meshes[-2]
    verts, faces, _ = M.extract(fuser.tsdf.tsdf_values.numpy(), single_mesh=True)
    assert len(faces) > 100
    assert np.array_equal(mesh.kw["faces"], faces)
    world = (tsdf_pred.origin.half().float().view(1, 3) + torch.from_numpy(verts) * 0.12).numpy()
    assert np.array_equal(mesh.kw["vertices"], world)
    tv, _, _ = T.new_volume(gt_bounds(gt, 0.12), 0.12)
    assert tv.shape == tsdf_pred.tsdf_values.shape


def gt_bounds(mesh, voxel):
    lo, hi = mesh.vertices.min(0) - 3 * voxel, mesh.vertices.max(0) + 3 * voxel
    return {"xmin": lo[0], "xmax": hi[0], "ymin": lo[1], "ymax": hi[1], "zmin": lo[2], "zmax": hi[2]}
