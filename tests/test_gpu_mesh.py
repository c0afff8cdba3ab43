"""GPU: marching-cubes extraction (csrc/srcv_mesh.cuh) on fused rooms, bit for bit against
oracle/mesh_oracle.py, and TSDF.to_mesh / save through a recording stand-in for trimesh."""
import types

import numpy as np
import pytest
import torch

import simplerecon_b200 as S
from oracle import mesh_oracle as M
from simplerecon_b200.synthetic import make_tsdf_case
from tests.test_emu_mesh import _sphere, check_sphere

pytestmark = pytest.mark.gpu


def _fused(voxel, room=(4.0, 3.0, 2.6), frames=4, seed=11, hw=(120, 160)):
    c = make_tsdf_case(seed=seed, frames=frames, voxel_size=voxel, height=hw[0], width=hw[1], room=room)
    vol = S.TSDF.from_bounds(c["bounds"], voxel)
    fuser = S.TSDFFuser(vol, max_depth=c["max_depth"])
    fuser.integrate_depth(c["depth"].cuda(), c["cam_T_world"].cuda(), c["K"].cuda())
    return vol, fuser, c


def _assert_oracle(vol, single):
    verts, faces, normals = vol.extract_mesh(single_mesh=single)
    torch.cuda.synchronize()
    ov, of, on = M.extract(vol.tsdf_values.cpu().numpy(), single_mesh=single)
    assert faces.shape == of.shape and verts.shape == ov.shape
    assert np.array_equal(faces.cpu().numpy(), of)
    assert np.array_equal(verts.cpu().numpy().view(np.uint32), ov.view(np.uint32))
    assert np.array_equal(normals.cpu().numpy().view(np.uint32), on.view(np.uint32))
    return verts, faces, normals


@pytest.mark.parametrize("voxel", [0.04, 0.02])
@pytest.mark.parametrize("single", [False, True])
def test_fused_room_matches_oracle(voxel, single):
    vol, _, _ = _fused(voxel)
    _, f, _ = _assert_oracle(vol, single)
    assert len(f) > 10000


def test_room_larger_than_l2_repeat_and_more_frames():
    vol, fuser, c = _fused(0.01, room=(6.0, 5.0, 3.0), frames=2, seed=100, hw=(240, 320))
    assert tuple(vol.tsdf_values.shape) == (608, 512, 312)
    assert vol.tsdf_values.numel() * 2 >= 128 * 2**20
    a = _assert_oracle(vol, True)
    b = vol.extract_mesh(single_mesh=True)
    for x, y in zip(a, b):                                     # same bytes on a second run
        assert torch.equal(x.view(torch.int32), y.view(torch.int32))
    d = make_tsdf_case(seed=101, frames=2, voxel_size=0.01, height=240, width=320, room=(6.0, 5.0, 3.0))
    fuser.integrate_depth(d["depth"].cuda(), d["cam_T_world"].cuda(), d["K"].cuda())
    _, f, _ = _assert_oracle(vol, False)
    assert len(f) > len(a[1])


def test_sphere_256():
    c, r = (127.4, 128.3, 126.8), 90.5
    v = torch.from_numpy(_sphere(256, c, r)).cuda()
    vol = S.TSDF(v, torch.zeros_like(v), 0.01, torch.zeros(3))
    verts, faces, normals = (t.cpu().numpy() for t in vol.extract_mesh())
    check_sphere(verts, faces, normals, c, r)


def test_to_mesh_and_save_with_a_stand_in_trimesh(monkeypatch, tmp_path):
    calls = []

    class Trimesh:
        def __init__(self, **kw):
            self.kw = kw

    def export_mesh(mesh, path, file_type=None):
        calls.append((mesh, path, file_type))

    fake = types.ModuleType("trimesh")
    fake.Trimesh = Trimesh
    fake.exchange = types.SimpleNamespace(export=types.SimpleNamespace(export_mesh=export_mesh))
    monkeypatch.setitem(__import__("sys").modules, "trimesh", fake)
    vol, _, _ = _fused(0.04)
    m = vol.to_mesh(export_single_mesh=True)
    verts, faces, normals = vol.extract_mesh(single_mesh=True)
    world = vol.origin.half().float().view(1, 3) + verts.cpu() * vol.voxel_size
    assert set(m.kw) == {"vertices", "faces", "normals"}
    assert np.array_equal(m.kw["vertices"], world.numpy())
    assert np.array_equal(m.kw["faces"], faces.cpu().numpy())
    vol.save(str(tmp_path / "out"), "scene.bin")
    assert calls[-1][1] == str(tmp_path / "out" / "scene.ply") and calls[-1][2] == "ply"
    assert vol.tsdf_values.is_cuda and vol.tsdf_weights.is_cuda
