"""CPU: the mesh-extraction kernels (csrc/srcv_mesh.cuh) compiled for the host (tests/emu) through
TSDF.extract_mesh / to_mesh, bit for bit against oracle/mesh_oracle.py, plus analytic surfaces
and the C ABI's argument checks."""
import contextlib
import ctypes as C
import types

import numpy as np
import pytest
import torch

from oracle import mesh_oracle as M
from oracle import tsdf_oracle as T
from simplerecon_b200 import _native, tsdf as tsdf_mod
from simplerecon_b200.synthetic import make_tsdf_case
from tests import emu
from tests.parity import load_reference_outputs


@pytest.fixture()
def emulated(monkeypatch):
    lib = emu.load_or_skip()
    monkeypatch.setattr(_native, "_lib", lib)
    monkeypatch.setattr(tsdf_mod, "_require_cuda", lambda t: None)
    monkeypatch.setattr(torch.cuda, "device", lambda dev: contextlib.nullcontext())
    monkeypatch.setattr(torch.cuda, "current_stream", lambda dev=None: types.SimpleNamespace(cuda_stream=0))
    real_empty = torch.empty

    def aligned_empty(*size, **kw):
        if kw.get("dtype") is torch.uint8 and len(size) == 1 and isinstance(size[0], int):
            buf = real_empty(size[0] + 256, **kw)
            off = (-buf.data_ptr()) % 256
            return buf[off:off + size[0]]
        return real_empty(*size, **kw)

    monkeypatch.setattr(torch, "empty", aligned_empty)
    return lib


def _volume(values) -> tsdf_mod.TSDF:
    v = torch.as_tensor(values).half()
    return tsdf_mod.TSDF(v, torch.zeros_like(v), 0.04, torch.zeros(3))


def assert_matches_oracle(values, single_mesh):
    vol = _volume(values)
    verts, faces, normals = vol.extract_mesh(single_mesh=single_mesh)
    ov, of, on = M.extract(vol.tsdf_values.numpy(), single_mesh=single_mesh)
    assert verts.dtype == torch.float32 and faces.dtype == torch.int32 and normals.dtype == torch.float32
    assert faces.shape == of.shape and verts.shape == ov.shape, (faces.shape, of.shape, verts.shape, ov.shape)
    assert np.array_equal(faces.numpy(), of)
    assert np.array_equal(verts.numpy().view(np.uint32), ov.view(np.uint32))
    assert np.array_equal(normals.numpy().view(np.uint32), on.view(np.uint32))
    return verts, faces, normals


def test_every_single_cell_configuration(emulated):
    g = np.random.default_rng(0)
    for config in range(256):
        mag = g.uniform(0.05, 1.0, 8).astype(np.float32)
        mag[g.random(8) < 0.25] = 1.0                   # exact +-1 corners exercise single_mesh
        vals = np.empty((2, 2, 2), np.float32)
        for c in range(8):
            i, j, k = M.CORNER_OFF[c]
            vals[i, j, k] = -mag[c] if config >> c & 1 else mag[c]
        for single in (False, True):
            _, f, _ = assert_matches_oracle(vals, single)
            if not single:
                assert len(f) == len(M.G.TABLE[config])


@pytest.mark.parametrize("seed,single", [(1, False), (1, True), (3, True)])
def test_reference_fused_volumes(emulated, seed, single):
    R = load_reference_outputs("tsdf")
    _, f, _ = assert_matches_oracle(R[f"c{seed}_r1_values"], single)
    assert len(f) > 1000


@pytest.mark.parametrize("z", [29, 31])
@pytest.mark.parametrize("single", [False, True])
def test_fused_case_odd_sizes(emulated, z, single):
    c = make_tsdf_case(seed=5, frames=2, voxel_size=0.11, height=48, width=64)
    tv, tw, origin = T.new_volume(c["bounds"], 0.11)
    T.integrate(tv, tw, origin, 0.11, c["depth"], c["cam_T_world"], c["K"], max_depth=c["max_depth"])
    vals = tv[:-1, :, :z].contiguous()                         # odd X, Z % 8 != 0
    _, f, _ = assert_matches_oracle(vals, single)
    assert len(f) > 100


def _merged(verts, faces):
    """Vertices merged where they coincide exactly; faces re-indexed, degenerate ones dropped."""
    u, inv = np.unique(verts, axis=0, return_inverse=True)
    f = inv.reshape(-1)[faces]
    f = f[(f[:, 0] != f[:, 1]) & (f[:, 1] != f[:, 2]) & (f[:, 0] != f[:, 2])]
    return u, f


def _topology(verts, faces):
    v, f = _merged(verts, faces)
    e = np.sort(np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]]), 1)
    ue, cnt = np.unique(e, axis=0, return_counts=True)
    directed = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])
    assert len(np.unique(directed, axis=0)) == len(directed)          # consistently oriented
    return v, f, len(v) - len(ue) + len(f), cnt


def _sphere(n, c, r):
    x = np.arange(n, dtype=np.float64)
    d = np.sqrt(((x[:, None, None] - c[0]) ** 2 + (x[None, :, None] - c[1]) ** 2 + (x[None, None, :] - c[2]) ** 2))
    return np.clip((d - r) / 3.0, -1, 1).astype(np.float16)


def check_sphere(verts, faces, normals, c, r):
    v, f, chi, cnt = _topology(verts, faces)
    assert np.all(cnt == 2) and chi == 2                        # closed 2-manifold, sphere
    p = v[f]
    vol = np.einsum("ij,ij->i", p[:, 0], np.cross(p[:, 1], p[:, 2])).sum() / 6.0
    assert abs(vol / (4.0 / 3.0 * np.pi * r ** 3) - 1) < 0.01
    # normals: along the analytic normal, and on the side the faces wind toward
    radial = verts - np.asarray(c)
    radial /= np.linalg.norm(radial, axis=1, keepdims=True)
    assert np.einsum("ij,ij->i", normals, radial).min() > 0.99
    fn = np.cross(verts[faces[:, 1]] - verts[faces[:, 0]], verts[faces[:, 2]] - verts[faces[:, 0]])
    assert np.all(np.einsum("ij,ij->i", fn, normals[faces].sum(1)) > 0)


def test_sphere_and_torus(emulated):
    c, r = (12.3, 11.7, 12.1), 8.2
    vol = _volume(_sphere(25, c, r))
    verts, faces, normals = (t.numpy() for t in vol.extract_mesh())
    check_sphere(verts, faces, normals, c, r)
    x = np.arange(28, dtype=np.float64) - 13.6
    X, Y, Z = np.meshgrid(x, x, x - 0.3, indexing="ij")
    d = np.sqrt((np.sqrt(X ** 2 + Y ** 2) - 8.0) ** 2 + Z ** 2) - 3.1
    verts, faces, _ = (t.numpy() for t in _volume(np.clip(d / 3, -1, 1)).extract_mesh())
    _, _, chi, cnt = _topology(verts, faces)
    assert np.all(cnt == 2) and chi == 0


def test_plane_through_exact_zeros_has_no_degenerate_face(emulated):
    x = np.arange(10, dtype=np.float32)
    vals = np.broadcast_to(((x - 4.0) / 4.0)[None, None, :], (9, 7, 10)).copy()   # exactly 0 at z = 4
    vals[:, :, 2] = -0.25
    verts, faces, _ = assert_matches_oracle(vals, False)
    v, f = verts.numpy(), faces.numpy()
    assert len(f) > 0
    area = np.linalg.norm(np.cross(v[f[:, 1]] - v[f[:, 0]], v[f[:, 2]] - v[f[:, 0]]), axis=1)
    assert area.min() > 0
    assert np.array_equal(np.unique(f), np.arange(len(v)))       # every vertex referenced


def test_empty_volume(emulated):
    vol = tsdf_mod.TSDF.from_bounds({"xmin": 0, "xmax": 0.3, "ymin": 0, "ymax": 0.3, "zmin": 0, "zmax": 0.3},
                                    0.04, device="cpu")
    verts, faces, normals = vol.extract_mesh()
    assert verts.shape == (0, 3) and faces.shape == (0, 3) and normals.shape == (0, 3)
    with pytest.raises(ValueError):
        vol.to_mesh()


def test_abi_argument_checks(emulated):
    lib = emulated
    v = torch.zeros((4, 4, 4), dtype=torch.float16)
    counts = torch.zeros(4, dtype=torch.int64)
    ws = torch.empty(1 << 16, dtype=torch.uint8)
    good = _native.MeshVolume(v.data_ptr(), 4, 4, 4, 0)
    n = lib.srcv_mesh_workspace_bytes(C.byref(good))
    assert 0 < n <= 1 << 16

    def count(vol, cnt=counts.data_ptr(), w=ws.data_ptr(), nb=n):
        return lib.srcv_mesh_count_f16(C.byref(vol) if vol is not None else None, cnt, w, nb, None)

    assert count(good) == 0
    assert count(None) == 1
    assert count(_native.MeshVolume(None, 4, 4, 4, 0)) == 1
    assert count(good, cnt=None) == 1
    assert count(good, w=None) == 1
    for dims in ((1, 4, 4), (4, 1, 4), (4, 4, 1), (0, 4, 4), (-3, 4, 4)):
        assert count(_native.MeshVolume(v.data_ptr(), *dims, 0)) == 2
    assert count(_native.MeshVolume(v.data_ptr(), 4, 4, 4, 2)) == 2
    assert count(_native.MeshVolume(v.data_ptr() + 1, 4, 4, 4, 0)) == 4         # misaligned values
    assert count(good, cnt=counts.data_ptr() + 4) == 4
    assert count(good, nb=n - 1) == 3                                           # workspace too small
    assert count(good, w=ws.data_ptr() + 1) == 3                                # misaligned workspace
    sb = lib.srcv_mesh_scratch_bytes(8)
    sc = torch.empty(sb, dtype=torch.uint8)
    out = torch.empty(64, dtype=torch.float32)
    f = torch.empty(64, dtype=torch.int32)

    def emit(nc=8, nf=4, verts=out.data_ptr(), sbytes=sb):
        return lib.srcv_mesh_emit_f16(C.byref(good), nc, nf, verts, out.data_ptr(), f.data_ptr(), counts.data_ptr(),
                                      ws.data_ptr(), n, sc.data_ptr(), sbytes, None)

    assert emit(-1) == 2 and emit(8, -1) == 2
    assert emit(8, 2**31 // 3 + 1) == 2                                         # 3 F overflows int32
    assert emit(verts=None) == 1
    assert emit(verts=out.data_ptr() + 2) == 4
    assert emit(sbytes=sb - 1) == 3
    assert lib.srcv_mesh_scratch_bytes(-1) == 0
