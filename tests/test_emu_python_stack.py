"""The Python layer (manager classes, autograd Functions, ctypes marshalling) driven on the
CPU against the host-emulated C-ABI library (tests/emu), checked against the oracle.

The product refuses CPU tensors (`cost_volume._require_cuda`) and loads only the nvcc-built
library; this test monkeypatches exactly those two things — the device gate and the loaded
library handle — plus the torch.cuda calls the managers make (and the workspace alignment a CUDA allocation has), so that the very same
`forward` / autograd code that runs on the GPU runs here.  Nothing in the product takes this
path by itself."""
import contextlib
import types

import pytest
import torch

import simplerecon_b200 as S
from oracle import costvolume_oracle as O
from simplerecon_b200 import _native, cost_volume
from simplerecon_b200.synthetic import make_tuple, mlp_state
from tests import emu
from tests.parity import assert_cost_close, assert_lowest_close, assert_mask_close, load_reference_outputs


@pytest.fixture()
def emulated(monkeypatch):
    lib = emu.load_or_skip()
    lib.emu_set_sms(4)
    lib.srcv_set_variant(_native.VARIANT_AUTO)
    monkeypatch.setattr(_native, "_lib", lib)
    monkeypatch.setattr(cost_volume, "_require_cuda", lambda dev: None)
    monkeypatch.setattr(torch.cuda, "device", lambda dev: contextlib.nullcontext())
    monkeypatch.setattr(torch.cuda, "current_stream", lambda dev=None: types.SimpleNamespace(cuda_stream=0))
    # CUDA allocations are >= 256-byte aligned (the C ABI requires it of the workspace); CPU ones are not
    real_empty = torch.empty

    def aligned_empty(*size, **kw):
        if kw.get("dtype") is torch.uint8 and len(size) == 1 and isinstance(size[0], int):
            buf = real_empty(size[0] + 256, **kw)
            off = (-buf.data_ptr()) % 256
            return buf[off:off + size[0]]
        return real_empty(*size, **kw)

    monkeypatch.setattr(torch, "empty", aligned_empty)
    return lib


def _rel(a, b):
    a, b = a.double(), b.double()
    return ((a - b).abs().max() / (b.abs().max() + 1e-30)).item()


def _hero(K, C, H, W, D, fast=False):
    cls = S.FastFeatureVolumeManager if fast else S.FeatureVolumeManager
    m = cls(H, W, num_depth_bins=D, mlp_channels=[0, 128, 128, 1], matching_dim_size=C, num_source_views=K)
    m.load_state_dict({**m.state_dict(), **mlp_state(views=K, channels=C, seed=1)})
    return m


def test_dot_manager_forward_and_training(emulated):
    B, K, C, H, W, D = 2, 3, 16, 10, 12, 8
    t = make_tuple(B, K, H, W, channels=C, seed=7)
    m = S.CostVolumeManager(H, W, num_depth_bins=D)
    with torch.no_grad():
        cost, lowest, planes, mask = m(**t)
    oc, ol, op, _ = O.forward_dot(**t, num_depth_bins=D)
    assert mask is None and planes.shape == (B, D, H, W) and planes.stride()[2:] == (0, 0)
    assert_cost_close("dot", cost, oc, what="manager/emu")
    assert_lowest_close("dot", lowest, planes, oc, what="manager/emu")
    # training path: _DotVolumeFunction
    g = torch.randn(B, D, H, W, generator=torch.Generator().manual_seed(8))
    ours, ref = dict(t), dict(t)
    for d in (ours, ref):
        d["cur_feats"] = t["cur_feats"].clone().requires_grad_(True)
        d["src_feats"] = t["src_feats"].clone().requires_grad_(True)
    c2, l2, _, _ = m(**ours)
    assert c2.requires_grad and not l2.requires_grad and torch.equal(c2.detach(), cost)
    (c2 * g).sum().backward()
    rc, *_ = O.forward_dot(**ref, num_depth_bins=D)
    (rc * g).sum().backward()
    for k in ("cur_feats", "src_feats"):
        assert _rel(ours[k].grad, ref[k].grad) < 5e-5, k


@pytest.mark.parametrize("fast,return_mask", [(False, True), (True, False)])
def test_hero_manager_forward(emulated, fast, return_mask):
    B, K, C, H, W, D = 1, 3, 8, 9, 11, 3
    t = make_tuple(B, K, H, W, channels=C, seed=9)
    m = _hero(K, C, H, W, D, fast)
    with torch.no_grad():
        cost, lowest, planes, mask = m(**t, return_mask=return_mask)
    wts = O.mlp_weights_from_state_dict(m.state_dict())
    oc, ol, op, om = O.forward_mlp(**t, weights=wts, num_depth_bins=D, return_mask=True)
    assert_cost_close("mlp", cost, oc, what="hero manager/emu")
    assert_lowest_close("mlp", lowest, planes, oc, what="hero manager/emu")
    if return_mask:
        assert mask.dtype == torch.bool
        assert_mask_close(mask, om, what="hero manager/emu")
    else:
        assert mask is None


@pytest.mark.parametrize("per_pixel", [False, True])
def test_hero_manager_training(emulated, per_pixel):
    """FeatureVolumeManager under autograd: _MlpVolumeFunction -> srcv_mlp_backward_f32; gradients
    of both feature inputs and all six MLP parameters against autograd through the oracle."""
    B, K, C, H, W, D = 1, 2, 8, 8, 10, 3
    t = make_tuple(B, K, H, W, channels=C, seed=13)
    g = torch.Generator().manual_seed(14)
    gcost = torch.randn(B, D, H, W, generator=g)
    planes = (0.3 + 4.0 * torch.rand(B, D, H, W, generator=g)) if per_pixel else None
    m = _hero(K, C, H, W, D).train()
    ours = dict(t)
    ours["cur_feats"] = t["cur_feats"].clone().requires_grad_(True)
    ours["src_feats"] = t["src_feats"].clone().requires_grad_(True)
    cost, lowest, planes_ret, mask = m(**ours, depth_planes_bdhw=planes, return_mask=True)
    assert cost.requires_grad and not lowest.requires_grad and mask.dtype == torch.bool and not mask.requires_grad
    (cost * gcost).sum().backward()
    # fp64 oracle gradients (the fp32 composite flips LeakyReLU kinks more often than the kernel)
    ref = {k: v.double() for k, v in t.items()}
    ref["cur_feats"] = ref["cur_feats"].clone().requires_grad_(True)
    ref["src_feats"] = ref["src_feats"].clone().requires_grad_(True)
    wo = [w.detach().double().clone().requires_grad_(True) for w in O.mlp_weights_from_state_dict(m.state_dict())]
    oc, *_ = O.forward_mlp(**ref, weights=tuple(wo), num_depth_bins=D,
                           depth_planes_bdhw=None if planes is None else planes.double())
    (oc * gcost.double()).sum().backward()
    oc = oc.float()
    assert_cost_close("mlp", cost, oc.detach(), what="hero training forward")
    assert _rel(ours["cur_feats"].grad, ref["cur_feats"].grad) < 2e-5
    assert _rel(ours["src_feats"].grad, ref["src_feats"].grad) < 2e-5
    params = [p for i in (0, 2, 4) for p in (m.mlp.net[i].weight, m.mlp.net[i].bias)]
    for p, w in zip(params, wo):
        assert p.grad is not None and p.grad.shape == w.grad.shape
        assert _rel(p.grad, w.grad) < 2e-5
    # only the MLP parameters require grad (features detached): still differentiable
    m.zero_grad()
    c3, *_ = m(**t, depth_planes_bdhw=planes)
    assert c3.requires_grad
    (c3 * gcost).sum().backward()
    assert _rel(m.mlp.net[0].weight.grad, wo[0].grad) < 2e-5
    # inference calls on the same manager take the plain fused path
    with torch.no_grad():
        c4, *_ = m(**t, depth_planes_bdhw=planes)
    assert not c4.requires_grad and torch.equal(c4, cost.detach())


def test_warp_features_method(emulated):
    B, K, C, H, W = 1, 2, 8, 9, 12
    t = make_tuple(B, K, H, W, channels=C, seed=15)
    m = S.CostVolumeManager(H, W, num_depth_bins=4)
    plane = torch.full((B, 1, 1, 1), 1.7).expand(B, 1, H, W)
    world, depths, warped, mask = m.warp_features(t["src_feats"].reshape(B * K, C, H, W), t["src_extrinsics"],
                                                  t["src_Ks"], t["cur_invK"], plane, B, K, C)
    X = 1.7 * O.backproject_rays(t["cur_invK"], H, W)
    px, py, zp = O.project(X, t["src_Ks"], t["src_extrinsics"])
    ref = O.sample_bilinear_zeros(t["src_feats"], px, py).reshape(B, K, C, H, W)
    assert (warped - ref).abs().max().item() <= 4e-5 * ref.abs().max().item() + 1e-6
    assert world.shape == (B * K, 4, H * W)


@pytest.mark.parametrize("kind", ["dot", "mlp"])
def test_training_with_strided_views_and_half_inputs(emulated, kind):
    """ADVICE r1: (high) the reference caller passes VIEWS of one encoder output — cur_feats =
    matching_feats[:, 0] is non-contiguous for B > 1 (experiment_modules/depth_model.py:242) — so
    the backward must run on the dense copies the forward read; (medium) half / bf16 features
    are upcast in the no-grad path exactly as in the autograd Functions."""
    B, K, C, H, W, D = 2, 2, 8, 8, 10, 3
    t = make_tuple(B, K, H, W, channels=C, seed=21)
    g = torch.Generator().manual_seed(22)
    feats = torch.randn(B, 1 + K, C, H, W, generator=g)
    gcost = torch.randn(B, D, H, W, generator=g)
    m = (S.CostVolumeManager(H, W, num_depth_bins=D) if kind == "dot" else _hero(K, C, H, W, D)).train()
    fo = feats.clone().requires_grad_(True)
    ours = dict(t)
    ours["cur_feats"], ours["src_feats"] = fo[:, 0], fo[:, 1:]
    assert not ours["cur_feats"].is_contiguous()
    cost, *_ = m(**ours)
    (cost * gcost).sum().backward()
    f64 = feats.double().requires_grad_(True)
    ref = {k: v.double() for k, v in t.items()}
    ref["cur_feats"], ref["src_feats"] = f64[:, 0], f64[:, 1:]
    if kind == "dot":
        oc, *_ = O.forward_dot(**ref, num_depth_bins=D)
    else:
        wo = tuple(w.detach().double() for w in O.mlp_weights_from_state_dict(m.state_dict()))
        oc, *_ = O.forward_mlp(**ref, weights=wo, num_depth_bins=D)
    (oc * gcost.double()).sum().backward()
    assert _rel(fo.grad, f64.grad) < 5e-5
    # half inputs without grad (Lightning validation under autocast): upcast, same result as fp32 of the
    # rounded values; with grad: gradients come back in the inputs' dtype
    for dt in (torch.float16, torch.bfloat16):
        fh = feats.to(dt)
        with torch.no_grad():
            ch, *_ = m(**{**t, "cur_feats": fh[:, 0], "src_feats": fh[:, 1:]})
            cf, *_ = m(**{**t, "cur_feats": fh[:, 0].float(), "src_feats": fh[:, 1:].float()})
        assert ch.dtype == torch.float32 and torch.equal(ch, cf)
        fhg = fh.clone().requires_grad_(True)
        cg, *_ = m(**{**t, "cur_feats": fhg[:, 0], "src_feats": fhg[:, 1:]})
        (cg * gcost).sum().backward()
        assert fhg.grad.dtype == dt and torch.isfinite(fhg.grad.float()).all()


def test_unsupported_training_shape_fails_in_forward(emulated):
    """The dot backward kernel serves C in {8, 16, 32}: a C = 4 training call is refused when the
    graph is built, not at backward() time (ADVICE r1)."""
    B, K, C, H, W, D = 1, 2, 4, 6, 8, 3
    t = make_tuple(B, K, H, W, channels=C, seed=23)
    m = S.CostVolumeManager(H, W, num_depth_bins=D)
    with torch.no_grad():
        m(**t)                                  # inference is fine (generic kernel)
    t["cur_feats"] = t["cur_feats"].clone().requires_grad_(True)
    with pytest.raises(NotImplementedError):
        m(**t)


def test_per_frame_depth_range_and_weight_image_cache(emulated):
    B, K, C, H, W, D = 2, 7, 16, 6, 16, 4
    t = make_tuple(B, K, H, W, channels=C, seed=24)
    t["min_depth"] = torch.tensor([0.25, 0.6]).view(B, 1, 1, 1)
    t["max_depth"] = torch.tensor([5.0, 3.0]).view(B, 1, 1, 1)
    m = _hero(K, C, H, W, D)
    with torch.no_grad():
        cost, lowest, planes, _ = m(**t)
        key0 = m.__dict__["_srcv_packed"][0]
        cost2, *_ = m(**t)
        assert m.__dict__["_srcv_packed"][0] == key0 and torch.equal(cost, cost2)     # image reused
        m.mlp.net[0].bias.add_(0.25)                                                  # in-place update: new version
        cost3, *_ = m(**t)
        assert m.__dict__["_srcv_packed"][0] != key0 and not torch.equal(cost3, cost)
    assert "_srcv_packed" not in m.state_dict() and len(m.state_dict()) == 9
    wts = O.mlp_weights_from_state_dict(m.state_dict())
    oc, ol, op, _ = O.forward_mlp(**t, weights=wts, num_depth_bins=D)
    assert torch.allclose(planes, op, rtol=3e-7, atol=0)
    assert_cost_close("mlp", cost3, oc, what="per-frame range, tcgen05/emu")


def test_fast_manager_warp_features_five_tuple(emulated):
    """FastFeatureVolumeManager.warp_features (reference modules/cost_volume.py:812-964): all planes
    at once, 5-tuple (world points, depths, warped, mask, pixel coordinates) — against the oracle,
    and against the reference class's output (tests/golden/make_golden_reference.py)."""
    B, K, C, H, W, D = 2, 3, 8, 9, 12, 4
    t = make_tuple(B, K, H, W, channels=C, seed=31)
    m = _hero(K, C, H, W, D, fast=True)
    planes = m.generate_depth_planes(B, t["min_depth"], t["max_depth"])
    world, depths, warped, mask, pix = m.warp_features(t["src_feats"], t["src_extrinsics"], t["src_Ks"],
                                                       t["cur_invK"], planes, B, K, C, None)
    assert world.shape == (B, K, D, 4, H, W) and depths.shape == (B, K, D, H, W)
    assert warped.shape == (B, K, D, C, H, W) and mask.shape == (B, K, D, H, W) and pix.shape == (B, K, D, 2, H, W)
    rays = O.backproject_rays(t["cur_invK"], H, W)
    for d in range(D):
        X = planes[:, d, 0, 0].view(B, 1, 1) * rays
        px, py, zp = O.project(X, t["src_Ks"], t["src_extrinsics"])
        ref = O.sample_bilinear_zeros(t["src_feats"], px, py).reshape(B, K, C, H, W)
        assert (warped[:, :, d] - ref).abs().max().item() <= 4e-5 * ref.abs().max().item() + 1e-6
        assert torch.allclose(depths[:, :, d].reshape(B, K, -1), zp, rtol=2e-6, atol=1e-6)
        assert torch.allclose(pix[:, :, d, 0].reshape(B, K, -1), px, rtol=0, atol=2e-4)
        assert torch.allclose(pix[:, :, d, 1].reshape(B, K, -1), py, rtol=0, atol=2e-4)
        assert torch.equal(mask[:, :, d].reshape(B, K, -1), (zp > 0).float())
        assert torch.allclose(world[:, 0, d, :3].reshape(B, 3, -1), X, rtol=1e-6, atol=1e-7)
    R = load_reference_outputs("python_layer")
    rw, rd, rf, rm, rp = (R[f"warp_{k}"] for k in ("world", "depths", "feats", "mask", "pix"))
    assert torch.allclose(world, rw, rtol=1e-6, atol=1e-7) and torch.equal(mask, rm)
    assert torch.allclose(depths, rd, rtol=2e-6, atol=1e-6) and torch.allclose(pix, rp, rtol=0, atol=2e-4)
    assert (warped - rf).abs().max().item() <= 4e-5 * rf.abs().max().item() + 1e-6


def test_producer_side_fusion_chunk_planar_and_raw_poses(emulated):
    """SURVEY §8f-2: (1) instance_norm_to_chunk_planar == nn.InstanceNorm2d(16) (reference
    modules/networks.py:201) written in the gather layout; (2) both sweeps on chunk-planar inputs
    equal the NCHW path bit for bit (same values, no prep copy); (3) raw poses: the prep kernel's
    relative transforms (depth_model.py:324-332) reproduce the call with PyTorch-side products."""
    B, K, C, H, W, D = 2, 7, 16, 10, 16, 4
    t = make_tuple(B, K, H, W, channels=C, seed=41)
    g = torch.Generator().manual_seed(42)
    x = 3.0 * torch.randn(B, 1 + K, C, H, W, generator=g) + 0.7
    cur_c4, src_c4 = S.instance_norm_to_chunk_planar(x)
    ref = torch.nn.InstanceNorm2d(C)(x.reshape(B * (1 + K), C, H, W)).reshape(B, 1 + K, C, H, W)
    back = lambda c4: c4.movedim(-1, -3).flatten(-4, -3)        # (..., C/4, H, W, 4) -> (..., C, H, W)
    assert cur_c4.shape == (B, C // 4, H, W, 4) and src_c4.shape == (B, K, C // 4, H, W, 4)
    assert (back(cur_c4) - ref[:, 0]).abs().max().item() < 3e-6
    assert (back(src_c4) - ref[:, 1:]).abs().max().item() < 3e-6
    nchw = dict(t, cur_feats=back(cur_c4).contiguous(), src_feats=back(src_c4).contiguous())
    c4 = dict(t, cur_feats=cur_c4, src_feats=src_c4)
    # world poses whose products are the tuple's relative transforms
    world_T_cur = torch.linalg.inv(make_tuple(B, 1, H, W, seed=43)["src_extrinsics"][:, 0].double())
    cur_T_world = torch.linalg.inv(world_T_cur)
    raw = dict(src_cam_T_world=(t["src_extrinsics"].double() @ cur_T_world[:, None]).float(),
               src_world_T_cam=(world_T_cur[:, None] @ t["src_poses"].double()).float(),
               cur_cam_T_world=cur_T_world.float(), cur_world_T_cam=world_T_cur.float())
    for m in (S.CostVolumeManager(H, W, num_depth_bins=D), _hero(K, C, H, W, D)):
        with torch.no_grad():
            a = m(**nchw, return_mask=True)
            b = m(**c4, return_mask=True)
            r = m(**{**nchw, "src_extrinsics": None, "src_poses": None}, return_mask=True, raw_poses=raw)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
        if a[3] is not None:
            assert torch.equal(a[3], b[3])
        tol = 2e-4 * float(a[0].abs().max())      # the raw poses went through an fp32 round trip
        assert (r[0] - a[0]).abs().max().item() <= tol
    # gradients are refused on the chunk-planar path (the backward kernels take NCHW)
    c4g = dict(c4, cur_feats=cur_c4.clone().requires_grad_(True))
    with pytest.raises(NotImplementedError):
        S.CostVolumeManager(H, W, num_depth_bins=D)(**c4g)
