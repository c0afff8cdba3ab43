"""GPU parity: the sm_100a kernels (through the C ABI, via the manager classes)
against (1) the committed golden vectors of the unmodified reference, (2) the CPU
oracle on seeded inputs, (3) size-independent properties at BASELINE.json's full
sizes.  Tolerances are stated in tests/parity.py."""
import pytest
import torch

import simplerecon_b200 as S
from oracle import costvolume_oracle as O
from simplerecon_b200 import _native
from simplerecon_b200.synthetic import CONFIGS, make_tuple, make_workload_tuple, mlp_state, to_device
from tests.parity import (assert_cost_close, assert_lowest_close, assert_mask_close, cost_tol,
                          golden_fullsize_names, golden_names, load_golden, load_golden_fullsize)

pytestmark = pytest.mark.gpu

VARIANTS = {"generic": _native.VARIANT_GENERIC, "fast": _native.VARIANT_FAST, "auto": _native.VARIANT_AUTO}


@pytest.fixture(autouse=True)
def _reset_variant(cuda_device):
    yield
    _native.set_variant(_native.VARIANT_AUTO)


def make_manager(kind, K, C, H, W, D, sd=None, device="cuda", fast_cls=False):
    if kind == "dot":
        m = S.CostVolumeManager(H, W, num_depth_bins=D)
    else:
        cls = S.FastFeatureVolumeManager if fast_cls else S.FeatureVolumeManager
        m = cls(H, W, num_depth_bins=D, mlp_channels=[0, 128, 128, 1], matching_dim_size=C,
                num_source_views=K)
        m.load_state_dict({**m.state_dict(), **sd})
    return m.to(device).eval()


def run_gpu(kind, inputs, D, sd=None, variant="auto", return_mask=True, fast_cls=False):
    B, K, C, H, W = inputs["src_feats"].shape
    m = make_manager(kind, K, C, H, W, D, sd, fast_cls=fast_cls)
    _native.set_variant(VARIANTS[variant])
    with torch.inference_mode():
        out = m(**to_device(inputs, "cuda"), return_mask=return_mask)
    torch.cuda.synchronize()
    return out, _native.last_variant()


def fast_ok(kind, inputs):
    B, K, C, H, W = inputs["src_feats"].shape
    if kind == "dot":
        return C == 16                      # chunk-planar gather kernel
    return C == 16 and K == 7               # tcgen05 kernel: hero layout (hidden widths 128/128)


# --------------------------------------------------------------------------- #
# 1. golden vectors of the unmodified reference                               #
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize("variant", ["generic", "fast"])
@pytest.mark.parametrize("name", golden_names())
def test_golden(name, variant):
    g, inputs, sd = load_golden(name)
    kind = g["kind"]
    if variant == "fast" and not fast_ok(kind, inputs):
        pytest.skip("fast variant does not cover this shape")
    (cost, lowest, planes, mask), used = run_gpu(kind, inputs, g["D"], sd, variant)
    assert (("fast" in used) or ("tc" in used)) == (variant == "fast"), used
    assert cost.is_contiguous() and cost.dtype == torch.float32 and cost.is_cuda
    assert_cost_close(kind, cost, g["ref_cost"], g["ref_cost64"], what=f"{name}/{variant}")
    ref_planes = g["ref_planes"]
    if ref_planes.dim() == 2:
        assert planes.stride()[2:] == (0, 0)                       # expanded view, like the reference
        assert torch.allclose(planes[:, :, 0, 0].cpu(), ref_planes, rtol=3e-7, atol=0)
    else:
        assert torch.equal(planes.cpu(), ref_planes)               # caller-supplied planes are handed back
    assert_lowest_close(kind, lowest, planes, g["ref_cost"], what=name)
    if kind == "mlp":
        assert_mask_close(mask, g["ref_mask"], what=name)
    else:
        assert mask is None


@pytest.mark.parametrize("variant", ["generic", "fast"])
@pytest.mark.parametrize("name", golden_fullsize_names())
def test_golden_full_size(name, variant):
    """The unmodified reference's outputs at the bench feature-map size (120 x 160, 7 views): the fast
    variants run their compile-time 160 x 120 instantiations here (the dot sweep and the tcgen05 kernel)."""
    g, inputs, sd = load_golden_fullsize(name)
    kind = g["kind"]
    (cost, lowest, planes, mask), used = run_gpu(kind, inputs, g["D"], sd, variant)
    assert (("fast" in used) or ("tc" in used)) == (variant == "fast"), used
    assert_cost_close(kind, cost, g["ref_cost"], g["ref_cost64"], what=f"{name}/{variant}", e_ref=g["err32v64"])
    assert torch.allclose(planes[:, :, 0, 0].cpu(), g["ref_planes"], rtol=3e-7, atol=0)
    assert_lowest_close(kind, lowest, planes, g["ref_cost"], what=name)
    if kind == "mlp":
        assert_mask_close(mask, g["ref_mask"], what=name)


# --------------------------------------------------------------------------- #
# 2. CPU oracle on seeded inputs                                              #
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize("variant", ["generic", "fast"])
@pytest.mark.parametrize("B,K,H,W,D,seed,smooth", [
    (2, 7, 60, 80, 32, 3, False),
    (1, 2, 48, 64, 16, 1234, False),
    (3, 5, 33, 47, 9, 8, True),        # odd sizes: partial warps and tiles
    (1, 8, 17, 160, 4, 9, False),
])
def test_dot_vs_oracle(B, K, H, W, D, seed, smooth, variant):
    t = make_tuple(B, K, H, W, seed=seed, smooth=smooth)
    (cost, lowest, planes, mask), used = run_gpu("dot", t, D, variant=variant)
    oc, ol, op, _ = O.forward_dot(**t, num_depth_bins=D)
    assert_cost_close("dot", cost, oc, what=f"dot {used}")
    assert torch.allclose(planes.cpu()[:, :, 0, 0], op[:, :, 0, 0], rtol=3e-7)
    assert_lowest_close("dot", lowest, planes, oc, what="dot")
    assert mask is None


@pytest.mark.parametrize("variant", ["generic", "fast"])
@pytest.mark.parametrize("B,K,C,H,W,D,seed", [
    (1, 7, 16, 30, 40, 16, 5),
    (2, 7, 16, 37, 53, 3, 15),         # partial 16x8 tiles on both borders
    (2, 3, 16, 21, 19, 5, 6),
    (1, 2, 8, 16, 24, 4, 7),           # C != 16
])
def test_mlp_vs_oracle(B, K, C, H, W, D, seed, variant):
    t = make_tuple(B, K, H, W, channels=C, seed=seed)
    if variant == "fast" and not fast_ok("mlp", t):
        pytest.skip("tensor-core variant covers the hero layout only")
    sd = mlp_state(K, C, seed=seed)
    (cost, lowest, planes, mask), used = run_gpu("mlp", t, D, sd, variant)
    assert ("tc" in used) == (variant == "fast"), used
    w = O.mlp_weights_from_state_dict(sd)
    oc, ol, op, om = O.forward_mlp(**t, weights=w, num_depth_bins=D, return_mask=True)
    assert_cost_close("mlp", cost, oc, what=f"mlp {used}")
    assert_mask_close(mask, om)
    # without return_mask the mask is None, like the reference
    (c2, _, _, m2), _ = run_gpu("mlp", t, D, sd, variant, return_mask=False)
    assert m2 is None and torch.equal(c2, cost)


def test_mlp_other_hidden_widths():
    # reference API allows any mlp_channels list; widths <= 128 run on the generic kernel
    t = make_tuple(1, 3, 12, 16, seed=21)
    m = S.FeatureVolumeManager(12, 16, 4, mlp_channels=[0, 64, 24, 1], matching_dim_size=16,
                               num_source_views=3).cuda().eval()
    with torch.inference_mode():
        cost, lowest, planes, mask = m(**to_device(t, "cuda"), return_mask=True)
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    oc, *_ = O.forward_mlp(**t, weights=O.mlp_weights_from_state_dict(sd), num_depth_bins=4, return_mask=True)
    assert_cost_close("mlp", cost, oc)


# --------------------------------------------------------------------------- #
# 3. BASELINE.json full sizes: properties + one frame against the oracle      #
# --------------------------------------------------------------------------- #
def test_full_size_dot_cfg1():
    w = CONFIGS[1]
    t = make_workload_tuple(w)
    (cost, lowest, planes, _), used = run_gpu("dot", t, w.planes, variant="auto")
    assert "fast" in used and cost.shape == (4, 64, 120, 160)
    # (a) frame 0 against the CPU oracle at full size
    t0 = {k: (v[:1] if v.dim() > 0 and v.shape[0] == w.batch else v) for k, v in t.items()}
    oc, ol, op, _ = O.forward_dot(**t0, num_depth_bins=w.planes)
    oc64, *_ = O.forward_dot(**{k: v.double() for k, v in t0.items()}, num_depth_bins=w.planes)
    assert_cost_close("dot", cost[:1], oc, oc64, what="cfg1 frame0")
    # (b) both variants agree
    (cost_g, lowest_g, _, _), _ = run_gpu("dot", t, w.planes, variant="generic")
    assert (cost - cost_g).abs().max().item() <= cost_tol("dot", oc)
    # (c) shard invariance: frames 2..3 alone == the same frames inside the batch (bit-exact)
    th = {k: (v[2:] if v.dim() > 0 and v.shape[0] == w.batch else v) for k, v in t.items()}
    (cost_h, lowest_h, _, _), _ = run_gpu("dot", th, w.planes)
    assert torch.equal(cost_h, cost[2:]) and torch.equal(lowest_h, lowest[2:])
    # (d) homogeneity: scaling the reference features by 2 scales the volume by exactly 2
    t2 = dict(t); t2["cur_feats"] = t["cur_feats"] * 2
    (cost2, lowest2, _, _), _ = run_gpu("dot", t2, w.planes)
    assert torch.equal(cost2, cost * 2) and torch.equal(lowest2, lowest)
    # (e) lowest_cost is the plane at the argmax of our own volume
    idx = cost.argmax(1, keepdim=True)
    assert torch.equal(torch.gather(planes.expand_as(cost), 1, idx).squeeze(1), lowest)
    # (f) determinism
    (cost_r, _, _, _), _ = run_gpu("dot", t, w.planes)
    assert torch.equal(cost_r, cost)


def test_full_size_hero_cfg2_two_frames():
    w = CONFIGS[2]
    t = make_workload_tuple(w, batch=2)
    sd = mlp_state(7, 16, seed=0)
    (cost, lowest, planes, mask), used = run_gpu("mlp", t, w.planes, sd)
    assert "tc" in used, used
    assert cost.shape == (2, 64, 120, 160) and mask.shape == (2, 120, 160) and mask.dtype == torch.bool
    t0 = {k: (v[:1] if v.dim() > 0 and v.shape[0] == 2 else v) for k, v in t.items()}
    wts = O.mlp_weights_from_state_dict(sd)
    oc, ol, op, om = O.forward_mlp(**t0, weights=wts, num_depth_bins=w.planes, return_mask=True)
    oc64, *_ = O.forward_mlp(**{k: v.double() for k, v in t0.items()},
                             weights=tuple(x.double() for x in wts), num_depth_bins=w.planes)
    assert_cost_close("mlp", cost[:1], oc, oc64, what="cfg2 frame0")
    assert_mask_close(mask[:1], om)
    # shard invariance + argmax consistency + the fast class runs the same sweep
    t1 = {k: (v[1:] if v.dim() > 0 and v.shape[0] == 2 else v) for k, v in t.items()}
    (cost1, lowest1, _, mask1), _ = run_gpu("mlp", t1, w.planes, sd)
    assert torch.equal(cost1, cost[1:]) and torch.equal(mask1, mask[1:])
    idx = cost.argmax(1, keepdim=True)
    assert torch.equal(torch.gather(planes.expand_as(cost), 1, idx).squeeze(1), lowest)
    (cost_f, _, _, mask_f), _ = run_gpu("mlp", t, w.planes, sd, fast_cls=True)
    assert torch.equal(cost_f, cost) and torch.equal(mask_f, mask)
    # the fp32 SIMT variant agrees with the tensor-core variant
    (cost_g, _, _, mask_g), used_g = run_gpu("mlp", t, w.planes, sd, variant="generic")
    assert "generic" in used_g and torch.equal(mask_g, mask)
    assert (cost_g - cost).abs().max().item() <= cost_tol("mlp", oc)


# --------------------------------------------------------------------------- #
# 4. interface behaviour on the device                                        #
# --------------------------------------------------------------------------- #
def test_interface_contract_on_device():
    t = make_tuple(2, 3, 12, 16, seed=31)
    d = to_device(t, "cuda")
    m = make_manager("dot", 3, 16, 12, 16, 6)
    with torch.no_grad():
        cost, lowest, planes, mask = m(**d)
        c3, p3, m3 = m.build_cost_volume(**d)
    assert cost.shape == (2, 6, 12, 16) and lowest.shape == (2, 12, 16) and planes.shape == (2, 6, 12, 16)
    assert mask is None and m3 is None and torch.equal(c3, cost) and torch.equal(p3, planes)
    # planes equal what generate_depth_planes (plain torch ops, as in the reference) gives
    gen = m.generate_depth_planes(2, d["min_depth"], d["max_depth"])
    assert torch.allclose(planes, gen, rtol=3e-7, atol=0)
    # caller-supplied expanded planes take the per-plane path and give the same volume
    with torch.no_grad():
        cost_p, _, planes_p, _ = m(**d, depth_planes_bdhw=planes)
    assert planes_p is planes and torch.equal(cost_p, cost)
    # a non-default stream is honoured
    s = torch.cuda.Stream()
    with torch.cuda.stream(s), torch.no_grad():
        cost_s, *_ = m(**d)
    s.synchronize()
    assert torch.equal(cost_s, cost)
    # non-contiguous features are accepted
    d2 = dict(d); d2["cur_feats"] = d["cur_feats"].permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2)
    with torch.no_grad():
        cost_nc, *_ = m(**d2)
    assert torch.equal(cost_nc, cost)


def test_errors_on_device():
    t = to_device(make_tuple(1, 2, 12, 16, seed=32), "cuda")
    m = make_manager("dot", 2, 16, 12, 16, 4)
    with torch.no_grad():
        with pytest.raises(ValueError):
            S.CostVolumeManager(10, 16, 4).cuda()(**t)                      # wrong H
        # half features are the autocast contract (upcast, computed in fp32): same result as fp32 of
        # the rounded values; other dtypes are refused
        half = dict(t); half["src_feats"] = t["src_feats"].half()
        full = dict(t); full["src_feats"] = t["src_feats"].half().float()
        assert torch.equal(m(**half)[0], m(**full)[0])
        bad = dict(t); bad["src_feats"] = t["src_feats"].double()
        with pytest.raises(ValueError):
            m(**bad)
        bad = dict(t); bad["src_Ks"] = t["src_Ks"][:, :1]
        with pytest.raises(ValueError):
            m(**bad)
    # MLP input width inconsistent with K, C
    f = S.FeatureVolumeManager(12, 16, 4, matching_dim_size=16, num_source_views=7).cuda()
    with torch.no_grad(), pytest.raises(ValueError):
        f(**t)
    # (gradient-requiring calls of the metadata-MLP volume: tests/test_zzz_gpu_mlp_backward.py)
    _native.set_variant(_native.VARIANT_FAST)
    t8 = to_device(make_tuple(1, 2, 12, 16, channels=8, seed=33), "cuda")
    with torch.no_grad(), pytest.raises(_native.SrcvError):
        m(**t8)


def test_warp_features_helper_matches_oracle():
    """CostVolumeManager.warp_features (reference modules/cost_volume.py:139-234): the
    materialising single-plane helper."""
    B, K, H, W = 2, 3, 21, 19
    t = make_tuple(B, K, H, W, seed=44)
    d = to_device(t, "cuda")
    m = make_manager("dot", K, 16, H, W, 4)
    plane = torch.full((B, 1, 1, 1), 1.7, device="cuda").expand(B, 1, H, W)
    with torch.no_grad():
        pts, depths, warped, mask = m.warp_features(d["src_feats"], d["src_extrinsics"], d["src_Ks"],
                                                    d["cur_invK"], plane, B, K, 16, None)
    assert pts.shape == (B * K, 4, H * W) and warped.shape == (B, K, 16, H, W)
    rays = O.backproject_rays(t["cur_invK"], H, W)
    px, py, zp = O.project(1.7 * rays, t["src_Ks"], t["src_extrinsics"])
    ow = O.sample_bilinear_zeros(t["src_feats"], px, py).reshape(B, K, 16, H, W)
    assert (warped.cpu() - ow).abs().max().item() <= 5e-5 * float(ow.abs().max())
    assert torch.allclose(depths.cpu().reshape(B, K, -1), zp, rtol=1e-5, atol=1e-6)
    assert torch.equal(mask.cpu().reshape(B, K, -1), (zp > 0).float())
    assert torch.allclose(pts.cpu().reshape(B, K, 4, -1)[:, 0, :3], 1.7 * rays, rtol=1e-5, atol=1e-6)
    # per-pixel plane
    g = torch.Generator().manual_seed(3)
    pp = (0.5 + 3 * torch.rand(B, 1, H, W, generator=g))
    with torch.no_grad():
        _, depths2, warped2, _ = m.warp_features(d["src_feats"], d["src_extrinsics"], d["src_Ks"],
                                                 d["cur_invK"], pp.cuda(), B, K, 16, None)
    px, py, zp = O.project(pp.reshape(B, 1, -1) * rays, t["src_Ks"], t["src_extrinsics"])
    ow = O.sample_bilinear_zeros(t["src_feats"], px, py).reshape(B, K, 16, H, W)
    assert (warped2.cpu() - ow).abs().max().item() <= 5e-5 * float(ow.abs().max())


def test_host_streamer_matches_direct_calls():
    from simplerecon_b200.pipeline import HostStreamer
    m = make_manager("dot", 3, 16, 24, 32, 6)
    batches = [{k: v.pin_memory() for k, v in make_tuple(2, 3, 24, 32, seed=60 + i).items()} for i in range(5)]
    st = HostStreamer(m, "cuda")
    got = [[t.clone() for t in out] for out in st.run(batches)]
    assert len(got) == 5
    with torch.inference_mode():
        for b, out in zip(batches, got):
            cost, lowest, _, _ = m(**to_device(b, "cuda"))
            assert torch.equal(out[0], cost.cpu()) and torch.equal(out[1], lowest.cpu())


def test_hero_cfg3_planes_96_and_batch_shards():
    """BASELINE configs[3]: hero, D = 96, sharded 4 frames per GPU — one shard here, checked for
    shard invariance and against the oracle on a plane subset (caller-supplied planes)."""
    w = CONFIGS[3]
    t = make_workload_tuple(w, batch=4)
    sd = mlp_state(7, 16, seed=0)
    (cost, lowest, planes, mask), used = run_gpu("mlp", t, w.planes, sd)
    assert "tc" in used and cost.shape == (4, 96, 120, 160)
    t1 = {k: (v[3:] if v.dim() > 0 and v.shape[0] == 4 else v) for k, v in t.items()}
    (cost1, lowest1, _, mask1), _ = run_gpu("mlp", t1, w.planes, sd)
    assert torch.equal(cost1, cost[3:]) and torch.equal(lowest1, lowest[3:]) and torch.equal(mask1, mask[3:])
    # oracle on planes 90..95 of frame 3 via explicit per-plane depths
    sub = planes[3:, 90:].cpu().contiguous()
    wts = O.mlp_weights_from_state_dict(sd)
    oc, ol, op, om = O.forward_mlp(**t1, weights=wts, num_depth_bins=6, depth_planes_bdhw=sub, return_mask=True)
    oc64, *_ = O.forward_mlp(**{k: v.double() for k, v in t1.items()}, weights=tuple(x.double() for x in wts),
                             num_depth_bins=6, depth_planes_bdhw=sub.double())
    assert_cost_close("mlp", cost[3:, 90:], oc, oc64, what="cfg3 planes 90-95")
    assert_mask_close(mask[3:], om)


def test_hero_at_the_reference_training_resolution():
    """512x384 frames (the reference's default, options.py:70-71): the 96x128 feature map runs the
    tensor-core kernel's <false, 128, 96> instantiation.  B = 2, D = 64, planes from the range;
    frame 0 against the oracle on every ninth plane (ending with the last, whose mask is the
    volume's), frame 1 alone against frame 1 in the batch, and the SIMT kernel against both."""
    B, K, H, W, D = 2, 7, 96, 128, 64
    t = make_tuple(B, K, H, W, seed=131)
    sd = mlp_state(K, 16, seed=7)
    (cost, lowest, planes, mask), used = run_gpu("mlp", t, D, sd, variant="fast")
    assert "tc" in used and cost.shape == (B, D, H, W) and mask.shape == (B, H, W)
    sub = list(range(0, D, 9))
    assert sub[-1] == D - 1
    t0 = {k: (v[:1] if v.dim() > 0 and v.shape[0] == B else v) for k, v in t.items()}
    p0 = planes[:1, sub].cpu().contiguous()
    wts = O.mlp_weights_from_state_dict(sd)
    oc, _, _, om = O.forward_mlp(**t0, weights=wts, num_depth_bins=len(sub), depth_planes_bdhw=p0, return_mask=True)
    oc64, *_ = O.forward_mlp(**{k: v.double() for k, v in t0.items()}, weights=tuple(x.double() for x in wts),
                             num_depth_bins=len(sub), depth_planes_bdhw=p0.double())
    assert_cost_close("mlp", cost[:1, sub], oc, oc64, what="96x128 frame 0")
    assert_mask_close(mask[:1], om)
    idx = cost.argmax(1, keepdim=True)
    assert torch.equal(torch.gather(planes.expand_as(cost), 1, idx).squeeze(1), lowest)
    t1 = {k: (v[1:] if v.dim() > 0 and v.shape[0] == B else v) for k, v in t.items()}
    (cost1, lowest1, _, mask1), _ = run_gpu("mlp", t1, D, sd, variant="fast")
    assert torch.equal(cost1, cost[1:]) and torch.equal(lowest1, lowest[1:]) and torch.equal(mask1, mask[1:])
    (cost_g, lowest_g, _, mask_g), used_g = run_gpu("mlp", t, D, sd, variant="generic")
    assert "generic" in used_g and torch.equal(mask_g, mask)
    assert (cost_g - cost).abs().max().item() <= cost_tol("mlp", oc)
    assert_lowest_close("mlp", lowest, planes, cost_g.cpu(), what="96x128 lowest vs the SIMT volume")


def test_bench_gpu_arm_prints_one_json_line():
    """bench.py (ours, N=1, default workload): stdout is exactly ONE JSON line with the contract's
    keys, kernels were launched, and the roofline / e2e / clock blocks are populated."""
    import json
    import subprocess
    import sys
    from pathlib import Path
    root = Path(__file__).resolve().parents[1]
    r = subprocess.run([sys.executable, str(root / "bench.py"), "--steps", "10", "--warmup", "3"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "roofline", "cpu_baseline", "e2e",
              "gpu_launches", "clocks"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 10 and d["value"] > 0 and d["gpu_launches"] >= 20
    # default workload = hero model, 8 frames per GPU (BASELINE configs[2]; configs[4] at 8 GPUs)
    assert d["config"]["workload"].startswith("cfg2_hero") and d["config"]["batch_per_gpu"] == 8
    assert d["dtype"] == "f32" and d["scaling"] == "weak" and "tcgen05" in d["kernel_variant"]
    rf = d["roofline"]
    assert rf["bound"] == "tensor" and 0 < rf["frac"] < 1.2 and rf["peak"] > 500 and rf["achieved"] > 0
    assert 0 < rf["hbm"]["frac"] < 1.5 and rf["issued_mma"]["achieved"] > 2.8 * rf["achieved"]
    assert d["e2e"]["h2d_bytes_per_step"] > 7.8e7 and d["e2e"]["d2h_bytes_per_step"] > 3.9e7
    assert 0 < d["e2e"]["value"] <= d["value"] * 1.05 and len(d["e2e"]["windows_ms_per_step"]) == 3
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] > 0
    assert d["clocks"]["sm_max_mhz"] and not (set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"})
    # the dot-product configuration (BASELINE configs[1]) rides in the same line
    (name, a), = d["also"].items()
    assert name.startswith("cfg1_dot") and a["value"] > 0 and a["roofline"]["bound"] == "hbm"
    assert 0 < a["roofline"]["frac"] < 1.5 and a["e2e"]["h2d_bytes_per_step"] > 3.9e7


@pytest.mark.parametrize("B,K,C,H,W,D,seed,per_pixel", [
    (2, 3, 16, 14, 18, 5, 71, False),
    (1, 7, 16, 24, 32, 8, 72, False),
    (1, 2, 8, 10, 12, 4, 73, True),
    (2, 7, 16, 96, 128, 8, 74, True),      # fast forward at its 512x384-frame size, C = 16 per-pixel backward
    (1, 7, 16, 120, 160, 4, 75, True),
    (1, 3, 32, 11, 13, 4, 76, False),      # C = 32 (generic forward), both plane modes
    (2, 3, 32, 11, 13, 3, 77, True),
])
def test_dot_backward_matches_autograd_of_the_oracle(B, K, C, H, W, D, seed, per_pixel):
    """Training path of CostVolumeManager: dL/dcur_feats and dL/dsrc_feats from the backward
    kernel against CPU autograd through the oracle (the composite the reference differentiates,
    modules/cost_volume.py:305-333)."""
    t = make_tuple(B, K, H, W, channels=C, seed=seed)
    g = torch.Generator().manual_seed(seed)
    gcost = torch.randn(B, D, H, W, generator=g)
    planes = (0.3 + 4.0 * torch.rand(B, D, H, W, generator=g)) if per_pixel else None
    # oracle + autograd (CPU)
    tc = dict(t)
    tc["cur_feats"] = t["cur_feats"].clone().requires_grad_(True)
    tc["src_feats"] = t["src_feats"].clone().requires_grad_(True)
    oc, *_ = O.forward_dot(**tc, num_depth_bins=D, depth_planes_bdhw=planes)
    (oc * gcost).sum().backward()
    # fused forward + backward kernel (GPU)
    d = to_device(t, "cuda")
    d["cur_feats"] = d["cur_feats"].clone().requires_grad_(True)
    d["src_feats"] = d["src_feats"].clone().requires_grad_(True)
    m = make_manager("dot", K, C, H, W, D)
    cost, lowest, planes_ret, mask = m(**d, depth_planes_bdhw=planes.cuda() if per_pixel else None)
    assert cost.requires_grad and not lowest.requires_grad and mask is None
    assert _native.last_variant() == ("dot_fast_c4planar" if C == 16 else "dot_generic")
    assert_cost_close("dot", cost, oc.detach())
    (cost * gcost.cuda()).sum().backward()
    assert _native.last_variant() == "dot_backward_atomic"
    for name in ("cur_feats", "src_feats"):
        ours, ref = d[name].grad.cpu(), tc[name].grad
        tol = 5e-5 * float(ref.abs().max()) + 1e-6
        assert (ours - ref).abs().max().item() <= tol, name
    # inference calls on the same manager still take the plain fused path
    with torch.no_grad():
        c2, *_ = m(**{k: v.detach() for k, v in d.items()}, depth_planes_bdhw=planes.cuda() if per_pixel else None)
    assert torch.equal(c2, cost.detach())


def test_dot_large_batch_unsplit_plane_loop():
    """B = 64 small frames: enough warps that the plane loop is NOT split, i.e. the argmax is
    fused in the sweep itself (the other tests run the split, last-arriver form)."""
    B, K, H, W, D = 64, 2, 60, 80, 8
    t = make_tuple(B, K, H, W, seed=91)
    (cost, lowest, planes, _), used = run_gpu("dot", t, D, variant="fast")
    oc, ol, op, _ = O.forward_dot(**t, num_depth_bins=D)
    assert_cost_close("dot", cost, oc, what="B=64")
    assert_lowest_close("dot", lowest, planes, oc, what="B=64")
    idx = cost.argmax(1, keepdim=True)
    assert torch.equal(torch.gather(planes.expand_as(cost), 1, idx).squeeze(1), lowest)


def _edge_views(t):
    """View 1 looks backwards (every plane point behind the camera: mask 0, features still
    sampled), view 2 is shifted 40 m sideways (every sample outside the frustum)."""
    E = t["src_extrinsics"].clone()
    E[:, 1] = torch.tensor([[-1., 0, 0, 0.05], [0, 1, 0, 0], [0, 0, -1, -0.1], [0, 0, 0, 1]])
    E[:, 2, :3, :3] = torch.eye(3)
    E[:, 2, :3, 3] = torch.tensor([40.0, 0.0, 0.0])
    t = dict(t)
    t["src_extrinsics"] = E
    t["src_poses"] = torch.linalg.inv(E.double()).float()
    return t


@pytest.mark.parametrize("variant,H,W", [
    pytest.param(v, H, W, id=v if (H, W) == (19, 27) else f"{v}-{H}x{W}")
    for H, W in [(19, 27), (96, 128), (120, 160)] for v in ("generic", "fast")])
def test_hero_k7_edge_views_and_per_pixel_planes(variant, H, W):
    """The tensor-core kernel (and the SIMT one) on the reference's corner cases at the hero
    layout: behind-camera and out-of-frustum source views, caller-supplied per-pixel depth
    hypotheses (including a non-positive one), partial tiles — at a generic map size and at both
    sizes the tensor-core kernel is instantiated for (512x384 and 640x480 frames)."""
    B, K, D = 1, 7, 4
    t = _edge_views(make_tuple(B, K, H, W, seed=81))
    sd = mlp_state(K, 16, seed=5)
    g = torch.Generator().manual_seed(82)
    planes = 0.3 + 4.0 * torch.rand(B, D, H, W, generator=g)
    planes[0, 1, 3, 4] = 0.0          # degenerate hypothesis: the point is the camera centre
    planes[0, 2, 5, 6] = -1.0         # behind the reference camera
    w = O.mlp_weights_from_state_dict(sd)
    for dp in (None, planes):
        kw = dict(t)
        if dp is not None:
            kw["depth_planes_bdhw"] = dp
        (cost, lowest, pl, mask), used = run_gpu("mlp", kw, D, sd, variant)
        assert ("tc" in used) == (variant == "fast")
        oc, ol, op, om = O.forward_mlp(**t, weights=w, num_depth_bins=D, depth_planes_bdhw=dp, return_mask=True)
        oc64, *_ = O.forward_mlp(**{k: v.double() for k, v in t.items()}, weights=tuple(x.double() for x in w),
                                 num_depth_bins=D, depth_planes_bdhw=None if dp is None else dp.double())
        assert torch.isfinite(cost).all()
        assert_cost_close("mlp", cost, oc, oc64, what=f"edge {variant} per_pixel={dp is not None}")
        assert_mask_close(mask, om, max_frac=5e-3)


# --------------------------------------------------------------------------- #
# training-side contract: strided views and autocast (half / bf16) inputs      #
# --------------------------------------------------------------------------- #
def _assert_grad_close(ours, ref, rtol):
    """max-abs within rtol * max|ref|, or — LeakyReLU has a kink at 0 and a pre-activation of ~1e-7
    takes either sign in fp32 (tests/test_zzz_gpu_mlp_backward.py, DESIGN §2): a handful of entries
    may then move — the difference is small in norm.  A wrong-layout bug (ADVICE r1: relative error
    1.3) fails both."""
    a, b = ours.detach().double().cpu(), ref.detach().double().cpu()
    if (a - b).abs().max().item() <= rtol * float(b.abs().max()) + 1e-6:
        return
    rel = ((a - b).norm() / (b.norm() + 1e-30)).item()
    assert rel < 2e-2, f"gradient differs: norm-relative {rel:.2e}, max-abs {(a - b).abs().max().item():.2e}"


def _feats_like_the_reference_caller(B, K, C, H, W, seed, dtype=torch.float32):
    """The reference hands the managers VIEWS of one (B, 1+K, C, H, W) encoder output:
    cur_feats = matching_feats[:, 0] is non-contiguous for B > 1, src_feats = matching_feats[:, 1:]
    (experiment_modules/depth_model.py:242-243)."""
    g = torch.Generator().manual_seed(seed)
    feats = torch.randn(B, 1 + K, C, H, W, generator=g)
    return feats.to(dtype)


@pytest.mark.parametrize("kind", ["dot", "mlp"])
def test_backward_with_strided_views_of_one_encoder_output(kind):
    """ADVICE r1 (high): the saved tensors of the autograd Functions must be the dense copies the
    forward kernel read, not the caller's strided views.  B = 2, cur = feats[:, 0]."""
    B, K, C, H, W, D = 2, 7 if kind == "mlp" else 3, 16, 12, 16, 4
    t = make_tuple(B, K, H, W, channels=C, seed=101)
    feats_cpu = _feats_like_the_reference_caller(B, K, C, H, W, 102).requires_grad_(True)
    sd = mlp_state(K, C, seed=3) if kind == "mlp" else None
    g = torch.Generator().manual_seed(103)
    gcost = torch.randn(B, D, H, W, generator=g)
    # CPU autograd through the oracle, fp64 (see DESIGN §2: LeakyReLU kinks)
    tc = {k: (v.double() if torch.is_tensor(v) else v) for k, v in t.items()}
    f64 = feats_cpu.detach().double().requires_grad_(True)
    tc["cur_feats"], tc["src_feats"] = f64[:, 0], f64[:, 1:]
    if kind == "dot":
        oc, *_ = O.forward_dot(**tc, num_depth_bins=D)
    else:
        w64 = tuple(x.double() for x in O.mlp_weights_from_state_dict(sd))
        oc, *_ = O.forward_mlp(**tc, weights=w64, num_depth_bins=D)
    (oc * gcost.double()).sum().backward()
    # GPU: the same views of one leaf tensor
    d = to_device(t, "cuda")
    fg = feats_cpu.detach().cuda().requires_grad_(True)
    d["cur_feats"], d["src_feats"] = fg[:, 0], fg[:, 1:]
    assert not d["cur_feats"].is_contiguous()
    m = make_manager(kind, K, C, H, W, D, sd).train()
    cost, *_ = m(**d)
    (cost * gcost.cuda()).sum().backward()
    ref = f64.grad
    _assert_grad_close(fg.grad, ref, 1e-4)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("kind", ["dot", "mlp"])
def test_autocast_half_inputs_forward_and_backward(kind, dtype):
    """Training at precision=16 (reference train.py:132): under torch.autocast the matching
    features arrive in fp16 / bf16 and carry grad (modules/cost_volume.py:208,597 cast the grid
    with type_as(src_feats)).  The kernels upcast, compute in fp32 and return gradients in the
    inputs' dtype.  Compared with fp64 autograd through the oracle ON THE SAME (rounded) inputs."""
    B, K, C, H, W, D = 2, 7 if kind == "mlp" else 2, 16, 10, 14, 4
    t = make_tuple(B, K, H, W, channels=C, seed=111)
    feats = _feats_like_the_reference_caller(B, K, C, H, W, 112, dtype)
    sd = mlp_state(K, C, seed=4) if kind == "mlp" else None
    g = torch.Generator().manual_seed(113)
    gcost = torch.randn(B, D, H, W, generator=g)
    tc = {k: (v.double() if torch.is_tensor(v) else v) for k, v in t.items()}
    f64 = feats.double().requires_grad_(True)               # exactly the values the GPU upcasts
    tc["cur_feats"], tc["src_feats"] = f64[:, 0], f64[:, 1:]
    if kind == "dot":
        oc, *_ = O.forward_dot(**tc, num_depth_bins=D)
    else:
        oc, *_ = O.forward_mlp(**tc, weights=tuple(x.double() for x in O.mlp_weights_from_state_dict(sd)),
                               num_depth_bins=D)
    (oc * gcost.double()).sum().backward()
    d = to_device(t, "cuda")
    fg = feats.cuda().requires_grad_(True)
    d["cur_feats"], d["src_feats"] = fg[:, 0], fg[:, 1:]
    m = make_manager(kind, K, C, H, W, D, sd).train()
    with torch.autocast("cuda", dtype=dtype):
        cost, lowest, planes, mask = m(**d)
    assert cost.dtype == torch.float32 and cost.requires_grad
    assert_cost_close(kind, cost.detach(), oc.detach().float())
    (cost * gcost.cuda()).sum().backward()
    assert fg.grad.dtype == dtype
    ref = f64.grad
    eps = 2.0 ** -10 if dtype == torch.float16 else 2.0 ** -7   # the gradient is rounded to the input dtype
    _assert_grad_close(fg.grad, ref, eps)
    # the no-grad (validation) path takes half inputs too (ADVICE r1, medium)
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
        c2, *_ = m.eval()(**{k: (v.detach() if torch.is_tensor(v) else v) for k, v in d.items()})
    assert torch.equal(c2, cost.detach())


def test_per_frame_depth_ranges():
    """min_depth / max_depth of shape (B,1,1,1): generate_depth_planes broadcasts a per-frame range
    (reference modules/cost_volume.py:124-127)."""
    B, K, H, W, D = 3, 2, 12, 16, 6
    t = make_tuple(B, K, H, W, seed=121)
    t["min_depth"] = torch.tensor([0.25, 0.5, 0.3]).view(B, 1, 1, 1)
    t["max_depth"] = torch.tensor([5.0, 8.0, 2.0]).view(B, 1, 1, 1)
    (cost, lowest, planes, _), _ = run_gpu("dot", t, D)
    oc, ol, op, _ = O.forward_dot(**t, num_depth_bins=D)
    assert torch.allclose(planes.cpu(), op, rtol=3e-7, atol=0)
    assert_cost_close("dot", cost, oc, what="per-frame ranges")
