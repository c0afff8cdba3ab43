"""Coverage of what the other parity tests hold fixed.

1. Per-frame camera data.  `make_tuple` gives every view of every frame the same intrinsics and
   one depth range; a kernel or the prep pass that read frame 0's `cur_invK`, view 0's `K` or
   frame 0's planes for the whole batch would pass every test built on it.  Here every
   (frame, view) has its own intrinsics and every frame its own `cur_invK` and depth range, at
   every compile-time map size of the sweeps (`COMPILE_TIME_MAP_SIZES`) and at one odd size that
   takes the generic instantiations, against the fp32 and fp64 oracle.
2. Batch-permutation equivariance: reversing the frames reverses the outputs, bit for bit.
3. The same camera cases on the CPU tier (host emulation, tests/emu) at tiny sizes.
4. The cache of the tensor-core kernel's packed weight image
   (`FeatureVolumeManager._attach_packed_image`): reused while the MLP parameters are unchanged,
   re-packed when they change — also for fp16 weights and under `inference_mode`.
5. An inventory guard: the compile-time size arms in the kernel sources are exactly
   `COMPILE_TIME_MAP_SIZES`, so a new instantiation cannot land without the cases of 1."""
import re
from pathlib import Path

import pytest
import torch
from torch import nn

import simplerecon_b200 as S
from oracle import costvolume_oracle as O
from simplerecon_b200 import _native
from simplerecon_b200.synthetic import make_tuple, matching_intrinsics, mlp_state, to_device
from tests.parity import assert_cost_close, assert_lowest_close, assert_mask_close
from tests.test_emu_python_stack import emulated  # noqa: F401  (fixture)
from tests.test_zzz_gpu_mlp_backward import _grad_close, _oracle_grads, _rel

CSRC = Path(__file__).resolve().parents[1] / "simplerecon_b200" / "csrc"

# (H, W) feature maps with their own instantiations of the tensor-core MLP sweep (SRCV_TC_SIZES in
# srcv_mlp_tc.cu) and of the chunk-planar dot sweep (SRCV_SIZED in srcv_dot.cu): 640x480, 512x384
# and 256x192 frames.  Any other size runs the generic <0, 0> instantiations.
COMPILE_TIME_MAP_SIZES = [(120, 160), (96, 128), (48, 64)]
GENERIC_MAP_SIZE = (37, 53)
PLANE_MODES = ["range", "per_pixel"]
K, C = 7, 16                      # the hero layout: every kind below runs on the same inputs

# kind -> (variant to force, what _native.last_variant() must then report, oracle kind)
KINDS = {
    "tc": (_native.VARIANT_FAST, "mlp_tc_tcgen05_f16x3", "mlp"),
    "mlp_generic": (_native.VARIANT_GENERIC, "mlp_generic_fp32", "mlp"),
    "dot": (_native.VARIANT_FAST, "dot_fast_c4planar", "dot"),
}
SD = mlp_state(K, C, seed=5)


@pytest.fixture()
def gpu(cuda_device):
    yield "cuda"
    _native.set_variant(_native.VARIANT_AUTO)


@pytest.fixture(params=[pytest.param("cuda", marks=pytest.mark.gpu), "emulated"])
def device(request):
    """The B200, or the host emulation of the same kernel sources driven through the same
    Python layer (tests/test_emu_python_stack.py)."""
    if request.param == "cuda":
        request.getfixturevalue("cuda_device")
        yield "cuda"
        _native.set_variant(_native.VARIANT_AUTO)
    else:
        request.getfixturevalue("emulated")
        yield "cpu"


def per_frame_cameras(t, seed):
    """`t` (a `make_tuple` result) with camera data that differs between frames and views: every
    (frame, view) its own `src_Ks` (fx, fy scaled independently by up to +-15 %, cx, cy moved by
    up to 2 pixels), every frame its own `cur_invK` (the inverse of another such K) and its own
    `min_depth` / `max_depth` of shape (B,1,1,1)."""
    B, Kv, _, H, W = t["src_feats"].shape
    g = torch.Generator().manual_seed(seed)
    u = lambda *s: 2 * torch.rand(*s, generator=g, dtype=torch.float64) - 1          # U(-1, 1)

    def jittered(n):
        Ks = matching_intrinsics(H, W).repeat(n, 1, 1)       # bottom row stays [0, 0, 0, 1]
        Ks[:, 0, 0] *= 1 + 0.15 * u(n)
        Ks[:, 1, 1] *= 1 + 0.15 * u(n)
        Ks[:, 0, 2] += 2.0 * u(n)
        Ks[:, 1, 2] += 2.0 * u(n)
        return Ks

    t = dict(t)
    t["src_Ks"] = jittered(B * Kv).reshape(B, Kv, 4, 4).float().contiguous()
    t["cur_invK"] = torch.linalg.inv(jittered(B)).float().contiguous()
    t["min_depth"] = (0.2 + 0.4 * torch.rand(B, generator=g)).view(B, 1, 1, 1)
    t["max_depth"] = (2.5 + 4.0 * torch.rand(B, generator=g)).view(B, 1, 1, 1)
    return t


def camera_case(B, H, W, D, planes_mode, seed):
    """Inputs with per-frame cameras, and per-pixel planes drawn inside each frame's range."""
    t = per_frame_cameras(make_tuple(B, K, H, W, channels=C, seed=seed), seed + 1)
    planes = None
    if planes_mode == "per_pixel":
        g = torch.Generator().manual_seed(seed + 2)
        planes = t["min_depth"] + (t["max_depth"] - t["min_depth"]) * torch.rand(B, D, H, W, generator=g)
    return t, planes


def make_manager(kind, H, W, D, device):
    if kind == "dot":
        m = S.CostVolumeManager(H, W, num_depth_bins=D)
    else:
        m = S.FeatureVolumeManager(H, W, num_depth_bins=D, mlp_channels=[0, 128, 128, 1], matching_dim_size=C,
                                   num_source_views=K)
        m.load_state_dict({**m.state_dict(), **SD})
    return m.to(device)


def run(kind, t, D, planes, device):
    """One inference call with the variant of `kind` forced; outputs on the CPU."""
    H, W = t["src_feats"].shape[-2:]
    m = make_manager(kind, H, W, D, device).eval()
    _native.set_variant(KINDS[kind][0])
    with torch.inference_mode():
        out = m(**to_device(t, device), depth_planes_bdhw=None if planes is None else planes.to(device),
                return_mask=True)
    used = _native.last_variant()
    assert used == KINDS[kind][1], used
    return [None if x is None else x.cpu() for x in out]


def oracle(kind, t, D, planes, dtype):
    tt = {k: v.to(dtype) for k, v in t.items()}
    dp = None if planes is None else planes.to(dtype)
    if KINDS[kind][2] == "dot":
        return O.forward_dot(**tt, num_depth_bins=D, depth_planes_bdhw=dp)
    w = tuple(x.to(dtype) for x in O.mlp_weights_from_state_dict(SD))
    return O.forward_mlp(**tt, weights=w, num_depth_bins=D, depth_planes_bdhw=dp, return_mask=True)


def check_forward(kind, B, H, W, D, planes_mode, device, seed):
    t, planes = camera_case(B, H, W, D, planes_mode, seed)
    cost, lowest, pl, mask = run(kind, t, D, planes, device)
    oc, _, op, om = oracle(kind, t, D, planes, torch.float32)
    oc64 = oracle(kind, t, D, planes, torch.float64)[0]
    okind, what = KINDS[kind][2], f"{kind} {H}x{W} {planes_mode}"
    if planes is None:
        assert torch.allclose(pl, op, rtol=3e-7, atol=0), what          # each frame its own range
    assert_cost_close(okind, cost, oc, oc64, what=what)
    assert_lowest_close(okind, lowest, pl, oc, what=what)
    if okind == "mlp":
        assert_mask_close(mask, om, what=what)
    else:
        assert mask is None


FORWARD_CASES = ([("tc", H, W) for H, W in [*COMPILE_TIME_MAP_SIZES, GENERIC_MAP_SIZE]]
                 + [("dot", H, W) for H, W in [*COMPILE_TIME_MAP_SIZES, GENERIC_MAP_SIZE]]
                 + [("mlp_generic", *GENERIC_MAP_SIZE)])


@pytest.mark.gpu
@pytest.mark.parametrize("planes_mode", PLANE_MODES)
@pytest.mark.parametrize("kind,H,W", FORWARD_CASES)
def test_per_frame_cameras_forward(gpu, kind, H, W, planes_mode):
    """Every forward arm (kernel x compile-time size x plane mode) on per-frame cameras, B = 2."""
    check_forward(kind, 2, H, W, 8, planes_mode, "cuda", seed=200 + H)


@pytest.mark.parametrize("planes_mode", PLANE_MODES)
@pytest.mark.parametrize("kind", list(KINDS))
def test_per_frame_cameras_forward_emulated(emulated, kind, planes_mode):
    """The same on the CPU tier: the prep pass and the kernels' per-frame / per-view indexing."""
    check_forward(kind, 3, 9, 13, 4, planes_mode, "cpu", seed=300)


@pytest.mark.parametrize("planes_mode", PLANE_MODES)
@pytest.mark.parametrize("kind", ["dot", "mlp"])
def test_per_frame_cameras_backward(device, kind, planes_mode):
    """Both backward kernels on per-frame cameras against fp64 autograd through the oracle
    (tolerance of tests/test_zzz_gpu_mlp_backward.py)."""
    B, H, W, D = 2, 11, 14, 3
    t, planes = camera_case(B, H, W, D, planes_mode, seed=400)
    gcost = torch.randn(B, D, H, W, generator=torch.Generator().manual_seed(401))
    m = make_manager(kind, H, W, D, device).train()
    d = to_device(t, device)
    d["cur_feats"] = d["cur_feats"].clone().requires_grad_(True)
    d["src_feats"] = d["src_feats"].clone().requires_grad_(True)
    cost, *_ = m(**d, depth_planes_bdhw=None if planes is None else planes.to(device))
    (cost * gcost.to(device)).sum().backward()
    if kind == "dot":
        assert _native.last_variant() == "dot_backward_atomic"
        tc = {k: v.double() for k, v in t.items()}
        tc["cur_feats"] = tc["cur_feats"].requires_grad_(True)
        tc["src_feats"] = tc["src_feats"].requires_grad_(True)
        oc, *_ = O.forward_dot(**tc, num_depth_bins=D, depth_planes_bdhw=None if planes is None else planes.double())
        (oc * gcost.double()).sum().backward()
        ours, ref = [d["cur_feats"].grad, d["src_feats"].grad], [tc["cur_feats"].grad, tc["src_feats"].grad]
        names = ("cur", "src")
    else:
        assert _native.last_variant() == "mlp_backward_fp32_recompute"
        params = [p for i in (0, 2, 4) for p in (m.mlp.net[i].weight, m.mlp.net[i].bias)]
        oc, ref = _oracle_grads(t, params, D, gcost, planes)
        ours = [d["cur_feats"].grad, d["src_feats"].grad] + [p.grad for p in params]
        names = ("cur", "src", "w1", "b1", "w2", "b2", "w3", "b3")
    assert_cost_close(kind, cost, oc.detach().float(), what=f"{kind} training forward")
    for name, o, r in zip(names, ours, ref):
        assert o is not None and tuple(o.shape) == tuple(r.shape), name
        assert _grad_close(o, r), f"grad {name}: rel err {_rel(o, r):.2e}"


@pytest.mark.parametrize("kind", list(KINDS))
def test_batch_permutation_equivariance(device, kind):
    """Reversing the frame order of every per-frame input (features, poses, intrinsics, depth
    ranges, per-pixel planes) reverses cost, lowest and mask bit for bit.  Frames that share no
    camera data make a kernel that mixes frames up visible without any oracle."""
    B, H, W, D = (3, 96, 128, 8) if device == "cuda" else (3, 9, 13, 4)
    for planes_mode in PLANE_MODES:
        t, planes = camera_case(B, H, W, D, planes_mode, seed=500)
        rev = {k: v.flip(0) for k, v in t.items()}
        out = run(kind, t, D, planes, device)
        out_r = run(kind, rev, D, None if planes is None else planes.flip(0), device)
        for name, a, b in zip(("cost", "lowest", "planes", "mask"), out, out_r):
            if a is None:
                assert b is None
                continue
            assert torch.equal(b, a.flip(0)), f"{kind} {planes_mode}: {name} of the reversed batch"


# --------------------------------------------------------------------------- #
# the tensor-core kernel's packed weight image                                #
# --------------------------------------------------------------------------- #
CACHE_H, CACHE_W, CACHE_D = 12, 16, 4


def _cache_manager(device, seed):
    m = S.FeatureVolumeManager(CACHE_H, CACHE_W, num_depth_bins=CACHE_D, mlp_channels=[0, 128, 128, 1],
                               matching_dim_size=C, num_source_views=K)
    m.load_state_dict({**m.state_dict(), **mlp_state(K, C, seed=seed)})
    return m.to(device).eval()


def _cache_inputs(device):
    return to_device(make_tuple(1, K, CACHE_H, CACHE_W, channels=C, seed=600), device)


def _params(m):
    return [p for i in (0, 2, 4) for p in (m.mlp.net[i].weight, m.mlp.net[i].bias)]


def _two_calls_share_one_image(m, t):
    """Two calls with unchanged weights: the second one reuses the first one's image (same tensor,
    one kernel launch fewer: no pack)."""
    n0 = _native.launch_count()
    c1 = m(**t)[0]
    n1 = _native.launch_count()
    image = m.__dict__["_srcv_packed"][1]
    c2 = m(**t)[0]
    n2 = _native.launch_count()
    assert _native.last_variant() == "mlp_tc_tcgen05_f16x3"
    assert m.__dict__["_srcv_packed"][1] is image, "unchanged weights were re-packed"
    assert n2 - n1 == (n1 - n0) - 1, (n1 - n0, n2 - n1)
    assert torch.equal(c1, c2)
    return c1


def _assert_matches_oracle(m, t, cost, what):
    tc = to_device(t, "cpu")
    w = tuple(p.detach().float().cpu() for p in _params(m))       # the values the kernel upcasts
    oc, *_ = O.forward_mlp(**tc, weights=w, num_depth_bins=CACHE_D)
    assert_cost_close("mlp", cost, oc, what=what)


def test_weight_image_cache_half_weights_no_grad(device):
    """fp16 weights (`model.half()`): `_f32c` upcasts them into fresh fp32 tensors at version 0 on
    every call, so a key built from those copies either misses every call or — when the
    allocator hands back the same addresses — misses a `load_state_dict`.  Keyed on the
    parameters, the image is reused while they are unchanged and re-packed when they change."""
    t = _cache_inputs(device)
    m = _cache_manager(device, seed=1)
    m.mlp.half()
    with torch.no_grad():
        c1 = _two_calls_share_one_image(m, t)
        m.load_state_dict({**m.state_dict(), **mlp_state(K, C, seed=2)})
        c3 = m(**t)[0]
    assert not torch.equal(c3, c1)
    _assert_matches_oracle(m, t, c3, "fp16 weights after load_state_dict")


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16], ids=["fp32", "fp16"])
def test_weight_image_cache_under_inference_mode(device, dtype):
    """Under `inference_mode` the fp32 copies `_f32c` makes of fp16 weights are inference tensors
    without a version counter; the parameters are not, so the image is still reused while they
    are unchanged."""
    t = _cache_inputs(device)
    m = _cache_manager(device, seed=3)
    m.mlp.to(dtype)
    with torch.inference_mode():
        c1 = _two_calls_share_one_image(m, t)
    _assert_matches_oracle(m, t, c1, f"inference_mode {dtype}")


def test_weight_image_cache_sees_optimizer_steps_and_new_parameters(device):
    t = _cache_inputs(device)
    m = _cache_manager(device, seed=4)
    with torch.no_grad():
        c1 = m(**t)[0]
    g = torch.Generator().manual_seed(601)
    for p in m.mlp.parameters():
        p.grad = (0.05 * torch.randn(p.shape, generator=g)).to(device)
    torch.optim.SGD(m.mlp.parameters(), lr=1.0).step()
    with torch.no_grad():
        c2 = m(**t)[0]
    assert not torch.equal(c2, c1)
    _assert_matches_oracle(m, t, c2, "after an optimizer step")
    w = mlp_state(K, C, seed=5)["mlp.net.2.weight"]
    m.mlp.net[2].weight = nn.Parameter(w.to(device))
    with torch.no_grad():
        c3 = m(**t)[0]
    assert not torch.equal(c3, c2)
    _assert_matches_oracle(m, t, c3, "after replacing a Parameter")


# --------------------------------------------------------------------------- #
# inventory guard                                                             #
# --------------------------------------------------------------------------- #
def test_compile_time_map_sizes_are_all_exercised():
    """The size arms of the tensor-core launcher (SRCV_TC_SIZES) and of the chunk-planar dot
    launcher (SRCV_SIZED) are exactly COMPILE_TIME_MAP_SIZES, which the camera cases above run in
    both plane modes.

    Exempt: the dot sweep's 32-wide warp tile (`SRCV_DOT_TILE_W=32`) instantiates the same sizes
    with another tile shape.  It is a tuning knob read once per process, so a test process cannot
    switch to it; the suite runs the default 16-wide tile."""
    tc = (CSRC / "srcv_mlp_tc.cu").read_text()
    body = re.search(r"#define SRCV_TC_SIZES\(PP\)((?:[^\n]*\\\n)*[^\n]*)", tc)
    assert body, "SRCV_TC_SIZES not found in srcv_mlp_tc.cu"
    tc_sizes = {(int(h), int(w)) for w, h in re.findall(r"s\.W == (\d+) && s\.H == (\d+)", body.group(1))}
    dot = (CSRC / "srcv_dot.cu").read_text()
    dot_sizes = {(int(h), int(w)) for w, h in re.findall(r"^\s*SRCV_SIZED\((\d+),\s*(\d+)\)", dot, re.M)}
    assert tc_sizes and dot_sizes
    assert tc_sizes | dot_sizes == set(COMPILE_TIME_MAP_SIZES), (tc_sizes, dot_sizes)
    assert GENERIC_MAP_SIZE not in tc_sizes | dot_sizes
