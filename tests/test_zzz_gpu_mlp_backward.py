"""GPU: training path of the metadata-MLP managers — fused forward + `srcv_mlp_backward_f32`
(recompute kernel) against CPU autograd through the oracle, i.e. the composite the reference
differentiates (modules/cost_volume.py:451-736, modules/networks.py:129-147).

The same kernel source is checked on the CPU tier by tests/test_emu_kernels.py /
tests/test_emu_python_stack.py (host emulation); this file is its run on real hardware.
(File name sorts last on purpose: written after the round-1 GPU budget was spent, so its
first execution is the round-end GPU tier.)

Tolerance: gradients are fp32 sums of up to D*H*W*K atomically accumulated terms; the order
differs between runs and from the CPU: rel. 1e-4 of the largest entry of the fp64 oracle gradient.
Why fp64: LeakyReLU has a kink at 0 and a pre-activation of ~1e-7 takes either sign depending on
the fp32 summation order.  scripts/emu_fuzz.py sees it in ~8 % of random cases — almost always on
the side of the fp32 composite (the reference's own arithmetic) while the kernel matches the fp64
gradients on every entry; rarely on the kernel's side, where a bounded set of entries moves by up to
~1e-2 of the maximum.  That rare case passes if the relative L2 error stays below 2e-2; an
indexing or protocol bug does not."""
import pytest
import torch

import simplerecon_b200 as S
import simplerecon_b200.torch_ops  # noqa: F401
from oracle import costvolume_oracle as O
from simplerecon_b200 import _native
from simplerecon_b200.synthetic import make_tuple, mlp_state, to_device
from tests.parity import assert_cost_close

pytestmark = pytest.mark.gpu
RTOL = 1e-4


def _rel(a, b):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    return ((a - b).abs().max() / (b.abs().max() + 1e-30)).item()


def _grad_close(a, b):
    if _rel(a, b) < RTOL:
        return True
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    return ((a - b).norm() / (b.norm() + 1e-30)).item() < 2e-2      # LeakyReLU kink flip on our side, see the docstring


def _manager(K, C, H, W, D, hidden=(128, 128), fast=False):
    cls = S.FastFeatureVolumeManager if fast else S.FeatureVolumeManager
    m = cls(H, W, num_depth_bins=D, mlp_channels=[0, *hidden, 1], matching_dim_size=C, num_source_views=K)
    m.load_state_dict({**m.state_dict(), **mlp_state(views=K, channels=C, hidden=hidden, seed=1)})
    return m.cuda().train()


def _oracle_grads(t, wts, D, gcost, planes, dtype=torch.float64):
    """Autograd through the oracle in fp64 (see the module docstring: the fp32 composite — the
    reference's own arithmetic — flips LeakyReLU kinks more often than the kernel does)."""
    tc = {k: (v.to(dtype) if torch.is_tensor(v) else v) for k, v in t.items()}
    tc["cur_feats"] = tc["cur_feats"].clone().requires_grad_(True)
    tc["src_feats"] = tc["src_feats"].clone().requires_grad_(True)
    wo = [w.detach().cpu().to(dtype).clone().requires_grad_(True) for w in wts]
    oc, *_ = O.forward_mlp(**tc, weights=tuple(wo), num_depth_bins=D,
                           depth_planes_bdhw=None if planes is None else planes.to(dtype))
    (oc * gcost.to(dtype)).sum().backward()
    return oc.detach(), [tc["cur_feats"].grad, tc["src_feats"].grad] + [w.grad for w in wo]


@pytest.mark.parametrize("B,K,C,H,W,D,hidden,per_pixel,fast", [
    (1, 7, 16, 16, 20, 4, (128, 128), False, False),   # hero layout: tcgen05 forward, fp32 recompute backward
    (2, 2, 8, 13, 17, 3, (128, 128), True, False),     # generic forward, per-pixel planes, ragged tiles
    (1, 3, 16, 12, 16, 5, (96, 64), False, True),      # narrow hidden layers, Fast manager class
    (1, 7, 16, 13, 17, 3, (128, 128), True, False),    # 202 input features per-pixel: backward <true, 13>
    (1, 3, 16, 12, 16, 4, (96, 64), True, False),      # 98 input features per-pixel: backward <true, 8>
    (1, 7, 16, 96, 128, 8, (128, 128), False, False),  # 512x384 frames: tcgen05 forward <false, 128, 96>
])
def test_hero_training_matches_oracle_autograd(cuda_device, B, K, C, H, W, D, hidden, per_pixel, fast):
    t = make_tuple(B, K, H, W, channels=C, seed=31)
    g = torch.Generator().manual_seed(32)
    gcost = torch.randn(B, D, H, W, generator=g)
    planes = (0.3 + 4.0 * torch.rand(B, D, H, W, generator=g)) if per_pixel else None
    m = _manager(K, C, H, W, D, hidden, fast)
    d = to_device(t, "cuda")
    d["cur_feats"] = d["cur_feats"].clone().requires_grad_(True)
    d["src_feats"] = d["src_feats"].clone().requires_grad_(True)
    cost, lowest, planes_ret, mask = m(**d, depth_planes_bdhw=planes.cuda() if per_pixel else None,
                                       return_mask=True)
    assert cost.requires_grad and not lowest.requires_grad and mask.dtype == torch.bool
    hero = (K, C, tuple(hidden)) == (7, 16, (128, 128))
    assert _native.last_variant() == ("mlp_tc_tcgen05_f16x3" if hero else "mlp_generic_fp32")
    (cost * gcost.cuda()).sum().backward()
    torch.cuda.synchronize()
    assert _native.last_variant() == "mlp_backward_fp32_recompute"
    params = [p for i in (0, 2, 4) for p in (m.mlp.net[i].weight, m.mlp.net[i].bias)]
    oc64, ref = _oracle_grads(t, params, D, gcost, planes)
    oc, *_ = O.forward_mlp(**t, weights=tuple(p.detach().cpu() for p in params), num_depth_bins=D,
                           depth_planes_bdhw=planes)
    assert_cost_close("mlp", cost, oc, oc64, what="hero training forward")
    ours = [d["cur_feats"].grad, d["src_feats"].grad] + [p.grad for p in params]
    for name, o, r in zip(("cur", "src", "w1", "b1", "w2", "b2", "w3", "b3"), ours, ref):
        assert o is not None and tuple(o.shape) == tuple(r.shape), name
        assert _grad_close(o, r), f"grad {name}: rel err {_rel(o, r):.2e}"
    # inference on the same manager still takes the plain fused path
    with torch.no_grad():
        c2, *_ = m(**{k: v.detach() for k, v in d.items()}, depth_planes_bdhw=planes.cuda() if per_pixel else None)
    assert not c2.requires_grad and torch.equal(c2, cost.detach())


def test_mlp_torch_op_autograd(cuda_device):
    B, K, C, H, W, D = 1, 2, 8, 10, 12, 3
    t = make_tuple(B, K, H, W, channels=C, seed=33)
    gcost = torch.randn(B, D, H, W, generator=torch.Generator().manual_seed(34))
    sd = mlp_state(views=K, channels=C, seed=1)
    wts = [sd[f"mlp.net.{i}.{n}"].cuda().requires_grad_(True) for i in (0, 2, 4) for n in ("weight", "bias")]
    planes_bd = torch.linspace(0.5, 4.0, D).repeat(B, 1)
    d = to_device(t, "cuda")
    cur = d["cur_feats"].clone().requires_grad_(True)
    src = d["src_feats"].clone().requires_grad_(True)
    cost, lowest, mask = torch.ops.b200cv.mlp_forward(cur, src, d["src_extrinsics"], d["src_poses"], d["src_Ks"],
                                                      d["cur_invK"], planes_bd.cuda(), *wts)
    assert cost.requires_grad and not lowest.requires_grad and mask.dtype == torch.bool
    (cost * gcost.cuda()).sum().backward()
    torch.cuda.synchronize()
    _, ref = _oracle_grads(t, wts, D, gcost, planes_bd.view(B, D, 1, 1).expand(B, D, H, W))
    for name, o, r in zip(("cur", "src", "w1", "b1", "w2", "b2", "w3", "b3"), [cur.grad, src.grad] + [w.grad for w in wts], ref):
        assert _grad_close(o, r), f"grad {name}: rel err {_rel(o, r):.2e}"
