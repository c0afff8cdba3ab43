"""CPU: the oracle against the reference classes' outputs on randomised shapes, as recorded from the
unmodified reference by tests/golden/make_golden_reference.py."""
import pytest
import torch

from oracle import costvolume_oracle as O
from simplerecon_b200.synthetic import make_tuple, mlp_state
from tests.parity import assert_cost_close, load_reference_outputs


@pytest.fixture(scope="module")
def ref():
    return load_reference_outputs("cost_volume")


@pytest.mark.parametrize("B,K,H,W,D,seed", [(2, 3, 20, 28, 6, 1), (1, 7, 15, 21, 5, 2), (3, 1, 8, 8, 3, 3)])
def test_dot_matches_live_reference(ref, B, K, H, W, D, seed):
    t = make_tuple(B, K, H, W, seed=seed)
    rc, rl, rp = ref[f"dot{seed}_cost"], ref[f"dot{seed}_lowest"], ref[f"dot{seed}_planes"]
    oc, ol, op, om = O.forward_dot(**t, num_depth_bins=D, sampler="aten")
    assert torch.equal(op.contiguous(), rp)
    assert (oc - rc).abs().max().item() <= 2e-6 * float(rc.abs().max())
    assert torch.equal(ol, rl) and om is None
    oc2, *_ = O.forward_dot(**t, num_depth_bins=D, sampler="explicit")
    assert_cost_close("dot", oc2, rc)


@pytest.mark.parametrize("B,K,H,W,D,seed", [(2, 3, 12, 16, 4, 4), (1, 7, 10, 14, 3, 5)])
def test_mlp_matches_live_reference_slow_and_fast(ref, B, K, H, W, D, seed):
    t = make_tuple(B, K, H, W, seed=seed)
    sd = mlp_state(K, 16, seed=seed)
    rc, rl, rm = ref[f"mlp{seed}_cost"], ref[f"mlp{seed}_lowest"], ref[f"mlp{seed}_mask"]
    fc, fm = ref[f"mlp{seed}_fast_cost"], ref[f"mlp{seed}_fast_mask"]
    w = O.mlp_weights_from_state_dict(sd)
    oc, ol, op, om = O.forward_mlp(**t, weights=w, num_depth_bins=D, return_mask=True, sampler="aten")
    for c in (rc, fc):
        assert (oc - c).abs().max().item() <= 5e-6 * float(c.abs().max()) + 1e-7
    assert torch.equal(om, rm) and torch.equal(om, fm)
    assert torch.equal(ol, rl)


def test_pose_distance_matches_live_reference(ref):
    t = make_tuple(3, 5, 4, 4, seed=9)
    comb, r, tm = O.pose_distance(t["src_poses"])
    assert torch.allclose(comb.reshape(-1), ref["pose_combined"]) and torch.allclose(r.reshape(-1), ref["pose_r"])
    assert torch.allclose(tm.reshape(-1), ref["pose_t"])


def test_dot_gradients_match_live_reference_autograd(ref):
    """The oracle's autograd (which the GPU backward kernel is tested against) equals autograd
    through the reference's own CostVolumeManager for the two feature inputs."""
    B, K, H, W, D = 2, 3, 10, 14, 4
    t = make_tuple(B, K, H, W, seed=17)
    g = torch.randn(B, D, H, W, generator=torch.Generator().manual_seed(1))
    t["cur_feats"].requires_grad_(True)
    t["src_feats"].requires_grad_(True)
    cost, *_ = O.forward_dot(**t, num_depth_bins=D, sampler="explicit")
    (cost * g).sum().backward()
    for a, b in ((ref["grad_cur_feats"], t["cur_feats"].grad), (ref["grad_src_feats"], t["src_feats"].grad)):
        assert (a - b).abs().max().item() <= 2e-5 * float(a.abs().max()) + 1e-6


def test_per_frame_depth_range_matches_live_reference(ref):
    """(B,1,1,1) min/max depth: the reference's generate_depth_planes broadcasts one range per
    frame (modules/cost_volume.py:124-127); the oracle restates that."""
    B, K, H, W, D = 3, 2, 10, 12, 5
    t = make_tuple(B, K, H, W, seed=31)
    t["min_depth"] = torch.tensor([0.25, 0.5, 0.3]).view(B, 1, 1, 1)
    t["max_depth"] = torch.tensor([5.0, 8.0, 2.0]).view(B, 1, 1, 1)
    rc, rl, rp = ref["range_cost"], ref["range_lowest"], ref["range_planes"]
    oc, ol, op, _ = O.forward_dot(**t, num_depth_bins=D, sampler="aten")
    assert torch.equal(op.contiguous(), rp)
    assert (oc - rc).abs().max().item() <= 2e-6 * float(rc.abs().max()) and torch.equal(ol, rl)
