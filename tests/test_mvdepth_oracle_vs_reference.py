"""CPU: the multi-view depth-loss oracle against the reference's ``losses.MVDepthLoss``
(losses.py:79-208), value and gradient, as recorded from the unmodified reference by
tests/golden/make_golden_reference.py."""
import pytest
import torch

from oracle import mvdepth_oracle as M
from simplerecon_b200.synthetic import make_mvloss_batch
from tests.parity import load_reference_outputs


@pytest.fixture(scope="module")
def ref():
    return load_reference_outputs("mvdepth_loss")


@pytest.mark.parametrize("seed,B,K,hw", [(0, 2, 3, (24, 32)), (1, 1, 7, (30, 40)), (2, 3, 2, (17, 23))])
def test_loss_and_gradient_match_live_reference(ref, seed, B, K, hw):
    t = make_mvloss_batch(seed, B, K, *hw)
    l_ref, g_ref = ref[f"s{seed}_loss"], ref[f"s{seed}_grad"]
    p_ora = t["depth_pred_b1hw"].clone().requires_grad_(True)
    l_ora = M.mv_depth_loss(**{**t, "depth_pred_b1hw": p_ora})
    assert torch.isfinite(l_ref) and l_ref.item() > 1e-3
    assert l_ora.item() == l_ref.item()                      # same ops in the same order: bit-equal
    l_ora.backward()
    assert torch.equal(g_ref, p_ora.grad) and g_ref.abs().sum() > 0


def test_valid_mask_matches_live_reference(ref):
    t = make_mvloss_batch(5, 2, 2, 20, 28)
    a = (t["cur_depth_b1hw"], t["src_depth_bk1hw"][:, 1], t["cur_invK_b44"], t["src_K_bk44"][:, 1],
         t["cur_world_T_cam_b44"], t["src_cam_T_world_bk44"][:, 1])
    vm_r, s_r = ref["valid_mask"], ref["valid_mask_src"]
    vm_o, s_o = M.valid_mask(*a)
    assert torch.equal(vm_r, vm_o) and torch.equal(s_r, s_o)
    assert 0.05 < vm_r.float().mean().item() < 0.98


def test_prediction_behind_a_source_camera_is_dropped_from_the_mean_but_poisons_its_gradient(ref):
    """z_pred <= 0 makes log() NaN / -inf: nanmean drops NaN terms from the VALUE (losses.py:173); what the
    reference's autograd does with such a pixel is recorded here (the kernel follows it)."""
    t = make_mvloss_batch(7, 1, 2, 16, 20)
    vm, _ = M.valid_mask(t["cur_depth_b1hw"], t["src_depth_bk1hw"][:, 0], t["cur_invK_b44"], t["src_K_bk44"][:, 0],
                         t["cur_world_T_cam_b44"], t["src_cam_T_world_bk44"][:, 0])
    idx = vm.flatten().nonzero()[0].item()
    p = t["depth_pred_b1hw"].clone()
    p.view(-1)[idx] = -50.0                        # a (nonsensical) negative prediction at a valid pixel
    p_ora = p.clone().requires_grad_(True)
    l_ref, g_ref = ref["behind_loss"], ref["behind_grad"]
    l_ora = M.mv_depth_loss(**{**t, "depth_pred_b1hw": p_ora})
    assert torch.isfinite(l_ref) and l_ora.item() == l_ref.item()
    l_ora.backward()
    assert torch.equal(torch.isnan(g_ref), torch.isnan(p_ora.grad))
    print("grad at the behind-camera pixel:", g_ref.view(-1)[idx].item(), "NaNs:", torch.isnan(g_ref).sum().item())
