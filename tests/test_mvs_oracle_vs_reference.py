"""CPU: the multi-view consistency oracle against the reference's process_depth
(tools/torch_point_cloud_fusion.py), as recorded from the unmodified reference by
tests/golden/make_golden_reference.py."""
import numpy as np
import pytest
import torch

from oracle import mvs_oracle as M
from simplerecon_b200.synthetic import make_mvs_scene
from tests.parity import load_reference_outputs


@pytest.mark.parametrize("seed,n,hw", [(1, 5, (24, 32)), (2, 9, (30, 40))])
def test_process_depth_matches_live_reference(seed, n, hw):
    R = load_reference_outputs("mvs")
    sc = make_mvs_scene(seed=seed, frames=n, height=hw[0], width=hw[1])
    depths, images, P, K = sc["depths"], sc["images"], sc["cam_T_world"], sc["K"]
    for ref_idx in (0, n // 2):
        src = torch.arange(n) != ref_idx
        rp, rrgb, rvalid = (R[f"s{seed}_r{ref_idx}_{k}"].numpy() for k in ("points", "rgb", "valid"))
        pts_avg, n_valid, valid = M.process_depth_dense(depths[ref_idx], depths[src], P[ref_idx], P[src],
                                                        K[ref_idx], K[src], 0.1, 3)
        assert np.array_equal(valid.numpy(), rvalid) and 0.05 < valid.float().mean().item() < 0.99
        op, orgb = M.compact(pts_avg, valid, images[ref_idx])
        assert np.allclose(op.numpy(), rp, rtol=0, atol=1e-6) and np.array_equal(orgb.numpy(), rrgb)
