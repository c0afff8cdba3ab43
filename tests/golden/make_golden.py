"""Generates the golden vectors in tests/golden/*.npz from the UNMODIFIED reference.

Run in the build container (needs /root/reference):

    python tests/golden/make_golden.py

Every case stores the exact inputs, the reference classes' fp32 outputs and — for
error budgeting — the outputs of the same classes evaluated in fp64
(``.double()``).  The reference holds no golden vectors of its own (SURVEY.md §4,
§8c); these files are the pin.  Inputs come from simplerecon_b200.synthetic
(seeded), edge cases are built explicitly below.
"""
from __future__ import annotations

import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from oracle.ref_import import load_reference  # noqa: E402
from simplerecon_b200.synthetic import make_tuple, mlp_state  # noqa: E402

OUT = Path(__file__).resolve().parent
INPUT_KEYS = ("cur_feats", "src_feats", "src_extrinsics", "src_poses", "src_Ks", "cur_invK",
              "min_depth", "max_depth")


def run_case(R, name, kind, tup, D, mlp_sd=None, depth_planes=None, return_mask=True):
    B, K, C, H, W = tup["src_feats"].shape
    kw = dict(tup)
    if depth_planes is not None:
        kw["depth_planes_bdhw"] = depth_planes
    if kind == "dot":
        mgr = R.CostVolumeManager(H, W, num_depth_bins=D)
    else:
        mgr = R.FeatureVolumeManager(H, W, num_depth_bins=D, mlp_channels=[0, 128, 128, 1],
                                     matching_dim_size=C, num_source_views=K)
        mgr.load_state_dict({**mgr.state_dict(), **mlp_sd})
    with torch.no_grad():
        cost, lowest, planes, mask = mgr(**kw, return_mask=return_mask)
        mgr64 = mgr.double()
        kw64 = {k: (v.double() if torch.is_tensor(v) else v) for k, v in kw.items()}
        cost64, lowest64, _, mask64 = mgr64(**kw64, return_mask=return_mask)
        if kind == "mlp":
            # the reference's own claim: fast == slow (cost_volume.py:750-756)
            fast = mgr.float().to_fast()
            fc, fl, _, fm = fast(**kw, return_mask=return_mask)
            assert (fc - cost).abs().max() < 1e-5 and bool((fm == mask).all())
    out = {k: tup[k].numpy() for k in INPUT_KEYS}
    out.update(kind=np.array(kind), D=np.array(D), ref_cost=cost.numpy(), ref_lowest=lowest.numpy(),
               ref_planes=planes[:, :, 0, 0].numpy() if depth_planes is None else planes.contiguous().numpy(),
               ref_cost64_minus_ref_cost=(cost64 - cost.double()).float().numpy(),  # keeps files < 1 MB
               ref_lowest64=lowest64.numpy())
    if depth_planes is not None:
        out["depth_planes_bdhw"] = depth_planes.contiguous().numpy()
    if mask is not None:
        out["ref_mask"] = mask.numpy()
    if mlp_sd is not None:
        out.update({k.replace(".", "_"): v.numpy() for k, v in mlp_sd.items()})
    np.savez_compressed(OUT / f"{name}.npz", **out)
    print(f"{name}: cost {tuple(cost.shape)} max|c|={cost.abs().max():.4f} "
          f"err32v64={float((cost.double() - cost64).abs().max()):.3e} "
          f"mask_mean={float(mask.float().mean()) if mask is not None else -1:.3f}")


def edge_tuple(seed=77):
    """K=3 views on an odd-sized map: view 0 ordinary; view 1 looks backwards
    (every plane point behind the camera -> mask 0 but features still sampled);
    view 2 translated so far sideways that all samples fall outside the frustum."""
    t = make_tuple(1, 3, 13, 17, seed=seed)
    E = t["src_extrinsics"].clone()
    E[0, 1] = torch.tensor([[-1., 0, 0, 0.05], [0, 1, 0, 0], [0, 0, -1, -0.1], [0, 0, 0, 1]])
    E[0, 2, :3, :3] = torch.eye(3)
    E[0, 2, :3, 3] = torch.tensor([40.0, 0.0, 0.0])
    t["src_extrinsics"] = E
    t["src_poses"] = torch.linalg.inv(E.double()).float()
    return t


def main():
    R = load_reference()
    torch.manual_seed(0)
    # BASELINE.json configs[0]: dot, 1+2 views, 256x192 -> 48x64, D=16, B=1
    run_case(R, "cfg0_dot_48x64_D16_K2", "dot", make_tuple(1, 2, 48, 64, seed=1234), 16)
    # hero mini: the BASELINE hero layout (K=7, C=16, F=202) on a small map
    run_case(R, "hero_mini_24x32_D8_K7", "mlp", make_tuple(1, 7, 24, 32, seed=4321), 8,
             mlp_sd=mlp_state(7, 16, seed=0))
    # dot with K=7 smooth features
    run_case(R, "dot_mini_24x32_D8_K7_smooth", "dot", make_tuple(2, 7, 24, 32, seed=99, smooth=True), 8)
    # edge cases: behind-camera view, out-of-frustum view, odd H/W, K=3
    et = edge_tuple()
    run_case(R, "edge_dot_13x17_D5_K3", "dot", et, 5)
    run_case(R, "edge_hero_13x17_D5_K3", "mlp", et, 5, mlp_sd=mlp_state(3, 16, seed=2))
    # D=1, K=1
    run_case(R, "k1_d1_hero_9x11", "mlp", make_tuple(2, 1, 9, 11, seed=5), 1, mlp_sd=mlp_state(1, 16, seed=3))
    # caller-supplied per-pixel depth hypotheses (modules/cost_volume.py:247, :297-299)
    t = make_tuple(1, 2, 12, 16, seed=6)
    g = torch.Generator().manual_seed(7)
    dp = 0.3 + 4.0 * torch.rand(1, 6, 12, 16, generator=g)
    run_case(R, "perpixel_planes_dot_12x16_D6_K2", "dot", t, 6, depth_planes=dp)
    run_case(R, "perpixel_planes_hero_12x16_D6_K2", "mlp", t, 6, mlp_sd=mlp_state(2, 16, seed=4), depth_planes=dp)
    # non-default channel count (generic kernels)
    run_case(R, "c8_dot_10x12_D4_K2", "dot", make_tuple(1, 2, 10, 12, channels=8, seed=8), 4)


if __name__ == "__main__":
    main()
