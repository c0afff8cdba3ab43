"""Depth-map parity through the reference's own U-Net (BASELINE target: depth Abs-Diff <= 1e-4).

The reference's `CVEncoder` + `DepthDecoderPP` (reference modules/networks.py:20-127) turn a
cost volume + image-prior features into the depth map.  They live only in /root/reference
(build container, CPU); our kernels run only on the GPU box.  So the check has two halves:

    # on the GPU box (through gpurun): our cost volumes for seeded 640x480 tuples
    python scripts/depth_parity.py dump        ->  gpurun_out/depth_parity_ours.npz

    # in the build container: reference cost volumes (CPU, reference classes) for the SAME
    # tuples, then the reference decoder on both, Abs-Diff of depth_pred_s0_b1hw
    python scripts/depth_parity.py eval        ->  profiles/depth_parity_r02.json

Round 2: a BATCH per model — 8 hero frames (one B = 8 call, BASELINE configs[2]'s shard) and 4
dot frames (configs[1]) at 640x480 — with the Abs-Diff reported per frame.  tests/test_gpu_depth_parity.py
runs the first half (into a temporary directory) and checks the dump's shapes and kernel variants.

Seeded random weights everywhere (no checkpoint exists in this environment, SURVEY.md §8c);
image-prior pyramid = seeded random tensors with EfficientNetV2-S channel counts
[24,48,64,160,256] at strides 2..32 (reference depth_model.py:108-116).  Abs-Diff is
`mean|a-b|` (reference utils/metrics_utils.py:38).
"""
from __future__ import annotations

import json
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from simplerecon_b200.synthetic import make_tuple, mlp_state  # noqa: E402

H, W, D, K, C = 120, 160, 64, 7, 16
SEEDS = {"dot": 2024, "hero": 2025}
FRAMES = {"dot": 4, "hero": 8}          # 4 x 19.7 MB + 8 x 4.9 MB... fp32 volumes: 59 MB < gpurun_out's 64 MiB
DUMP = ROOT / "gpurun_out" / "depth_parity_ours.npz"
REPORT = ROOT / "profiles" / "depth_parity_r02.json"


def dump(path: Path = DUMP):
    import simplerecon_b200 as S
    from simplerecon_b200 import _native
    from simplerecon_b200.synthetic import to_device
    out = {}
    with torch.inference_mode():
        for kind, seed in SEEDS.items():
            t = to_device(make_tuple(FRAMES[kind], K, H, W, seed=seed, smooth=True), "cuda")
            if kind == "dot":
                m = S.CostVolumeManager(H, W, D).cuda()
            else:
                m = S.FeatureVolumeManager(H, W, D, [0, 128, 128, 1], C, K)
                m.load_state_dict({**m.state_dict(), **mlp_state(K, C, seed=0)})
                m = m.cuda()
            cost, lowest, planes, mask = m(**t, return_mask=True)
            out[f"{kind}_cost"] = cost.cpu().numpy()
            out[f"{kind}_lowest"] = lowest.cpu().numpy()
            out[f"{kind}_variant"] = np.array(_native.last_variant())
    path.parent.mkdir(exist_ok=True)
    np.savez_compressed(path, **out)
    print("wrote", path, {k: getattr(v, "shape", None) for k, v in out.items()})


def evaluate(write: bool = True) -> dict:
    from oracle.ref_import import load_reference
    R = load_reference()
    z = np.load(DUMP)
    torch.manual_seed(0)
    enc_ch = [24, 48, 64, 160, 256]                      # EfficientNetV2-S feature_info.channels()
    cv_net = R.CVEncoder(num_ch_cv=D, num_ch_enc=enc_ch[1:], num_ch_outs=[64, 128, 256, 384]).eval()
    dec = R.DepthDecoderPP(enc_ch[:1] + cv_net.num_ch_enc).eval()
    g = torch.Generator().manual_seed(7)
    nmax = max(FRAMES.values())
    img_feats = [torch.randn(nmax, c, 4 * H // (2 ** (i + 1)), 4 * W // (2 ** (i + 1)), generator=g)
                 for i, c in enumerate(enc_ch)]

    def depth_from(cv):
        n = cv.shape[0]
        with torch.no_grad():
            feats = [img_feats[0][:n]] + cv_net(cv, [f[:n] for f in img_feats[1:]])
            outs = dec(feats)
        return torch.exp(outs["log_depth_pred_s0_b1hw"].float())

    report = {}
    for kind, seed in SEEDS.items():
        n = FRAMES[kind]
        t = make_tuple(n, K, H, W, seed=seed, smooth=True)
        if kind == "dot":
            ref = R.CostVolumeManager(H, W, num_depth_bins=D)
        else:
            ref = R.FeatureVolumeManager(H, W, num_depth_bins=D, mlp_channels=[0, 128, 128, 1],
                                         matching_dim_size=C, num_source_views=K)
            ref.load_state_dict({**ref.state_dict(), **mlp_state(K, C, seed=0)})
        with torch.no_grad():
            rc, rl, _, _ = ref(**t, return_mask=True)
            # the reference's own fp32 noise floor, on the first frame only (the fp64 run is slow)
            t1 = {k: (v[:1] if v.dim() > 0 and v.shape[0] == n else v).double() for k, v in t.items()}
            rc64, _, _, _ = ref.double()(**t1, return_mask=True)
            ref.float()
        ours = torch.from_numpy(z[f"{kind}_cost"])
        assert ours.shape == rc.shape, (ours.shape, rc.shape)
        d_ref, d_ours = depth_from(rc), depth_from(ours)
        d_64 = depth_from(rc64.float())
        per_frame = (d_ours - d_ref).abs().mean(dim=(1, 2, 3))
        report[kind] = {
            "kernel_variant": str(z[f"{kind}_variant"]), "frames": n,
            "cost_max_abs": float(rc.abs().max()),
            "cost_err_ours_vs_ref32": float((ours - rc).abs().max()),
            "cost_err_ours_vs_ref64_frame0": float((ours[:1].double() - rc64).abs().max()),
            "cost_err_ref32_vs_ref64_frame0": float((rc[:1].double() - rc64).abs().max()),
            # argmax plane index (plane VALUES differ by an ulp between the CPU's and the GPU's exp/log)
            "argmax_plane_mismatch_px": int((ours.argmax(1) != rc.argmax(1)).sum()),
            "depth_shape": list(d_ref.shape), "depth_mean": float(d_ref.mean()),
            "depth_abs_diff_per_frame": [float(x) for x in per_frame],
            "depth_abs_diff_ours_vs_ref": float(per_frame.mean()),
            "depth_abs_diff_worst_frame": float(per_frame.max()),
            "depth_max_diff_ours_vs_ref": float((d_ours - d_ref).abs().max()),
            # the reference's own fp32-vs-fp64 cost-volume noise pushed through the same decoder
            "depth_abs_diff_ref32_vs_ref64cv_frame0": float((d_ref[:1] - d_64).abs().mean()),
            "target_abs_diff": 1e-4,
        }
        report[kind]["pass"] = report[kind]["depth_abs_diff_worst_frame"] <= 1e-4
    if write:
        REPORT.write_text(json.dumps(report, indent=1))
    print(json.dumps(report, indent=1))
    return report


if __name__ == "__main__":
    {"dump": dump, "eval": evaluate}[sys.argv[1]]()
