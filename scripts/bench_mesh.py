"""Timing + roofline of the marching-cubes extraction (TSDF.extract_mesh), one JSON line.

    python scripts/bench_mesh.py [--voxel 0.01] [--steps 20]
    python scripts/bench_mesh.py --live [--steps 20]

Default workload: the 1 cm room of scripts/bench_tsdf.py (608 x 512 x 312 voxels, 194 MB of fp16
values, larger than the 126 MB L2), fused from 8 frames, extracted with single_mesh.
--live: the 504^3 volume OurFuser builds without a ground-truth mesh (+-10 m at 4 cm); each step
integrates one frame and then extracts, as visualize_live_meshing.py does per frame.

Compulsory bytes of one extraction: 2 B per voxel of values read + the outputs written
(24 B per vertex, 12 B per face).  The host alternatives are measured on the same volume and
labelled for what they are: the device-to-host copy of the clamped fp32 volume the reference
makes before scikit-image runs, and the numpy oracle's time, which stands in for scikit-image
(not installed) and is not scikit-image.
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import torch  # noqa: E402

import simplerecon_b200 as S  # noqa: E402
from oracle import mesh_oracle as M  # noqa: E402
from simplerecon_b200.synthetic import make_tsdf_case  # noqa: E402

HBM_PEAK_GBS = 7700.0      # HGX B200 data sheet, one GPU, 1000 W

ap = argparse.ArgumentParser()
ap.add_argument("--voxel", type=float, default=0.01)
ap.add_argument("--steps", type=int, default=20)
ap.add_argument("--live", action="store_true")
ap.add_argument("--no-host", action="store_true", help="skip the host alternatives")
a = ap.parse_args()

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()[0]
ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

if a.live:
    vol = S.TSDF.from_bounds({k: (-10.0 if "min" in k else 10.0) for k in
                              ("xmin", "xmax", "ymin", "ymax", "zmin", "zmax")}, 0.04)
    fuser = S.TSDFFuser(vol, max_depth=3.0)
    frames = []
    for i in range(8):
        c = make_tsdf_case(seed=200 + i, frames=1, voxel_size=0.04, height=192, width=256, room=(6.0, 5.0, 3.0))
        frames.append((c["depth"].cuda(), c["cam_T_world"].cuda(), c["K"].cuda()))
    for i in range(3):
        fuser.integrate_depth(*frames[i % 8])
        vol.extract_mesh(single_mesh=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(a.steps):
        fuser.integrate_depth(*frames[i % 8])
        verts, faces, _ = vol.extract_mesh(single_mesh=True)
    torch.cuda.synchronize()
    s = (time.perf_counter() - t0) / a.steps
    print(json.dumps({"workload": "live 504^3 at 4 cm: integrate 1 frame (192x256) + extract_mesh(single_mesh)",
                      "gpu": gpu, "volume": list(vol.tsdf_values.shape), "vertices": len(verts), "faces": len(faces),
                      "ms_per_frame": s * 1e3, "frames_per_s": 1.0 / s}))
    sys.exit(0)

cases = [make_tsdf_case(seed=100 + i, frames=2, voxel_size=a.voxel, height=240, width=320, room=(6.0, 5.0, 3.0))
         for i in range(4)]
vol = S.TSDF.from_bounds(cases[0]["bounds"], a.voxel)
fuser = S.TSDFFuser(vol, max_depth=3.0)
for c in cases:
    fuser.integrate_depth(c["depth"].cuda(), c["cam_T_world"].cuda(), c["K"].cuda())
for _ in range(3):
    verts, faces, normals = vol.extract_mesh(single_mesh=True)
torch.cuda.synchronize()
e0, e1 = ev(), ev()
e0.record()
for _ in range(a.steps):
    verts, faces, normals = vol.extract_mesh(single_mesh=True)
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / a.steps
nvox = vol.tsdf_values.numel()
V, F = len(verts), len(faces)
compulsory = 2 * nvox + 24 * V + 12 * F
out = {"workload": f"fused room at {a.voxel * 100:g} cm, extract_mesh(single_mesh=True)", "gpu": gpu,
       "volume": list(vol.tsdf_values.shape), "values_MB": 2 * nvox / 1e6, "vertices": V, "faces": F,
       "ms_per_extract": ms, "compulsory_bytes": compulsory, "achieved_GBps": compulsory / (ms * 1e-3) / 1e9,
       "frac_of_hbm_peak": compulsory / (ms * 1e-3) / 1e9 / HBM_PEAK_GBS,
       "hbm_peak_GBps": HBM_PEAK_GBS, "timing": "CUDA events around steps extractions (2 host syncs each), after 3 warm-up"}
if not a.no_host:
    e0.record()
    host = vol.tsdf_values.float().clamp(-1, 1).cpu()
    e1.record()
    torch.cuda.synchronize()
    out["host_copy_clamped_fp32_ms"] = e0.elapsed_time(e1)
    out["host_copy_note"] = "the reference's .cpu().float().clamp() before marching cubes (clamp on device here)"
    t0 = time.perf_counter()
    M.extract(vol.tsdf_values.cpu().numpy(), single_mesh=True)
    out["numpy_oracle_s"] = time.perf_counter() - t0
    out["numpy_oracle_note"] = "vectorised numpy restatement of the contract, one CPU thread; stands in for skimage, is not skimage"
print(json.dumps(out))
