"""CPU: the reference arm of bench.py runs here (it is the CPU port) and prints the contract's
JSON line; the GPU arm's helpers are importable."""
import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]


def test_reference_arm_prints_contract_line():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--workload", "cfg0",
                        "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step",
              "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["unit"] == "frames/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
    assert line["config"]["workload"].startswith("cfg0")


def test_reference_arm_stays_bounded_at_many_steps():
    """At large step counts (the no-flag default is 100) a step becomes a plane subset of one frame, the
    metric stays per frame and the run stays within its budget."""
    import os
    env = dict(os.environ, SRCV_REF_BUDGET_S="0.02", SRCV_CPU_THREADS="2")
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--workload", "cfg0",
                        "--steps", "12", "--warmup", "3"], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    cb = line["cpu_baseline"]
    assert "planes of one frame per step" in cb["sample"] and 0 < cb["frames_per_step_timed"] < 1
    assert line["steps"] == 12 and line["value"] > 0 and line["config"]["workload"].startswith("cfg0")


def test_algorithmic_bytes_match_survey():
    sys.path.insert(0, str(ROOT))
    import bench
    from simplerecon_b200.synthetic import CONFIGS
    # SURVEY.md §8(d): cfgA 14.82 MB (dot) / 14.84 MB (hero) per frame
    assert abs(bench.algorithmic_bytes_per_frame(CONFIGS[1], False, True) - 14.82e6) < 0.02e6
    assert abs(bench.algorithmic_bytes_per_frame(CONFIGS[2], True, True) - 14.84e6) < 0.02e6
    assert abs(bench.algorithmic_bytes_per_frame(CONFIGS[3], True, True) - 17.30e6) < 0.03e6


def test_mlp_flops_match_survey_and_configs_agree_between_arms():
    sys.path.insert(0, str(ROOT))
    import bench
    from simplerecon_b200.synthetic import CONFIGS
    # SURVEY.md §8(d): 104.1 GFLOP (MLP) per frame at cfgA, 156.2 at cfgB
    assert abs(bench.mlp_flops_per_frame(CONFIGS[2], False) - 104.1e9) < 0.1e9
    assert abs(bench.mlp_flops_per_frame(CONFIGS[3], False) - 156.2e9) < 0.15e9
    # what the tcgen05 kernel issues: 3 MMAs per product, layer-1 K = 192 (pose measures as a bias)
    assert bench.mlp_flops_per_frame(CONFIGS[2], True) > 3 * 0.95 * bench.mlp_flops_per_frame(CONFIGS[2], False)
    # the default workload is the hero configuration at 8 frames per GPU: N = 1 is BASELINE configs[2],
    # N = 8 is configs[4]; both arms print the same `config`
    assert bench.DEFAULT_WORKLOAD == "cfg2" and bench.PER_GPU["cfg2"] == 8
    w = next(c for c in CONFIGS if c.name.startswith(bench.DEFAULT_WORKLOAD))
    c1, _ = bench.workload_config(w, bench.PER_GPU["cfg2"], 8)
    assert c1["global_batch"] == 64 and c1["matching"] == "mlp" and c1["planes"] == 64


def test_dump_outputs_samples_past_the_budget(tmp_path, monkeypatch):
    """Under the budget every array is written whole; past it each becomes the same seeded sample."""
    import numpy as np
    import torch
    sys.path.insert(0, str(ROOT))
    import bench
    a = torch.arange(6000, dtype=torch.float32).reshape(2, 3000)
    b = torch.ones(4, 5, dtype=torch.float64)
    info = bench.dump_outputs(str(tmp_path / "whole"), {"a": a, "b": b})
    assert info == {"a": [2, 3000], "b": [4, 5]}
    assert np.array_equal(np.load(tmp_path / "whole" / "a.npy"), a.numpy())
    assert np.load(tmp_path / "whole" / "b.npy").dtype == np.float32
    monkeypatch.setattr(bench, "DUMP_BYTES", 4 * 1200)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), {"a": a})
    s1, s2 = np.load(tmp_path / "s1" / "a.npy"), np.load(tmp_path / "s2" / "a.npy")
    assert s1.shape == (1200,) and np.array_equal(s1, s2)
    assert np.all(np.diff(s1) > 0)                      # distinct elements, in storage order


@pytest.mark.gpu
def test_dump_outputs_holds_the_last_timed_step(tmp_path):
    """`--dump-outputs` writes what the last of `--steps` timed steps returned: its input set is the
    seeded tuple of that step, so the dump equals the oracle's volume for that tuple."""
    import numpy as np
    sys.path.insert(0, str(ROOT))
    from oracle import costvolume_oracle as O
    from simplerecon_b200.synthetic import CONFIGS, make_workload_tuple
    steps = 3
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--workload", "cfg0", "--steps", str(steps),
                        "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and set(line["dumped_outputs"]["arrays"]) == {
        "cfg0_cost_volume", "cfg0_lowest_cost", "cfg0_depth_planes"}
    w = CONFIGS[0]
    t = make_workload_tuple(w, seed_offset=steps - 1, batch=1)       # sets rotate: step i uses set i
    oc, ol, op, _ = O.forward_dot(**t, num_depth_bins=w.planes)
    cost = np.load(tmp_path / "cfg0_cost_volume.npy")
    assert cost.dtype == np.float32 and cost.shape == tuple(oc.shape)
    assert np.abs(cost - oc.numpy()).max() <= 4e-5 * float(oc.abs().max()) + 1e-6
    assert np.load(tmp_path / "cfg0_depth_planes.npy").shape == (1, w.planes, 1, 1)
