"""GPU half of the depth-map parity check (BASELINE target: depth Abs-Diff <= 1e-4 through the
reference's U-Net): our cost volumes for a batch of seeded 640x480 tuples — 8 hero frames in one
B = 8 call, 4 dot frames — as `scripts/depth_parity.py dump` writes them.  The evaluation through the
reference's decoder is `scripts/depth_parity.py eval`, run where a SimpleRecon checkout is available."""
import importlib.util
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]


def test_dump_cost_volumes_for_depth_parity(cuda_device, tmp_path):
    spec = importlib.util.spec_from_file_location("depth_parity", ROOT / "scripts" / "depth_parity.py")
    dp = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(dp)
    dp.dump(tmp_path / dp.DUMP.name)
    z = np.load(tmp_path / dp.DUMP.name)
    assert z["hero_cost"].shape == (8, 64, 120, 160) and z["dot_cost"].shape == (4, 64, 120, 160)
    assert np.isfinite(z["hero_cost"]).all() and np.isfinite(z["dot_cost"]).all()
    assert "tcgen05" in str(z["hero_variant"]) and "fast" in str(z["dot_variant"])
