"""CPU: the TSDF oracle against the reference TSDFFuser (tools/tsdf.py), bit for bit in fp16, on
volumes recorded from the unmodified reference by tests/golden/make_golden_reference.py."""
import pytest
import torch

from oracle import tsdf_oracle as T
from simplerecon_b200.synthetic import make_tsdf_case
from tests.parity import load_reference_outputs


@pytest.mark.parametrize("seed,frames,voxel,masked", [(1, 1, 0.08, False), (2, 3, 0.05, False), (3, 2, 0.06, True)])
def test_integrate_matches_live_reference_bitwise(seed, frames, voxel, masked):
    R = load_reference_outputs("tsdf")
    c = make_tsdf_case(seed=seed, frames=frames, voxel_size=voxel, height=48, width=64, masked=masked)
    tv, tw, origin = T.new_volume(c["bounds"], voxel)
    assert tuple(tv.shape) == tuple(R[f"c{seed}_r0_values"].shape)
    # voxels whose fp16 sampling coordinate overflows: undefined in the CPU run of the reference
    # (see tsdf_oracle.overflow_voxels); a handful next to each camera's principal plane
    skip = T.overflow_voxels(origin, tuple(tv.shape), voxel, c["cam_T_world"], c["K"], c["depth"].shape[2:])
    assert skip.float().mean().item() < 1e-2
    keep = ~skip
    for rep in range(2):          # two rounds: the second one starts from non-trivial weights
        rv, rw = R[f"c{seed}_r{rep}_values"], R[f"c{seed}_r{rep}_weights"]
        T.integrate(tv, tw, origin, voxel, c["depth"], c["cam_T_world"], c["K"], c["mask"],
                    min_depth=float(R[f"c{seed}_min_depth"]), max_depth=c["max_depth"])
        touched = int((rw > 0).sum())
        assert touched > 1000, touched
        assert torch.equal(tw[keep], rw[keep]), (tw.float() - rw.float())[keep].abs().max()
        assert torch.equal(tv[keep], rv[keep]), (tv.float() - rv.float())[keep].abs().max()
        # keep the two states identical for the next round (the skipped voxels differ by construction)
        tv[skip], tw[skip] = rv[skip], rw[skip]
