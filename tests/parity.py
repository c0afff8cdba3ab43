"""Shared parity helpers: golden-case loading and the stated tolerances.

Tolerances (fp32, SURVEY.md §8c).  The reference's own fp32 result differs from its
fp64 evaluation — fp32 rounding of ~100-pixel coordinates feeding bilinear weights —
by up to ~1.5e-5 of max|cost| (dot) and, at the BASELINE 120x160 / D=64 size, 3.4e-5
of max|cost| (MLP volume: measured 1.5e-5 abs on max|cost| 0.45).  Hence:

* cost volume, element-wise:
      |ours - ref32| <= max(RTOL_MAX[kind] * max|ref| + 1e-6,  2 * max|ref32 - ref64|)
  (the second term only where the fp64 evaluation of the reference is available);
* against the fp64 reference (where available) ours must not be further off than twice
  the reference's own fp32 result:  max|ours - ref64| <= 2 max|ref32 - ref64| + 1e-6 max|ref|
  (the centred-coordinate kernels are in fact closer to fp64 than the reference is);
* lowest_cost (argmax depth): a pixel may pick another plane only on a near tie, i.e.
  ref cost at our plane within 2x the cost tolerance of the ref maximum; at most 0.5 % of pixels;
* overall mask: at most 0.1 % of pixels differ (strict-inequality tests on fp32 coordinates).
"""
from __future__ import annotations

from pathlib import Path

import numpy as np
import torch

GOLDEN = Path(__file__).resolve().parent / "golden"
RTOL_MAX = {"dot": 4e-5, "mlp": 2e-5}
INPUT_KEYS = ("cur_feats", "src_feats", "src_extrinsics", "src_poses", "src_Ks", "cur_invK",
              "min_depth", "max_depth")


def golden_names(kind=None):
    names = sorted(p.stem for p in GOLDEN.glob("*.npz"))
    if kind:
        names = [n for n in names if str(np.load(GOLDEN / f"{n}.npz")["kind"]) == kind]
    return names


def load_golden(name):
    z = np.load(GOLDEN / f"{name}.npz")
    g = {k: (torch.from_numpy(z[k]) if z[k].dtype.kind == "f" or z[k].dtype.kind == "b" else z[k])
         for k in z.files}
    g["kind"] = str(z["kind"])
    g["D"] = int(z["D"])
    if "ref_cost64_minus_ref_cost" in g:     # stored as an fp32 residual where the fp64 volume is large
        g["ref_cost64"] = g["ref_cost"].double() + g.pop("ref_cost64_minus_ref_cost").double()
    inputs = {k: g[k] for k in INPUT_KEYS}
    if "depth_planes_bdhw" in g:
        inputs["depth_planes_bdhw"] = g["depth_planes_bdhw"]
    sd = {k.replace("mlp_net_", "mlp.net.").replace("_weight", ".weight").replace("_bias", ".bias"): v
          for k, v in g.items() if k.startswith("mlp_net_")}
    return g, inputs, sd


def golden_fullsize_names():
    return sorted(p.stem for p in (GOLDEN / "fullsize").glob("*.npz"))


def load_golden_fullsize(name):
    """Fixtures at the bench feature-map size (tests/golden/make_golden_fullsize.py): the inputs are
    REGENERATED from the stored generator call and checked against the stored SHA-256; outputs are the
    unmodified reference's.  Returns (g, inputs, state_dict or None) like load_golden; g["ref_cost64"]
    is the fp64 evaluation rounded to fp32 and g["err32v64"] the reference's own max|fp32 - fp64|."""
    import ast
    import hashlib

    from simplerecon_b200.synthetic import make_tuple, mlp_state
    z = np.load(GOLDEN / "fullsize" / f"{name}.npz")
    gen = dict(ast.literal_eval(str(z["gen"])))
    inputs = make_tuple(**gen)
    h = hashlib.sha256()
    for k in INPUT_KEYS:
        h.update(np.ascontiguousarray(inputs[k].numpy()).tobytes())
    if h.hexdigest() != str(z["sha256"]):
        raise RuntimeError(f"{name}: regenerated inputs do not hash to the stored value (generator drift)")
    g = {k: torch.from_numpy(z[k]) for k in ("ref_cost", "ref_cost64_as_f32", "ref_lowest", "ref_planes")}
    g["ref_cost64"] = g.pop("ref_cost64_as_f32").double()
    g["err32v64"] = float(z["err32v64"])
    g["kind"], g["D"] = str(z["kind"]), int(z["D"])
    if "ref_mask" in z.files:
        g["ref_mask"] = torch.from_numpy(z["ref_mask"])
    sd = mlp_state(gen["views"], gen["channels"], seed=gen["seed"]) if g["kind"] == "mlp" else None
    return g, inputs, sd


def load_reference_outputs(name):
    """What the unmodified reference computed for the cases of one test module
    (tests/golden/make_golden_reference.py), as CPU tensors; string arrays stay numpy."""
    z = np.load(GOLDEN / "reference" / f"{name}.npz")
    return {k: (z[k] if z[k].dtype.kind == "U" else torch.from_numpy(z[k])) for k in z.files}


def cost_tol(kind, ref):
    return RTOL_MAX[kind] * float(ref.abs().max()) + 1e-6


def assert_cost_close(kind, ours, ref32, ref64=None, what="", e_ref=None):
    """`e_ref`: the reference's own max|fp32 - fp64| when `ref64` is stored rounded to fp32."""
    ours = ours.detach().cpu()
    tol = cost_tol(kind, ref32)
    if ref64 is not None:
        e_ref = (ref32.double() - ref64).abs().max().item() if e_ref is None else e_ref
        tol = max(tol, 2 * e_ref)
    err = (ours - ref32).abs().max().item()
    assert err <= tol, f"{what}: cost max-abs err {err:.3e} > tol {tol:.3e}"
    if ref64 is not None:
        e_ours = (ours.double() - ref64).abs().max().item()
        bound = 2 * e_ref + 1e-6 * float(ref64.abs().max()) + 1e-7
        assert e_ours <= bound, f"{what}: err vs fp64 {e_ours:.3e} > 2x reference's own {e_ref:.3e}"
        print(f"[parity] {what}: |ours-ref32|={err:.3e} |ours-ref64|={e_ours:.3e} |ref32-ref64|={e_ref:.3e}")
    return err


def assert_lowest_close(kind, ours_lowest, ours_planes_bdhw, ref_cost, what="", max_frac=5e-3):
    """`ours_lowest` must be the plane depth at (a near-tie of) the argmax of the
    reference volume.  Works on plane INDICES so that a 1-ulp difference between the
    CPU's and the GPU's exp/log plane values does not matter."""
    ours_lowest = ours_lowest.detach().cpu()
    planes = ours_planes_bdhw.detach().cpu().expand_as(ref_cost)
    idx_ours = (planes - ours_lowest.unsqueeze(1)).abs().argmin(1)
    picked = torch.gather(planes, 1, idx_ours.unsqueeze(1)).squeeze(1)
    assert torch.equal(picked, ours_lowest), f"{what}: lowest_cost is not one of the plane depths"
    idx_ref = ref_cost.argmax(1)
    diff = idx_ours != idx_ref
    n = int(diff.sum())
    if n == 0:
        return 0
    assert n <= max(1, int(max_frac * diff.numel())), f"{what}: {n} argmax-depth mismatches"
    tol = 2 * cost_tol(kind, ref_cost)
    at_ours = torch.gather(ref_cost, 1, idx_ours.unsqueeze(1)).squeeze(1)
    bad = diff & ((ref_cost.max(1).values - at_ours) > tol)
    assert int(bad.sum()) == 0, f"{what}: {int(bad.sum())} argmax mismatches are not near ties"
    return n


def assert_mask_close(ours_mask, ref_mask, what="", max_frac=1e-3):
    ours_mask = ours_mask.detach().cpu()
    assert ours_mask.dtype == torch.bool and ours_mask.shape == ref_mask.shape
    n = int((ours_mask != ref_mask).sum())
    assert n <= max(1, int(max_frac * ref_mask.numel())), f"{what}: {n} mask mismatches"
    return n
