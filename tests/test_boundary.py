"""CPU: the Python mirror keeps the reference's interface (SURVEY.md §8b) — class
names, constructor / forward signatures, buffers, state_dict keys, to_fast(),
install() — and refuses to run anywhere but on the CUDA path."""
import inspect
import sys
import types

import pytest
import torch

import simplerecon_b200 as S
from simplerecon_b200.synthetic import CONFIGS, make_tuple, mlp_state

FWD_ARGS = ["self", "cur_feats", "src_feats", "src_extrinsics", "src_poses", "src_Ks", "cur_invK",
            "min_depth", "max_depth", "depth_planes_bdhw", "return_mask"]


def test_constructor_signatures_match_reference():
    # reference modules/cost_volume.py:27-34, :398-404, :757-763
    p = list(inspect.signature(S.CostVolumeManager.__init__).parameters)
    assert p == ["self", "matching_height", "matching_width", "num_depth_bins", "matching_dim_size",
                 "num_source_views"]
    for cls in (S.FeatureVolumeManager, S.FastFeatureVolumeManager):
        sig = inspect.signature(cls.__init__)
        assert list(sig.parameters) == ["self", "matching_height", "matching_width", "num_depth_bins",
                                        "mlp_channels", "matching_dim_size", "num_source_views"]
        assert sig.parameters["num_depth_bins"].default == 64
        assert sig.parameters["matching_dim_size"].default == 16
        assert sig.parameters["num_source_views"].default == 7


@pytest.mark.parametrize("cls", [S.CostVolumeManager, S.FeatureVolumeManager, S.FastFeatureVolumeManager])
def test_forward_and_build_signatures(cls):
    # the reference's parameters, in its order; forward() may append OPTIONAL extensions after them
    # (raw_poses, SURVEY §8f-2) — a caller written against the reference never sees those
    fwd = inspect.signature(cls.forward).parameters
    assert list(fwd)[:len(FWD_ARGS)] == FWD_ARGS
    assert all(p.default is None for n, p in fwd.items() if n not in FWD_ARGS)
    assert list(inspect.signature(cls.build_cost_volume).parameters) == FWD_ARGS
    for m in ("generate_depth_planes", "get_mask", "indices_to_disparity", "warp_features",
              "initialise_for_projection"):
        assert callable(getattr(cls, m))


def test_state_dict_keys_and_shapes():
    # SURVEY.md §5: keys a Lightning checkpoint of the reference holds for this module
    m = S.FeatureVolumeManager(120, 160, num_depth_bins=64, matching_dim_size=16, num_source_views=7)
    sd = m.state_dict()
    exp = {
        "linear_ramp_1d11": (1, 64, 1, 1), "backprojector.pix_coords_13N": (1, 3, 19200),
        "projector.eps": (1, 1, 1), "mlp.net.0.weight": (128, 202), "mlp.net.0.bias": (128,),
        "mlp.net.2.weight": (128, 128), "mlp.net.2.bias": (128,), "mlp.net.4.weight": (1, 128),
        "mlp.net.4.bias": (1,),
    }
    assert {k: tuple(v.shape) for k, v in sd.items()} == exp
    assert sum(p.numel() for p in m.parameters()) == 42625
    d = S.CostVolumeManager(48, 64, 16)
    assert sorted(d.state_dict()) == ["backprojector.pix_coords_13N", "linear_ramp_1d11", "projector.eps"]
    m.load_state_dict({**sd, **mlp_state(7, 16)}, strict=True)


def test_hierarchy_to_fast_and_quirks():
    m = S.FeatureVolumeManager(12, 16, 8, matching_dim_size=16, num_source_views=3)
    assert isinstance(m, S.CostVolumeManager)
    f = m.to_fast()
    assert isinstance(f, S.FastFeatureVolumeManager) and isinstance(f, S.FeatureVolumeManager)
    assert f.mlp is m.mlp and f.num_depth_bins == 8 and (f.matching_height, f.matching_width) == (12, 16)
    # mlp_channels[0] is overwritten from K and C (reference :429)
    ch = [0, 32, 16, 1]
    S.FeatureVolumeManager(4, 4, 2, ch, 8, 2)
    assert ch[0] == 8 * 3 + 10 * 2 + 4


def test_helper_methods_match_oracle():
    from oracle import costvolume_oracle as O
    m = S.CostVolumeManager(6, 8, 5)
    mn, mx = torch.tensor(0.25).view(1, 1, 1, 1), torch.tensor(5.0).view(1, 1, 1, 1)
    planes = m.generate_depth_planes(2, mn, mx)
    assert planes.shape == (2, 5, 6, 8) and planes.stride()[2:] == (0, 0)
    assert torch.allclose(planes[0, :, 0, 0], O.depth_planes(0.25, 5.0, 5))
    pix = torch.tensor([[[[1.0, 3.0, 7.0]], [[3.0, 3.0, 3.0]]]]).view(1, 1, 2, 1, 3)
    assert m.get_mask(pix).flatten().tolist() == [False, True, False]
    idx = torch.tensor([[[0, 4]]])
    assert torch.equal(m.indices_to_disparity(idx.expand(2, 1, 2), planes[:, :, :1, :2]),
                       planes[:, [0, 4], 0, 0].view(2, 1, 2))
    # geometry helper modules agree with the oracle's restatement
    t = make_tuple(1, 2, 6, 8, seed=3)
    rays = O.backproject_rays(t["cur_invK"], 6, 8)
    pts = m.backprojector(planes[:1, 2:3], t["cur_invK"])
    assert torch.allclose(pts[:, :3], planes[0, 2, 0, 0] * rays, atol=1e-6)
    cam = m.projector(pts, t["src_Ks"][:, 0], t["src_extrinsics"][:, 0])
    px, py, zp = O.project(pts[:, :3], t["src_Ks"], t["src_extrinsics"])
    assert torch.allclose(cam[:, 0], px[:, 0], atol=1e-4) and torch.allclose(cam[:, 2], zp[:, 0], atol=1e-6)


def test_cpu_tensors_are_refused_not_silently_computed():
    m = S.CostVolumeManager(6, 8, 4)
    t = make_tuple(1, 2, 6, 8, seed=1)
    with torch.no_grad(), pytest.raises(RuntimeError, match="no CPU fallback"):
        m(**t)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.warp_features(t["src_feats"], t["src_extrinsics"], t["src_Ks"], t["cur_invK"],
                        torch.ones(1, 1, 6, 8), 1, 2, 16, None)


def test_product_package_never_imports_the_oracle():
    import pathlib
    pkg = pathlib.Path(S.__file__).parent
    for p in pkg.rglob("*.py"):
        src = p.read_text()
        assert "import oracle" not in src and "from oracle" not in src, p


def test_install_patches_reference_namespace(monkeypatch):
    fake_pkg = types.ModuleType("modules")
    fake_pkg.__path__ = []
    fake_cv = types.ModuleType("modules.cost_volume")
    for n in ("CostVolumeManager", "FeatureVolumeManager", "FastFeatureVolumeManager"):
        setattr(fake_cv, n, type(n, (), {}))
    fake_dm = types.ModuleType("experiment_modules.depth_model")
    fake_dm.CostVolumeManager, fake_dm.FeatureVolumeManager = fake_cv.CostVolumeManager, fake_cv.FeatureVolumeManager
    monkeypatch.setitem(sys.modules, "modules", fake_pkg)
    monkeypatch.setitem(sys.modules, "modules.cost_volume", fake_cv)
    monkeypatch.setitem(sys.modules, "experiment_modules.depth_model", fake_dm)
    orig = fake_cv.CostVolumeManager
    patched = S.install()
    assert patched == ["modules.cost_volume", "experiment_modules.depth_model"]
    assert fake_cv.FeatureVolumeManager is S.FeatureVolumeManager
    assert fake_dm.CostVolumeManager is S.CostVolumeManager
    assert fake_cv.FastFeatureVolumeManager is S.FastFeatureVolumeManager
    S.uninstall()
    assert fake_cv.CostVolumeManager is orig


def test_synthetic_tuples_are_deterministic_and_shaped():
    a, b = make_tuple(2, 7, 12, 16, seed=11), make_tuple(2, 7, 12, 16, seed=11)
    for k in a:
        assert torch.equal(a[k], b[k])
    assert a["src_feats"].shape == (2, 7, 16, 12, 16) and a["cur_invK"].shape == (2, 4, 4)
    # poses are mutual inverses and sorted by pose distance
    I = a["src_extrinsics"].double() @ a["src_poses"].double()
    assert torch.allclose(I, torch.eye(4, dtype=torch.float64).expand_as(I), atol=1e-5)
    from oracle.costvolume_oracle import pose_distance
    comb, _, _ = pose_distance(a["src_poses"])
    assert bool((comb[:, 1:] >= comb[:, :-1] - 1e-6).all())
    # BASELINE.json configs at feature-map resolution
    assert [(c.kind, c.batch, c.views, c.height, c.width, c.planes) for c in CONFIGS] == [
        ("dot", 1, 2, 48, 64, 16), ("dot", 4, 7, 120, 160, 64), ("mlp", 8, 7, 120, 160, 64),
        ("mlp", 16, 7, 120, 160, 96), ("mlp", 64, 7, 120, 160, 64)]


def _reference_like_module(monkeypatch, name, class_names):
    """A module under the reference's import name holding stand-ins for `class_names`, for install()."""
    mod = types.ModuleType(name)
    for n in class_names:
        setattr(mod, n, type(n, (torch.nn.Module,), {}))
    if "." in name:
        pkg = types.ModuleType(name.split(".")[0])
        pkg.__path__ = []
        monkeypatch.setitem(sys.modules, pkg.__name__, pkg)
    monkeypatch.setitem(sys.modules, name, mod)
    monkeypatch.delitem(sys.modules, "experiment_modules.depth_model", raising=False)
    return mod


def test_install_against_the_real_reference_module(monkeypatch):
    """install() on the reference's modules.cost_volume namespace: the three names resolve to our
    classes, `isinstance` / `to_fast()` as used by test.py:196-198 keep working, the state_dict the
    unmodified reference's FeatureVolumeManager produces (recorded by tests/golden/make_golden_reference.py)
    loads strictly into ours, and uninstall() restores the reference's classes."""
    from tests.parity import load_reference_outputs
    R = load_reference_outputs("python_layer")
    ref_state = {k[len("state_dict/"):]: v for k, v in R.items() if k.startswith("state_dict/")}
    names = ("CostVolumeManager", "FeatureVolumeManager", "FastFeatureVolumeManager")
    ref_cv = _reference_like_module(monkeypatch, "modules.cost_volume", names)
    orig = {n: getattr(ref_cv, n) for n in names}
    try:
        patched = S.install()
        assert "modules.cost_volume" in patched
        assert ref_cv.CostVolumeManager is S.CostVolumeManager
        assert ref_cv.FeatureVolumeManager is S.FeatureVolumeManager
        assert ref_cv.FastFeatureVolumeManager is S.FastFeatureVolumeManager
        # what experiment_modules/depth_model.py:162-176 does, by keyword
        cv = ref_cv.FeatureVolumeManager(matching_height=12, matching_width=16, num_depth_bins=8,
                                         matching_dim_size=16, num_source_views=7)
        cv.load_state_dict(ref_state, strict=True)                     # Lightning loads strictly
        assert isinstance(cv, ref_cv.FeatureVolumeManager)              # test.py:196
        fast = cv.to_fast()                                             # test.py:198
        assert isinstance(fast, ref_cv.FastFeatureVolumeManager) and fast.mlp is cv.mlp
        assert set(cv.state_dict()) == set(ref_state)
    finally:
        S.uninstall()
    for n, c in orig.items():
        assert getattr(ref_cv, n) is c


def test_install_swaps_the_real_reference_loss_class(monkeypatch):
    """install(losses=True) on the reference's losses namespace: MVDepthLoss resolves to the kernel-backed
    mirror, whose constructor / forward / helper signatures are those of the unmodified reference's
    (recorded by tests/golden/make_golden_reference.py); uninstall() restores it."""
    from tests.parity import load_reference_outputs
    ref_sigs = {s.split()[0]: s.split()[1:] for s in load_reference_outputs("mvdepth_loss")["signatures"]}
    _reference_like_module(monkeypatch, "modules.cost_volume", ())
    ref_losses = _reference_like_module(monkeypatch, "losses", ("MVDepthLoss",))
    orig = ref_losses.MVDepthLoss
    try:
        patched = S.install(losses=True)
        assert "losses" in patched and ref_losses.MVDepthLoss is S.MVDepthLoss
        for name in ("__init__", "forward", "get_valid_mask", "get_error_for_pair"):
            assert list(inspect.signature(getattr(S.MVDepthLoss, name)).parameters) == ref_sigs[name], name
        loss = ref_losses.MVDepthLoss(192, 256)                     # depth_model.py:144-147
        assert loss.height == 192 and loss.width == 256
        with pytest.raises(RuntimeError):                           # CPU tensors: refused, no fallback
            loss(*[torch.zeros(1)] * 7)
    finally:
        S.uninstall()
    assert ref_losses.MVDepthLoss is orig
