"""Drop-in cost-volume managers backed by the sm_100a kernels.

Class names, constructor signatures, method names, ``forward`` signature / return
tuple, buffers and ``state_dict`` keys follow the reference's
``modules/cost_volume.py`` (``CostVolumeManager`` :13-380, ``FeatureVolumeManager``
:383-746, ``FastFeatureVolumeManager`` :749-1164) so that
``experiment_modules/depth_model.py:162-176, 362-372`` and the ``isinstance`` /
``to_fast()`` swaps in ``test.py:196-198`` work unchanged.  The sweep itself is one
call into ``libsrcv_b200.so`` (include/srcv_b200.h) on the current CUDA stream.

Contract at the boundary (SURVEY.md §8b): fp32 CUDA tensors, inference only.
Anything else raises — there is no PyTorch / CPU fallback on this path.
"""
from __future__ import annotations

import ctypes as C

import torch
from torch import Tensor, nn

from . import _native
from .geometry import BackprojectDepth, Project3D
from .networks import MLP


def _require_cuda(dev) -> None:
    """The one device gate of the managers: CUDA tensors only, no CPU / PyTorch fallback.
    (tests/test_emu_python_stack.py patches exactly this to drive the Python layer against the
    host-emulated library; the product never bypasses it.)"""
    if dev.type != "cuda":
        raise RuntimeError(
            "simplerecon_b200 cost volumes run on CUDA (sm_100a) only; got tensors on "
            f"{dev}.  There is no CPU fallback.")


def _ptr(t: Tensor | None):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _f32c(t: Tensor, name: str, device) -> Tensor:
    if not torch.is_tensor(t):
        raise TypeError(f"{name} must be a tensor")
    if t.dtype in (torch.float16, torch.bfloat16):
        # autocast producers (the reference trains and validates at precision=16, train.py:132, and
        # casts its sampling grid with type_as(src_feats), modules/cost_volume.py:208,597): the
        # kernels compute in fp32, so half inputs are upcast — in the no-grad path exactly as in
        # the autograd Functions below
        t = t.float()
    if t.dtype != torch.float32:
        raise ValueError(f"{name} must be float32, float16 or bfloat16 (got {t.dtype})")
    if t.device != device:
        raise ValueError(f"{name} is on {t.device}, expected {device}")
    t = t.contiguous()
    if t.data_ptr() % 16 != 0:      # the kernels use 16-byte vector loads
        t = t.clone()
    return t


def _check_backward_supported(kind: str, src_shape, hidden) -> None:
    """Unsupported training shapes fail in forward(), not at backward() time."""
    lib = _native.load()
    B, K, Cc, H, W = src_shape
    shape = _native.Shape(B, K, Cc, H, W, 1)
    if kind == "dot":
        if lib.srcv_dot_backward_supported(C.byref(shape)) == 0:
            raise NotImplementedError(f"dot-product volume backward is built for C in {{8, 16, 32}}, got C={Cc}")
    else:
        if lib.srcv_mlp_backward_supported(C.byref(shape), int(hidden[0]), int(hidden[1])) == 0:
            raise NotImplementedError(
                "metadata-MLP volume backward: at most 208 input features and hidden widths <= 128 "
                f"(K={K}, C={Cc}, hidden={tuple(hidden)})")


def instance_norm_to_chunk_planar(x_bvchw: Tensor, eps: float = 1e-5):
    """The matching encoder's final ``nn.InstanceNorm2d(C)`` (reference modules/networks.py:201:
    no affine, biased variance, eps 1e-5) fused with the layout pass of the sweeps.

    ``x_bvchw``: the conv output for the stacked images, ``(B, 1+K, C, H, W)`` (reference frame
    first, as depth_model.py:220-243 arranges it).  Returns ``(cur_feats, src_feats)`` as
    chunk-planar tensors ``(B,C/4,H,W,4)`` / ``(B,K,C/4,H,W,4)`` that the managers' ``forward``
    accepts in place of the NCHW ones — the normalised NCHW tensor and the prep pass's re-layout
    copy never exist."""
    if not torch.is_tensor(x_bvchw) or x_bvchw.dim() != 5:
        raise ValueError("expected a (B, 1+K, C, H, W) tensor")
    dev = x_bvchw.device
    _require_cuda(dev)
    x = _f32c(x_bvchw, "x", dev)
    B, V, Cc, H, W = x.shape
    if Cc % 4 != 0:
        raise ValueError("the chunk-planar layout needs C % 4 == 0")
    lib = _native.load()
    with torch.cuda.device(dev):
        cur = torch.empty(B, Cc // 4, H, W, 4, device=dev, dtype=torch.float32)
        src = torch.empty(B, max(V - 1, 0), Cc // 4, H, W, 4, device=dev, dtype=torch.float32)
        _native.check(lib.srcv_instnorm_to_chunk_planar_f32(
            _ptr(x), B, V, Cc, H, W, float(eps), _ptr(cur), _ptr(src) if V > 1 else C.c_void_p(0),
            C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return cur, src


class _DotVolumeFunction(torch.autograd.Function):
    """Differentiable wrapper of the dot-product sweep: fused forward, and a backward kernel
    (``srcv_dot_backward_f32``) for the two feature inputs — what autograd of the reference's
    grid_sample / mul / sum composite (modules/cost_volume.py:305-333) yields for them.
    Cameras and plane depths get no gradient.  fp16 / bf16 features (autocast) are upcast."""

    @staticmethod
    def forward(ctx, mgr, cur_feats, src_feats, src_extrinsics, src_Ks, cur_invK, min_depth, max_depth,
                depth_planes_bdhw):
        dev = src_feats.device
        # What is saved for the backward kernel is what the forward kernel read: dense, 16-byte
        # aligned fp32 copies.  The caller's own tensors may be strided views — the reference
        # passes cur_feats = matching_feats[:, 0] (experiment_modules/depth_model.py:242) — and the
        # kernels index them as dense NCHW.
        cur32, src32 = _f32c(cur_feats, "cur_feats", dev), _f32c(src_feats, "src_feats", dev)
        E32, Ks32 = _f32c(src_extrinsics, "src_extrinsics", dev), _f32c(src_Ks, "src_Ks", dev)
        invK32 = _f32c(cur_invK, "cur_invK", dev)
        _check_backward_supported("dot", src32.shape, None)
        cost, lowest, planes_ret, _ = mgr._run_fused(
            cur32, src32, E32, None, Ks32, invK32, min_depth,
            max_depth, depth_planes_bdhw, True, allow_grad=True)
        B, D, H, W = cost.shape
        st = planes_ret.stride()
        per_pixel = not ((st[2] == 0 or H == 1) and (st[3] == 0 or W == 1))
        planes = planes_ret[:, :D].contiguous() if per_pixel else planes_ret[:, :D, 0, 0].contiguous()
        ctx.save_for_backward(cur32, src32, E32, Ks32, invK32, planes)
        ctx.per_pixel = per_pixel
        ctx.in_dtypes = (cur_feats.dtype, src_feats.dtype)
        ctx.mark_non_differentiable(lowest, planes_ret)
        return cost, lowest, planes_ret

    @staticmethod
    def backward(ctx, grad_cost, _grad_lowest, _grad_planes):
        cur, src, E, Ks, invK, planes = ctx.saved_tensors
        lib = _native.load()
        dev = cur.device
        B, K, Cc, H, W = src.shape
        D = grad_cost.shape[1]
        shape = _native.Shape(B, K, Cc, H, W, D)
        # saved tensors are the dense aligned copies the forward made (see forward)
        cams = _native.Cameras(E.data_ptr(), None, Ks.data_ptr(), invK.data_ptr())
        pl = _native.Planes()
        pl.mode = _native.PLANES_PER_PIXEL if ctx.per_pixel else _native.PLANES_PER_PLANE
        pl.planes = planes.data_ptr()
        pl.min_depth = pl.max_depth = pl.ramp = pl.planes_out = None
        g = grad_cost.float().contiguous()
        with torch.cuda.device(dev):
            gcur = torch.empty_like(cur)
            gsrc = torch.empty_like(src)
            n = lib.srcv_dot_backward_workspace_bytes(C.byref(shape))
            ws = torch.empty(n, device=dev, dtype=torch.uint8)
            _native.check(lib.srcv_dot_backward_f32(
                C.byref(shape), _ptr(cur), _ptr(src), C.byref(cams), C.byref(pl), _ptr(g), _ptr(gcur),
                _ptr(gsrc), _ptr(ws), n, C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
        return (None, gcur.to(ctx.in_dtypes[0]), gsrc.to(ctx.in_dtypes[1]), None, None, None, None, None, None)


class _MlpVolumeFunction(torch.autograd.Function):
    """Differentiable wrapper of the metadata-MLP sweep: fused forward (tcgen05 where the
    shape allows), and ``srcv_mlp_backward_f32`` — a recompute kernel, nothing but the inputs
    is saved — for the two feature inputs and the six MLP parameters: what autograd of the
    reference composite (modules/cost_volume.py:451-736, modules/networks.py:129-147) yields.
    Cameras and plane depths get no gradient.  fp16 / bf16 features (autocast) are upcast."""

    @staticmethod
    def forward(ctx, mgr, return_mask, cur_feats, src_feats, src_extrinsics, src_poses, src_Ks, cur_invK,
                min_depth, max_depth, depth_planes_bdhw, w1, b1, w2, b2, w3, b3):
        dev = src_feats.device
        cur32, src32 = _f32c(cur_feats, "cur_feats", dev), _f32c(src_feats, "src_feats", dev)
        cams = [_f32c(t, n, dev) for t, n in ((src_extrinsics, "src_extrinsics"), (src_poses, "src_poses"),
                                              (src_Ks, "src_Ks"), (cur_invK, "cur_invK"))]
        _check_backward_supported("mlp", src32.shape, (w1.shape[0], w2.shape[0]))
        cost, lowest, planes_ret, mask = mgr._run_fused(
            cur32, src32, cams[0], cams[1], cams[2], cams[3], min_depth, max_depth, depth_planes_bdhw,
            return_mask, True, allow_grad=True)
        B, D, H, W = cost.shape
        st = planes_ret.stride()
        per_pixel = not ((st[2] == 0 or H == 1) and (st[3] == 0 or W == 1))
        planes = planes_ret[:, :D].contiguous() if per_pixel else planes_ret[:, :D, 0, 0].contiguous()
        ctx.save_for_backward(cur32, src32, *cams, planes, w1, b1, w2, b2, w3, b3)
        ctx.per_pixel = per_pixel
        ctx.in_dtypes = (cur_feats.dtype, src_feats.dtype)
        if mask is None:
            mask = torch.empty(0, dtype=torch.bool, device=cost.device)
        ctx.mark_non_differentiable(lowest, planes_ret, mask)
        return cost, lowest, planes_ret, mask

    @staticmethod
    def backward(ctx, grad_cost, _gl, _gp, _gm):
        cur, src, E, P, Ks, invK, planes, *wts = ctx.saved_tensors
        lib = _native.load()
        dev = cur.device
        B, K, Cc, H, W = src.shape
        D = grad_cost.shape[1]
        shape = _native.Shape(B, K, Cc, H, W, D)
        cams = _native.Cameras(E.data_ptr(), P.data_ptr(), Ks.data_ptr(), invK.data_ptr())
        pl = _native.Planes()
        pl.mode = _native.PLANES_PER_PIXEL if ctx.per_pixel else _native.PLANES_PER_PLANE
        pl.planes = planes.data_ptr()
        pl.min_depth = pl.max_depth = pl.ramp = pl.planes_out = None
        wc = [_f32c(t.detach(), "mlp parameter", dev) for t in wts]
        w = _native.MlpWeights(*[t.data_ptr() for t in wc], wc[0].shape[0], wc[2].shape[0], None)
        g = grad_cost.float().contiguous()
        with torch.cuda.device(dev):
            gcur, gsrc = torch.empty_like(cur), torch.empty_like(src)
            gw = [torch.empty_like(t) for t in wc]
            grads = _native.MlpGrads(*[t.data_ptr() for t in gw])
            n = lib.srcv_mlp_backward_workspace_bytes(C.byref(shape), C.byref(w))
            if n == 0:
                raise NotImplementedError("metadata-MLP backward: at most 208 input features, hidden widths <= 128")
            ws = torch.empty(n, device=dev, dtype=torch.uint8)
            _native.check(lib.srcv_mlp_backward_f32(
                C.byref(shape), _ptr(cur), _ptr(src), C.byref(cams), C.byref(pl), C.byref(w), _ptr(g),
                _ptr(gcur), _ptr(gsrc), C.byref(grads), _ptr(ws), n,
                C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
        gw = [a.to(b.dtype) for a, b in zip(gw, wts)]
        return (None, None, gcur.to(ctx.in_dtypes[0]), gsrc.to(ctx.in_dtypes[1]), None, None, None, None,
                None, None, None, *gw)


class CostVolumeManager(nn.Module):
    """Dot-product plane-sweep cost volume (reference modules/cost_volume.py:13-380).

    ``matching_dim_size`` and ``num_source_views`` are accepted and ignored, as in
    the reference (:27-34).
    """

    def __init__(self, matching_height, matching_width, num_depth_bins=64,
                 matching_dim_size=None, num_source_views=None):
        super().__init__()
        self.num_depth_bins = num_depth_bins
        self.matching_height = matching_height
        self.matching_width = matching_width
        self.initialise_for_projection()

    # -- reference :58-74 -----------------------------------------------------
    def initialise_for_projection(self):
        ramp = torch.linspace(0, 1, self.num_depth_bins).view(1, self.num_depth_bins, 1, 1)
        self.register_buffer("linear_ramp_1d11", ramp)
        self.backprojector = BackprojectDepth(height=self.matching_height, width=self.matching_width)
        self.projector = Project3D()

    # -- reference :77-97 -----------------------------------------------------
    def get_mask(self, pix_coords_bk2hw):
        x, y = pix_coords_bk2hw[:, :, 0], pix_coords_bk2hw[:, :, 1]
        return (x > 2) & (x < self.matching_width - 2) & (y > 2) & (y < self.matching_height - 2)

    # -- reference :100-136 ---------------------------------------------------
    def generate_depth_planes(self, batch_size: int, min_depth: Tensor, max_depth: Tensor) -> Tensor:
        ramp = self.linear_ramp_1d11.expand(batch_size, self.num_depth_bins, 1, 1)
        planes = torch.exp(torch.log(min_depth) + torch.log(max_depth / min_depth) * ramp)
        return planes.expand(batch_size, self.num_depth_bins, self.matching_height, self.matching_width)

    # -- reference :139-234 ---------------------------------------------------
    def warp_features(self, src_feats, src_extrinsics, src_Ks, cur_invK, depth_plane_b1hw,
                      batch_size, num_src_frames, num_feat_channels, uv_scale=None):
        """Warps every source view to the reference view at ONE depth plane and returns
        ``(world_points_B4N, depths, src_feat_warped, mask)`` like the reference helper.
        This is the materialising form the fused sweeps avoid; it is kept because the
        reference exposes it.  ``uv_scale`` is accepted and unused (the kernel works in
        pixel coordinates)."""
        lib = _native.load()
        dev = src_feats.device
        _require_cuda(dev)
        B, K, Cc = batch_size, num_src_frames, num_feat_channels
        H, W = self.matching_height, self.matching_width
        src = _f32c(src_feats, "src_feats", dev).reshape(B, K, Cc, H, W)
        E, Ks = _f32c(src_extrinsics, "src_extrinsics", dev), _f32c(src_Ks, "src_Ks", dev)
        invK = _f32c(cur_invK, "cur_invK", dev)
        plane = depth_plane_b1hw
        st = plane.stride()
        per_pixel = not ((st[2] == 0 or H == 1) and (st[3] == 0 or W == 1))
        plane_c = plane.contiguous().reshape(B, H * W) if per_pixel else plane[:, 0, 0, 0].contiguous()
        shape = _native.Shape(B, K, Cc, H, W, 1)
        cams = _native.Cameras(E.data_ptr(), None, Ks.data_ptr(), invK.data_ptr())
        with torch.cuda.device(dev):
            warped = torch.empty(B, K, Cc, H, W, device=dev, dtype=torch.float32)
            depths = torch.empty(B, K, H, W, device=dev, dtype=torch.float32)
            mask = torch.empty(B, K, H, W, device=dev, dtype=torch.float32)
            n = lib.srcv_warp_workspace_bytes(C.byref(shape))
            ws = torch.empty(n, device=dev, dtype=torch.uint8)
            _native.check(lib.srcv_warp_features_f32(
                C.byref(shape), _ptr(src), C.byref(cams), _ptr(plane_c), int(per_pixel), _ptr(warped),
                _ptr(depths), _ptr(mask), _ptr(ws), n,
                C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
        world_points_b4N = self.backprojector(depth_plane_b1hw.expand(B, 1, H, W), invK)
        return world_points_b4N.repeat_interleave(K, dim=0), depths, warped, mask

    # -- reference :338-342 ---------------------------------------------------
    def indices_to_disparity(self, indices, depth_planes_bdhw):
        return torch.gather(depth_planes_bdhw, dim=1, index=indices.unsqueeze(1)).squeeze(1)

    # ------------------------------------------------------------------------
    # shared argument handling
    # ------------------------------------------------------------------------
    def _prepare(self, cur_feats, src_feats, src_extrinsics, src_poses, src_Ks, cur_invK,
                 min_depth, max_depth, depth_planes_bdhw, need_poses, allow_grad=False, raw_poses=None):
        # chunk-planar features (B,K,C/4,H,W,4) / (B,C/4,H,W,4), e.g. from
        # instance_norm_to_chunk_planar(): gathered in place, the prep pass makes no copy
        chunk_planar = torch.is_tensor(src_feats) and src_feats.dim() == 6 and src_feats.shape[-1] == 4
        if chunk_planar:
            if cur_feats.dim() != 5 or cur_feats.shape[-1] != 4:
                raise ValueError("chunk-planar src_feats (B,K,C/4,H,W,4) need chunk-planar cur_feats (B,C/4,H,W,4)")
            if allow_grad or (torch.is_grad_enabled() and (cur_feats.requires_grad or src_feats.requires_grad)):
                raise NotImplementedError("the backward kernels take the reference's NCHW features")
            src_view = src_feats.permute(0, 1, 2, 5, 3, 4).flatten(2, 3)      # logical (B,K,C,H,W) view: shapes only
            cur_view = cur_feats.permute(0, 1, 4, 2, 3).flatten(1, 2)
        else:
            src_view, cur_view = src_feats, cur_feats
        if not torch.is_tensor(src_feats) or src_view.dim() != 5:
            raise ValueError("src_feats must be a (B,K,C,H,W) tensor")
        dev = src_feats.device
        _require_cuda(dev)
        if not allow_grad and torch.is_grad_enabled() and (
                cur_feats.requires_grad or src_feats.requires_grad
                or any(p.requires_grad for p in self.parameters())
        ):
            raise RuntimeError("internal: a gradient-requiring call reached the plain fused path")
        B, K, Cc, H, W = src_view.shape
        if (H, W) != (self.matching_height, self.matching_width):
            raise ValueError(f"feature map {H}x{W} does not match the manager's "
                             f"{self.matching_height}x{self.matching_width}")
        if tuple(cur_view.shape) != (B, Cc, H, W):
            raise ValueError(f"cur_feats shape {tuple(cur_view.shape)} != {(B, Cc, H, W)}")
        raw = raw_poses is not None
        checks = [("src_Ks", src_Ks, (B, K, 4, 4)), ("cur_invK", cur_invK, (B, 4, 4))]
        if raw:
            # the prep kernel forms src_cam_T_cur_cam / cur_cam_T_src_cam itself (depth_model.py:324-332)
            checks += [("src_cam_T_world", raw_poses["src_cam_T_world"], (B, K, 4, 4)),
                       ("src_world_T_cam", raw_poses["src_world_T_cam"], (B, K, 4, 4)),
                       ("cur_cam_T_world", raw_poses["cur_cam_T_world"], (B, 4, 4)),
                       ("cur_world_T_cam", raw_poses["cur_world_T_cam"], (B, 4, 4))]
        else:
            checks.append(("src_extrinsics", src_extrinsics, (B, K, 4, 4)))
            if need_poses:
                checks.append(("src_poses", src_poses, (B, K, 4, 4)))
        for name, tt, shp in checks:
            if tuple(tt.shape) != shp:
                raise ValueError(f"{name} shape {tuple(tt.shape)} != {shp}")
        t = dict(
            cur=_f32c(cur_feats, "cur_feats", dev), src=_f32c(src_feats, "src_feats", dev),
            E=None if raw else _f32c(src_extrinsics, "src_extrinsics", dev), Ks=_f32c(src_Ks, "src_Ks", dev),
            invK=_f32c(cur_invK, "cur_invK", dev),
            poses=_f32c(src_poses, "src_poses", dev) if (need_poses and not raw) else None,
        )
        if raw:
            for k in ("src_cam_T_world", "src_world_T_cam", "cur_cam_T_world", "cur_world_T_cam"):
                t[k] = _f32c(raw_poses[k], k, dev)
        D = self.num_depth_bins
        pl = _native.Planes()
        keep = []
        if depth_planes_bdhw is None:
            mn = _f32c(min_depth.to(dev), "min_depth", dev).reshape(-1)
            mx = _f32c(max_depth.to(dev), "max_depth", dev).reshape(-1)
            # one range for the batch ((1,1,1,1), depth_model.py:358-359) or one per frame
            # ((B,1,1,1): generate_depth_planes broadcasts it, reference :124-127)
            if mn.numel() != mx.numel() or mn.numel() not in (1, B):
                raise ValueError("min_depth / max_depth must hold one value or one value per frame "
                                 f"(got {mn.numel()} / {mx.numel()} for a batch of {B})")
            pl.range_per_frame = int(mn.numel() == B and B > 1)
            ramp = _f32c(self.linear_ramp_1d11, "linear_ramp_1d11", dev).reshape(-1)
            planes_bd = torch.empty(B, D, device=dev, dtype=torch.float32)
            pl.mode = _native.PLANES_FROM_RANGE
            pl.planes, pl.min_depth, pl.max_depth = None, mn.data_ptr(), mx.data_ptr()
            pl.ramp, pl.planes_out = ramp.data_ptr(), planes_bd.data_ptr()
            keep += [mn, mx, ramp]
            planes_ret = planes_bd.view(B, D, 1, 1).expand(B, D, H, W)   # expanded view, like :129-134
        else:
            if depth_planes_bdhw.dim() != 4 or tuple(depth_planes_bdhw.shape[::2]) != (B, H) \
                    or depth_planes_bdhw.shape[3] != W:
                raise ValueError("depth_planes_bdhw must be (B,D,H,W)")
            # the per-plane managers sweep the first `num_depth_bins` planes (:305, :557);
            # the fast one takes the tensor's own plane count (:1065)
            D = depth_planes_bdhw.shape[1] if isinstance(self, FastFeatureVolumeManager) \
                else self.num_depth_bins
            if depth_planes_bdhw.shape[1] < D:
                raise ValueError(f"depth_planes_bdhw holds {depth_planes_bdhw.shape[1]} planes, "
                                 f"the manager sweeps {D}")
            if depth_planes_bdhw.dtype != torch.float32 or depth_planes_bdhw.device != dev:
                raise ValueError("depth_planes_bdhw must be float32 on the features' device")
            st = depth_planes_bdhw.stride()
            if (st[2] == 0 or H == 1) and (st[3] == 0 or W == 1):
                per = depth_planes_bdhw[:, :D, 0, 0].contiguous()
                pl.mode = _native.PLANES_PER_PLANE
            else:
                per = depth_planes_bdhw[:, :D].contiguous()
                pl.mode = _native.PLANES_PER_PIXEL
            pl.planes = per.data_ptr()
            pl.min_depth = pl.max_depth = pl.ramp = pl.planes_out = None
            keep.append(per)
            planes_ret = depth_planes_bdhw
        shape = _native.Shape(B, K, Cc, H, W, D,
                              _native.LAYOUT_CHUNK_PLANAR if chunk_planar else _native.LAYOUT_NCHW)
        if raw:
            cams = _native.Cameras(None, None, t["Ks"].data_ptr(), t["invK"].data_ptr(),
                                   t["src_cam_T_world"].data_ptr(), t["cur_world_T_cam"].data_ptr(),
                                   t["cur_cam_T_world"].data_ptr(), t["src_world_T_cam"].data_ptr())
        else:
            cams = _native.Cameras(t["E"].data_ptr(), t["poses"].data_ptr() if need_poses else None,
                                   t["Ks"].data_ptr(), t["invK"].data_ptr())
        return dev, shape, t, cams, pl, planes_ret, keep

    # -- reference :237-335 ---------------------------------------------------
    def build_cost_volume(self, cur_feats: Tensor, src_feats: Tensor, src_extrinsics: Tensor,
                          src_poses: Tensor, src_Ks: Tensor, cur_invK: Tensor, min_depth: Tensor,
                          max_depth: Tensor, depth_planes_bdhw: Tensor = None,
                          return_mask: bool = False):
        cost, _, planes, mask = self._run(cur_feats, src_feats, src_extrinsics, src_poses, src_Ks,
                                          cur_invK, min_depth, max_depth, depth_planes_bdhw,
                                          return_mask, want_lowest=False)
        return cost, planes, mask

    def _run(self, cur_feats, src_feats, src_extrinsics, src_poses, src_Ks, cur_invK, min_depth,
             max_depth, depth_planes_bdhw, return_mask, want_lowest, raw_poses=None):
        # `src_poses` and `return_mask` are ignored by the dot-product volume (:286)
        if torch.is_grad_enabled() and (cur_feats.requires_grad or src_feats.requires_grad):
            if raw_poses is not None or cur_feats.dim() != 4:
                raise NotImplementedError("raw_poses / chunk-planar features are inference-path options")
            # training: same fused forward, gradients w.r.t. the features by the backward kernel
            cost, lowest, planes_ret = _DotVolumeFunction.apply(
                self, cur_feats, src_feats, src_extrinsics, src_Ks, cur_invK, min_depth, max_depth,
                depth_planes_bdhw)
            return cost, (lowest if want_lowest else None), planes_ret, None
        return self._run_fused(cur_feats, src_feats, src_extrinsics, src_poses, src_Ks, cur_invK,
                               min_depth, max_depth, depth_planes_bdhw, want_lowest, raw_poses=raw_poses)

    def _run_fused(self, cur_feats, src_feats, src_extrinsics, src_poses, src_Ks, cur_invK, min_depth,
                   max_depth, depth_planes_bdhw, want_lowest, allow_grad=False, raw_poses=None):
        lib = _native.load()
        dev, shape, t, cams, pl, planes_ret, keep = self._prepare(
            cur_feats, src_feats, src_extrinsics, src_poses, src_Ks, cur_invK, min_depth,
            max_depth, depth_planes_bdhw, need_poses=False, allow_grad=allow_grad, raw_poses=raw_poses)
        with torch.cuda.device(dev):
            cost = torch.empty(shape.B, shape.D, shape.H, shape.W, device=dev, dtype=torch.float32)
            lowest = torch.empty(shape.B, shape.H, shape.W, device=dev, dtype=torch.float32) \
                if want_lowest else None
            nbytes = lib.srcv_dot_workspace_bytes(C.byref(shape))
            ws = torch.empty(nbytes, device=dev, dtype=torch.uint8)
            stream = torch.cuda.current_stream(dev).cuda_stream
            _native.check(lib.srcv_dot_forward_f32(
                C.byref(shape), _ptr(t["cur"]), _ptr(t["src"]), C.byref(cams), C.byref(pl),
                _ptr(cost), _ptr(lowest), _ptr(ws), nbytes, C.c_void_p(stream)))
        return cost, lowest, planes_ret, None

    # -- reference :345-380 ---------------------------------------------------
    def forward(self, cur_feats, src_feats, src_extrinsics, src_poses, src_Ks, cur_invK,
                min_depth, max_depth, depth_planes_bdhw=None, return_mask=False, raw_poses=None):
        """Returns ``(cost_volume, lowest_cost, depth_planes_bdhw, overall_mask_bhw)``.
        ``lowest_cost`` is the plane depth at the ARGMAX of the volume, as in the
        reference (:374-378).

        Two producer-side extensions beyond the reference's call (SURVEY.md §8f-2), both optional:
        ``cur_feats`` / ``src_feats`` may be CHUNK-PLANAR tensors ``(B,C/4,H,W,4)`` / ``(B,K,C/4,H,W,4)``
        (``instance_norm_to_chunk_planar``), which the kernels gather in place; and ``raw_poses`` =
        ``dict(src_cam_T_world, src_world_T_cam, cur_cam_T_world, cur_world_T_cam)`` makes the prep
        kernel form the relative transforms of experiment_modules/depth_model.py:324-332 itself
        (``src_extrinsics`` / ``src_poses`` are then ignored and may be None)."""
        return self._run(cur_feats, src_feats, src_extrinsics, src_poses, src_Ks, cur_invK,
                         min_depth, max_depth, depth_planes_bdhw, return_mask, want_lowest=True,
                         raw_poses=raw_poses)


class FeatureVolumeManager(CostVolumeManager):
    """Metadata-MLP plane-sweep volume (reference modules/cost_volume.py:383-746)."""

    _banner = "FeatureVolumeManager"

    def __init__(self, matching_height, matching_width, num_depth_bins=64,
                 mlp_channels=[202, 128, 128, 1], matching_dim_size=16, num_source_views=7):
        super().__init__(matching_height, matching_width, num_depth_bins)
        # channel bookkeeping of :420-435.  The shared default list is updated in place,
        # exactly like the reference (:429) — callers relying on that quirk keep working.
        mlp_channels[0] = (matching_dim_size * (1 + num_source_views)   # visual
                           + (1 + num_source_views)                      # depths
                           + 3 * (1 + num_source_views)                  # rays
                           + num_source_views                            # ray angles
                           + num_source_views                            # masks
                           + num_source_views                            # dots
                           + 3 * num_source_views)                       # pose measures
        self.mlp = MLP(channel_list=mlp_channels, disable_final_activation=True)
        print(f" simplerecon_b200 {self._banner}: {num_source_views} source views, "
              f"MLP channels {mlp_channels} (sm_100a fused sweep) ")

    def _mlp_weights(self, dev, n_features):
        lin = [m for m in self.mlp.net if isinstance(m, nn.Linear)]
        acts = [m for m in self.mlp.net if not isinstance(m, nn.Linear)]
        if len(lin) != 3 or len(self.mlp.net) != 5 or not all(isinstance(a, nn.LeakyReLU) for a in acts) \
                or any(abs(a.negative_slope - 0.01) > 0 for a in acts) or lin[2].out_features != 1:
            raise NotImplementedError(
                "the fused kernels implement the reference's F->H1->H2->1 LeakyReLU(0.01) MLP; "
                f"got {self.mlp.net}")
        if lin[0].in_features != n_features:
            raise ValueError(f"MLP expects {lin[0].in_features} input channels but K and C of the "
                             f"inputs give {n_features}")
        ts = []
        for l in lin:
            if l.bias is None:
                raise NotImplementedError("MLP layers without bias are not supported")
            ts += [_f32c(l.weight.detach(), "mlp weight", dev), _f32c(l.bias.detach(), "mlp bias", dev)]
        w = _native.MlpWeights(*[x.data_ptr() for x in ts], lin[0].out_features, lin[1].out_features, None)
        return w, ts

    def _attach_packed_image(self, dev, shape, w):
        """Points ``w.packed_image`` at the tensor-core kernel's fp16 weight image, re-packing it
        (``srcv_mlp_pack_weights``) only when a parameter changed.  The cache key is, for every
        ``weight`` / ``bias`` of the MLP's linear layers, the Parameter's identity, storage
        address, version counter and dtype — of the parameters themselves, not of the fp32
        copies ``_f32c`` makes of fp16 / bf16 weights, which are fresh tensors at version 0 on
        every call.  So replacing a Parameter, ``load_state_dict``, an optimizer step or any
        other in-place update re-packs, also under ``no_grad`` / ``inference_mode``.  Writes
        through ``.data`` bypass the version counter and are not seen.  Returns what must
        stay alive."""
        lib = _native.load()
        nbytes = lib.srcv_mlp_packed_bytes(C.byref(shape), C.byref(w))
        if nbytes == 0:
            return None                                   # SIMT variant: nothing to pack
        params = [p for l in self.mlp.net if isinstance(l, nn.Linear) for p in (l.weight, l.bias)]
        try:
            key = (str(dev), tuple((id(p), p.data_ptr(), p._version, p.dtype) for p in params))
        except RuntimeError:                              # parameters created under inference_mode
            key = None                                    # carry no version counter: pack every call
        cache = self.__dict__.get("_srcv_packed")
        if key is None or cache is None or cache[0] != key:
            with torch.cuda.device(dev):
                image = torch.empty(nbytes, device=dev, dtype=torch.uint8)
                _native.check(lib.srcv_mlp_pack_weights(
                    C.byref(shape), C.byref(w), _ptr(image),
                    C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
            cache = (key, image)
            self.__dict__["_srcv_packed"] = cache         # plain attribute: not a buffer, not in state_dict
        w.packed_image = cache[1].data_ptr()
        return cache[1]

    def _run(self, cur_feats, src_feats, src_extrinsics, src_poses, src_Ks, cur_invK, min_depth,
             max_depth, depth_planes_bdhw, return_mask, want_lowest, raw_poses=None):
        if torch.is_grad_enabled() and (cur_feats.requires_grad or src_feats.requires_grad
                                        or any(p.requires_grad for p in self.mlp.parameters())):
            if raw_poses is not None or cur_feats.dim() != 4:
                raise NotImplementedError("raw_poses / chunk-planar features are inference-path options")
            # training: same fused forward; gradients for features and MLP parameters by the
            # recompute backward kernel (srcv_mlp_backward_f32)
            lin = [m for m in self.mlp.net if isinstance(m, nn.Linear)]
            if len(lin) != 3 or any(l.bias is None for l in lin):
                raise NotImplementedError("the fused kernels implement the reference's three-layer MLP with biases")
            cost, lowest, planes_ret, mask = _MlpVolumeFunction.apply(
                self, bool(return_mask), cur_feats, src_feats, src_extrinsics, src_poses, src_Ks, cur_invK,
                min_depth, max_depth, depth_planes_bdhw, lin[0].weight, lin[0].bias, lin[1].weight,
                lin[1].bias, lin[2].weight, lin[2].bias)
            return cost, (lowest if want_lowest else None), planes_ret, (mask if return_mask else None)
        return self._run_fused(cur_feats, src_feats, src_extrinsics, src_poses, src_Ks, cur_invK, min_depth,
                               max_depth, depth_planes_bdhw, return_mask, want_lowest, raw_poses=raw_poses)

    def _run_fused(self, cur_feats, src_feats, src_extrinsics, src_poses, src_Ks, cur_invK, min_depth,
                   max_depth, depth_planes_bdhw, return_mask, want_lowest, allow_grad=False, raw_poses=None):
        lib = _native.load()
        dev, shape, t, cams, pl, planes_ret, keep = self._prepare(
            cur_feats, src_feats, src_extrinsics, src_poses, src_Ks, cur_invK, min_depth,
            max_depth, depth_planes_bdhw, need_poses=True, allow_grad=allow_grad, raw_poses=raw_poses)
        n_features = shape.C * (shape.K + 1) + 10 * shape.K + 4
        w, wkeep = self._mlp_weights(dev, n_features)
        wkeep.append(self._attach_packed_image(dev, shape, w))
        with torch.cuda.device(dev):
            cost = torch.empty(shape.B, shape.D, shape.H, shape.W, device=dev, dtype=torch.float32)
            lowest = torch.empty(shape.B, shape.H, shape.W, device=dev, dtype=torch.float32) \
                if want_lowest else None
            mask = torch.empty(shape.B, shape.H, shape.W, device=dev, dtype=torch.uint8) \
                if return_mask else None
            nbytes = lib.srcv_mlp_workspace_bytes(C.byref(shape), C.byref(w))
            if nbytes == 0:
                raise NotImplementedError(
                    f"MLP widths ({w.hidden1},{w.hidden2}) are not supported by the fused kernels")
            ws = torch.empty(nbytes, device=dev, dtype=torch.uint8)
            stream = torch.cuda.current_stream(dev).cuda_stream
            _native.check(lib.srcv_mlp_forward_f32(
                C.byref(shape), _ptr(t["cur"]), _ptr(t["src"]), C.byref(cams), C.byref(pl),
                C.byref(w), _ptr(cost), _ptr(lowest), _ptr(mask), _ptr(ws), nbytes,
                C.c_void_p(stream)))
        return cost, lowest, planes_ret, (mask.bool() if mask is not None else None)

    # -- reference :739-746 ---------------------------------------------------
    def to_fast(self) -> "FastFeatureVolumeManager":
        manager = FastFeatureVolumeManager(self.matching_height, self.matching_width,
                                           num_depth_bins=self.num_depth_bins)
        manager.mlp = self.mlp
        return manager


class FastFeatureVolumeManager(FeatureVolumeManager):
    """Same volume as ``FeatureVolumeManager``; in the reference (:749-1164) this class
    trades 550 MB + 993 MB of materialised tensors per frame for fewer launches.  The
    fused kernel has neither cost, so both classes run the same sweep; the subclass
    exists because ``test.py:196-198`` swaps it in via ``to_fast()``."""

    _banner = "FastFeatureVolumeManager"

    def __init__(self, matching_height, matching_width, num_depth_bins=64,
                 mlp_channels=[202, 128, 128, 1], matching_dim_size=16, num_source_views=7):
        super().__init__(matching_height, matching_width, num_depth_bins, mlp_channels,
                         matching_dim_size, num_source_views)

    # -- reference :812-964 ---------------------------------------------------
    def warp_features(self, src_feats, src_extrinsics, src_Ks, cur_invK, depth_plane_bdhw,
                      batch_size, num_src_frames, num_feat_channels, uv_scale=None):
        """Warps every source view to the reference view at EVERY plane of ``depth_plane_bdhw``
        and returns the reference's 5-tuple ``(world_points_bkd4hw, depths_bkdhw,
        src_feat_warped_bkdfhw, mask_bkdhw, pix_coords_bkd2hw)``.  This is the materialising
        form (550 MB per frame at the hero shape) the fused sweep avoids; it exists because the
        reference exposes it.  ``uv_scale`` is accepted and unused (the kernel works in pixel
        coordinates)."""
        lib = _native.load()
        dev = src_feats.device
        _require_cuda(dev)
        B, K, Cc = batch_size, num_src_frames, num_feat_channels
        H, W = self.matching_height, self.matching_width
        D = depth_plane_bdhw.shape[1]
        src = _f32c(src_feats, "src_feats", dev).reshape(B, K, Cc, H, W)
        E, Ks = _f32c(src_extrinsics, "src_extrinsics", dev), _f32c(src_Ks, "src_Ks", dev)
        invK = _f32c(cur_invK, "cur_invK", dev)
        st = depth_plane_bdhw.stride()
        per_pixel = not ((st[2] == 0 or H == 1) and (st[3] == 0 or W == 1))
        planes = _f32c(depth_plane_bdhw if per_pixel else depth_plane_bdhw[:, :, 0, 0], "depth_plane_bdhw", dev)
        shape = _native.Shape(B, K, Cc, H, W, D)
        cams = _native.Cameras(E.data_ptr(), None, Ks.data_ptr(), invK.data_ptr())
        with torch.cuda.device(dev):
            warped = torch.empty(B, K, D, Cc, H, W, device=dev, dtype=torch.float32)
            depths = torch.empty(B, K, D, H, W, device=dev, dtype=torch.float32)
            mask = torch.empty(B, K, D, H, W, device=dev, dtype=torch.float32)
            pix = torch.empty(B, K, D, 2, H, W, device=dev, dtype=torch.float32)
            n = lib.srcv_warp_workspace_bytes(C.byref(shape))
            ws = torch.empty(n, device=dev, dtype=torch.uint8)
            _native.check(lib.srcv_warp_features_planes_f32(
                C.byref(shape), _ptr(src), C.byref(cams), _ptr(planes), int(per_pixel), _ptr(warped),
                _ptr(depths), _ptr(mask), _ptr(pix), _ptr(ws), n,
                C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
        # world points of every plane (:857-873): X = depth * (invK3 @ p), homogeneous
        world = self.backprojector(depth_plane_bdhw.reshape(B * D, 1, H, W).expand(B * D, 1, H, W),
                                   invK.repeat_interleave(D, dim=0))
        world = world.reshape(B, 1, D, 4, H, W).expand(B, K, D, 4, H, W)
        return world, depths, warped, mask, pix
