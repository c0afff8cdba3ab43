/*
 * srcv_b200 — C ABI of the B200-native plane-sweep cost-volume library.
 *
 * This is the drop-in boundary for SimpleRecon's cost-volume hot path.  The
 * reference has no native layer (it is pure PyTorch), so each entry point below
 * names the reference *Python* interface it replaces; the Python classes in
 * simplerecon_b200/cost_volume.py bind these symbols through ctypes and keep the
 * reference's class / method signatures (see INTEGRATION.md for the binding a
 * maintainer of the reference would add).
 *
 * Conventions
 *   - plain C types only: device pointers, sizes, an opaque stream handle
 *     (a cudaStream_t passed as void*; NULL = legacy default stream);
 *   - all tensors are fp32, contiguous, row-major in the reference's layouts;
 *   - outputs and the workspace are caller-allocated (the Python side hands
 *     PyTorch caching-allocator memory); nothing is allocated, freed or retained
 *     by the library, and no call synchronises the device: work is enqueued on
 *     `stream` and the call returns;
 *   - every function returns an srcv_status (0 = ok).  Argument errors are
 *     detected on the host before anything is launched; CUDA launch errors are
 *     returned as SRCV_ERR_CUDA with the text available from srcv_last_error().
 */
#ifndef SRCV_B200_H_
#define SRCV_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SRCV_ABI_VERSION 2

typedef enum srcv_status {
  SRCV_OK = 0,
  SRCV_ERR_NULL = 1,        /* a required pointer is NULL                      */
  SRCV_ERR_SHAPE = 2,       /* a dimension is <= 0 or out of the supported set */
  SRCV_ERR_WORKSPACE = 3,   /* workspace too small or misaligned               */
  SRCV_ERR_UNSUPPORTED = 4, /* valid request this build cannot serve           */
  SRCV_ERR_CUDA = 5,        /* CUDA runtime error (see srcv_last_error)        */
  SRCV_ERR_DEVICE = 6       /* current device is not an sm_100 part            */
} srcv_status;

/* Problem shape.  Mirrors the tensor contract of
 * CostVolumeManager.forward (reference modules/cost_volume.py:345-380):
 *   cur_feats (B,C,H,W)  src_feats (B,K,C,H,W)  cost (B,D,H,W).          */
typedef struct srcv_shape {
  int32_t B; /* reference frames in this call (batch)                        */
  int32_t K; /* source views per frame                                       */
  int32_t C; /* matching-feature channels                                    */
  int32_t H; /* matching feature-map height                                  */
  int32_t W; /* matching feature-map width                                   */
  int32_t D; /* depth planes                                                 */
  int32_t layout; /* srcv_feature_layout of cur_feats / src_feats (0 = the reference's NCHW)  */
} srcv_shape;

/* Memory layout of the two feature inputs.  CHUNK_PLANAR is what the gather kernels read
 * internally — cur_feats (B,C/4,H,W,4), src_feats (B,K,C/4,H,W,4): a texel's 4-channel chunk is
 * one 16-byte vector — and what srcv_instnorm_to_chunk_planar_f32 produces: a caller that
 * hands it over skips the re-layout copy of the prep pass (SURVEY.md §8f-2).  Served by the
 * chunk-planar dot sweep (C == 16) and the tensor-core MLP sweep (K == 7, C == 16, 128/128);
 * other shapes return SRCV_ERR_UNSUPPORTED.                                               */
typedef enum srcv_feature_layout {
  SRCV_LAYOUT_NCHW = 0,
  SRCV_LAYOUT_CHUNK_PLANAR = 1
} srcv_feature_layout;

/* How the depth hypotheses are given. */
typedef enum srcv_planes_mode {
  /* planes == NULL on input: the library evaluates
   *   d_i = exp(log(min) + log(max/min) * ramp_i)
   * (reference modules/cost_volume.py:100-136) from the DEVICE scalars
   * min_depth / max_depth and the DEVICE ramp (D floats, the module buffer
   * `linear_ramp_1d11`) and writes the (B,D) result to planes_out.          */
  SRCV_PLANES_FROM_RANGE = 0,
  /* planes is a DEVICE (B,D) array: one depth per plane and frame.         */
  SRCV_PLANES_PER_PLANE = 1,
  /* planes is a DEVICE (B,D,H,W) array: caller-supplied per-pixel
   * hypotheses (the `depth_planes_bdhw` argument, modules/cost_volume.py:247) */
  SRCV_PLANES_PER_PIXEL = 2
} srcv_planes_mode;

typedef struct srcv_planes {
  int32_t mode;            /* srcv_planes_mode                               */
  const float* planes;     /* (B,D) or (B,D,H,W); NULL for FROM_RANGE        */
  const float* min_depth;  /* device scalar, FROM_RANGE only                 */
  const float* max_depth;  /* device scalar, FROM_RANGE only                 */
  const float* ramp;       /* device (D), FROM_RANGE only                    */
  float* planes_out;       /* device (B,D), FROM_RANGE only (may be NULL)    */
  int32_t range_per_frame; /* FROM_RANGE: 0 = min/max_depth are single scalars (the
                            * (1,1,1,1) tensors of depth_model.py:358-359); 1 = B values each,
                            * one range per frame (generate_depth_planes broadcasts a
                            * (B,1,1,1) range, modules/cost_volume.py:124-127)  */
} srcv_planes;

/* Camera block shared by both volumes (all DEVICE pointers). */
typedef struct srcv_cameras {
  const float* src_extrinsics; /* (B,K,4,4) src_cam_T_cur_cam               */
  const float* src_poses;      /* (B,K,4,4) cur_cam_T_src_cam (MLP volume only; may be NULL for dot) */
  const float* src_Ks;         /* (B,K,4,4) source intrinsics at matching scale */
  const float* cur_invK;       /* (B,4,4) inverse intrinsics of the reference frame */
  /* Optional raw poses (SURVEY.md §8f-2).  When src_extrinsics is NULL the prep kernel forms
   *   src_cam_T_cur_cam = src_cam_T_world @ cur_world_T_cam          (-> src_extrinsics)
   *   cur_cam_T_src_cam = cur_cam_T_world @ src_world_T_cam          (-> src_poses)
   * itself — the two batched 4x4 products experiment_modules/depth_model.py:324-332 runs in
   * PyTorch before the call — evaluated in fp64 and rounded to fp32.  All four DEVICE pointers
   * are then required ((B,K,4,4), (B,4,4), (B,4,4), (B,K,4,4)); ignored otherwise.        */
  const float* src_cam_T_world;
  const float* cur_world_T_cam;
  const float* cur_cam_T_world;
  const float* src_world_T_cam;
} srcv_cameras;

/* Weights of the matching MLP — the parameters of the reference's
 * `MLP([F,H1,H2,1], disable_final_activation=True)` (modules/networks.py:129-147),
 * in nn.Linear layout (out_features, in_features), LeakyReLU slope 0.01.    */
typedef struct srcv_mlp_weights {
  const float* w1; const float* b1; /* (H1,F), (H1)  F = C*(K+1)+10*K+4       */
  const float* w2; const float* b2; /* (H2,H1), (H2)                          */
  const float* w3; const float* b3; /* (1,H2), (1)                            */
  int32_t hidden1;                  /* H1                                     */
  int32_t hidden2;                  /* H2                                     */
  /* Optional: DEVICE image written by srcv_mlp_pack_weights for exactly these weights
   * (srcv_mlp_packed_bytes bytes, 256-byte aligned).  NULL = the forward call packs the
   * weights itself, into its workspace, on every call.  A caller whose parameters change
   * rarely (inference; one optimiser step per forward in training) packs once per change.  */
  const void* packed_image;
} srcv_mlp_weights;

/* ---- library / device ------------------------------------------------- */
int32_t srcv_abi_version(void);
/* 0 if the CURRENT CUDA device can run this library (compute capability 10.x),
 * else SRCV_ERR_DEVICE / SRCV_ERR_CUDA.                                      */
int32_t srcv_check_device(void);
const char* srcv_status_string(int32_t status);
/* Thread-local text of the last SRCV_ERR_* raised on this thread.           */
const char* srcv_last_error(void);

/* ---- dot-product volume ----------------------------------------------- *
 * Replaces CostVolumeManager.build_cost_volume + the argmax in
 * CostVolumeManager.forward (reference modules/cost_volume.py:237-335,
 * :345-380): per plane, homography-warp every source feature map into the
 * reference frustum (bilinear, zeros padding, align_corners=False), dot it with
 * the reference features, mask by depth validity, sum over views.
 *   cost   (B,D,H,W) out
 *   lowest (B,H,W)   out, plane depth at argmax_d cost (first index on ties);
 *                    NULL to skip.                                           */
size_t srcv_dot_workspace_bytes(const srcv_shape* shape);
int32_t srcv_dot_forward_f32(const srcv_shape* shape,
                             const float* cur_feats, const float* src_feats,
                             const srcv_cameras* cams, const srcv_planes* planes,
                             float* cost, float* lowest,
                             void* workspace, size_t workspace_bytes,
                             void* stream);

/* ---- backward of the dot-product volume (training) ----------------------- *
 * Gradients of a scalar loss w.r.t. the FEATURE inputs of srcv_dot_forward_f32, given
 * grad_cost = dL/dcost (B,D,H,W) — what autograd of the reference's composite
 * (modules/cost_volume.py:305-333: grid_sample, mul, sum) yields for cur_feats and
 * src_feats.  Cameras and plane depths get no gradient.  C must be 8, 16 or 32.
 *   grad_cur (B,C,H,W) out      grad_src (B,K,C,H,W) out (zeroed here, then accumulated
 *   with float atomics: reproducible to fp32 rounding, not bit-for-bit)           */
size_t srcv_dot_backward_workspace_bytes(const srcv_shape* shape);
/* 1 if srcv_dot_backward_f32 serves this shape (C in {8,16,32}), else 0 — lets the caller
 * refuse an unsupported training shape in forward() instead of at backward() time.          */
int32_t srcv_dot_backward_supported(const srcv_shape* shape);
int32_t srcv_dot_backward_f32(const srcv_shape* shape, const float* cur_feats, const float* src_feats,
                              const srcv_cameras* cams, const srcv_planes* planes,
                              const float* grad_cost, float* grad_cur, float* grad_src,
                              void* workspace, size_t workspace_bytes, void* stream);

/* ---- single-plane warp -------------------------------------------------- *
 * Replaces CostVolumeManager.warp_features (reference modules/cost_volume.py:139-234),
 * the helper that MATERIALISES the warped source features of one depth plane; the
 * sweeps above never call it (they keep the warped values in registers / TMEM), it is
 * exported because the reference exposes it as a method.  shape->D is ignored.
 *   depth_plane  DEVICE (B) one depth per frame, or (B,H,W) when per_pixel != 0
 *   warped (B,K,C,H,W)  depths (B,K,H,W) = z' of the plane point in each source camera
 *   mask   (B,K,H,W)    1.0 where z' > 0                                         */
size_t srcv_warp_workspace_bytes(const srcv_shape* shape);
int32_t srcv_warp_features_f32(const srcv_shape* shape, const float* src_feats,
                               const srcv_cameras* cams, const float* depth_plane,
                               int32_t per_pixel, float* warped, float* depths, float* mask,
                               void* workspace, size_t workspace_bytes, void* stream);

/* All planes at once: replaces FastFeatureVolumeManager.warp_features (reference
 * modules/cost_volume.py:812-964), which materialises the warped features of EVERY plane
 * (550 MB per frame at the hero shape) — exported for callers of that method; the sweeps
 * never call it.  shape->D = number of planes.
 *   depth_planes DEVICE (B,D), or (B,D,H,W) when per_pixel != 0
 *   warped (B,K,D,C,H,W)   depths, mask (B,K,D,H,W)
 *   pix_coords (B,K,D,2,H,W): the projected pixel coordinates (x, y); NULL to skip        */
int32_t srcv_warp_features_planes_f32(const srcv_shape* shape, const float* src_feats,
                                      const srcv_cameras* cams, const float* depth_planes,
                                      int32_t per_pixel, float* warped, float* depths, float* mask,
                                      float* pix_coords, void* workspace, size_t workspace_bytes,
                                      void* stream);

/* ---- metadata-MLP volume ---------------------------------------------- *
 * Replaces FeatureVolumeManager.build_cost_volume /
 * FastFeatureVolumeManager.build_cost_volume + the argmax in forward
 * (reference modules/cost_volume.py:451-736, :967-1164): builds the per
 * (plane,pixel) metadata vector (warped features, reference features, validity,
 * source depths, plane depth, per-view dot, ray angle, rays, pose measures —
 * order of :698-723) and runs the matching MLP on it, without materialising it.
 *   overall_mask (B,H,W) uint8 out (1 = some source view sees the pixel at the
 *   LAST plane, :625-637); NULL when return_mask is False.                   */
size_t srcv_mlp_workspace_bytes(const srcv_shape* shape, const srcv_mlp_weights* w);
/* Size of the packed weight image of the tensor-core variant for this shape / these widths
 * (0 when that variant does not serve them and there is nothing to pack), and the packing
 * itself: `image` DEVICE, 256-byte aligned, srcv_mlp_packed_bytes bytes.                   */
size_t srcv_mlp_packed_bytes(const srcv_shape* shape, const srcv_mlp_weights* w);
int32_t srcv_mlp_pack_weights(const srcv_shape* shape, const srcv_mlp_weights* w, void* image,
                              void* stream);
int32_t srcv_mlp_forward_f32(const srcv_shape* shape,
                             const float* cur_feats, const float* src_feats,
                             const srcv_cameras* cams, const srcv_planes* planes,
                             const srcv_mlp_weights* weights,
                             float* cost, float* lowest, uint8_t* overall_mask,
                             void* workspace, size_t workspace_bytes,
                             void* stream);

/* ---- metadata-MLP volume, backward ------------------------------------ *
 * What autograd of the reference composite (modules/cost_volume.py:451-736 with the
 * MLP of modules/networks.py:129-147; used for training by
 * experiment_modules/depth_model.py:362-372 under train.py) yields for the two feature
 * inputs and the six MLP parameters, given dL/dcost.  Nothing of the forward is saved:
 * the kernel recomputes the metadata tile and the activations per 64-row tile.  Every
 * output is OVERWRITTEN (zeroed, then accumulated with fp32 atomics — the summation
 * order, hence the last bits, may differ between calls).  Cameras and plane depths get
 * no gradient.  Supported: C (K+1) + 10 K + 4 <= 208 features, hidden widths <= 128.
 *   grad_cost (B,D,H,W)   grad_cur (B,C,H,W)   grad_src (B,K,C,H,W)
 *   grads     DEVICE pointers shaped like the parameters in srcv_mlp_weights        */
typedef struct srcv_mlp_grads {
  float* w1; float* b1;
  float* w2; float* b2;
  float* w3; float* b3;
} srcv_mlp_grads;
size_t srcv_mlp_backward_workspace_bytes(const srcv_shape* shape, const srcv_mlp_weights* w);
/* 1 if srcv_mlp_backward_f32 serves this shape and these hidden widths, else 0.             */
int32_t srcv_mlp_backward_supported(const srcv_shape* shape, int32_t hidden1, int32_t hidden2);
int32_t srcv_mlp_backward_f32(const srcv_shape* shape,
                              const float* cur_feats, const float* src_feats,
                              const srcv_cameras* cams, const srcv_planes* planes,
                              const srcv_mlp_weights* weights, const float* grad_cost,
                              float* grad_cur, float* grad_src, const srcv_mlp_grads* grads,
                              void* workspace, size_t workspace_bytes, void* stream);

/* ---- producer-side fusion: encoder tail -> chunk-planar features -------------------- *
 * Replaces the last op of the reference's matching encoder, nn.InstanceNorm2d(C) without
 * affine (modules/networks.py:201; biased variance), AND the re-layout pass of the sweeps:
 *   x        DEVICE (B, V, C, H, W) fp32 — the conv output for the stacked (reference frame,
 *            K = V-1 source views) images, as depth_model.py:220-243 produces it
 *   cur_c4   DEVICE (B, C/4, H, W, 4)        normalised features of view 0
 *   src_c4   DEVICE (B, V-1, C/4, H, W, 4)   normalised features of views 1..V-1
 * Pass both to the forward calls with shape->layout = SRCV_LAYOUT_CHUNK_PLANAR.  C % 4 == 0. */
int32_t srcv_instnorm_to_chunk_planar_f32(const float* x, int32_t B, int32_t V, int32_t C, int32_t H,
                                          int32_t W, float eps, float* cur_c4, float* src_c4, void* stream);

/* ---- TSDF integration of depth maps (the consumer of the predicted depth) ---- *
 * Replaces TSDFFuser.integrate_depth + project_to_camera (reference tools/tsdf.py:221-320,
 * :204-219) as OurFuser.fuse_frames drives them (tools/fusers_helper.py:64-71): a dense
 * (X,Y,Z) fp16 volume of truncated signed distances and running-average weights, z fastest,
 * updated in place with a batch of depth maps applied IN ORDER.  All tensors are fp16, as in
 * the reference (which `.half()`s depth, intrinsics and extrinsics): the arithmetic is the
 * reference's op for op, every operation rounded to fp16.  One launch per <= 16 frames; a
 * voxel's 4 bytes are read and written at most once per launch.
 *   tsdf_values, tsdf_weights  DEVICE (X,Y,Z) fp16, updated in place (16-byte aligned and
 *                              Z % 8 == 0 take the vector path; anything else a scalar path)
 *   origin                     world position of voxel (0,0,0) (fp32, TSDF.from_bounds :85)
 *   depth        DEVICE (B,H,W) fp16     cam_T_world, K  DEVICE (B,4,4) fp16
 *   depth_mask   DEVICE (B,H,W) uint8 (0 = invalid pixel, :251-253) or NULL             */
typedef struct srcv_tsdf_volume {
  void* tsdf_values;
  void* tsdf_weights;
  int32_t X, Y, Z;
  float origin[3];
  float voxel_size;
  float truncation_voxels; /* TSDFFuser.truncation_size (3.0), :181 */
  float max_weight;        /* TSDFFuser.maxW (100.0), :182          */
} srcv_tsdf_volume;
typedef struct srcv_tsdf_frames {
  const void* depth;
  const void* cam_T_world;
  const void* K;
  const uint8_t* depth_mask;
  int32_t B, H, W;
  float min_depth; /* TSDFFuser(min_depth=0.5)  */
  float max_depth; /* TSDFFuser(max_depth=5.0)  */
} srcv_tsdf_frames;
size_t srcv_tsdf_workspace_bytes(const srcv_tsdf_frames* frames);
int32_t srcv_tsdf_integrate_f16(const srcv_tsdf_volume* volume, const srcv_tsdf_frames* frames,
                                void* workspace, size_t workspace_bytes, void* stream);

/* ---- marching-cubes mesh extraction from the fused volume ---------------------------- *
 * Replaces the host half of TSDF.to_mesh (reference tools/tsdf.py:125-157: a copy of the volume
 * to the host and scikit-image's marching_cubes(level=0, allow_degenerate=False)).  Reads
 * tsdf_values in place, clamped to [-1, 1] in fp32; a corner is below iff its value is < 0.
 * Triangles whose vertices coincide in fp32 are dropped; with single_mesh, so is every triangle
 * that needs a vertex on an edge from exactly -1 to exactly +1 (the boundary between observed free
 * space and never-observed voxels).  Output in voxel-index space (axis 0, 1, 2):
 *   verts, normals (V,3) fp32: one vertex per crossing edge a kept triangle uses, ordered by the
 *                   owning voxel's linear index, then axis; normals = the normalised, linearly
 *                   interpolated central-difference gradient (toward increasing values)
 *   faces (F,3) int32: ordered by cell, then table order; counter-clockwise seen from above
 * Two calls, two host synchronisations:
 *   1. srcv_mesh_count_f16 writes counts[0] = candidate vertices, counts[1] = F, and counts[2] bit 0 /
 *      bit 1 = the volume has a value >= 0 / <= 0 (level 0 inside [min, max] iff both are set);
 *   2. the caller reads them, allocates faces (F,3) and verts / normals with room for counts[0]
 *      rows, and srcv_mesh_emit_f16 (same volume, same workspace, untouched in between) writes
 *      them and counts[3] = V <= counts[0]: rows V.. of verts / normals are unused.
 * counts: DEVICE int64[4], 8-byte aligned.  Candidate and face counts must fit int32.
 * scratch: DEVICE, srcv_mesh_scratch_bytes(counts[0]) bytes, 256-byte aligned.               */
typedef struct srcv_mesh_volume {
  const void* tsdf_values; /* DEVICE (X,Y,Z) fp16, z fastest, 2-byte aligned               */
  int32_t X, Y, Z;         /* each >= 2                                                    */
  int32_t single_mesh;     /* 0 / 1                                                        */
} srcv_mesh_volume;
size_t srcv_mesh_workspace_bytes(const srcv_mesh_volume* volume);
size_t srcv_mesh_scratch_bytes(int32_t n_candidates);
int32_t srcv_mesh_count_f16(const srcv_mesh_volume* volume, int64_t* counts, void* workspace,
                            size_t workspace_bytes, void* stream);
int32_t srcv_mesh_emit_f16(const srcv_mesh_volume* volume, int32_t n_candidates, int32_t n_faces,
                           float* verts, float* normals, int32_t* faces, int64_t* counts,
                           void* workspace, size_t workspace_bytes, void* scratch, size_t scratch_bytes,
                           void* stream);

/* ---- multi-view depth consistency (point-cloud fusion) ------------------------------ *
 * Replaces process_depth of the reference's 3DVNet-style fuser (tools/torch_point_cloud_fusion.py
 * :12-97), which pc_fusion.py:158 runs for every frame of a scan against all the others: for each
 * pixel of frame `ref_index`, un-project, re-project into every other frame, nearest-sample its
 * depth, count the frames that agree within z_thresh, and average the back-projected consistent
 * samples with the pixel's own point.  fp32, the reference's operation order.
 *   scan: N frames — depths (N,H,W), K and K_inv (N,3,3), cam_T_world and world_T_cam (N,4,4)
 *         (the caller inverts once per scan; the reference inverts per call, :25-27), all DEVICE
 *   pts_avg (H*W,3) out    n_valid (H*W) int32 out    valid (H*W) uint8 out (n_valid >= n_consistent)
 * The workspace keeps the staged per-frame matrices: pass frames_ready != 0 on every call after
 * the first of a scan to skip re-staging them.                                              */
typedef struct srcv_mvs_scan {
  const float* depths;
  const float* K;
  const float* K_inv;
  const float* cam_T_world;
  const float* world_T_cam;
  int32_t N, H, W;
} srcv_mvs_scan;
size_t srcv_mvs_workspace_bytes(const srcv_mvs_scan* scan);
int32_t srcv_mvs_consistency_f32(const srcv_mvs_scan* scan, int32_t ref_index, float z_thresh,
                                 int32_t n_consistent, float* pts_avg, int32_t* n_valid, uint8_t* valid,
                                 void* workspace, size_t workspace_bytes, int32_t frames_ready, void* stream);

/* ---- multi-view depth regression loss (training) ------------------------------------- *
 * Replaces MVDepthLoss.forward of the reference (losses.py:180-208, with get_valid_mask :90-135
 * and get_error_for_pair :138-178; called from experiment_modules/depth_model.py:477-485): for every
 * source view, the whole-batch mean over valid pixels of |log s - log z|, s = the view's depth
 * nearest-sampled where the GROUND-TRUTH depth projects, z = the depth of the PREDICTED point in
 * that view; the loss is the mean over the views.  NaN terms are dropped (nanmean).  fp32, the
 * reference's operation order.  All pointers DEVICE memory, dense:
 *   depth_pred, cur_depth (B,1,H,W)   src_depth (B,K,1,H,W)
 *   cur_invK, cur_world_T_cam (B,4,4)   src_K, src_cam_T_world (B,K,4,4)          K <= 16
 * forward : loss (1 float) out; optional valid_mask (B,K,H,W) uint8 and src_depth_sampled
 *           (B,K,H,W) float outputs = get_valid_mask of every view (NULL: not written).
 * backward: grad_depth_pred (B,1,H,W) out = grad_loss[0] * d loss / d depth_pred; `workspace` must
 *           be the one the forward call of the same arguments filled (it keeps the per-view counts).
 * Deterministic: per-CTA partial sums reduced in a fixed order.                                 */
typedef struct srcv_mvloss_args {
  const float* depth_pred;
  const float* cur_depth;
  const float* src_depth;
  const float* cur_invK;
  const float* src_K;
  const float* cur_world_T_cam;
  const float* src_cam_T_world;
  int32_t B, K, H, W;
} srcv_mvloss_args;
size_t srcv_mvloss_workspace_bytes(const srcv_mvloss_args* args);
int32_t srcv_mvloss_forward_f32(const srcv_mvloss_args* args, float* loss, uint8_t* valid_mask,
                                float* src_depth_sampled, void* workspace, size_t workspace_bytes,
                                void* stream);
int32_t srcv_mvloss_backward_f32(const srcv_mvloss_args* args, const float* grad_loss,
                                 float* grad_depth_pred, const void* workspace, size_t workspace_bytes,
                                 void* stream);

/* ---- tuning / introspection ------------------------------------------- *
 * Selects the kernel variant used by the two forward calls on this thread's
 * next invocations (process-global).  0 = automatic choice.  Used by the tests
 * to exercise every variant against the oracle and by bench.py to report which
 * one ran.  Unknown values are rejected with SRCV_ERR_UNSUPPORTED.           */
typedef enum srcv_variant {
  SRCV_VARIANT_AUTO = 0,
  SRCV_VARIANT_GENERIC = 1, /* shape-generic SIMT kernels                     */
  SRCV_VARIANT_FAST = 2     /* chunk-planar gather / tcgen05 kernels          */
} srcv_variant;
int32_t srcv_set_variant(int32_t variant);
/* Name of the kernel variant the last forward call on this process launched. */
const char* srcv_last_variant(void);
/* Number of kernel launches issued by the library since load (monotonic).    */
uint64_t srcv_launch_count(void);


/* ---- tensor-core self-test (test support) -------------------------------- *
 * D (128,128) = A (128,Kp) W^T, W (128,Kp), all DEVICE fp32, Kp a multiple of 16
 * and <= 256, through the same TMEM / descriptor / mbarrier machinery as the
 * metadata-MLP kernel (fp16 hi/lo split, three MMAs).  `scratch` = 512*Kp bytes.  */
int32_t srcv_tc_selftest_f32(const float* A, const float* W, int32_t Kp, float* D, void* scratch,
                             void* stream);

/* ---- per-kernel timing (benchmark support) ---------------------------- *
 * Between srcv_profile_begin and srcv_profile_end every forward call records
 * CUDA events on ITS stream around the prep pass and around the sweep kernel(s)
 * (at most max_records calls are recorded; later ones run unrecorded).
 * srcv_profile_end waits for the recorded events, returns the summed device
 * times in milliseconds and the number of recorded calls, and releases the
 * events.  Outside a begin/end pair nothing is recorded.                     */
int32_t srcv_profile_begin(int32_t max_records);
int32_t srcv_profile_end(double* prep_ms_total, double* sweep_ms_total, int32_t* n_records);

#ifdef __cplusplus
}
#endif
#endif /* SRCV_B200_H_ */
