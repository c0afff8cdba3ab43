// extern "C" surface of libsrcv_b200.so — see include/srcv_b200.h for the contract
// and the reference interfaces each entry point stands in for.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <vector>

#include "srcv_kernels.h"

namespace srcv {

static std::atomic<uint64_t> g_launches{0};
static std::atomic<int> g_variant{SRCV_VARIANT_AUTO};
static std::atomic<const char*> g_last_variant{"none"};   // process-global, like g_variant
static thread_local char g_err[512] = "";

void note_launch(int n) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

static int32_t fail(int32_t code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

static int32_t cuda_fail(cudaError_t e, const char* where) {
  return fail(SRCV_ERR_CUDA, "%s: %s (%s)", where, cudaGetErrorName(e), cudaGetErrorString(e));
}

// ---- optional per-kernel timing ------------------------------------------------
struct ProfRecord { cudaEvent_t e[3]; };
static std::vector<ProfRecord> g_prof;
static int g_prof_used = 0;
static bool g_prof_on = false;
static std::mutex g_prof_mu;

static ProfRecord* prof_next() {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (!g_prof_on || g_prof_used >= (int)g_prof.size()) return nullptr;
  return &g_prof[g_prof_used++];
}

static int32_t check_shape(const srcv_shape* s) {
  if (!s) return fail(SRCV_ERR_NULL, "shape is NULL");
  if (s->B <= 0 || s->K <= 0 || s->C <= 0 || s->H <= 0 || s->W <= 0 || s->D <= 0)
    return fail(SRCV_ERR_SHAPE, "non-positive dimension B=%d K=%d C=%d H=%d W=%d D=%d", s->B, s->K,
                s->C, s->H, s->W, s->D);
  if ((long long)s->H * s->W > (1ll << 26) || s->K > 64 || s->C > 1024 ||
      (long long)s->B * s->D * s->H * s->W > (1ll << 40))
    return fail(SRCV_ERR_SHAPE, "dimension out of supported range");
  if (s->layout != SRCV_LAYOUT_NCHW && s->layout != SRCV_LAYOUT_CHUNK_PLANAR)
    return fail(SRCV_ERR_UNSUPPORTED, "unknown feature layout %d", s->layout);
  if (s->layout == SRCV_LAYOUT_CHUNK_PLANAR && (s->C % 4) != 0)
    return fail(SRCV_ERR_SHAPE, "chunk-planar features need C %% 4 == 0");
  return SRCV_OK;
}

static int32_t check_common(const srcv_shape* s, const float* cur, const float* src,
                            const srcv_cameras* cams, const srcv_planes* pl, const float* cost,
                            bool need_poses) {
  if (int32_t e = check_shape(s)) return e;
  if (!cur || !src || !cost) return fail(SRCV_ERR_NULL, "cur_feats/src_feats/cost is NULL");
  if (((reinterpret_cast<uintptr_t>(cur) | reinterpret_cast<uintptr_t>(src)) & 15u) != 0)
    return fail(SRCV_ERR_UNSUPPORTED, "cur_feats / src_feats must be 16-byte aligned");
  if (!cams || !cams->src_Ks || !cams->cur_invK) return fail(SRCV_ERR_NULL, "camera block incomplete");
  if (!cams->src_extrinsics) {
    // raw poses: the prep kernel forms the relative transforms itself
    if (!cams->src_cam_T_world || !cams->cur_world_T_cam || !cams->cur_cam_T_world || !cams->src_world_T_cam)
      return fail(SRCV_ERR_NULL, "src_extrinsics is NULL and the raw pose block is incomplete");
  } else if (need_poses && !cams->src_poses) {
    return fail(SRCV_ERR_NULL, "src_poses is NULL");
  }
  if (!pl) return fail(SRCV_ERR_NULL, "planes descriptor is NULL");
  switch (pl->mode) {
    case SRCV_PLANES_FROM_RANGE:
      if (!pl->min_depth || !pl->max_depth || !pl->ramp)
        return fail(SRCV_ERR_NULL, "FROM_RANGE needs min_depth, max_depth and ramp");
      break;
    case SRCV_PLANES_PER_PLANE:
    case SRCV_PLANES_PER_PIXEL:
      if (!pl->planes) return fail(SRCV_ERR_NULL, "planes pointer is NULL");
      break;
    default:
      return fail(SRCV_ERR_UNSUPPORTED, "unknown planes mode %d", pl->mode);
  }
  return SRCV_OK;
}

static int32_t check_workspace(void* ws, size_t have, size_t need) {
  if (!ws) return fail(SRCV_ERR_NULL, "workspace is NULL (need %zu bytes)", need);
  if ((reinterpret_cast<uintptr_t>(ws) & 255u) != 0)
    return fail(SRCV_ERR_WORKSPACE, "workspace must be 256-byte aligned");
  if (have < need) return fail(SRCV_ERR_WORKSPACE, "workspace too small: %zu < %zu", have, need);
  return SRCV_OK;
}

static bool use_fast_dot(const srcv_shape& s) {
  const int v = g_variant.load();
  if (v == SRCV_VARIANT_GENERIC) return false;
  return dot_fast_supported(s);
}

}  // namespace srcv

using namespace srcv;

extern "C" {

int32_t srcv_abi_version(void) { return SRCV_ABI_VERSION; }

int32_t srcv_check_device(void) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return cuda_fail(e, "cudaGetDevice");
  int major = 0;
  e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (e != cudaSuccess) return cuda_fail(e, "cudaDeviceGetAttribute");
  if (major != 10) return fail(SRCV_ERR_DEVICE, "device %d has compute capability %d.x; this library is built for sm_100a only", dev, major);
  return SRCV_OK;
}

const char* srcv_status_string(int32_t st) {
  switch (st) {
    case SRCV_OK: return "ok";
    case SRCV_ERR_NULL: return "null pointer";
    case SRCV_ERR_SHAPE: return "bad shape";
    case SRCV_ERR_WORKSPACE: return "bad workspace";
    case SRCV_ERR_UNSUPPORTED: return "unsupported";
    case SRCV_ERR_CUDA: return "cuda error";
    case SRCV_ERR_DEVICE: return "unsupported device";
    default: return "unknown status";
  }
}

const char* srcv_last_error(void) { return g_err; }

int32_t srcv_set_variant(int32_t v) {
  if (v != SRCV_VARIANT_AUTO && v != SRCV_VARIANT_GENERIC && v != SRCV_VARIANT_FAST)
    return fail(SRCV_ERR_UNSUPPORTED, "unknown variant %d", v);
  g_variant.store(v);
  return SRCV_OK;
}

const char* srcv_last_variant(void) { return g_last_variant.load(); }

uint64_t srcv_launch_count(void) { return g_launches.load(); }

size_t srcv_dot_workspace_bytes(const srcv_shape* s) {
  if (check_shape(s) != SRCV_OK) return 0;
  return carve_workspace(*s, nullptr, dot_fast_supported(*s), 0).bytes;
}

int32_t srcv_dot_forward_f32(const srcv_shape* s, const float* cur, const float* src,
                             const srcv_cameras* cams, const srcv_planes* pl, float* cost,
                             float* lowest, void* workspace, size_t workspace_bytes, void* stream_) {
  if (int32_t e = check_common(s, cur, src, cams, pl, cost, false)) return e;
  const bool fast = use_fast_dot(*s);
  if (g_variant.load() == SRCV_VARIANT_FAST && !fast)
    return fail(SRCV_ERR_UNSUPPORTED, "fast dot variant needs C == 16 and K <= 8");
  if (s->layout == SRCV_LAYOUT_CHUNK_PLANAR && !fast)
    return fail(SRCV_ERR_UNSUPPORTED, "chunk-planar features are served by the chunk-planar dot sweep only (C == 16, variant != generic)");
  const Workspace need = carve_workspace(*s, nullptr, dot_fast_supported(*s), 0);
  if (int32_t e = check_workspace(workspace, workspace_bytes, need.bytes)) return e;
  Workspace ws = carve_workspace(*s, workspace, dot_fast_supported(*s), 0);
  if (!fast) { ws.src_c4 = nullptr; ws.tile_done = nullptr; }  // skip the chunk-planar copies
  ws.cur_c4 = nullptr;             // the dot kernel keeps the reference features in registers
  if (s->layout == SRCV_LAYOUT_CHUNK_PLANAR) ws.src_c4 = const_cast<float*>(src);   // gathered in place, no copy
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ProfRecord* pr = prof_next();
  if (pr) cudaEventRecord(pr->e[0], stream);
  cudaError_t err = launch_prep(*s, *cams, *pl, src, cur, ws, false, stream);
  if (err != cudaSuccess) return cuda_fail(err, "prep");
  if (pr) cudaEventRecord(pr->e[1], stream);
  const bool per_pixel = pl->mode == SRCV_PLANES_PER_PIXEL;
  const float* planes = pl->mode == SRCV_PLANES_FROM_RANGE ? ws.planes : pl->planes;
  if (fast) {
    g_last_variant.store("dot_fast_c4planar");
    err = launch_dot_fast(*s, cur, ws, planes, per_pixel, cost, lowest, stream);
  } else {
    g_last_variant.store("dot_generic");
    err = launch_dot_generic(*s, cur, src, ws, planes, per_pixel, cost, lowest, stream);
  }
  if (err != cudaSuccess) return cuda_fail(err, g_last_variant.load());
  if (pr) cudaEventRecord(pr->e[2], stream);
  return SRCV_OK;
}

size_t srcv_dot_backward_workspace_bytes(const srcv_shape* s) {
  if (check_shape(s) != SRCV_OK) return 0;
  return carve_workspace(*s, nullptr, false, 0).bytes;
}

int32_t srcv_dot_backward_supported(const srcv_shape* s) {
  return (check_shape(s) == SRCV_OK && dot_backward_supported(*s)) ? 1 : 0;
}

int32_t srcv_dot_backward_f32(const srcv_shape* s, const float* cur, const float* src,
                              const srcv_cameras* cams, const srcv_planes* pl, const float* grad_cost,
                              float* grad_cur, float* grad_src, void* workspace,
                              size_t workspace_bytes, void* stream_) {
  if (int32_t e = check_common(s, cur, src, cams, pl, grad_cost, false)) return e;
  if (!grad_cur || !grad_src) return fail(SRCV_ERR_NULL, "grad_cur / grad_src is NULL");
  if (!dot_backward_supported(*s))
    return fail(SRCV_ERR_UNSUPPORTED, "dot backward is built for C in {8, 16, 32}, got %d", s->C);
  if (s->layout != SRCV_LAYOUT_NCHW) return fail(SRCV_ERR_UNSUPPORTED, "the backward kernels take NCHW features");
  const Workspace need = carve_workspace(*s, nullptr, false, 0);
  if (int32_t e = check_workspace(workspace, workspace_bytes, need.bytes)) return e;
  Workspace ws = carve_workspace(*s, workspace, false, 0);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  cudaError_t err = launch_prep(*s, *cams, *pl, src, cur, ws, false, stream);
  if (err != cudaSuccess) return cuda_fail(err, "prep");
  err = cudaMemsetAsync(grad_src, 0, sizeof(float) * (size_t)s->B * s->K * s->C * s->H * s->W, stream);
  if (err != cudaSuccess) return cuda_fail(err, "memset grad_src");
  const bool per_pixel = pl->mode == SRCV_PLANES_PER_PIXEL;
  const float* planes = pl->mode == SRCV_PLANES_FROM_RANGE ? ws.planes : pl->planes;
  g_last_variant.store("dot_backward_atomic");
  err = launch_dot_backward(*s, cur, src, ws, planes, per_pixel, grad_cost, grad_cur, grad_src, stream);
  if (err != cudaSuccess) return cuda_fail(err, g_last_variant.load());
  return SRCV_OK;
}

size_t srcv_warp_workspace_bytes(const srcv_shape* s) {
  if (check_shape(s) != SRCV_OK) return 0;
  return carve_workspace(*s, nullptr, false, 0).bytes;
}

static int32_t warp_planes_impl(const srcv_shape* s, const float* src, const srcv_cameras* cams,
                                const float* planes, int32_t per_pixel, float* warped, float* depths,
                                float* mask, float* pix, void* workspace, size_t workspace_bytes,
                                void* stream_) {
  if (int32_t e = check_shape(s)) return e;
  if (!src || !planes || !warped || !depths || !mask)
    return fail(SRCV_ERR_NULL, "warp_features pointer is NULL");
  if (!cams || !cams->src_extrinsics || !cams->src_Ks || !cams->cur_invK)
    return fail(SRCV_ERR_NULL, "camera block incomplete");
  if (s->layout != SRCV_LAYOUT_NCHW) return fail(SRCV_ERR_UNSUPPORTED, "warp_features takes NCHW features");
  if (s->D > 65535) return fail(SRCV_ERR_SHAPE, "at most 65535 planes per warp call");
  const Workspace need = carve_workspace(*s, nullptr, false, 0);
  if (int32_t e = check_workspace(workspace, workspace_bytes, need.bytes)) return e;
  Workspace ws = carve_workspace(*s, workspace, false, 0);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  srcv_planes pl{};
  pl.mode = SRCV_PLANES_PER_PLANE;   // the planes come straight from the caller
  pl.planes = planes;
  cudaError_t err = launch_prep(*s, *cams, pl, src, nullptr, ws, false, stream);
  if (err != cudaSuccess) return cuda_fail(err, "prep");
  g_last_variant.store("warp_planes");
  err = launch_warp_planes(*s, src, ws, planes, per_pixel != 0, warped, depths, mask, pix, stream);
  if (err != cudaSuccess) return cuda_fail(err, g_last_variant.load());
  return SRCV_OK;
}

int32_t srcv_warp_features_f32(const srcv_shape* s, const float* src, const srcv_cameras* cams,
                               const float* depth_plane, int32_t per_pixel, float* warped,
                               float* depths, float* mask, void* workspace, size_t workspace_bytes,
                               void* stream_) {
  if (!s) return fail(SRCV_ERR_NULL, "shape is NULL");
  srcv_shape one = *s;
  one.D = 1;                         // shape->D is ignored: one plane
  return warp_planes_impl(&one, src, cams, depth_plane, per_pixel, warped, depths, mask, nullptr, workspace,
                          workspace_bytes, stream_);
}

int32_t srcv_warp_features_planes_f32(const srcv_shape* s, const float* src, const srcv_cameras* cams,
                                      const float* depth_planes, int32_t per_pixel, float* warped,
                                      float* depths, float* mask, float* pix_coords, void* workspace,
                                      size_t workspace_bytes, void* stream_) {
  return warp_planes_impl(s, src, cams, depth_planes, per_pixel, warped, depths, mask, pix_coords, workspace,
                          workspace_bytes, stream_);
}

static int32_t check_weights(const srcv_shape* s, const srcv_mlp_weights* w) {
  if (!w) return fail(SRCV_ERR_NULL, "weights is NULL");
  if (!w->w1 || !w->b1 || !w->w2 || !w->b2 || !w->w3 || !w->b3)
    return fail(SRCV_ERR_NULL, "a weight pointer is NULL");
  if (w->hidden1 <= 0 || w->hidden2 <= 0) return fail(SRCV_ERR_SHAPE, "hidden widths must be positive");
  if (!mlp_generic_supported(*s, *w))
    return fail(SRCV_ERR_UNSUPPORTED, "MLP widths (%d,%d) / feature count not supported by this build (hidden <= 128)", w->hidden1, w->hidden2);
  return SRCV_OK;
}

static bool use_tc_mlp(const srcv_shape& s, const srcv_mlp_weights& w) {
  if (g_variant.load() == SRCV_VARIANT_GENERIC) return false;
  return mlp_tc_supported(s, w);
}

static size_t mlp_extra_bytes(const srcv_shape& s, const srcv_mlp_weights& w) {
  size_t e = mlp_generic_extra_bytes(s, w);
  if (mlp_tc_supported(s, w) && mlp_tc_extra_bytes(s) > e) e = mlp_tc_extra_bytes(s);
  return e;
}

size_t srcv_mlp_workspace_bytes(const srcv_shape* s, const srcv_mlp_weights* w) {
  if (check_shape(s) != SRCV_OK || !w) return 0;
  if (!mlp_generic_supported(*s, *w)) return 0;
  return carve_workspace(*s, nullptr, mlp_tc_supported(*s, *w), mlp_extra_bytes(*s, *w)).bytes;
}

size_t srcv_mlp_packed_bytes(const srcv_shape* s, const srcv_mlp_weights* w) {
  if (check_shape(s) != SRCV_OK || !w) return 0;
  return mlp_tc_supported(*s, *w) ? mlp_tc_image_bytes() : 0;
}

int32_t srcv_mlp_pack_weights(const srcv_shape* s, const srcv_mlp_weights* w, void* image, void* stream_) {
  if (int32_t e = check_shape(s)) return e;
  if (int32_t e = check_weights(s, w)) return e;
  if (!mlp_tc_supported(*s, *w))
    return fail(SRCV_ERR_UNSUPPORTED, "only the tensor-core variant (K == 7, C == 16, hidden 128/128) has a packed image");
  if (!image) return fail(SRCV_ERR_NULL, "image is NULL");
  if ((reinterpret_cast<uintptr_t>(image) & 255u) != 0)
    return fail(SRCV_ERR_WORKSPACE, "image must be 256-byte aligned");
  cudaError_t err = launch_mlp_tc_pack(*w, image, static_cast<cudaStream_t>(stream_));
  if (err != cudaSuccess) return cuda_fail(err, "pack");
  return SRCV_OK;
}

int32_t srcv_mlp_forward_f32(const srcv_shape* s, const float* cur, const float* src,
                             const srcv_cameras* cams, const srcv_planes* pl,
                             const srcv_mlp_weights* w, float* cost, float* lowest,
                             uint8_t* overall_mask, void* workspace, size_t workspace_bytes,
                             void* stream_) {
  if (int32_t e = check_common(s, cur, src, cams, pl, cost, true)) return e;
  if (int32_t e = check_weights(s, w)) return e;
  const bool tc = use_tc_mlp(*s, *w);
  if (g_variant.load() == SRCV_VARIANT_FAST && !tc)
    return fail(SRCV_ERR_UNSUPPORTED, "tensor-core MLP variant needs K == 7, C == 16, hidden widths 128/128");
  if (s->layout == SRCV_LAYOUT_CHUNK_PLANAR && !tc)
    return fail(SRCV_ERR_UNSUPPORTED, "chunk-planar features are served by the tensor-core MLP sweep only (K == 7, C == 16, 128/128, variant != generic)");
  const size_t extra = mlp_extra_bytes(*s, *w);
  const bool c4 = mlp_tc_supported(*s, *w);
  const Workspace need = carve_workspace(*s, nullptr, c4, extra);
  if (int32_t e = check_workspace(workspace, workspace_bytes, need.bytes)) return e;
  Workspace ws = carve_workspace(*s, workspace, c4, extra);
  if (!tc) ws.src_c4 = nullptr;  // skip the chunk-planar copy
  ws.tile_done = nullptr;        // only the dot sweep uses the tile counters
  if (s->layout == SRCV_LAYOUT_CHUNK_PLANAR) {   // gathered in place, no copy
    ws.src_c4 = const_cast<float*>(src);
    ws.cur_c4 = const_cast<float*>(cur);
  }
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ProfRecord* pr = prof_next();
  if (pr) cudaEventRecord(pr->e[0], stream);
  cudaError_t err = launch_prep(*s, *cams, *pl, src, cur, ws, true, stream);
  if (err != cudaSuccess) return cuda_fail(err, "prep");
  if (pr) cudaEventRecord(pr->e[1], stream);
  const bool per_pixel = pl->mode == SRCV_PLANES_PER_PIXEL;
  const float* planes = pl->mode == SRCV_PLANES_FROM_RANGE ? ws.planes : pl->planes;
  if (tc) {
    g_last_variant.store("mlp_tc_tcgen05_f16x3");
    err = launch_mlp_tc(*s, cur, ws, planes, per_pixel, *w, cost, lowest, overall_mask, stream);
  } else {
    g_last_variant.store("mlp_generic_fp32");
    err = launch_mlp_generic(*s, cur, src, ws, planes, per_pixel, *w, cost, lowest, overall_mask, stream);
  }
  if (err != cudaSuccess) return cuda_fail(err, g_last_variant.load());
  if (pr) cudaEventRecord(pr->e[2], stream);
  return SRCV_OK;
}

size_t srcv_mlp_backward_workspace_bytes(const srcv_shape* s, const srcv_mlp_weights* w) {
  if (check_shape(s) != SRCV_OK || !w) return 0;
  if (!mlp_backward_supported(*s, *w)) return 0;
  return carve_workspace(*s, nullptr, false, mlp_backward_extra_bytes(*s, *w)).bytes;
}

int32_t srcv_mlp_backward_supported(const srcv_shape* s, int32_t hidden1, int32_t hidden2) {
  if (check_shape(s) != SRCV_OK) return 0;
  srcv_mlp_weights w{};
  w.hidden1 = hidden1;
  w.hidden2 = hidden2;
  return mlp_backward_supported(*s, w) ? 1 : 0;
}

int32_t srcv_mlp_backward_f32(const srcv_shape* s, const float* cur, const float* src,
                              const srcv_cameras* cams, const srcv_planes* pl,
                              const srcv_mlp_weights* w, const float* grad_cost, float* grad_cur,
                              float* grad_src, const srcv_mlp_grads* g, void* workspace,
                              size_t workspace_bytes, void* stream_) {
  if (int32_t e = check_common(s, cur, src, cams, pl, grad_cost, true)) return e;
  if (int32_t e = check_weights(s, w)) return e;
  if (!grad_cur || !grad_src) return fail(SRCV_ERR_NULL, "grad_cur / grad_src is NULL");
  if (!g || !g->w1 || !g->b1 || !g->w2 || !g->b2 || !g->w3 || !g->b3)
    return fail(SRCV_ERR_NULL, "a parameter-gradient pointer is NULL");
  if (!mlp_backward_supported(*s, *w))
    return fail(SRCV_ERR_UNSUPPORTED, "MLP backward supports at most 208 input features and hidden widths <= 128");
  if (s->layout != SRCV_LAYOUT_NCHW) return fail(SRCV_ERR_UNSUPPORTED, "the backward kernels take NCHW features");
  const size_t extra = mlp_backward_extra_bytes(*s, *w);
  const Workspace need = carve_workspace(*s, nullptr, false, extra);
  if (int32_t e = check_workspace(workspace, workspace_bytes, need.bytes)) return e;
  Workspace ws = carve_workspace(*s, workspace, false, extra);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  cudaError_t err = launch_prep(*s, *cams, *pl, src, cur, ws, true, stream);
  if (err != cudaSuccess) return cuda_fail(err, "prep");
  const size_t F = (size_t)s->C * (s->K + 1) + 10 * (size_t)s->K + 4;
  const size_t HW = (size_t)s->H * s->W;
  struct { void* p; size_t n; } zero[] = {
      {grad_cur, (size_t)s->B * s->C * HW}, {grad_src, (size_t)s->B * s->K * s->C * HW},
      {g->w1, (size_t)w->hidden1 * F}, {g->b1, (size_t)w->hidden1},
      {g->w2, (size_t)w->hidden2 * w->hidden1}, {g->b2, (size_t)w->hidden2},
      {g->w3, (size_t)w->hidden2}, {g->b3, 1}};
  for (auto& z : zero) {
    err = cudaMemsetAsync(z.p, 0, sizeof(float) * z.n, stream);
    if (err != cudaSuccess) return cuda_fail(err, "memset gradients");
  }
  const bool per_pixel = pl->mode == SRCV_PLANES_PER_PIXEL;
  const float* planes = pl->mode == SRCV_PLANES_FROM_RANGE ? ws.planes : pl->planes;
  g_last_variant.store("mlp_backward_fp32_recompute");
  err = launch_mlp_backward(*s, cur, src, ws, planes, per_pixel, *w, grad_cost, grad_cur, grad_src, *g, stream);
  if (err != cudaSuccess) return cuda_fail(err, g_last_variant.load());
  return SRCV_OK;
}

int32_t srcv_instnorm_to_chunk_planar_f32(const float* x, int32_t B, int32_t V, int32_t C, int32_t H, int32_t W,
                                          float eps, float* cur_c4, float* src_c4, void* stream_) {
  if (!x || !cur_c4 || (V > 1 && !src_c4)) return fail(SRCV_ERR_NULL, "instnorm pointer is NULL");
  if (B <= 0 || V <= 0 || C <= 0 || H <= 0 || W <= 0 || (C % 4) != 0 || (long long)H * W > (1ll << 26) ||
      (long long)B * V * (C / 4) > 2147483647ll)
    return fail(SRCV_ERR_SHAPE, "bad shape B=%d V=%d C=%d H=%d W=%d (C must be a multiple of 4)", B, V, C, H, W);
  if (!(eps >= 0.f)) return fail(SRCV_ERR_SHAPE, "eps must be non-negative");
  if (((reinterpret_cast<uintptr_t>(cur_c4) | reinterpret_cast<uintptr_t>(src_c4)) & 15u) != 0)
    return fail(SRCV_ERR_UNSUPPORTED, "chunk-planar outputs must be 16-byte aligned");
  g_last_variant.store("instnorm_chunk_planar");
  cudaError_t err = launch_instnorm_c4(x, B, V, C, H, W, eps, cur_c4, src_c4, static_cast<cudaStream_t>(stream_));
  if (err != cudaSuccess) return cuda_fail(err, "instnorm_to_chunk_planar");
  return SRCV_OK;
}

size_t srcv_tsdf_workspace_bytes(const srcv_tsdf_frames* f) {
  if (!f || f->B <= 0) return 0;
  return tsdf_workspace_bytes(f->B);
}

int32_t srcv_tsdf_integrate_f16(const srcv_tsdf_volume* v, const srcv_tsdf_frames* f, void* workspace,
                                size_t workspace_bytes, void* stream_) {
  if (!v || !f) return fail(SRCV_ERR_NULL, "volume / frames descriptor is NULL");
  if (!v->tsdf_values || !v->tsdf_weights) return fail(SRCV_ERR_NULL, "tsdf_values / tsdf_weights is NULL");
  if (!f->depth || !f->cam_T_world || !f->K) return fail(SRCV_ERR_NULL, "depth / cam_T_world / K is NULL");
  if (v->X <= 0 || v->Y <= 0 || v->Z <= 0 || (long long)v->X * v->Y * v->Z > (1ll << 40))
    return fail(SRCV_ERR_SHAPE, "bad volume dimensions %d x %d x %d", v->X, v->Y, v->Z);
  if (f->B <= 0 || f->H <= 0 || f->W <= 0 || f->W > 2048 || f->H > 2048)
    return fail(SRCV_ERR_SHAPE, "bad frame batch B=%d H=%d W=%d (image sizes up to 2048 are exact in fp16)", f->B, f->H, f->W);
  if (!(v->voxel_size > 0.f) || !(v->truncation_voxels > 0.f) || !(v->max_weight > 0.f) || !(f->max_depth > f->min_depth))
    return fail(SRCV_ERR_SHAPE, "voxel_size, truncation, max_weight must be positive and max_depth > min_depth");
  if (((reinterpret_cast<uintptr_t>(v->tsdf_values) | reinterpret_cast<uintptr_t>(v->tsdf_weights) |
        reinterpret_cast<uintptr_t>(f->depth) | reinterpret_cast<uintptr_t>(f->cam_T_world) |
        reinterpret_cast<uintptr_t>(f->K)) & 1u) != 0)
    return fail(SRCV_ERR_UNSUPPORTED, "fp16 arrays must be 2-byte aligned");
  if (int32_t e = check_workspace(workspace, workspace_bytes, tsdf_workspace_bytes(f->B))) return e;
  g_last_variant.store("tsdf_integrate_f16");
  cudaError_t err = launch_tsdf_integrate(*v, *f, workspace, static_cast<cudaStream_t>(stream_));
  if (err != cudaSuccess) return cuda_fail(err, "tsdf_integrate");
  return SRCV_OK;
}

static int32_t check_mesh_volume(const srcv_mesh_volume* v) {
  if (!v) return fail(SRCV_ERR_NULL, "mesh volume descriptor is NULL");
  if (!v->tsdf_values) return fail(SRCV_ERR_NULL, "tsdf_values is NULL");
  if (v->X < 2 || v->Y < 2 || v->Z < 2 || v->X >= (1 << 24) || v->Y >= (1 << 24) || v->Z >= (1 << 24) ||
      (long long)v->X * v->Y > 2147483647ll || (long long)v->X * v->Y * v->Z > (1ll << 40))
    return fail(SRCV_ERR_SHAPE, "bad mesh volume dimensions %d x %d x %d (each must be >= 2)", v->X, v->Y, v->Z);
  if (v->single_mesh != 0 && v->single_mesh != 1) return fail(SRCV_ERR_SHAPE, "single_mesh must be 0 or 1");
  if ((reinterpret_cast<uintptr_t>(v->tsdf_values) & 1u) != 0)
    return fail(SRCV_ERR_UNSUPPORTED, "tsdf_values must be 2-byte aligned");
  return SRCV_OK;
}

size_t srcv_mesh_workspace_bytes(const srcv_mesh_volume* v) {
  if (!v || v->X < 2 || v->Y < 2 || v->Z < 2) return 0;
  return mesh_workspace_bytes(*v);
}

size_t srcv_mesh_scratch_bytes(int32_t n_candidates) {
  return n_candidates < 0 ? 0 : mesh_scratch_bytes(n_candidates);
}

int32_t srcv_mesh_count_f16(const srcv_mesh_volume* v, int64_t* counts, void* workspace, size_t workspace_bytes,
                            void* stream_) {
  if (int32_t e = check_mesh_volume(v)) return e;
  if (!counts) return fail(SRCV_ERR_NULL, "counts is NULL");
  if ((reinterpret_cast<uintptr_t>(counts) & 7u) != 0) return fail(SRCV_ERR_UNSUPPORTED, "counts must be 8-byte aligned");
  if (int32_t e = check_workspace(workspace, workspace_bytes, mesh_workspace_bytes(*v))) return e;
  g_last_variant.store("mesh_count_f16");
  cudaError_t err = launch_mesh_count(*v, reinterpret_cast<long long*>(counts), workspace,
                                      static_cast<cudaStream_t>(stream_));
  if (err != cudaSuccess) return cuda_fail(err, "mesh_count");
  return SRCV_OK;
}

int32_t srcv_mesh_emit_f16(const srcv_mesh_volume* v, int32_t n_candidates, int32_t n_faces, float* verts,
                           float* normals, int32_t* faces, int64_t* counts, void* workspace, size_t workspace_bytes,
                           void* scratch, size_t scratch_bytes, void* stream_) {
  if (int32_t e = check_mesh_volume(v)) return e;
  if (n_candidates < 0 || n_faces < 0 || n_faces > 2147483647 / 3)
    return fail(SRCV_ERR_SHAPE, "bad counts: %d candidate vertices, %d faces (int32 overflow?)", n_candidates, n_faces);
  if (!counts) return fail(SRCV_ERR_NULL, "counts is NULL");
  if ((n_candidates > 0 && (!verts || !normals)) || (n_faces > 0 && !faces))
    return fail(SRCV_ERR_NULL, "verts / normals / faces is NULL");
  if (((reinterpret_cast<uintptr_t>(verts) | reinterpret_cast<uintptr_t>(normals) |
        reinterpret_cast<uintptr_t>(faces)) & 3u) != 0 || (reinterpret_cast<uintptr_t>(counts) & 7u) != 0)
    return fail(SRCV_ERR_UNSUPPORTED, "verts / normals / faces must be 4-byte aligned, counts 8-byte aligned");
  if (int32_t e = check_workspace(workspace, workspace_bytes, mesh_workspace_bytes(*v))) return e;
  if (int32_t e = check_workspace(scratch, scratch_bytes, mesh_scratch_bytes(n_candidates))) return e;
  g_last_variant.store("mesh_emit_f16");
  cudaError_t err = launch_mesh_emit(*v, n_candidates, n_faces, verts, normals, faces,
                                     reinterpret_cast<long long*>(counts), workspace, scratch,
                                     static_cast<cudaStream_t>(stream_));
  if (err != cudaSuccess) return cuda_fail(err, "mesh_emit");
  return SRCV_OK;
}

size_t srcv_mvs_workspace_bytes(const srcv_mvs_scan* s) {
  if (!s || s->N <= 0) return 0;
  return mvs_workspace_bytes(s->N);
}

int32_t srcv_mvs_consistency_f32(const srcv_mvs_scan* s, int32_t ref, float z_thresh, int32_t n_consistent,
                                 float* pts_avg, int32_t* n_valid, uint8_t* valid, void* workspace,
                                 size_t workspace_bytes, int32_t frames_ready, void* stream_) {
  if (!s) return fail(SRCV_ERR_NULL, "scan descriptor is NULL");
  if (!s->depths || !s->K || !s->K_inv || !s->cam_T_world || !s->world_T_cam)
    return fail(SRCV_ERR_NULL, "a scan pointer is NULL");
  if (!pts_avg || !n_valid || !valid) return fail(SRCV_ERR_NULL, "an output pointer is NULL");
  if (s->N <= 0 || s->H <= 1 || s->W <= 1 || (long long)s->H * s->W > (1ll << 26) ||
      (long long)s->N * s->H * s->W > (1ll << 40))
    return fail(SRCV_ERR_SHAPE, "bad scan shape N=%d H=%d W=%d", s->N, s->H, s->W);
  if (ref < 0 || ref >= s->N) return fail(SRCV_ERR_SHAPE, "ref_index %d out of range [0,%d)", ref, s->N);
  if (int32_t e = check_workspace(workspace, workspace_bytes, mvs_workspace_bytes(s->N))) return e;
  g_last_variant.store("mvs_consistency_f32");
  cudaError_t err = launch_mvs_consistency(*s, ref, z_thresh, n_consistent, pts_avg, n_valid, valid, workspace,
                                           frames_ready != 0, static_cast<cudaStream_t>(stream_));
  if (err != cudaSuccess) return cuda_fail(err, "mvs_consistency");
  return SRCV_OK;
}

static int32_t check_mvloss(const srcv_mvloss_args* a) {
  if (!a) return fail(SRCV_ERR_NULL, "loss arguments are NULL");
  if (!a->depth_pred || !a->cur_depth || !a->src_depth || !a->cur_invK || !a->src_K || !a->cur_world_T_cam ||
      !a->src_cam_T_world)
    return fail(SRCV_ERR_NULL, "a loss input pointer is NULL");
  if (a->B <= 0 || a->K <= 0 || a->H <= 0 || a->W <= 0 || (long long)a->H * a->W > (1ll << 26) ||
      (long long)a->B * a->K * a->H * a->W > (1ll << 40) || a->B > 65535)
    return fail(SRCV_ERR_SHAPE, "bad loss shape B=%d K=%d H=%d W=%d", a->B, a->K, a->H, a->W);
  if (a->K > mvloss_max_views())
    return fail(SRCV_ERR_UNSUPPORTED, "at most %d source views per call (got %d)", mvloss_max_views(), a->K);
  return SRCV_OK;
}

size_t srcv_mvloss_workspace_bytes(const srcv_mvloss_args* a) {
  if (!a || a->B <= 0 || a->K <= 0 || a->H <= 0 || a->W <= 0) return 0;
  return mvloss_workspace_bytes(*a);
}

int32_t srcv_mvloss_forward_f32(const srcv_mvloss_args* a, float* loss, uint8_t* valid_mask, float* sampled,
                                void* workspace, size_t workspace_bytes, void* stream_) {
  if (int32_t e = check_mvloss(a)) return e;
  if (!loss) return fail(SRCV_ERR_NULL, "loss output pointer is NULL");
  if (int32_t e = check_workspace(workspace, workspace_bytes, mvloss_workspace_bytes(*a))) return e;
  g_last_variant.store("mvloss_forward_f32");
  cudaError_t err = launch_mvloss_forward(*a, loss, valid_mask, sampled, workspace, static_cast<cudaStream_t>(stream_));
  if (err != cudaSuccess) return cuda_fail(err, "mvloss_forward");
  return SRCV_OK;
}

int32_t srcv_mvloss_backward_f32(const srcv_mvloss_args* a, const float* grad_loss, float* grad_depth_pred,
                                 const void* workspace, size_t workspace_bytes, void* stream_) {
  if (int32_t e = check_mvloss(a)) return e;
  if (!grad_loss || !grad_depth_pred) return fail(SRCV_ERR_NULL, "grad_loss / grad_depth_pred is NULL");
  if (int32_t e = check_workspace(const_cast<void*>(workspace), workspace_bytes, mvloss_workspace_bytes(*a))) return e;
  g_last_variant.store("mvloss_backward_f32");
  cudaError_t err = launch_mvloss_backward(*a, grad_loss, grad_depth_pred, workspace, static_cast<cudaStream_t>(stream_));
  if (err != cudaSuccess) return cuda_fail(err, "mvloss_backward");
  return SRCV_OK;
}

int32_t srcv_tc_selftest_f32(const float* A, const float* Wm, int32_t Kp, float* D, void* scratch,
                             void* stream) {
  if (!A || !Wm || !D || !scratch) return fail(SRCV_ERR_NULL, "selftest pointer is NULL");
  cudaError_t err = launch_tc_selftest(A, Wm, Kp, D, scratch, static_cast<cudaStream_t>(stream));
  if (err != cudaSuccess) return cuda_fail(err, "tc_selftest");
  return SRCV_OK;
}

int32_t srcv_profile_begin(int32_t max_records) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (g_prof_on) return fail(SRCV_ERR_UNSUPPORTED, "profiling already active");
  if (max_records <= 0 || max_records > 100000) return fail(SRCV_ERR_SHAPE, "max_records out of range");
  g_prof.resize(max_records);
  for (auto& r : g_prof)
    for (auto& e : r.e) {
      cudaError_t err = cudaEventCreate(&e);
      if (err != cudaSuccess) { g_prof.clear(); return cuda_fail(err, "cudaEventCreate"); }
    }
  g_prof_used = 0;
  g_prof_on = true;
  return SRCV_OK;
}

int32_t srcv_profile_end(double* prep_ms_total, double* sweep_ms_total, int32_t* n_records) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (!g_prof_on) return fail(SRCV_ERR_UNSUPPORTED, "profiling not active");
  double prep = 0.0, sweep = 0.0;
  int32_t st = SRCV_OK;
  for (int i = 0; i < g_prof_used; ++i) {
    cudaError_t err = cudaEventSynchronize(g_prof[i].e[2]);
    float a = 0.f, b = 0.f;
    if (err == cudaSuccess) err = cudaEventElapsedTime(&a, g_prof[i].e[0], g_prof[i].e[1]);
    if (err == cudaSuccess) err = cudaEventElapsedTime(&b, g_prof[i].e[1], g_prof[i].e[2]);
    if (err != cudaSuccess) { st = cuda_fail(err, "profile events"); break; }
    prep += a; sweep += b;
  }
  if (prep_ms_total) *prep_ms_total = prep;
  if (sweep_ms_total) *sweep_ms_total = sweep;
  if (n_records) *n_records = g_prof_used;
  for (auto& r : g_prof) for (auto& e : r.e) cudaEventDestroy(e);
  g_prof.clear();
  g_prof_used = 0;
  g_prof_on = false;
  return st;
}

}  // extern "C"
