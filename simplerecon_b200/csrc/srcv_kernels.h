// Internal host-side launch interface between srcv_api.cu and the kernel files.
#pragma once
#ifdef SRCV_HOST_EMU
#include "emu_cuda.h"   // tests/emu: the kernels compiled as host C++ (one std::thread per CUDA thread)
#else
#include <cuda_runtime.h>
#endif
#include <stddef.h>
#include <stdint.h>

#include "../../include/srcv_b200.h"
#include "srcv_common.cuh"

// One spelling for a kernel launch, so that the host emulation (tests/emu) can run the same
// launcher code: a template kernel name with commas goes in parentheses.
#ifdef SRCV_HOST_EMU
#define SRCV_LAUNCH(kernel, grid, block, smem, stream, ...) \
  ::emu::launch(dim3(grid), dim3(block), (size_t)(smem), [&] { kernel(__VA_ARGS__); })
#else
#define SRCV_LAUNCH(kernel, grid, block, smem, stream, ...) kernel<<<grid, block, smem, stream>>>(__VA_ARGS__)
#endif

namespace srcv {

// Workspace carve-up (all offsets 256-byte aligned).
struct Workspace {
  float* planes;        // (B,D) plane depths (FROM_RANGE / PER_PLANE copy)
  ViewParams* views;    // (B,K)
  FrameParams* frames;  // (B)
  float* src_c4;        // (B,K,C/4,H,W,4) chunk-planar copy of src_feats, or nullptr
  float* cur_c4;        // (B,C/4,H,W,4) chunk-planar copy of cur_feats, or nullptr
  unsigned* tile_done;  // per (frame, pixel tile) completion counters, zeroed by the prep pass
  size_t tile_done_count;
  float* extra;         // variant-specific scratch, or nullptr
  size_t bytes;         // total bytes needed
};

Workspace carve_workspace(const srcv_shape& s, void* base, bool want_c4, size_t extra_bytes);

// counts kernel launches for srcv_launch_count()
void note_launch(int n = 1);

// prep: view/frame params, plane depths, optional chunk-planar copy of src_feats.
cudaError_t launch_prep(const srcv_shape& s, const srcv_cameras& cams, const srcv_planes& pl,
                        const float* src_feats, const float* cur_feats, const Workspace& ws,
                        bool need_poses, cudaStream_t stream);

// dot-product volume
cudaError_t launch_dot_generic(const srcv_shape& s, const float* cur, const float* src,
                               const Workspace& ws, const float* planes, bool per_pixel,
                               float* cost, float* lowest, cudaStream_t stream);
bool dot_fast_supported(const srcv_shape& s);
size_t dot_fast_tile_counters(const srcv_shape& s);
// `cur` is NCHW, or chunk-planar (B,C/4,H,W,4) when s.layout says so
cudaError_t launch_dot_fast(const srcv_shape& s, const float* cur, const Workspace& ws,
                            const float* planes, bool per_pixel, float* cost, float* lowest,
                            cudaStream_t stream);

// backward of the dot-product volume w.r.t. the feature inputs
bool dot_backward_supported(const srcv_shape& s);
cudaError_t launch_dot_backward(const srcv_shape& s, const float* cur, const float* src,
                                const Workspace& ws, const float* planes, bool per_pixel,
                                const float* gcost, float* gcur, float* gsrc, cudaStream_t stream);

// single-plane warp (the reference's warp_features helper)
cudaError_t launch_warp_planes(const srcv_shape& s, const float* src, const Workspace& ws,
                               const float* planes, bool per_pixel, float* warped, float* depths,
                               float* mask, float* pix, cudaStream_t stream);

// metadata-MLP volume
bool mlp_generic_supported(const srcv_shape& s, const srcv_mlp_weights& w);
size_t mlp_generic_extra_bytes(const srcv_shape& s, const srcv_mlp_weights& w);
cudaError_t launch_mlp_generic(const srcv_shape& s, const float* cur, const float* src,
                               const Workspace& ws, const float* planes, bool per_pixel,
                               const srcv_mlp_weights& w, float* cost, float* lowest,
                               uint8_t* mask, cudaStream_t stream);

// backward of the metadata-MLP volume (fp32 SIMT, recompute)
bool mlp_backward_supported(const srcv_shape& s, const srcv_mlp_weights& w);
size_t mlp_backward_extra_bytes(const srcv_shape& s, const srcv_mlp_weights& w);
cudaError_t launch_mlp_backward(const srcv_shape& s, const float* cur, const float* src,
                                const Workspace& ws, const float* planes, bool per_pixel,
                                const srcv_mlp_weights& w, const float* gcost, float* gcur,
                                float* gsrc, const srcv_mlp_grads& g, cudaStream_t stream);

// tensor-core variant (tcgen05): K = 7, C = 16, 202 -> 128 -> 128 -> 1
bool mlp_tc_supported(const srcv_shape& s, const srcv_mlp_weights& w);
size_t mlp_tc_extra_bytes(const srcv_shape& s);
size_t mlp_tc_image_bytes();
cudaError_t launch_mlp_tc_pack(const srcv_mlp_weights& w, void* image, cudaStream_t stream);
cudaError_t launch_mlp_tc(const srcv_shape& s, const float* cur, const Workspace& ws,
                          const float* planes, bool per_pixel, const srcv_mlp_weights& w, float* cost,
                          float* lowest, uint8_t* mask, cudaStream_t stream);
cudaError_t launch_tc_selftest(const float* A, const float* Wm, int Kp, float* Dout, void* scratch,
                               cudaStream_t stream);

// producer-side fusion (csrc/srcv_producer.cu): InstanceNorm2d + chunk-planar layout
cudaError_t launch_instnorm_c4(const float* x, int B, int V, int C, int H, int W, float eps, float* cur_c4,
                               float* src_c4, cudaStream_t stream);

// dense-grid TSDF integration (csrc/srcv_tsdf.cu)
size_t tsdf_workspace_bytes(int frames);
cudaError_t launch_tsdf_integrate(const srcv_tsdf_volume& v, const srcv_tsdf_frames& f, void* workspace,
                                  cudaStream_t stream);

// marching-cubes mesh extraction (csrc/srcv_mesh.cuh)
size_t mesh_workspace_bytes(const srcv_mesh_volume& v);
size_t mesh_scratch_bytes(long long n_candidates);
cudaError_t launch_mesh_count(const srcv_mesh_volume& v, long long* counts, void* workspace, cudaStream_t stream);
cudaError_t launch_mesh_emit(const srcv_mesh_volume& v, long long n_candidates, long long n_faces, float* verts,
                             float* normals, int* faces, long long* counts, void* workspace, void* scratch,
                             cudaStream_t stream);

// multi-view depth consistency (csrc/srcv_mvs.cu)
size_t mvs_workspace_bytes(int n);
cudaError_t launch_mvs_consistency(const srcv_mvs_scan& s, int ref, float z_thresh, int n_consistent,
                                   float* pts_avg, int* n_valid, uint8_t* valid, void* workspace,
                                   bool frames_ready, cudaStream_t stream);

// multi-view depth regression loss (csrc/srcv_mvloss.cu)
int mvloss_max_views();
size_t mvloss_workspace_bytes(const srcv_mvloss_args& a);
cudaError_t launch_mvloss_forward(const srcv_mvloss_args& a, float* loss, uint8_t* valid, float* sampled,
                                  void* workspace, cudaStream_t stream);
cudaError_t launch_mvloss_backward(const srcv_mvloss_args& a, const float* grad_loss, float* grad_pred,
                                   const void* workspace, cudaStream_t stream);

// argmax over planes -> plane depth (used by variants that do not fuse it)
cudaError_t launch_argmax(const srcv_shape& s, const float* cost, const float* planes,
                          bool per_pixel, float* lowest, cudaStream_t stream);

}  // namespace srcv
