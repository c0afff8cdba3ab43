// Dense-grid TSDF integration of predicted depth maps — the step after the cost volume in the
// reference's product pipeline.
//
// Replaces TSDFFuser.integrate_depth / project_to_camera (reference tools/tsdf.py:221-320,
// :204-219) as driven by OurFuser.fuse_frames (tools/fusers_helper.py:64-71).  The reference
// runs the whole update in fp16 tensors — voxel coordinates, projection matrices, depth maps,
// confidences and the running averages are all halves, so every elementwise op rounds to fp16 —
// and makes ~40 full passes over the volume per frame (homogeneous coordinates, a (b,3,N)
// matmul, a grid_sample over an (X, Y*Z) "image", boolean-mask gathers and scatters).
//
// Here: ONE launch per batch of frames.  A thread owns eight consecutive voxels along z (the
// fastest axis: 16 bytes of tsdf values, 16 bytes of weights), projects them into every frame of
// the batch, applies the frames' updates IN ORDER in registers — the reference's per-frame loop
// (:298) is sequential because later frames see earlier frames' weights — and writes the 32
// bytes back only if something changed.  Voxel coordinates are recomputed from the grid index
// (the reference keeps a 6-bytes-per-voxel fp16 coordinate tensor plus a homogeneous copy).
// Arithmetic is the reference's, op for op: fp32 evaluation, one rounding to fp16 after every
// operation (r16), python scalars in fp32 for arithmetic and in fp16 for comparisons — pinned
// bit-for-bit by oracle/tsdf_oracle.py against the imported reference class.
//
// Culling: the camera-space coordinates are affine along a z column, so a column whose two end
// voxels are both clearly behind the camera / beyond max_depth / off the same image side (with a
// margin that covers the fp16 roundings) is skipped for that frame without touching memory.
#include "srcv_kernels.h"
#ifdef SRCV_HOST_EMU
#include "emu_tc.h"      // tests/emu: __half and its conversions on the host
#else
#include <cuda_fp16.h>
#endif

namespace srcv {

namespace {

constexpr int kVec = 8;                 // voxels per thread (one 16-byte vector of halves)
constexpr int kMaxFrames = 16;          // frames per launch (batches are split by the launcher)

struct TsdfFrame {
  float P[12];      // (K @ E)[:3, :4], every entry rounded to fp16 (tools/tsdf.py:211)
};

struct TsdfParams {
  int X, Y, Z, B, H, W;
  float ox, oy, oz, voxel_size;
  float min_depth, depth_span;          // fp32 scalars of the confidence (:264-266)
  float trunc;                          // fp32 scalar of dist / truncation (:270)
  float neg_trunc_h, max_depth_h;       // fp16-rounded scalars of the comparisons (:273-275)
  float max_w;                          // maxW (:313)
};

// eight halves as one 16-byte vector (a union: the punning is defined for nvcc and for the host
// compiler of the emulation build alike)
union Pack8 {
  uint4 u;
  __half2 h[4];
  __device__ Pack8() {}
};

__device__ __forceinline__ float r16(float x) { return __half2float(__float2half_rn(x)); }

// (K @ E)[:3] in fp16: fp32 accumulation over j, one rounding (a half matmul in PyTorch)
__global__ void tsdf_prep_kernel(const __half* __restrict__ K, const __half* __restrict__ E, int B,
                                 TsdfFrame* __restrict__ frames) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= B * 12) return;
  const int b = t / 12, i = (t % 12) / 4, k = t % 4;
  float acc = 0.f;
#pragma unroll
  for (int j = 0; j < 4; ++j)
    acc = __fmaf_rn(__half2float(K[b * 16 + i * 4 + j]), __half2float(E[b * 16 + j * 4 + k]), acc);
  frames[b].P[i * 4 + k] = r16(acc);
}

template <int VEC>
__global__ void __launch_bounds__(256)
tsdf_integrate_kernel(TsdfParams p, const TsdfFrame* __restrict__ frames, const __half* __restrict__ depth,
                      const uint8_t* __restrict__ mask, __half* __restrict__ tsdf, __half* __restrict__ weights) {
  // grid.y walks x; grid.x * blockDim.x covers the (y, z-column) plane: 32-bit index arithmetic only
  // (64-bit div/mod of a flat voxel index cost more than the projection of an empty column)
  const unsigned zcols = (unsigned)(p.Z / VEC);
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= zcols * (unsigned)p.Y) return;
  const int zc = (int)(t % zcols), iy = (int)(t / zcols), ix = (int)blockIdx.y;
  const int z0 = zc * VEC;
  const size_t base = ((size_t)ix * p.Y + iy) * p.Z + z0;
  // world coordinates: fp32 origin + index * voxel_size, then half (tools/tsdf.py:99-110, :92)
  const float wx = r16(__fadd_rn(p.ox, __fmul_rn((float)ix, p.voxel_size)));
  const float wy = r16(__fadd_rn(p.oy, __fmul_rn((float)iy, p.voxel_size)));
  const float Wf = (float)p.W, Hf = (float)p.H;
  // Conservative column cull, ALL frames first: camera-space coordinates are affine along the z
  // column, so if both end voxels are clearly behind the camera / beyond max_depth / off the same
  // image side (margins cover the fp16 roundings; sides are tested as x < -m z, no division), no
  // voxel of the column can be valid in that frame.  Most columns of a scene-sized volume leave
  // here after ~30 instructions per frame without touching memory.
  const float wza = r16(__fadd_rn(p.oz, __fmul_rn((float)z0, p.voxel_size)));
  const float wzb = r16(__fadd_rn(p.oz, __fmul_rn((float)(z0 + VEC - 1), p.voxel_size)));
  unsigned frame_mask = 0;
  for (int b = 0; b < p.B; ++b) {
    const float* P = frames[b].P;
    const float bz = __fmaf_rn(P[9], wy, __fmul_rn(P[8], wx));
    const float za = __fmaf_rn(P[10], wza, bz) + P[11], zb = __fmaf_rn(P[10], wzb, bz) + P[11];
    const float zmax = fmaxf(za, zb), zmin = fminf(za, zb);
    bool skip = (zmax < -0.01f) || (zmin > p.max_depth_h * 1.01f + 0.01f);
    if (!skip && zmin > 0.01f) {
      const float bx = __fmaf_rn(P[1], wy, __fmul_rn(P[0], wx));
      const float by = __fmaf_rn(P[5], wy, __fmul_rn(P[4], wx));
      const float xa = __fmaf_rn(P[2], wza, bx) + P[3], xb = __fmaf_rn(P[2], wzb, bx) + P[3];
      const float ya = __fmaf_rn(P[6], wza, by) + P[7], yb = __fmaf_rn(P[6], wzb, by) + P[7];
      // every voxel in between projects between the two ends' pixel coordinates u = x / z
      const float mx = 2.0f + 0.01f * Wf, my = 2.0f + 0.01f * Hf;
      skip = (xa < -mx * za && xb < -mx * zb) || (xa > (Wf + mx) * za && xb > (Wf + mx) * zb) ||
             (ya < -my * za && yb < -my * zb) || (ya > (Hf + my) * za && yb > (Hf + my) * zb);
    }
    if (!skip) frame_mask |= 1u << b;
  }
  if (frame_mask == 0u) return;

  float wz[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) wz[i] = r16(__fadd_rn(p.oz, __fmul_rn((float)(z0 + i), p.voxel_size)));

  float tv[VEC], tw[VEC];
  bool loaded = false, dirty = false;

  for (int b = 0; b < p.B; ++b) {
    if (!((frame_mask >> b) & 1u)) continue;
    const float* P = frames[b].P;
    // cam = P @ (x, y, z, 1): fp32 accumulation in k order, ONE rounding to half (:216)
    const float bx = __fmaf_rn(P[1], wy, __fmul_rn(P[0], wx));
    const float by = __fmaf_rn(P[5], wy, __fmul_rn(P[4], wx));
    const float bz = __fmaf_rn(P[9], wy, __fmul_rn(P[8], wx));
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const float cx = r16(__fadd_rn(__fmaf_rn(P[2], wz[i], bx), P[3]));
      const float cy = r16(__fadd_rn(__fmaf_rn(P[6], wz[i], by), P[7]));
      const float vz = r16(__fadd_rn(__fmaf_rn(P[10], wz[i], bz), P[11]));
      if (!(vz > 0.0f) || !(vz < p.max_depth_h)) continue;        // two of the validity terms (:273-275)
      const float px = r16(__fdiv_rn(cx, vz)), py = r16(__fdiv_rn(cy, vz));   // :217
      // 2 p / size - 1 (:249), then grid_sample's ((g + 1) size - 1) / 2 in half, nearest (half to even)
      const float gx = r16(__fadd_rn(r16(__fdiv_rn(r16(__fmul_rn(2.0f, px)), Wf)), -1.0f));
      const float gy = r16(__fadd_rn(r16(__fdiv_rn(r16(__fmul_rn(2.0f, py)), Hf)), -1.0f));
      const float sx = rintf(r16(__fmul_rn(r16(__fadd_rn(r16(__fmul_rn(r16(__fadd_rn(gx, 1.0f)), Wf)), -1.0f)), 0.5f)));
      const float sy = rintf(r16(__fmul_rn(r16(__fadd_rn(r16(__fmul_rn(r16(__fadd_rn(gy, 1.0f)), Hf)), -1.0f)), 0.5f)));
      if (!(sx >= 0.0f && sx <= Wf - 1.0f && sy >= 0.0f && sy <= Hf - 1.0f)) continue;   // zeros padding: ds = 0
      const size_t pix = ((size_t)b * p.H + (int)sy) * p.W + (int)sx;
      float ds = __half2float(depth[pix]);
      if (mask != nullptr && mask[pix] == 0) ds = -1.0f;           // :251-253
      if (!(ds > 0.0f)) continue;
      const float dist = r16(__fadd_rn(ds, -vz));                  // :269
      if (!(dist > p.neg_trunc_h)) continue;
      float conf = r16(__fadd_rn(1.0f, -r16(__fdiv_rn(r16(__fadd_rn(ds, -p.min_depth)), p.depth_span))));
      conf = fminf(fmaxf(conf, 0.0f), 1.0f);
      conf = r16(__fmul_rn(conf, conf));                           // :264-266
      if (!(conf > 0.0f)) continue;
      const float nt = fminf(fmaxf(r16(__fdiv_rn(dist, p.trunc)), -1.0f), 1.0f);   // :270
      if (!loaded) {
        // first valid voxel of this column: bring in the 2 x 16 bytes
        if (VEC == 8) {
          Pack8 a, w;
          a.u = *reinterpret_cast<const uint4*>(tsdf + base);
          w.u = *reinterpret_cast<const uint4*>(weights + base);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float2 fa = __half22float2(a.h[j]), fw = __half22float2(w.h[j]);
            tv[2 * j] = fa.x; tv[2 * j + 1] = fa.y; tw[2 * j] = fw.x; tw[2 * j + 1] = fw.y;
          }
        } else {
#pragma unroll
          for (int j = 0; j < VEC; ++j) { tv[j] = __half2float(tsdf[base + j]); tw[j] = __half2float(weights[base + j]); }
        }
        loaded = true;
      }
      // :307-318: running average with InfiniTAM's confidence-dependent rate
      const float rate = (conf < tw[i]) ? 2.0f : 5.0f;
      const float nw = r16(__fdiv_rn(r16(__fmul_rn(conf, rate)), p.max_w));
      const float total = r16(__fadd_rn(tw[i], nw));
      tv[i] = r16(__fdiv_rn(r16(__fadd_rn(r16(__fmul_rn(tv[i], tw[i])), r16(__fmul_rn(nt, nw)))), total));
      tw[i] = fminf(total, 1.0f);
      dirty = true;
    }
  }
  if (dirty) {
    if (VEC == 8) {
      Pack8 a, w;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        a.h[j] = __floats2half2_rn(tv[2 * j], tv[2 * j + 1]);
        w.h[j] = __floats2half2_rn(tw[2 * j], tw[2 * j + 1]);
      }
      *reinterpret_cast<uint4*>(tsdf + base) = a.u;
      *reinterpret_cast<uint4*>(weights + base) = w.u;
    } else {
#pragma unroll
      for (int j = 0; j < VEC; ++j) { tsdf[base + j] = __float2half_rn(tv[j]); weights[base + j] = __float2half_rn(tw[j]); }
    }
  }
}

}  // namespace

size_t tsdf_workspace_bytes(int frames) { return sizeof(TsdfFrame) * (size_t)(frames < kMaxFrames ? frames : kMaxFrames) + 256; }

cudaError_t launch_tsdf_integrate(const srcv_tsdf_volume& v, const srcv_tsdf_frames& f, void* workspace,
                                  cudaStream_t stream) {
  TsdfFrame* frames = reinterpret_cast<TsdfFrame*>(workspace);
  __half* tsdf = reinterpret_cast<__half*>(v.tsdf_values);
  __half* weights = reinterpret_cast<__half*>(v.tsdf_weights);
  const float trunc = v.truncation_voxels * v.voxel_size;
  for (int b0 = 0; b0 < f.B; b0 += kMaxFrames) {
    const int nb = (f.B - b0 < kMaxFrames) ? (f.B - b0) : kMaxFrames;
    const __half* K = reinterpret_cast<const __half*>(f.K) + (size_t)b0 * 16;
    const __half* E = reinterpret_cast<const __half*>(f.cam_T_world) + (size_t)b0 * 16;
    SRCV_LAUNCH(tsdf_prep_kernel, 1, 256, 0, stream, K, E, nb, frames);
    note_launch();
    TsdfParams p;
    p.X = v.X; p.Y = v.Y; p.Z = v.Z; p.B = nb; p.H = f.H; p.W = f.W;
    p.ox = v.origin[0]; p.oy = v.origin[1]; p.oz = v.origin[2]; p.voxel_size = v.voxel_size;
    p.min_depth = f.min_depth;
    p.depth_span = f.max_depth - f.min_depth;
    p.trunc = trunc;
    p.neg_trunc_h = -__half2float(__float2half_rn(trunc));
    p.max_depth_h = __half2float(__float2half_rn(f.max_depth));
    p.max_w = v.max_weight;
    const __half* depth = reinterpret_cast<const __half*>(f.depth) + (size_t)b0 * f.H * f.W;
    const uint8_t* mask = f.depth_mask ? f.depth_mask + (size_t)b0 * f.H * f.W : nullptr;
    const bool vec = (v.Z % kVec) == 0 && ((reinterpret_cast<uintptr_t>(tsdf) | reinterpret_cast<uintptr_t>(weights)) & 15u) == 0;
    const long long plane = (long long)v.Y * (vec ? v.Z / kVec : v.Z);
    if (plane > 2147483647ll || v.X > 65535) return cudaErrorInvalidValue;
    const dim3 grid((unsigned)((plane + 255) / 256), (unsigned)v.X);
    if (vec) SRCV_LAUNCH(tsdf_integrate_kernel<kVec>, grid, 256, 0, stream, p, frames, depth, mask, tsdf, weights);
    else SRCV_LAUNCH(tsdf_integrate_kernel<1>, grid, 256, 0, stream, p, frames, depth, mask, tsdf, weights);
    note_launch();
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return err;
  }
  return cudaSuccess;
}

}  // namespace srcv

// marching-cubes extraction from the same volume (TSDF.to_mesh)
#include "srcv_mesh.cuh"
