// What the projection translation units share (projection.cu: the pinhole kernels, the ABI entries and the camera-
// gradient finalize kernels; projection_ortho.cu / projection_fisheye.cu: the kernels of the other camera models):
// the kernel parameters, the launch geometry, and the staging / partial-sum helpers of the kernels.
#pragma once
#include "egs_common.cuh"
#include "egs_math.cuh"

namespace egs {

constexpr int kProjThreads = 256;

struct ProjFwdParams {
  int C, N, K, sh_degree, colors_per_camera;
  const float *means, *quats, *scales, *opacities, *sh, *viewmats, *Ks;
  float width, height, eps2d, near_plane, far_plane, radius_clip, tile_size;
  int tile_w, tile_h;
  int32_t* radii;
  float *means2d, *depths, *conics, *colors;
  int32_t* tiles_per_gauss;
  int32_t* tight_rects;  // nullable [C,N,2]: the TIGHT tile rectangle (tighten_tile_rect) of the blend kernels' own lists,
                         // packed {x0 | y0 << 16, w | h << 16} (w * h = 0 for a Gaussian that reaches no pixel)
  float4* splats;
  // raw-parameter mode (§8f-2): `scales` holds log-scales, `opacities` logits, `sh` the [N,1,3] DC band and
  // `sh_rest` the [N,15,3] remainder — exp / sigmoid / cat are folded into this kernel
  int raw;
  const float* sh_rest;
  // rasterize_mode="antialiased": opacity is multiplied by the compensation factor sqrt(det_orig / det_blur),
  // which is also written to compensations[C,N]
  int antialiased;
  float* compensations;
};

// exactly torch's CUDA elementwise formulas, so the folded path reproduces exp()/sigmoid() of the caller
__device__ __forceinline__ float act_exp(float x) { return expf(x); }
__device__ __forceinline__ float act_sigmoid(float x) { return 1.0f / (1.0f + expf(-x)); }

// Load the first `nfloats` floats of a per-Gaussian coefficient block into registers.
// VEC4: the block start is 16-byte aligned (K*3 % 4 == 0) -> 128-bit loads.
template <bool VEC4>
__device__ __forceinline__ void load_coeffs(const float* __restrict__ base, int nfloats, float (&c)[48]) {
  if (VEC4) {
    const float4* b4 = reinterpret_cast<const float4*>(base);
#pragma unroll
    for (int i = 0; i < 12; ++i) {
      if (i * 4 < nfloats) {
        float4 v = __ldg(b4 + i);
        c[i * 4 + 0] = v.x; c[i * 4 + 1] = v.y; c[i * 4 + 2] = v.z; c[i * 4 + 3] = v.w;
      } else {
        c[i * 4 + 0] = 0.f; c[i * 4 + 1] = 0.f; c[i * 4 + 2] = 0.f; c[i * 4 + 3] = 0.f;
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < 48; ++i) c[i] = (i < nfloats) ? __ldg(base + i) : 0.f;
  }
}



// ---- raw-parameter mode (§8f-2): the "cat" of sh_0 [N,1,3] and sh_rest [N,15,3] done in flight --------------------
// A warp's 32 rows are one contiguous, 16-byte aligned block in each source (32*45 and 32*3 floats), so the blocks
// travel with 128-bit global accesses; only the shared-memory side is scalar (row r, column c of the row tile
// <- element r*45 + (c-3) of the block).  Loads are unpredicated with a selected address (per-load predicates
// serialise them); blocks of the last, partial warp fall back to scalar accesses.
template <int RS>
__device__ __forceinline__ void load_rows_raw(float* __restrict__ tile, const float* __restrict__ sh0,
                                              const float* __restrict__ shrest, int n_base, int N, uint32_t row_mask,
                                              int lane) {
  const int rows = min(32, N - n_base);
  const float* b0 = sh0 + (size_t)n_base * 3;
  const float* b1 = shrest + (size_t)n_base * 45;
  if (rows == 32) {
#pragma unroll
    for (int i = 0; i < 12; ++i) {  // 360 float4 of the sh_rest block
      const int q = i * 32 + lane;
      if (q < 360) {
        const int e = q * 4, r0 = e / 45, r3 = (e + 3) / 45;
        const bool need = ((row_mask >> r0) | (row_mask >> r3)) & 1u;
        const float4 v = __ldg(reinterpret_cast<const float4*>(need ? b1 + e : b1));
        const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int ee = e + k, r = ee / 45, c = ee - r * 45;
          tile[r * RS + 3 + c] = vv[k];
        }
      }
    }
    if (lane < 24) {  // 24 float4 of the sh_0 block
      const int e = lane * 4;
      const float4 v = __ldg(reinterpret_cast<const float4*>(b0 + e));
      const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int ee = e + k, r = ee / 3, c = ee - r * 3;
        tile[r * RS + c] = vv[k];
      }
    }
  } else {
    for (int e = lane; e < rows * 45; e += 32) { const int r = e / 45, c = e - r * 45; tile[r * RS + 3 + c] = __ldg(b1 + e); }
    for (int e = lane; e < rows * 3; e += 32) { const int r = e / 3, c = e - r * 3; tile[r * RS + c] = __ldg(b0 + e); }
  }
}

template <int RS>
__device__ __forceinline__ void store_rows_raw(const float* __restrict__ tile, float* __restrict__ v_sh0,
                                               float* __restrict__ v_shrest, int n_base, int N, int lane) {
  const int rows = min(32, N - n_base);
  float* b0 = v_sh0 + (size_t)n_base * 3;
  float* b1 = v_shrest + (size_t)n_base * 45;
  if (rows == 32) {
#pragma unroll
    for (int i = 0; i < 12; ++i) {
      const int q = i * 32 + lane;
      if (q < 360) {
        const int e = q * 4;
        float vv[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int ee = e + k, r = ee / 45, c = ee - r * 45;
          vv[k] = tile[r * RS + 3 + c];
        }
        *reinterpret_cast<float4*>(b1 + e) = make_float4(vv[0], vv[1], vv[2], vv[3]);
      }
    }
    if (lane < 24) {
      const int e = lane * 4;
      float vv[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int ee = e + k, r = ee / 3, c = ee - r * 3;
        vv[k] = tile[r * RS + c];
      }
      *reinterpret_cast<float4*>(b0 + e) = make_float4(vv[0], vv[1], vv[2], vv[3]);
    }
  } else {
    for (int e = lane; e < rows * 45; e += 32) { const int r = e / 45, c = e - r * 45; b1[e] = tile[r * RS + 3 + c]; }
    for (int e = lane; e < rows * 3; e += 32) { const int r = e / 3, c = e - r * 3; b0[e] = tile[r * RS + c]; }
  }
}

constexpr int kPF2Threads = 128;
constexpr int kFwdRowStride = 52;  // floats; conflict-free float4 row reads for a quarter warp

struct ProjBwdParams {
  int C, N, K, sh_degree, colors_per_camera;
  const float *means, *quats, *scales, *sh, *viewmats, *Ks;
  float width, height, eps2d;
  const int32_t* radii;
  const float* colors;
  const float4* v_splats;
  const float* v_means2d_extra;
  float *v_means, *v_quats, *v_scales, *v_opacities, *v_sh;
  int raw;                    // see ProjFwdParams: inputs are raw parameters, outputs are their gradients
  const float* sh_rest;
  const float* opacities;     // logits (raw mode: needed for the sigmoid VJP) / opacities (antialiased mode)
  int antialiased;            // v_splats' opacity slot is d L / d (opacity * compensation)
  float* v_sh_rest;
  float2* absgrad;  // nullable [C,N]: sum over pixels of |d L / d means2d|, copied out of the gradient records
  // viewmat gradients (the VG instantiations only): per camera, one 16-float partial of the camera gradient
  // (egs_math.cuh kCamGradFloats, padded) per warp of the launch, camera-major: [C][gridDim.x * 4][16]; the counters
  // [C] of viewmat_grad_finalize_kernel are cleared by block 0.  The egs::ksgrad kernels store 20-float partials
  // (kCamGradFloats + kKsGradFloats, padded) for intrinsics_grad_finalize_kernel.
  float* cam_partials;
  int* cam_counters;
};

constexpr int kProjBwdThreads = 128;
constexpr int kMaxCamerasSmem = 64;

// ---- gradients w.r.t. the view matrices -------------------------------------------------------------------------------
// The camera gradient is a sum over all Gaussians per camera.  Each warp sums its 32 lanes' contributions to one camera
// with a fixed shuffle tree and lane 0 stores the warp's partial; viewmat_grad_finalize_kernel then sums the partials
// in a fixed order.  No float atomics anywhere: the same gradient records give bit-identical v_viewmats.
constexpr int kCamPartialFloats = 16;
// With intrinsics gradients (the egs::ksgrad kernels) a partial is 15 + 4 floats, padded to 20.
constexpr int kCamKsGradFloats = kCamGradFloats + kKsGradFloats;
constexpr int kCamKsPartialFloats = 20;
constexpr int kVgFinalizeThreads = 256;
constexpr int kVgMaxSlices = 32;

// Warp partials of a launch of the backward kernels (both run 4 warps per block).
inline int64_t vg_partial_slots(int64_t n_gauss) { return ceil_div(n_gauss, 128) * 4; }
// Blocks per camera of the finalize kernel: each sums one contiguous slice of the partials.
inline int vg_slices(int64_t slots) {
  const int64_t s = ceil_div(slots, 4 * kVgFinalizeThreads);
  return (int)(s < 1 ? 1 : s > kVgMaxSlices ? kVgMaxSlices : s);
}

// Warp-uniform `any`: false = no lane of the warp sees this camera, the partial is zero (no shuffles).
__device__ __forceinline__ void store_cam_partial(float (&v)[kCamGradFloats], bool any, float* __restrict__ dst, int lane) {
  if (any) {
#pragma unroll
    for (int k = 0; k < kCamGradFloats; ++k)
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) v[k] += __shfl_down_sync(0xffffffffu, v[k], off);
  }
  if (lane == 0) {
    float4* d = reinterpret_cast<float4*>(dst);
    if (any) {
      d[0] = make_float4(v[0], v[1], v[2], v[3]);
      d[1] = make_float4(v[4], v[5], v[6], v[7]);
      d[2] = make_float4(v[8], v[9], v[10], v[11]);
      d[3] = make_float4(v[12], v[13], v[14], 0.f);
    } else {
      const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      d[0] = z; d[1] = z; d[2] = z; d[3] = z;
    }
  }
}

// The same with the intrinsics gradient: 19 floats, stored as 20.
__device__ __forceinline__ void store_cam_partial(float (&v)[kCamKsGradFloats], bool any, float* __restrict__ dst, int lane) {
  if (any) {
#pragma unroll
    for (int k = 0; k < kCamKsGradFloats; ++k)
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) v[k] += __shfl_down_sync(0xffffffffu, v[k], off);
  }
  if (lane == 0) {
    float4* d = reinterpret_cast<float4*>(dst);
    if (any) {
      d[0] = make_float4(v[0], v[1], v[2], v[3]);
      d[1] = make_float4(v[4], v[5], v[6], v[7]);
      d[2] = make_float4(v[8], v[9], v[10], v[11]);
      d[3] = make_float4(v[12], v[13], v[14], v[15]);
      d[4] = make_float4(v[16], v[17], v[18], 0.f);
    } else {
      const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      d[0] = z; d[1] = z; d[2] = z; d[3] = z; d[4] = z;
    }
  }
}

// Partial of warp `warp` of this block for camera c; kStride floats per partial.
template <int kStride>
__device__ __forceinline__ float* cam_partial(const ProjBwdParams& p, int c, int warp) {
  const size_t slots = (size_t)gridDim.x * 4;
  return p.cam_partials + ((size_t)c * slots + (size_t)blockIdx.x * 4 + warp) * kStride;
}

__device__ __forceinline__ void clear_cam_counters(const ProjBwdParams& p) {
  if (blockIdx.x == 0)
    for (int c = threadIdx.x; c < p.C; c += blockDim.x) p.cam_counters[c] = 0;
}

// Store one SH gradient row of `total` = K * 3 floats: the 48 of bands 0..3 from registers, zeros past them.
template <bool VEC4>
__device__ __forceinline__ void store_coeff_grads(float* __restrict__ out, int total, const float (&vco)[48]) {
  if (VEC4) {
    float4* o4 = reinterpret_cast<float4*>(out);
#pragma unroll
    for (int i = 0; i < 12; ++i)
      if (i * 4 < total) o4[i] = make_float4(vco[4 * i + 0], vco[4 * i + 1], vco[4 * i + 2], vco[4 * i + 3]);
    for (int i = 48; i < total; ++i) out[i] = 0.f;  // K > 16: bands this kernel never activates
  } else {
#pragma unroll
    for (int i = 0; i < 48; ++i)
      if (i < total) out[i] = vco[i];
    for (int i = 48; i < total; ++i) out[i] = 0.f;
  }
}




// ------------------------------------------------------------------------------------------------
// Backward, K = 16 SH coefficients (the reference's layout): the 192-byte coefficient rows and the
// 192-byte gradient rows of a warp's 32 Gaussians are contiguous in HBM, so they travel through a
// shared-memory tile with fully coalesced 512-byte warp transactions instead of 32 strided 16-byte
// accesses per instruction; rows of Gaussians that no camera sees are not read.  Keeping the rows in
// shared memory also takes the 96 coefficient / gradient registers out of the thread (224 -> ~110),
// which triples the number of resident warps.  Row stride 52 floats makes the per-thread float4
// accesses of a quarter warp conflict free.
// ------------------------------------------------------------------------------------------------
constexpr int kRowFloats = 48;   // K * 3
constexpr int kRowStride = 52;
constexpr int kPB2Threads = 128;
constexpr int kPB2Warps = kPB2Threads / 32;

// 3 resident CTAs leave ptxas 149 registers (no spills): measured 0.339 ms per four views against 0.350 at the
// default 128 and 0.42 / 0.53 when squeezed to 96 / 80 (spills) — the kernel wants registers, not occupancy.
#ifndef EGS_PB_MIN_CTAS
#define EGS_PB_MIN_CTAS 3
#endif
// The per-camera-SH form with viewmat gradients holds the camera gradient and the staged rows' loop state at once: it
// runs 2 CTAs per SM (255 registers) instead of spilling at 168.  So do the forms with intrinsics gradients, whose 4
// more accumulators spill the classic form at 168.
#define EGS_PB_BOUNDS(TWO_CTAS) __launch_bounds__(kPB2Threads, (TWO_CTAS) ? 2 : EGS_PB_MIN_CTAS)

// Per-camera SH rows of a warp's 32 Gaussians (rows of camera c start at (c * N + n_base) * 48 floats), copied in and
// out with the same coalesced float4 pattern as the shared rows.
// Camera c's coefficient rows of the Gaussians in `mask` into `tile` (nothing to read for degree 0: only band 0's
// gradient is needed, which does not depend on the coefficients).
__device__ __forceinline__ void stage_sh_rows(float* __restrict__ tile, const float* __restrict__ sh, int sh_degree, int c,
                                              int N, int n_base, uint32_t mask, int lane) {
  const float4* src = reinterpret_cast<const float4*>(sh) + ((size_t)c * N + n_base) * (kRowFloats / 4);
#pragma unroll
  for (int i = 0; i < kRowFloats / 4; ++i) {
    const int f = i * 32 + lane;
    const int row = f / 12, c4 = f - row * 12;
    if (sh_degree >= 1 && ((mask >> row) & 1u)) *reinterpret_cast<float4*>(tile + row * kRowStride + c4 * 4) = __ldg(src + f);
  }
  __syncwarp();
}

// The accumulated gradient rows in `tile` -> camera c's rows of v_sh (rows past N are not stored), and `tile` cleared
// for the next camera.
__device__ __forceinline__ void store_sh_grad_rows(float* __restrict__ tile, float* __restrict__ v_sh, int c, int N,
                                                   int n_base, int lane) {
  __syncwarp();
  float4* dst = reinterpret_cast<float4*>(v_sh) + ((size_t)c * N + n_base) * (kRowFloats / 4);
#pragma unroll
  for (int i = 0; i < kRowFloats / 4; ++i) {
    const int f = i * 32 + lane;
    const int row = f / 12, c4 = f - row * 12;
    float4* t = reinterpret_cast<float4*>(tile + row * kRowStride + c4 * 4);
    if (n_base + row < N) dst[f] = *t;
    *t = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  __syncwarp();
}

// ------------------------------------------------------------------------------------------------
// SH degree 4 (K >= 25): the first 25 bands of a row are 75 floats, 300 B.  A warp stages the rows of its 32 Gaussians
// (rows row0 .. row0 + 31 of the [rows, K, 3] coefficient block: n_base, or c * N + n_base with per-camera rows) as a
// dense 32 x 75 tile; the odd row stride keeps a lane's row-wise reads conflict free.  For K = 25 the tile has the
// layout of the warp's 9600-byte span, so a full warp whose span is 16-byte aligned copies it with 19 128-bit accesses
// per lane, all in flight at once (a float4 that straddles two rows is needed when either row is).  Whether the span is
// aligned depends on the base pointer and, for per-camera rows, on N mod 4; unaligned spans, the last partial warp and
// K > 25 take 4-byte accesses, which are coalesced whatever the alignment (the latter skip the bands past 4).
// ------------------------------------------------------------------------------------------------
constexpr int kSh4RowFloats = kSh4Bands * 3;           // 75
constexpr int kSh4TileFloats = 32 * kSh4RowFloats;     // one warp's tile
constexpr int kSh4TileVec4 = kSh4TileFloats / 4;       // 600
constexpr int kSh4BwdMinCtas = 2;                      // 2 x 76.8 KB of tiles per SM

__device__ __forceinline__ bool sh4_span_vec4(const float* span, int K3, int rows) {
  return K3 == kSh4RowFloats && rows == 32 && (reinterpret_cast<uintptr_t>(span) & 15u) == 0;
}

// Rows in `mask` of the warp's `rows` into `tile` (other rows are zero-filled, nothing is read for them).
__device__ __forceinline__ void stage_sh4_rows(float* __restrict__ tile, const float* __restrict__ sh, size_t row0,
                                               int rows, int K3, uint32_t mask, int lane) {
  const float* src = sh + row0 * K3;
  if (sh4_span_vec4(src, K3, rows)) {
    const float4* s4 = reinterpret_cast<const float4*>(src);
    float4* t4 = reinterpret_cast<float4*>(tile);
#pragma unroll
    for (int i = 0; i < (kSh4TileVec4 + 31) / 32; ++i) {
      const int f = i * 32 + lane;
      if (f < kSh4TileVec4) {
        const int r0 = (4 * f) / kSh4RowFloats, r1 = (4 * f + 3) / kSh4RowFloats;
        const bool need = ((mask >> r0) | (mask >> r1)) & 1u;
        t4[f] = need ? __ldg(s4 + f) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
  } else {
#pragma unroll 5
    for (int e = lane; e < kSh4TileFloats; e += 32) {
      const int row = e / kSh4RowFloats, col = e - row * kSh4RowFloats;
      tile[e] = ((mask >> row) & 1u) ? __ldg(src + (size_t)row * K3 + col) : 0.f;
    }
  }
  __syncwarp();
}

// The warp's gradient tile -> rows row0 .. row0 + rows - 1 of v_sh, zeros for the bands past 4, and the tile cleared.
// Every element of those rows is written exactly once.
__device__ __forceinline__ void store_sh4_rows(float* __restrict__ tile, float* __restrict__ v_sh, size_t row0, int rows,
                                               int K3, int lane) {
  __syncwarp();
  float* dst = v_sh + row0 * K3;
  if (sh4_span_vec4(dst, K3, rows)) {
    float4* d4 = reinterpret_cast<float4*>(dst);
    float4* t4 = reinterpret_cast<float4*>(tile);
#pragma unroll
    for (int i = 0; i < (kSh4TileVec4 + 31) / 32; ++i) {
      const int f = i * 32 + lane;
      if (f < kSh4TileVec4) {
        d4[f] = t4[f];
        t4[f] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
  } else {
#pragma unroll 5
    for (int e = lane; e < kSh4TileFloats; e += 32) {
      const int row = e / kSh4RowFloats, col = e - row * kSh4RowFloats;
      if (row < rows) dst[(size_t)row * K3 + col] = tile[e];
      tile[e] = 0.f;
    }
    const int extra = K3 - kSh4RowFloats;
    if (extra > 0)
      for (int e = lane; e < rows * extra; e += 32) {
        const int row = e / extra;
        dst[(size_t)row * K3 + kSh4RowFloats + (e - row * extra)] = 0.f;
      }
  }
  __syncwarp();
}

// Kernel choice and launch of the camera models compiled in their own translation units (kOrtho, kFisheye): the
// forward (projection_fwd_launch.cuh) and the backward with the depth cotangent (projection_bwd_launch.cuh) of
// egs::ortho and egs::fisheye.
namespace ortho {
int launch_fwd(const ProjFwdParams& p, bool pc, bool vec4, cudaStream_t stream);
int launch_bwd(const ProjBwdParams& p, bool kg, bool vg, bool pc, bool vec4, bool antialiased, cudaStream_t stream);
}  // namespace ortho
namespace fisheye {
int launch_fwd(const ProjFwdParams& p, bool pc, bool vec4, cudaStream_t stream);
int launch_bwd(const ProjBwdParams& p, bool kg, bool vg, bool pc, bool vec4, bool antialiased, cudaStream_t stream);
}  // namespace fisheye

}  // namespace egs
