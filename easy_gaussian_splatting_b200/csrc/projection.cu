// g1 + g2 (+ tile count of g3) forward, and g8 + g9 backward: per-Gaussian streaming kernels.
//
// Both are HBM-bound (SURVEY.md §8d: 68 B/Gaussian projection + 204 B/visible Gaussian SH forward;
// 108 + 408 B backward), one thread per Gaussian, so the arithmetic is free and is written in the
// oracle's canonical fp32 order (this file is compiled with -fmad=false) to make radii, tile counts,
// means2d and depth bits bit-identical to the oracle.
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

template <bool VEC4>
__global__ void __launch_bounds__(kProjThreads) projection_fwd_kernel(const ProjFwdParams p) {
  __shared__ Camera cam;
  // camera fastest: the C blocks that read one chunk of Gaussians run back to back and share it through L2
  const int c = blockIdx.x % p.C, chunk = blockIdx.x / p.C;
  if (threadIdx.x == 0) load_camera(p.viewmats + (size_t)c * 16, p.Ks + (size_t)c * 9, cam);
  __syncthreads();
  const int n = chunk * kProjThreads + threadIdx.x;
  if (n >= p.N) return;
  const size_t idx = (size_t)c * p.N + n;

  float mean[3], quat[4], scale[3];
  mean[0] = __ldg(p.means + 3 * (size_t)n + 0);
  mean[1] = __ldg(p.means + 3 * (size_t)n + 1);
  mean[2] = __ldg(p.means + 3 * (size_t)n + 2);
  float4 q4 = __ldg(reinterpret_cast<const float4*>(p.quats) + n);
  quat[0] = q4.x; quat[1] = q4.y; quat[2] = q4.z; quat[3] = q4.w;
  scale[0] = __ldg(p.scales + 3 * (size_t)n + 0);
  scale[1] = __ldg(p.scales + 3 * (size_t)n + 1);
  scale[2] = __ldg(p.scales + 3 * (size_t)n + 2);

  ProjState st;
  ProjOut o;
  const bool vis = project_fwd(mean, quat, scale, cam, p.width, p.height, p.eps2d, p.near_plane, p.far_plane,
                               p.radius_clip, st, o);
  int32_t ntiles = 0;
  int2 tight = make_int2(0, 0);
  float rgb[3] = {0.f, 0.f, 0.f};
  if (vis) {
    int32_t x0, y0, x1, y1;
    tile_rect(o.m2x, o.m2y, o.radius, p.tile_size, p.tile_w, p.tile_h, x0, y0, x1, y1);
    ntiles = (x1 - x0) * (y1 - y0);
    if (p.sh_degree >= 0) {
      const int nb = (p.sh_degree + 1) * (p.sh_degree + 1);
      float co[48];
      load_coeffs<VEC4>(p.sh + (size_t)n * p.K * 3, nb * 3, co);
      sh_color_fwd(p.sh_degree, mean, cam, co, rgb);
    } else {
      const float* cp = p.sh + (p.colors_per_camera ? idx : (size_t)n) * 3;
      rgb[0] = __ldg(cp + 0); rgb[1] = __ldg(cp + 1); rgb[2] = __ldg(cp + 2);
    }
    float opac = __ldg(p.opacities + n);
    if (p.antialiased) opac = opac * o.comp;
    float4* s = p.splats + idx * 3;
    s[0] = make_float4(o.m2x, o.m2y, o.ca, o.cb);
    s[1] = make_float4(o.cc, opac, rgb[0], rgb[1]);
    const float cut = sigma_cutoff(opac);
    s[2] = make_float4(rgb[2], o.depth, 0.f, cut);
    if (p.tight_rects != nullptr) {
      tighten_tile_rect(o.m2x, o.m2y, o.ca, o.cb, o.cc, cut, p.tile_size, x0, y0, x1, y1);
      pack_tile_rect(x0, y0, x1, y1, tight.x, tight.y);
    }
  }
  p.radii[idx] = o.radius;
  p.tiles_per_gauss[idx] = ntiles;
  if (p.tight_rects != nullptr) reinterpret_cast<int2*>(p.tight_rects)[idx] = tight;
  reinterpret_cast<float2*>(p.means2d)[idx] = make_float2(o.m2x, o.m2y);
  p.depths[idx] = o.depth;
  p.conics[idx * 3 + 0] = o.ca; p.conics[idx * 3 + 1] = o.cb; p.conics[idx * 3 + 2] = o.cc;
  p.colors[idx * 3 + 0] = rgb[0]; p.colors[idx * 3 + 1] = rgb[1]; p.colors[idx * 3 + 2] = rgb[2];
  if (p.antialiased) p.compensations[idx] = o.comp;
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

// Forward, K = 16 SH coefficients (the reference's layout): only the coefficient rows of VISIBLE Gaussians
// are read, each as one contiguous 192-byte run by 12 lanes (a row-masked cooperative copy into a
// shared-memory tile), instead of twelve 16-byte loads per thread at a 192-byte lane stride.
constexpr int kPF2Threads = 128;
constexpr int kFwdRowStride = 52;  // floats; conflict-free float4 row reads for a quarter warp

__global__ void __launch_bounds__(kPF2Threads) projection_fwd_sh16_kernel(const ProjFwdParams p) {
  __shared__ Camera cam;
  __shared__ __align__(16) float tile[kPF2Threads / 32][32 * kFwdRowStride];
  // camera fastest: the C blocks that read one chunk of Gaussians (their 192 B of SH coefficients above all) run back
  // to back and share it through L2, instead of every camera streaming all Gaussians from HBM again
  const int c = blockIdx.x % p.C, chunk = blockIdx.x / p.C;
  if (threadIdx.x == 0) load_camera(p.viewmats + (size_t)c * 16, p.Ks + (size_t)c * 9, cam);
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n_base = chunk * kPF2Threads + warp * 32;
  const int n = n_base + lane;
  const bool in_range = n < p.N;
  const size_t idx = (size_t)c * p.N + (in_range ? n : 0);

  float mean[3] = {0.f, 0.f, 0.f};
  ProjOut o;
  o.m2x = 0.f; o.m2y = 0.f; o.depth = 0.f; o.ca = 0.f; o.cb = 0.f; o.cc = 0.f; o.radius = 0; o.lambda_max = 0.f; o.comp = 0.f;
  bool vis = false;
  if (in_range) {
    float quat[4], scale[3];
    mean[0] = __ldg(p.means + 3 * (size_t)n + 0);
    mean[1] = __ldg(p.means + 3 * (size_t)n + 1);
    mean[2] = __ldg(p.means + 3 * (size_t)n + 2);
    const float4 q4 = __ldg(reinterpret_cast<const float4*>(p.quats) + n);
    quat[0] = q4.x; quat[1] = q4.y; quat[2] = q4.z; quat[3] = q4.w;
    scale[0] = __ldg(p.scales + 3 * (size_t)n + 0);
    scale[1] = __ldg(p.scales + 3 * (size_t)n + 1);
    scale[2] = __ldg(p.scales + 3 * (size_t)n + 2);
    if (p.raw) { scale[0] = act_exp(scale[0]); scale[1] = act_exp(scale[1]); scale[2] = act_exp(scale[2]); }
    ProjState st;
    vis = project_fwd(mean, quat, scale, cam, p.width, p.height, p.eps2d, p.near_plane, p.far_plane, p.radius_clip, st, o);
  }
  const uint32_t vis_mask = __ballot_sync(0xffffffffu, vis);
  const int nb = (p.sh_degree + 1) * (p.sh_degree + 1);
  const int need4 = (nb * 3 + 3) / 4;  // float4s of a row that hold active bands
  if (!p.raw) {
    const float4* src = reinterpret_cast<const float4*>(p.sh) + (size_t)n_base * 12;
    float* t = tile[warp];
#pragma unroll
    for (int i = 0; i < 12; ++i) {
      const int f = i * 32 + lane;
      const int row = f / 12, c4 = f - row * 12;
      if (((vis_mask >> row) & 1u) && c4 < need4)
        *reinterpret_cast<float4*>(t + row * kFwdRowStride + c4 * 4) = __ldg(src + f);
    }
  } else {
    load_rows_raw<kFwdRowStride>(tile[warp], p.sh, p.sh_rest, n_base, p.N, vis_mask, lane);
  }
  __syncwarp();
  if (!in_range) return;
  int32_t ntiles = 0;
  int2 tight = make_int2(0, 0);
  float rgb[3] = {0.f, 0.f, 0.f};
  if (vis) {
    int32_t x0, y0, x1, y1;
    tile_rect(o.m2x, o.m2y, o.radius, p.tile_size, p.tile_w, p.tile_h, x0, y0, x1, y1);
    ntiles = (x1 - x0) * (y1 - y0);
    const float* row = tile[warp] + lane * kFwdRowStride;
    const float dx = mean[0] - cam.campos[0], dy = mean[1] - cam.campos[1], dz = mean[2] - cam.campos[2];
    const float inorm = 1.0f / sqrtf(dx * dx + dy * dy + dz * dz);
    float Y[16];
    sh_basis(p.sh_degree, dx * inorm, dy * inorm, dz * inorm, Y);
    float r = 0.f, g = 0.f, b = 0.f;
    // same accumulation order as sh_color_fwd: band by band
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (j * 4 < nb) {
        float cf[12];
#pragma unroll
        for (int q = 0; q < 3; ++q) {
          const float4 t4 = *reinterpret_cast<const float4*>(row + j * 12 + q * 4);
          cf[q * 4 + 0] = t4.x; cf[q * 4 + 1] = t4.y; cf[q * 4 + 2] = t4.z; cf[q * 4 + 3] = t4.w;
        }
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          const int k = j * 4 + kk;
          if (k < nb) {
            r += Y[k] * cf[3 * kk + 0];
            g += Y[k] * cf[3 * kk + 1];
            b += Y[k] * cf[3 * kk + 2];
          }
        }
      }
    }
    rgb[0] = fmaxf(r + 0.5f, 0.f);
    rgb[1] = fmaxf(g + 0.5f, 0.f);
    rgb[2] = fmaxf(b + 0.5f, 0.f);
    float opac = __ldg(p.opacities + n);
    if (p.raw) opac = act_sigmoid(opac);
    if (p.antialiased) opac = opac * o.comp;
    float4* s = p.splats + idx * 3;
    s[0] = make_float4(o.m2x, o.m2y, o.ca, o.cb);
    s[1] = make_float4(o.cc, opac, rgb[0], rgb[1]);
    const float cut = sigma_cutoff(opac);
    s[2] = make_float4(rgb[2], o.depth, 0.f, cut);
    if (p.tight_rects != nullptr) {
      tighten_tile_rect(o.m2x, o.m2y, o.ca, o.cb, o.cc, cut, p.tile_size, x0, y0, x1, y1);
      pack_tile_rect(x0, y0, x1, y1, tight.x, tight.y);
    }
  }
  p.radii[idx] = o.radius;
  p.tiles_per_gauss[idx] = ntiles;
  if (p.tight_rects != nullptr) reinterpret_cast<int2*>(p.tight_rects)[idx] = tight;
  reinterpret_cast<float2*>(p.means2d)[idx] = make_float2(o.m2x, o.m2y);
  p.depths[idx] = o.depth;
  p.conics[idx * 3 + 0] = o.ca; p.conics[idx * 3 + 1] = o.cb; p.conics[idx * 3 + 2] = o.cc;
  p.colors[idx * 3 + 0] = rgb[0]; p.colors[idx * 3 + 1] = rgb[1]; p.colors[idx * 3 + 2] = rgb[2];
  if (p.antialiased) p.compensations[idx] = o.comp;
}

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
  // [C] of viewmat_grad_finalize_kernel are cleared by block 0
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

__device__ __forceinline__ float* cam_partial(const ProjBwdParams& p, int c, int warp) {
  const size_t slots = (size_t)gridDim.x * 4;
  return p.cam_partials + ((size_t)c * slots + (size_t)blockIdx.x * 4 + warp) * kCamPartialFloats;
}

__device__ __forceinline__ void clear_cam_counters(const ProjBwdParams& p) {
  if (blockIdx.x == 0)
    for (int c = threadIdx.x; c < p.C; c += blockDim.x) p.cam_counters[c] = 0;
}

// grid (slices, C): block (s, c) sums slice s of camera c's warp partials (strided per thread, then a fixed tree) into
// slices[c][s]; the last block of a camera to finish sums the slices in order and writes v_viewmats[c] (16 floats).
__global__ void __launch_bounds__(kVgFinalizeThreads) viewmat_grad_finalize_kernel(
    int n_slots, const float* __restrict__ partials, float* __restrict__ slices, int* __restrict__ counters,
    const float* __restrict__ viewmats, float* __restrict__ v_viewmats) {
  __shared__ float red[kCamGradFloats][kVgFinalizeThreads];
  __shared__ bool last;
  const int s = blockIdx.x, S = gridDim.x, c = blockIdx.y, tid = threadIdx.x;
  const int per = (n_slots + S - 1) / S;
  const int begin = s * per, end = min(n_slots, begin + per);
  float acc[kCamGradFloats];
#pragma unroll
  for (int k = 0; k < kCamGradFloats; ++k) acc[k] = 0.f;
  const float4* src = reinterpret_cast<const float4*>(partials + (size_t)c * n_slots * kCamPartialFloats);
  for (int i = begin + tid; i < end; i += kVgFinalizeThreads) {
    const float4 a = src[(size_t)i * 4 + 0], b = src[(size_t)i * 4 + 1], d = src[(size_t)i * 4 + 2], e = src[(size_t)i * 4 + 3];
    acc[0] += a.x; acc[1] += a.y; acc[2] += a.z; acc[3] += a.w;
    acc[4] += b.x; acc[5] += b.y; acc[6] += b.z; acc[7] += b.w;
    acc[8] += d.x; acc[9] += d.y; acc[10] += d.z; acc[11] += d.w;
    acc[12] += e.x; acc[13] += e.y; acc[14] += e.z;
  }
#pragma unroll
  for (int k = 0; k < kCamGradFloats; ++k) red[k][tid] = acc[k];
  __syncthreads();
  for (int h = kVgFinalizeThreads / 2; h > 0; h >>= 1) {
    if (tid < h)
#pragma unroll
      for (int k = 0; k < kCamGradFloats; ++k) red[k][tid] += red[k][tid + h];
    __syncthreads();
  }
  float* my_slice = slices + ((size_t)c * S + s) * kCamPartialFloats;
  if (tid < kCamGradFloats) my_slice[tid] = red[tid][0];
  __threadfence();
  __syncthreads();
  if (tid == 0) last = atomicAdd(counters + c, 1) == S - 1;
  __syncthreads();
  if (!last) return;
  __threadfence();
  if (tid < kCamGradFloats) {
    float sum = 0.f;
    for (int j = 0; j < S; ++j) sum += __ldcg(slices + ((size_t)c * S + j) * kCamPartialFloats + tid);
    red[tid][0] = sum;
  }
  __syncthreads();
  if (tid == 0) {
    float vcam[kCamGradFloats], out[16];
#pragma unroll
    for (int k = 0; k < kCamGradFloats; ++k) vcam[k] = red[k][0];
    viewmat_grad_finalize(viewmats + (size_t)c * 16, vcam, out);
#pragma unroll
    for (int k = 0; k < 16; ++k) v_viewmats[(size_t)c * 16 + k] = out[k];
    counters[c] = 0;
  }
}

// One thread per Gaussian, looping over cameras: gradients summed over cameras stay in registers,
// so there are no atomics for any C.  Every output element is written exactly once (zeros for culled
// Gaussians and inactive SH bands), so the caller does not have to clear the gradient buffers.
// VG: also the view-matrix gradient partials (see store_cam_partial).  Every lane of a warp then runs the camera loop
// (the shuffles need all 32), lanes past N as if they saw nothing.
template <bool VEC4, bool VG = false>
__global__ void __launch_bounds__(kProjBwdThreads) projection_bwd_kernel(const ProjBwdParams p) {
  __shared__ Camera cams[kMaxCamerasSmem];
  for (int c = threadIdx.x; c < p.C && c < kMaxCamerasSmem; c += kProjBwdThreads)
    load_camera(p.viewmats + (size_t)c * 16, p.Ks + (size_t)c * 9, cams[c]);
  if constexpr (VG) clear_cam_counters(p);
  __syncthreads();
  const int n_lane = blockIdx.x * kProjBwdThreads + threadIdx.x;
  if (!VG && n_lane >= p.N) return;
  const bool in_range = !VG || n_lane < p.N;
  const int n = VG ? min(n_lane, p.N - 1) : n_lane;  // (VG) lanes past N read Gaussian N - 1 and write nothing
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

  float mean[3], quat[4], scale[3];
  mean[0] = __ldg(p.means + 3 * (size_t)n + 0);
  mean[1] = __ldg(p.means + 3 * (size_t)n + 1);
  mean[2] = __ldg(p.means + 3 * (size_t)n + 2);
  float4 q4 = __ldg(reinterpret_cast<const float4*>(p.quats) + n);
  quat[0] = q4.x; quat[1] = q4.y; quat[2] = q4.z; quat[3] = q4.w;
  scale[0] = __ldg(p.scales + 3 * (size_t)n + 0);
  scale[1] = __ldg(p.scales + 3 * (size_t)n + 1);
  scale[2] = __ldg(p.scales + 3 * (size_t)n + 2);

  const bool has_sh = p.sh_degree >= 0;
  const int nb = has_sh ? (p.sh_degree + 1) * (p.sh_degree + 1) : 0;
  float v_mean[3] = {0.f, 0.f, 0.f}, v_quat[4] = {0.f, 0.f, 0.f, 0.f}, v_scale[3] = {0.f, 0.f, 0.f};
  float v_opac = 0.f;
  float vco[48];
#pragma unroll
  for (int i = 0; i < 48; ++i) vco[i] = 0.f;
  float co[48];
  bool co_loaded = false;
  float v_rgb_sum[3] = {0.f, 0.f, 0.f};

  for (int c = 0; c < p.C; ++c) {
    const size_t idx = (size_t)c * p.N + n;
    const bool vis = in_range && p.radii[idx] > 0;
    float v_rgb[3] = {0.f, 0.f, 0.f};
    float vcam[kCamGradFloats];
    if constexpr (VG) {
#pragma unroll
      for (int k = 0; k < kCamGradFloats; ++k) vcam[k] = 0.f;
    }
    if (p.absgrad != nullptr && in_range) {
      float2 ag = make_float2(0.f, 0.f);
      if (vis) { const float4 g2a = p.v_splats[idx * 3 + 2]; ag = make_float2(g2a.y, g2a.z); }
      p.absgrad[idx] = ag;
    }
    if (vis) {
      Camera cam_local;
      const Camera* cam = &cams[c < kMaxCamerasSmem ? c : 0];
      if (c >= kMaxCamerasSmem) { load_camera(p.viewmats + (size_t)c * 16, p.Ks + (size_t)c * 9, cam_local); cam = &cam_local; }
      const float4 g0 = p.v_splats[idx * 3 + 0];
      const float4 g1 = p.v_splats[idx * 3 + 1];
      const float4 g2 = p.v_splats[idx * 3 + 2];
      float v_m2x = g0.x, v_m2y = g0.y;
      if (p.v_means2d_extra != nullptr) {
        v_m2x += p.v_means2d_extra[idx * 2 + 0];
        v_m2y += p.v_means2d_extra[idx * 2 + 1];
      }
      ProjState st;
      ProjOut o;
      project_fwd(mean, quat, scale, *cam, p.width, p.height, p.eps2d, 0.f, INFINITY, -1.f, st, o);
      // (culling thresholds are irrelevant here: visibility was decided by the forward pass; the
      //  off-screen test cannot fire differently because it only depends on the same values.)
      float v_comp = 0.f, w_opac = 1.f;
      if (p.antialiased) { v_comp = g1.y * __ldg(p.opacities + n); w_opac = o.comp; }
      if (o.radius > 0)
        project_bwd(st, scale, *cam, v_m2x, v_m2y, 0.f, g0.z, g0.w, g1.x, o, v_mean, v_quat, v_scale, v_comp, p.eps2d,
                    VG ? vcam : nullptr, mean);
      v_opac += g1.y * w_opac;
      v_rgb[0] = g1.z; v_rgb[1] = g1.w; v_rgb[2] = g2.x;
      if (has_sh) {
        if (!co_loaded) { load_coeffs<VEC4>(p.sh + (size_t)n * p.K * 3, nb * 3, co); co_loaded = true; }
        const float* col = p.colors + idx * 3;
        const float rgb_stored[3] = {col[0], col[1], col[2]};
        sh_color_bwd(p.sh_degree, mean, *cam, co, rgb_stored, v_rgb, vco, v_mean, VG ? vcam : nullptr);
      } else {
        v_rgb_sum[0] += v_rgb[0]; v_rgb_sum[1] += v_rgb[1]; v_rgb_sum[2] += v_rgb[2];
      }
    }
    if (!has_sh && p.colors_per_camera && in_range) {
      p.v_sh[idx * 3 + 0] = v_rgb[0]; p.v_sh[idx * 3 + 1] = v_rgb[1]; p.v_sh[idx * 3 + 2] = v_rgb[2];
    }
    if constexpr (VG) store_cam_partial(vcam, __ballot_sync(0xffffffffu, vis) != 0, cam_partial(p, c, warp), lane);
  }
  if (!in_range) return;

  p.v_means[3 * (size_t)n + 0] = v_mean[0]; p.v_means[3 * (size_t)n + 1] = v_mean[1]; p.v_means[3 * (size_t)n + 2] = v_mean[2];
  reinterpret_cast<float4*>(p.v_quats)[n] = make_float4(v_quat[0], v_quat[1], v_quat[2], v_quat[3]);
  p.v_scales[3 * (size_t)n + 0] = v_scale[0]; p.v_scales[3 * (size_t)n + 1] = v_scale[1]; p.v_scales[3 * (size_t)n + 2] = v_scale[2];
  p.v_opacities[n] = v_opac;
  if (has_sh) {
    float* out = p.v_sh + (size_t)n * p.K * 3;
    const int total = p.K * 3;
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
  } else if (!p.colors_per_camera) {
    p.v_sh[3 * (size_t)n + 0] = v_rgb_sum[0]; p.v_sh[3 * (size_t)n + 1] = v_rgb_sum[1]; p.v_sh[3 * (size_t)n + 2] = v_rgb_sum[2];
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
#define EGS_PB_BOUNDS __launch_bounds__(kPB2Threads, EGS_PB_MIN_CTAS)
// AA: rasterize_mode="antialiased" (a separate instantiation keeps the classic kernel at 128 registers).
// VG: also the view-matrix gradient partials (see store_cam_partial).  The camera loop then runs on every lane of a warp
// that has a seen Gaussian (the shuffles need all 32); lanes that see nothing only take part in the sums.
template <bool AA, bool VG = false>
__global__ void EGS_PB_BOUNDS projection_bwd_sh16_kernel(const ProjBwdParams p) {
  extern __shared__ __align__(16) float smem_pb[];
  __shared__ Camera cams[kMaxCamerasSmem];
  for (int c = threadIdx.x; c < p.C && c < kMaxCamerasSmem; c += kPB2Threads)
    load_camera(p.viewmats + (size_t)c * 16, p.Ks + (size_t)c * 9, cams[c]);
  if constexpr (VG) clear_cam_counters(p);
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* co_tile = smem_pb + (size_t)warp * 32 * kRowStride;                       // coefficients
  float* vc_tile = smem_pb + (size_t)(kPB2Warps + warp) * 32 * kRowStride;         // gradient accumulation
  const int n_base = blockIdx.x * kPB2Threads + warp * 32;
  const int n = n_base + lane;
  const bool in_range = n < p.N;
  const int nb = (p.sh_degree + 1) * (p.sh_degree + 1);

  // which of this warp's Gaussians does any camera see?
  bool seen = false;
  if (in_range)
    for (int c = 0; c < p.C; ++c) seen = seen || (p.radii[(size_t)c * p.N + n] > 0);
  const uint32_t seen_mask = __ballot_sync(0xffffffffu, seen);
  if constexpr (VG) {
    if (seen_mask == 0)  // the warp sees nothing: zero partials for every camera
      for (int c = lane; c < p.C; c += 32) {
        float4* d = reinterpret_cast<float4*>(cam_partial(p, c, warp));
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        d[0] = z; d[1] = z; d[2] = z; d[3] = z;
      }
  }

  // phase 1: coalesced load of the coefficient rows that are needed; zero the gradient rows
  if (!p.raw) {
    const float4* src = reinterpret_cast<const float4*>(p.sh) + (size_t)n_base * (kRowFloats / 4);
#pragma unroll
    for (int i = 0; i < kRowFloats / 4; ++i) {
      const int f = i * 32 + lane;           // float4 index inside the warp's 32 x 12 block
      const int row = f / 12, c4 = f - row * 12;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (p.sh_degree >= 1 && ((seen_mask >> row) & 1u)) v = __ldg(src + f);
      *reinterpret_cast<float4*>(co_tile + row * kRowStride + c4 * 4) = v;
      *reinterpret_cast<float4*>(vc_tile + row * kRowStride + c4 * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  } else {
    if (p.sh_degree >= 1) load_rows_raw<kRowStride>(co_tile, p.sh, p.sh_rest, n_base, p.N, seen_mask, lane);
#pragma unroll
    for (int i = 0; i < kRowFloats / 4; ++i) {
      const int f = i * 32 + lane;
      const int row = f / 12, c4 = f - row * 12;
      *reinterpret_cast<float4*>(vc_tile + row * kRowStride + c4 * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  __syncwarp();

  // phase 2: thread-private work on its own Gaussian / its own two rows
  float v_mean[3] = {0.f, 0.f, 0.f}, v_quat[4] = {0.f, 0.f, 0.f, 0.f}, v_scale[3] = {0.f, 0.f, 0.f};
  float v_opac = 0.f;
  if (in_range && p.absgrad != nullptr) {
    for (int c = 0; c < p.C; ++c) {
      const size_t idx = (size_t)c * p.N + n;
      float2 ag = make_float2(0.f, 0.f);
      if (p.radii[idx] > 0) { const float4 g2a = p.v_splats[idx * 3 + 2]; ag = make_float2(g2a.y, g2a.z); }
      p.absgrad[idx] = ag;
    }
  }
  if (VG ? seen_mask != 0 : seen) {
    const int nl = VG ? (in_range ? n : n_base) : n;  // (VG) a lane past the range reads the warp's first Gaussian
    float mean[3], quat[4], scale[3];
    mean[0] = __ldg(p.means + 3 * (size_t)nl + 0);
    mean[1] = __ldg(p.means + 3 * (size_t)nl + 1);
    mean[2] = __ldg(p.means + 3 * (size_t)nl + 2);
    const float4 q4 = __ldg(reinterpret_cast<const float4*>(p.quats) + nl);
    quat[0] = q4.x; quat[1] = q4.y; quat[2] = q4.z; quat[3] = q4.w;
    scale[0] = __ldg(p.scales + 3 * (size_t)nl + 0);
    scale[1] = __ldg(p.scales + 3 * (size_t)nl + 1);
    scale[2] = __ldg(p.scales + 3 * (size_t)nl + 2);
    if (p.raw) { scale[0] = act_exp(scale[0]); scale[1] = act_exp(scale[1]); scale[2] = act_exp(scale[2]); }
    const float* co = co_tile + lane * kRowStride;
    float* vc = vc_tile + lane * kRowStride;
    // The gradient record, stored colour and radius of camera c + 1 are requested before camera c is worked on: the
    // loop is a chain of dependent global loads otherwise (one exposed latency per camera; long-scoreboard stalls
    // were the kernel's top stall reason, profiles/r2p).  Records of culled entries are zero, loading them is safe.
    float4 ng0, ng1, ng2;
    float ncol[3];
    int nrad;
    auto fetch = [&](int c) {
      const size_t idx = (size_t)c * p.N + nl;
      nrad = p.radii[idx];
      if (VG && !in_range) nrad = 0;
      ng0 = p.v_splats[idx * 3 + 0];
      ng1 = p.v_splats[idx * 3 + 1];
      ng2 = p.v_splats[idx * 3 + 2];
      ncol[0] = p.colors[idx * 3 + 0]; ncol[1] = p.colors[idx * 3 + 1]; ncol[2] = p.colors[idx * 3 + 2];
    };
    fetch(0);
    for (int c = 0; c < p.C; ++c) {
      const size_t idx = (size_t)c * p.N + n;
      const int rad = nrad;
      const float4 g0 = ng0, g1 = ng1, g2 = ng2;
      const float col[3] = {ncol[0], ncol[1], ncol[2]};
      if (c + 1 < p.C) fetch(c + 1);
      float vcam[kCamGradFloats];
      if constexpr (VG) {
#pragma unroll
        for (int k = 0; k < kCamGradFloats; ++k) vcam[k] = 0.f;
      } else {
        if (!(rad > 0)) continue;
      }
      do {  // (VG: lanes that do not see camera c skip to the warp's sum below)
      if (VG && !(rad > 0)) break;
      Camera cam_local;
      const Camera* cam = &cams[c < kMaxCamerasSmem ? c : 0];
      if (c >= kMaxCamerasSmem) { load_camera(p.viewmats + (size_t)c * 16, p.Ks + (size_t)c * 9, cam_local); cam = &cam_local; }
      float v_m2x = g0.x, v_m2y = g0.y;
      if (p.v_means2d_extra != nullptr) {
        v_m2x += p.v_means2d_extra[idx * 2 + 0];
        v_m2y += p.v_means2d_extra[idx * 2 + 1];
      }
      {
        ProjState st;
        ProjOut o;
        project_fwd(mean, quat, scale, *cam, p.width, p.height, p.eps2d, 0.f, INFINITY, -1.f, st, o);
        if constexpr (AA) {
          float op = __ldg(p.opacities + n);
          if (p.raw) op = act_sigmoid(op);
          if (o.radius > 0)
            project_bwd(st, scale, *cam, v_m2x, v_m2y, 0.f, g0.z, g0.w, g1.x, o, v_mean, v_quat, v_scale, g1.y * op, p.eps2d,
                        VG ? vcam : nullptr, mean);
          v_opac += g1.y * o.comp;
        } else {
          if (o.radius > 0)
            project_bwd(st, scale, *cam, v_m2x, v_m2y, 0.f, g0.z, g0.w, g1.x, o, v_mean, v_quat, v_scale, 0.f, 0.f,
                        VG ? vcam : nullptr, mean);
          v_opac += g1.y;
        }
      }
      // SH: rgb = max(sum + 0.5, 0) -> gradient passes where the stored colour is > 0
      const float vr = (col[0] > 0.f) ? g1.z : 0.f, vg = (col[1] > 0.f) ? g1.w : 0.f, vb = (col[2] > 0.f) ? g2.x : 0.f;
      const float dx = mean[0] - cam->campos[0], dy = mean[1] - cam->campos[1], dz = mean[2] - cam->campos[2];
      const float inorm = 1.0f / sqrtf(dx * dx + dy * dy + dz * dz);
      const float x = dx * inorm, y = dy * inorm, z = dz * inorm;
      float Y[16], g[16];
      sh_basis(p.sh_degree, x, y, z, Y);
      // rows are walked 4 bands (= 12 floats = 3 float4) at a time
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float cf[12], out[12];
        if (p.sh_degree >= 1) {
#pragma unroll
          for (int q = 0; q < 3; ++q) {
            const float4 t = *reinterpret_cast<const float4*>(co + j * 12 + q * 4);
            cf[q * 4 + 0] = t.x; cf[q * 4 + 1] = t.y; cf[q * 4 + 2] = t.z; cf[q * 4 + 3] = t.w;
          }
        }
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          const int k = j * 4 + kk;
          const bool act = k < nb;
          g[k] = (act && p.sh_degree >= 1) ? (cf[3 * kk + 0] * vr + cf[3 * kk + 1] * vg + cf[3 * kk + 2] * vb) : 0.f;
          const float yk = act ? Y[k] : 0.f;
          out[3 * kk + 0] = yk * vr; out[3 * kk + 1] = yk * vg; out[3 * kk + 2] = yk * vb;
        }
        if (j * 4 < nb) {
#pragma unroll
          for (int q = 0; q < 3; ++q) {
            float4* dst = reinterpret_cast<float4*>(vc + j * 12 + q * 4);
            float4 acc = *dst;
            acc.x += out[q * 4 + 0]; acc.y += out[q * 4 + 1]; acc.z += out[q * 4 + 2]; acc.w += out[q * 4 + 3];
            *dst = acc;
          }
        }
      }
      if (p.sh_degree >= 1) {
        float vx, vy, vz;
        sh_basis_vjp(p.sh_degree, x, y, z, g, vx, vy, vz);
        const float dp = vx * x + vy * y + vz * z;
        const float d0 = (vx - dp * x) * inorm, d1 = (vy - dp * y) * inorm, d2 = (vz - dp * z) * inorm;
        v_mean[0] += d0;
        v_mean[1] += d1;
        v_mean[2] += d2;
        if constexpr (VG) { vcam[12] -= d0; vcam[13] -= d1; vcam[14] -= d2; }  // dir = mean - campos
      }
      } while (0);
      if constexpr (VG) store_cam_partial(vcam, __ballot_sync(0xffffffffu, rad > 0) != 0, cam_partial(p, c, warp), lane);
    }
  }
  __syncwarp();

  // VJPs of the folded activations: d exp = exp, d sigmoid = o (1 - o)
  if (p.raw && seen) {
    v_scale[0] *= act_exp(__ldg(p.scales + 3 * (size_t)n + 0));
    v_scale[1] *= act_exp(__ldg(p.scales + 3 * (size_t)n + 1));
    v_scale[2] *= act_exp(__ldg(p.scales + 3 * (size_t)n + 2));
    const float o_ = act_sigmoid(__ldg(p.opacities + n));
    v_opac *= o_ * (1.0f - o_);
  }
  // phase 3: coalesced store of the gradient rows; small per-Gaussian outputs directly
  if (!p.raw) {
    float4* dst = reinterpret_cast<float4*>(p.v_sh) + (size_t)n_base * (kRowFloats / 4);
#pragma unroll
    for (int i = 0; i < kRowFloats / 4; ++i) {
      const int f = i * 32 + lane;
      const int row = f / 12, c4 = f - row * 12;
      if (n_base + row < p.N) dst[f] = *reinterpret_cast<const float4*>(vc_tile + row * kRowStride + c4 * 4);
    }
  } else {
    store_rows_raw<kRowStride>(vc_tile, p.v_sh, p.v_sh_rest, n_base, p.N, lane);
  }
  if (in_range) {
    p.v_means[3 * (size_t)n + 0] = v_mean[0]; p.v_means[3 * (size_t)n + 1] = v_mean[1]; p.v_means[3 * (size_t)n + 2] = v_mean[2];
    reinterpret_cast<float4*>(p.v_quats)[n] = make_float4(v_quat[0], v_quat[1], v_quat[2], v_quat[3]);
    p.v_scales[3 * (size_t)n + 0] = v_scale[0]; p.v_scales[3 * (size_t)n + 1] = v_scale[1]; p.v_scales[3 * (size_t)n + 2] = v_scale[2];
    p.v_opacities[n] = v_opac;
  }
}

}  // namespace egs

using namespace egs;

static int projection_fwd_impl(int32_t C, int32_t N, const float* means, const float* quats, const float* scales,
                               const float* opacities, const float* sh_coeffs, const float* sh_rest, int32_t K,
                               int32_t sh_degree, int32_t colors_per_camera, const float* viewmats, const float* Ks,
                               int32_t width, int32_t height, float eps2d, float near_plane, float far_plane,
                               float radius_clip, int32_t tile_size, int32_t tile_width, int32_t tile_height,
                               int32_t* radii, float* means2d, float* depths, float* conics, float* colors,
                               int32_t* tiles_per_gauss, int32_t* tight_rects, float* splats, egs_stream_t stream,
                               float* compensations = nullptr) {
  const int raw = sh_rest != nullptr;
  EGS_REQUIRE(C >= 0 && N >= 0, "projection_fwd: negative sizes C=%d N=%d", C, N);
  EGS_REQUIRE(C <= 65535, "projection_fwd: C=%d exceeds 65535 cameras per call", C);
  EGS_REQUIRE(width >= 1 && height >= 1, "projection_fwd: width/height must be >= 1 (got %d x %d)", width, height);
  EGS_REQUIRE(tile_size >= 1 && (tile_size & (tile_size - 1)) == 0, "projection_fwd: tile_size must be a power of two");
  EGS_REQUIRE(sh_degree <= 3, "projection_fwd: sh_degree %d > 3 is not supported", sh_degree);
  EGS_REQUIRE(tight_rects == nullptr || (tile_width < 65536 && tile_height < 65536),
              "projection_fwd: tile grid %d x %d too large for the packed tight rectangles", tile_width, tile_height);
  EGS_REQUIRE(sh_degree < 0 || K >= (sh_degree + 1) * (sh_degree + 1), "projection_fwd: K=%d too small for sh_degree=%d", K, sh_degree);
  if (C == 0 || N == 0) return 0;
  ProjFwdParams p;
  p.C = C; p.N = N; p.K = K; p.sh_degree = sh_degree; p.colors_per_camera = colors_per_camera;
  p.means = means; p.quats = quats; p.scales = scales; p.opacities = opacities; p.sh = sh_coeffs;
  p.viewmats = viewmats; p.Ks = Ks;
  p.width = (float)width; p.height = (float)height; p.eps2d = eps2d; p.near_plane = near_plane;
  p.far_plane = far_plane; p.radius_clip = radius_clip; p.tile_size = (float)tile_size;
  p.tile_w = tile_width; p.tile_h = tile_height;
  p.radii = radii; p.means2d = means2d; p.depths = depths; p.conics = conics; p.colors = colors;
  p.tiles_per_gauss = tiles_per_gauss; p.tight_rects = tight_rects; p.splats = reinterpret_cast<float4*>(splats);
  p.raw = raw; p.sh_rest = sh_rest;
  p.antialiased = compensations != nullptr; p.compensations = compensations;
  const unsigned grid = (unsigned)(ceil_div(N, kProjThreads) * C);
  const bool vec4 = sh_degree >= 0 && (K * 3) % 4 == 0 && (reinterpret_cast<uintptr_t>(sh_coeffs) % 16 == 0);
  if (raw) {
    EGS_REQUIRE(K == 16 && sh_degree >= 0, "projection_fwd_raw: needs sh_0 [N,1,3] + sh_rest [N,15,3] and sh_degree >= 0");
  }
  if (raw || (vec4 && K == 16)) {
    const unsigned grid2 = (unsigned)(ceil_div(N, kPF2Threads) * C);
    projection_fwd_sh16_kernel<<<grid2, kPF2Threads, 0, (cudaStream_t)stream>>>(p);
    return check_launch("projection_fwd_sh16_kernel");
  }
  if (vec4) projection_fwd_kernel<true><<<grid, kProjThreads, 0, (cudaStream_t)stream>>>(p);
  else      projection_fwd_kernel<false><<<grid, kProjThreads, 0, (cudaStream_t)stream>>>(p);
  return check_launch("projection_fwd_kernel");
}

extern "C" int egs_projection_fwd(int32_t C, int32_t N, const float* means, const float* quats, const float* scales,
                                  const float* opacities, const float* sh_coeffs, int32_t K, int32_t sh_degree,
                                  int32_t colors_per_camera, const float* viewmats, const float* Ks, int32_t width,
                                  int32_t height, float eps2d, float near_plane, float far_plane, float radius_clip,
                                  int32_t tile_size, int32_t tile_width, int32_t tile_height, int32_t* radii,
                                  float* means2d, float* depths, float* conics, float* colors,
                                  int32_t* tiles_per_gauss, int32_t* tight_rects, float* splats, egs_stream_t stream) {
  return projection_fwd_impl(C, N, means, quats, scales, opacities, sh_coeffs, nullptr, K, sh_degree, colors_per_camera,
                             viewmats, Ks, width, height, eps2d, near_plane, far_plane, radius_clip, tile_size,
                             tile_width, tile_height, radii, means2d, depths, conics, colors, tiles_per_gauss, tight_rects,
                             splats, stream);
}

extern "C" int egs_projection_fwd_antialiased(
    int32_t C, int32_t N, const float* means, const float* quats, const float* scales, const float* opacities,
    const float* sh_coeffs, int32_t K, int32_t sh_degree, int32_t colors_per_camera, const float* viewmats,
    const float* Ks, int32_t width, int32_t height, float eps2d, float near_plane, float far_plane, float radius_clip,
    int32_t tile_size, int32_t tile_width, int32_t tile_height, int32_t* radii, float* means2d, float* depths,
    float* conics, float* colors, int32_t* tiles_per_gauss, int32_t* tight_rects, float* splats, float* compensations,
    egs_stream_t stream) {
  EGS_REQUIRE(compensations != nullptr, "projection_fwd_antialiased: compensations output is required");
  return projection_fwd_impl(C, N, means, quats, scales, opacities, sh_coeffs, nullptr, K, sh_degree, colors_per_camera,
                             viewmats, Ks, width, height, eps2d, near_plane, far_plane, radius_clip, tile_size,
                             tile_width, tile_height, radii, means2d, depths, conics, colors, tiles_per_gauss, tight_rects,
                             splats, stream, compensations);
}

extern "C" int egs_projection_fwd_raw(int32_t C, int32_t N, const float* means, const float* quats,
                                      const float* log_scales, const float* logit_opacities, const float* sh_0,
                                      const float* sh_rest, int32_t sh_degree, const float* viewmats, const float* Ks,
                                      int32_t width, int32_t height, float eps2d, float near_plane, float far_plane,
                                      float radius_clip, int32_t tile_size, int32_t tile_width, int32_t tile_height,
                                      int32_t* radii, float* means2d, float* depths, float* conics, float* colors,
                                      int32_t* tiles_per_gauss, int32_t* tight_rects, float* splats, egs_stream_t stream) {
  EGS_REQUIRE(sh_rest != nullptr && sh_0 != nullptr, "projection_fwd_raw: sh_0 and sh_rest are required");
  EGS_REQUIRE(reinterpret_cast<uintptr_t>(sh_0) % 16 == 0 && reinterpret_cast<uintptr_t>(sh_rest) % 16 == 0,
              "projection_fwd_raw: sh_0 and sh_rest must be 16-byte aligned");
  return projection_fwd_impl(C, N, means, quats, log_scales, logit_opacities, sh_0, sh_rest, 16, sh_degree, 0, viewmats,
                             Ks, width, height, eps2d, near_plane, far_plane, radius_clip, tile_size, tile_width,
                             tile_height, radii, means2d, depths, conics, colors, tiles_per_gauss, tight_rects, splats, stream);
}

static int projection_bwd_impl(int32_t C, int32_t N, const float* means, const float* quats, const float* scales,
                               const float* opacities_raw, const float* sh_coeffs, const float* sh_rest, int32_t K,
                               int32_t sh_degree, int32_t colors_per_camera, const float* viewmats, const float* Ks,
                               int32_t width, int32_t height, float eps2d, const int32_t* radii, const float* colors,
                               const float* v_splats, const float* v_means2d_extra, float* v_means, float* v_quats,
                               float* v_scales, float* v_opacities, float* v_sh_coeffs, float* v_sh_rest, float* absgrad,
                               egs_stream_t stream, int antialiased = 0, float* v_viewmats = nullptr,
                               void* workspace = nullptr, int64_t workspace_bytes = 0) {
  const int raw = sh_rest != nullptr;
  EGS_REQUIRE(C >= 0 && N >= 0, "projection_bwd: negative sizes C=%d N=%d", C, N);
  EGS_REQUIRE(sh_degree <= 3, "projection_bwd: sh_degree %d > 3 is not supported", sh_degree);
  EGS_REQUIRE(sh_degree < 0 || K >= (sh_degree + 1) * (sh_degree + 1), "projection_bwd: K=%d too small for sh_degree=%d", K, sh_degree);
  const bool vg = v_viewmats != nullptr;
  if (vg) {
    EGS_REQUIRE(C <= 65535, "projection_bwd: C=%d exceeds 65535 cameras per call", C);
    EGS_REQUIRE(workspace != nullptr && workspace_bytes >= egs_projection_bwd_viewmats_workspace_bytes(C, N),
                "projection_bwd: viewmat gradients need %lld workspace bytes (got %lld)",
                (long long)egs_projection_bwd_viewmats_workspace_bytes(C, N), (long long)workspace_bytes);
    if (N == 0 && C > 0) EGS_CUDA(cudaMemsetAsync(v_viewmats, 0, sizeof(float) * 16 * (size_t)C, (cudaStream_t)stream));
  }
  if (N == 0) return 0;
  ProjBwdParams p;
  p.C = C; p.N = N; p.K = K; p.sh_degree = sh_degree; p.colors_per_camera = colors_per_camera;
  p.means = means; p.quats = quats; p.scales = scales; p.sh = sh_coeffs; p.viewmats = viewmats; p.Ks = Ks;
  p.width = (float)width; p.height = (float)height; p.eps2d = eps2d;
  p.radii = radii; p.colors = colors; p.v_splats = reinterpret_cast<const float4*>(v_splats);
  p.v_means2d_extra = v_means2d_extra;
  p.v_means = v_means; p.v_quats = v_quats; p.v_scales = v_scales; p.v_opacities = v_opacities; p.v_sh = v_sh_coeffs;
  p.absgrad = reinterpret_cast<float2*>(absgrad);
  p.raw = raw; p.sh_rest = sh_rest; p.opacities = opacities_raw; p.v_sh_rest = v_sh_rest;
  p.antialiased = antialiased;
  p.cam_partials = nullptr; p.cam_counters = nullptr;
  EGS_REQUIRE(!antialiased || opacities_raw != nullptr, "projection_bwd: antialiased mode needs the opacities");
  const int64_t vg_slots = vg_partial_slots(N);
  if (vg) {
    p.cam_partials = static_cast<float*>(workspace);
    p.cam_counters = reinterpret_cast<int*>(p.cam_partials + (size_t)(C * vg_slots + C * vg_slices(vg_slots)) * kCamPartialFloats);
  }
  // viewmat_grad_finalize_kernel, after either backward kernel
  auto finalize = [&]() -> int {
    if (C == 0) return 0;
    const int S = vg_slices(vg_slots);
    float* slices = p.cam_partials + (size_t)C * vg_slots * kCamPartialFloats;
    viewmat_grad_finalize_kernel<<<dim3((unsigned)S, (unsigned)C), kVgFinalizeThreads, 0, (cudaStream_t)stream>>>(
        (int)vg_slots, p.cam_partials, slices, p.cam_counters, viewmats, v_viewmats);
    return check_launch("viewmat_grad_finalize_kernel");
  };
  const bool vec4 = sh_degree >= 0 && (K * 3) % 4 == 0 && (reinterpret_cast<uintptr_t>(sh_coeffs) % 16 == 0) &&
                    (reinterpret_cast<uintptr_t>(v_sh_coeffs) % 16 == 0);
  if (raw) {
    EGS_REQUIRE(K == 16 && sh_degree >= 0 && v_sh_rest != nullptr && opacities_raw != nullptr,
                "projection_bwd_raw: needs sh_0 / sh_rest (K = 16), logits and sh_degree >= 0");
  }
  if (raw || (vec4 && K == 16)) {
    // the reference's layout (K = 16): coalesced shared-memory staged rows
    constexpr int kSmem = 2 * kPB2Warps * 32 * kRowStride * (int)sizeof(float);
    auto kern = vg ? (antialiased ? projection_bwd_sh16_kernel<true, true> : projection_bwd_sh16_kernel<false, true>)
                   : (antialiased ? projection_bwd_sh16_kernel<true> : projection_bwd_sh16_kernel<false>);
    const cudaError_t attr_rc =  // per-device attribute: set on every call (cheap), not once per process
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
    if (attr_rc != cudaSuccess) return fail((int)attr_rc, "projection_bwd: shared memory opt-in failed: %s", cudaGetErrorString(attr_rc));
    kern<<<(unsigned)ceil_div(N, kPB2Threads), kPB2Threads, kSmem, (cudaStream_t)stream>>>(p);
    const int rc = check_launch("projection_bwd_sh16_kernel");
    return (rc != 0 || !vg) ? rc : finalize();
  }
  unsigned grid = (unsigned)ceil_div(N, kProjBwdThreads);
  if (vg) {
    if (vec4) projection_bwd_kernel<true, true><<<grid, kProjBwdThreads, 0, (cudaStream_t)stream>>>(p);
    else      projection_bwd_kernel<false, true><<<grid, kProjBwdThreads, 0, (cudaStream_t)stream>>>(p);
    const int rc = check_launch("projection_bwd_kernel");
    return rc != 0 ? rc : finalize();
  }
  if (vec4) projection_bwd_kernel<true><<<grid, kProjBwdThreads, 0, (cudaStream_t)stream>>>(p);
  else      projection_bwd_kernel<false><<<grid, kProjBwdThreads, 0, (cudaStream_t)stream>>>(p);
  return check_launch("projection_bwd_kernel");
}

extern "C" int egs_projection_bwd(int32_t C, int32_t N, const float* means, const float* quats, const float* scales,
                                  const float* sh_coeffs, int32_t K, int32_t sh_degree, int32_t colors_per_camera,
                                  const float* viewmats, const float* Ks, int32_t width, int32_t height, float eps2d,
                                  const int32_t* radii, const float* colors, const float* v_splats,
                                  const float* v_means2d_extra, float* v_means, float* v_quats, float* v_scales,
                                  float* v_opacities, float* v_sh_coeffs, float* absgrad, egs_stream_t stream) {
  return projection_bwd_impl(C, N, means, quats, scales, nullptr, sh_coeffs, nullptr, K, sh_degree, colors_per_camera,
                             viewmats, Ks, width, height, eps2d, radii, colors, v_splats, v_means2d_extra, v_means,
                             v_quats, v_scales, v_opacities, v_sh_coeffs, nullptr, absgrad, stream);
}

extern "C" int egs_projection_bwd_antialiased(
    int32_t C, int32_t N, const float* means, const float* quats, const float* scales, const float* opacities,
    const float* sh_coeffs, int32_t K, int32_t sh_degree, int32_t colors_per_camera, const float* viewmats,
    const float* Ks, int32_t width, int32_t height, float eps2d, const int32_t* radii, const float* colors,
    const float* v_splats, const float* v_means2d_extra, float* v_means, float* v_quats, float* v_scales,
    float* v_opacities, float* v_sh_coeffs, float* absgrad, egs_stream_t stream) {
  return projection_bwd_impl(C, N, means, quats, scales, opacities, sh_coeffs, nullptr, K, sh_degree, colors_per_camera,
                             viewmats, Ks, width, height, eps2d, radii, colors, v_splats, v_means2d_extra, v_means,
                             v_quats, v_scales, v_opacities, v_sh_coeffs, nullptr, absgrad, stream, 1);
}

extern "C" int egs_projection_bwd_raw(int32_t C, int32_t N, const float* means, const float* quats,
                                      const float* log_scales, const float* logit_opacities, const float* sh_0,
                                      const float* sh_rest, int32_t sh_degree, const float* viewmats, const float* Ks,
                                      int32_t width, int32_t height, float eps2d, const int32_t* radii,
                                      const float* colors, const float* v_splats, const float* v_means2d_extra,
                                      float* v_means, float* v_quats, float* v_log_scales, float* v_logit_opacities,
                                      float* v_sh_0, float* v_sh_rest, float* absgrad, egs_stream_t stream) {
  EGS_REQUIRE(sh_rest != nullptr && sh_0 != nullptr, "projection_bwd_raw: sh_0 and sh_rest are required");
  EGS_REQUIRE(reinterpret_cast<uintptr_t>(sh_0) % 16 == 0 && reinterpret_cast<uintptr_t>(sh_rest) % 16 == 0 &&
                  reinterpret_cast<uintptr_t>(v_sh_0) % 16 == 0 && reinterpret_cast<uintptr_t>(v_sh_rest) % 16 == 0,
              "projection_bwd_raw: sh_0 / sh_rest and their gradients must be 16-byte aligned");
  return projection_bwd_impl(C, N, means, quats, log_scales, logit_opacities, sh_0, sh_rest, 16, sh_degree, 0, viewmats,
                             Ks, width, height, eps2d, radii, colors, v_splats, v_means2d_extra, v_means, v_quats,
                             v_log_scales, v_logit_opacities, v_sh_0, v_sh_rest, absgrad, stream);
}

/* ---- gradients w.r.t. the view matrices ---- */
extern "C" int64_t egs_projection_bwd_viewmats_workspace_bytes(int32_t C, int32_t N) {
  if (C <= 0 || N < 0) return 0;
  const int64_t slots = vg_partial_slots(N);
  return (int64_t)C * (slots + vg_slices(slots)) * kCamPartialFloats * (int64_t)sizeof(float) + (int64_t)C * (int64_t)sizeof(int);
}

extern "C" int egs_projection_bwd_viewmats(
    int32_t C, int32_t N, const float* means, const float* quats, const float* scales, const float* opacities,
    const float* sh_coeffs, int32_t K, int32_t sh_degree, int32_t colors_per_camera, const float* viewmats,
    const float* Ks, int32_t width, int32_t height, float eps2d, const int32_t* radii, const float* colors,
    const float* v_splats, const float* v_means2d_extra, float* v_means, float* v_quats, float* v_scales,
    float* v_opacities, float* v_sh_coeffs, float* absgrad, int32_t antialiased, float* v_viewmats, void* workspace,
    int64_t workspace_bytes, egs_stream_t stream) {
  EGS_REQUIRE(v_viewmats != nullptr, "projection_bwd_viewmats: v_viewmats output is required");
  return projection_bwd_impl(C, N, means, quats, scales, antialiased ? opacities : nullptr, sh_coeffs, nullptr, K,
                             sh_degree, colors_per_camera, viewmats, Ks, width, height, eps2d, radii, colors, v_splats,
                             v_means2d_extra, v_means, v_quats, v_scales, v_opacities, v_sh_coeffs, nullptr, absgrad,
                             stream, antialiased ? 1 : 0, v_viewmats, workspace, workspace_bytes);
}

extern "C" int egs_projection_bwd_raw_viewmats(
    int32_t C, int32_t N, const float* means, const float* quats, const float* log_scales, const float* logit_opacities,
    const float* sh_0, const float* sh_rest, int32_t sh_degree, const float* viewmats, const float* Ks, int32_t width,
    int32_t height, float eps2d, const int32_t* radii, const float* colors, const float* v_splats,
    const float* v_means2d_extra, float* v_means, float* v_quats, float* v_log_scales, float* v_logit_opacities,
    float* v_sh_0, float* v_sh_rest, float* absgrad, float* v_viewmats, void* workspace, int64_t workspace_bytes,
    egs_stream_t stream) {
  EGS_REQUIRE(v_viewmats != nullptr, "projection_bwd_raw_viewmats: v_viewmats output is required");
  EGS_REQUIRE(sh_rest != nullptr && sh_0 != nullptr, "projection_bwd_raw: sh_0 and sh_rest are required");
  EGS_REQUIRE(reinterpret_cast<uintptr_t>(sh_0) % 16 == 0 && reinterpret_cast<uintptr_t>(sh_rest) % 16 == 0 &&
                  reinterpret_cast<uintptr_t>(v_sh_0) % 16 == 0 && reinterpret_cast<uintptr_t>(v_sh_rest) % 16 == 0,
              "projection_bwd_raw: sh_0 / sh_rest and their gradients must be 16-byte aligned");
  return projection_bwd_impl(C, N, means, quats, log_scales, logit_opacities, sh_0, sh_rest, 16, sh_degree, 0, viewmats,
                             Ks, width, height, eps2d, radii, colors, v_splats, v_means2d_extra, v_means, v_quats,
                             v_log_scales, v_logit_opacities, v_sh_0, v_sh_rest, absgrad, stream, 0, v_viewmats,
                             workspace, workspace_bytes);
}
