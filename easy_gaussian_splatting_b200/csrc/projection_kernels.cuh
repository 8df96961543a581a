// The projection kernels: the three forward kernels below (generic, K = 16, SH degree 4) and the three backward kernels
// of projection_bwd_kernels.cuh.  projection.cu includes this file twice: in namespace egs with kPerCameraSh = false (SH
// coefficients [N,K,3] shared by all cameras, or direct colours) and in egs::percam with kPerCameraSh = true (SH
// coefficients [C,N,K,3], one row per (camera, Gaussian)).  The per-camera code is behind `if constexpr`, so the
// shared-coefficient kernels keep their names and compile exactly as without it.
// kCameraModel (egs_math.cuh kPinhole / kOrtho / kFisheye) is the camera model of project_fwd / project_bwd: kPinhole in
// projection.cu; projection_ortho.cu and projection_fisheye.cu include this file in egs::ortho and egs::fisheye.
// (No include guard on purpose.)

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
  const bool vis = project_fwd<kCameraModel>(mean, quat, scale, cam, p.width, p.height, p.eps2d, p.near_plane, p.far_plane,
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
      load_coeffs<VEC4>(p.sh + (kPerCameraSh ? idx : (size_t)n) * p.K * 3, nb * 3, co);
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

// Forward, K = 16 SH coefficients (the reference's layout): only the coefficient rows of VISIBLE Gaussians
// are read, each as one contiguous 192-byte run by 12 lanes (a row-masked cooperative copy into a
// shared-memory tile), instead of twelve 16-byte loads per thread at a 192-byte lane stride.
__global__ void __launch_bounds__(kPF2Threads) projection_fwd_sh16_kernel(const ProjFwdParams p) {
  __shared__ Camera cam;
  __shared__ __align__(16) float tile[kPF2Threads / 32][32 * kFwdRowStride];
  // camera fastest: the C blocks that read one chunk of Gaussians (their 192 B of SH coefficients above all) run back
  // to back and share it through L2, instead of every camera streaming all Gaussians from HBM again (per-camera SH:
  // they share the Gaussians' geometry, each camera reads its own coefficient rows)
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
    vis = project_fwd<kCameraModel>(mean, quat, scale, cam, p.width, p.height, p.eps2d, p.near_plane, p.far_plane, p.radius_clip, st, o);
  }
  const uint32_t vis_mask = __ballot_sync(0xffffffffu, vis);
  const int nb = (p.sh_degree + 1) * (p.sh_degree + 1);
  const int need4 = (nb * 3 + 3) / 4;  // float4s of a row that hold active bands
  if (kPerCameraSh || !p.raw) {
    const float4* src = reinterpret_cast<const float4*>(p.sh) + ((kPerCameraSh ? (size_t)c * p.N : 0) + n_base) * 12;
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

// Forward, SH degree 4 (K >= 25): as projection_fwd_sh16_kernel, the coefficient rows of the warp's VISIBLE Gaussians
// go through a shared-memory tile (stage_sh4_rows), camera-fastest blocks.
__global__ void __launch_bounds__(kPF2Threads) projection_fwd_sh4_kernel(const ProjFwdParams p) {
  __shared__ Camera cam;
  __shared__ __align__(16) float tile[kPF2Threads / 32][kSh4TileFloats];
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
    ProjState st;
    vis = project_fwd<kCameraModel>(mean, quat, scale, cam, p.width, p.height, p.eps2d, p.near_plane, p.far_plane, p.radius_clip, st, o);
  }
  const uint32_t vis_mask = __ballot_sync(0xffffffffu, vis);
  if (vis_mask != 0)
    stage_sh4_rows(tile[warp], p.sh, (kPerCameraSh ? (size_t)c * p.N : 0) + n_base, min(32, p.N - n_base), p.K * 3,
                   vis_mask, lane);
  if (!in_range) return;
  int32_t ntiles = 0;
  int2 tight = make_int2(0, 0);
  float rgb[3] = {0.f, 0.f, 0.f};
  if (vis) {
    int32_t x0, y0, x1, y1;
    tile_rect(o.m2x, o.m2y, o.radius, p.tile_size, p.tile_w, p.tile_h, x0, y0, x1, y1);
    ntiles = (x1 - x0) * (y1 - y0);
    sh4_color_fwd(mean, cam, tile[warp] + lane * kSh4RowFloats, rgb);
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

#include "projection_bwd_kernels.cuh"
