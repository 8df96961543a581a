// g1 + g2 (+ tile count of g3) forward, and g8 + g9 backward: per-Gaussian streaming kernels.
//
// Both are HBM-bound (SURVEY.md §8d: 68 B/Gaussian projection + 204 B/visible Gaussian SH forward;
// 108 + 408 B backward), one thread per Gaussian, so the arithmetic is free and is written in the
// oracle's canonical fp32 order (this file is compiled with -fmad=false) to make radii, tile counts,
// means2d and depth bits bit-identical to the oracle.
#include "projection_common.cuh"

namespace egs {

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

// As viewmat_grad_finalize_kernel, for the 20-float partials of the egs::ksgrad kernels: writes v_Ks[c] (9 floats) and,
// when v_viewmats is not null, v_viewmats[c] (16 floats).
__global__ void __launch_bounds__(kVgFinalizeThreads) intrinsics_grad_finalize_kernel(
    int n_slots, const float* __restrict__ partials, float* __restrict__ slices, int* __restrict__ counters,
    const float* __restrict__ viewmats, float* __restrict__ v_viewmats, float* __restrict__ v_Ks) {
  __shared__ float red[kCamKsGradFloats][kVgFinalizeThreads];
  __shared__ bool last;
  const int s = blockIdx.x, S = gridDim.x, c = blockIdx.y, tid = threadIdx.x;
  const int per = (n_slots + S - 1) / S;
  const int begin = s * per, end = min(n_slots, begin + per);
  float acc[kCamKsGradFloats];
#pragma unroll
  for (int k = 0; k < kCamKsGradFloats; ++k) acc[k] = 0.f;
  const float4* src = reinterpret_cast<const float4*>(partials + (size_t)c * n_slots * kCamKsPartialFloats);
  for (int i = begin + tid; i < end; i += kVgFinalizeThreads) {
    const float4* q = src + (size_t)i * (kCamKsPartialFloats / 4);
    const float4 a = q[0], b = q[1], d = q[2], e = q[3], f = q[4];
    acc[0] += a.x; acc[1] += a.y; acc[2] += a.z; acc[3] += a.w;
    acc[4] += b.x; acc[5] += b.y; acc[6] += b.z; acc[7] += b.w;
    acc[8] += d.x; acc[9] += d.y; acc[10] += d.z; acc[11] += d.w;
    acc[12] += e.x; acc[13] += e.y; acc[14] += e.z; acc[15] += e.w;
    acc[16] += f.x; acc[17] += f.y; acc[18] += f.z;
  }
#pragma unroll
  for (int k = 0; k < kCamKsGradFloats; ++k) red[k][tid] = acc[k];
  __syncthreads();
  for (int h = kVgFinalizeThreads / 2; h > 0; h >>= 1) {
    if (tid < h)
#pragma unroll
      for (int k = 0; k < kCamKsGradFloats; ++k) red[k][tid] += red[k][tid + h];
    __syncthreads();
  }
  float* my_slice = slices + ((size_t)c * S + s) * kCamKsPartialFloats;
  if (tid < kCamKsGradFloats) my_slice[tid] = red[tid][0];
  __threadfence();
  __syncthreads();
  if (tid == 0) last = atomicAdd(counters + c, 1) == S - 1;
  __syncthreads();
  if (!last) return;
  __threadfence();
  if (tid < kCamKsGradFloats) {
    float sum = 0.f;
    for (int j = 0; j < S; ++j) sum += __ldcg(slices + ((size_t)c * S + j) * kCamKsPartialFloats + tid);
    red[tid][0] = sum;
  }
  __syncthreads();
  if (tid == 0) {
    float vcam[kCamGradFloats], vk[kKsGradFloats], out[16], kout[9];
#pragma unroll
    for (int k = 0; k < kCamGradFloats; ++k) vcam[k] = red[k][0];
#pragma unroll
    for (int k = 0; k < kKsGradFloats; ++k) vk[k] = red[kCamGradFloats + k][0];
    if (v_viewmats != nullptr) {
      viewmat_grad_finalize(viewmats + (size_t)c * 16, vcam, out);
#pragma unroll
      for (int k = 0; k < 16; ++k) v_viewmats[(size_t)c * 16 + k] = out[k];
    }
    ks_grad_finalize(vk, kout);
#pragma unroll
    for (int k = 0; k < 9; ++k) v_Ks[(size_t)c * 9 + k] = kout[k];
    counters[c] = 0;
  }
}


constexpr int kCameraModel = kPinhole;
constexpr bool kPerCameraSh = false;
constexpr bool kKsGrad = false;
constexpr bool kDepthGrad = false;
#include "projection_kernels.cuh"

namespace percam {
constexpr bool kPerCameraSh = true;
#include "projection_kernels.cuh"
}  // namespace percam

// Intrinsics gradients: only the VG forms of the backward kernels are instantiated here.  They are separate kernels so
// that the pose-only forms keep their registers (the classic sh16 one sits at the 168-register cap of 3 CTAs/SM).
namespace ksgrad {
constexpr bool kKsGrad = true;
#include "projection_bwd_kernels.cuh"

namespace percam {
constexpr bool kPerCameraSh = true;
#include "projection_bwd_kernels.cuh"
}  // namespace percam
}  // namespace ksgrad

#include "projection_fwd_launch.cuh"
#include "projection_bwd_launch.cuh"

// The backward kernels once more, with the depth cotangent of gradient-record slot 11 (render modes with expected
// depth): every form above, in a namespace of its own so that the kernels above keep their code and registers.
namespace depth {
constexpr bool kDepthGrad = true;
#include "projection_bwd_kernels.cuh"

namespace percam {
constexpr bool kPerCameraSh = true;
#include "projection_bwd_kernels.cuh"
}  // namespace percam

namespace ksgrad {
constexpr bool kKsGrad = true;
#include "projection_bwd_kernels.cuh"

namespace percam {
constexpr bool kPerCameraSh = true;
#include "projection_bwd_kernels.cuh"
}  // namespace percam
}  // namespace ksgrad

#include "projection_bwd_launch.cuh"
}  // namespace depth

}  // namespace egs

using namespace egs;

static int projection_fwd_impl(int32_t C, int32_t N, const float* means, const float* quats, const float* scales,
                               const float* opacities, const float* sh_coeffs, const float* sh_rest, int32_t K,
                               int32_t sh_degree, int32_t colors_per_camera, const float* viewmats, const float* Ks,
                               int32_t width, int32_t height, float eps2d, float near_plane, float far_plane,
                               float radius_clip, int32_t tile_size, int32_t tile_width, int32_t tile_height,
                               int32_t* radii, float* means2d, float* depths, float* conics, float* colors,
                               int32_t* tiles_per_gauss, int32_t* tight_rects, float* splats, egs_stream_t stream,
                               float* compensations = nullptr, int camera_model = kPinhole) {
  const int raw = sh_rest != nullptr;
  EGS_REQUIRE(C >= 0 && N >= 0, "projection_fwd: negative sizes C=%d N=%d", C, N);
  EGS_REQUIRE(C <= 65535, "projection_fwd: C=%d exceeds 65535 cameras per call", C);
  EGS_REQUIRE(width >= 1 && height >= 1, "projection_fwd: width/height must be >= 1 (got %d x %d)", width, height);
  EGS_REQUIRE(tile_size >= 1 && (tile_size & (tile_size - 1)) == 0, "projection_fwd: tile_size must be a power of two");
  EGS_REQUIRE(sh_degree <= 4, "projection_fwd: sh_degree %d > 4 is not supported", sh_degree);
  EGS_REQUIRE(tight_rects == nullptr || (tile_width < 65536 && tile_height < 65536),
              "projection_fwd: tile grid %d x %d too large for the packed tight rectangles", tile_width, tile_height);
  EGS_REQUIRE(sh_degree < 0 || K >= (sh_degree + 1) * (sh_degree + 1), "projection_fwd: K=%d too small for sh_degree=%d", K, sh_degree);
  EGS_REQUIRE(colors_per_camera == 0 || colors_per_camera == 1, "projection_fwd: colors_per_camera=%d must be 0 or 1",
              colors_per_camera);
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
  const bool vec4 = sh_degree >= 0 && (K * 3) % 4 == 0 && (reinterpret_cast<uintptr_t>(sh_coeffs) % 16 == 0);
  const bool pc = sh_degree >= 0 && colors_per_camera;  // per-camera SH coefficients [C,N,K,3]
  if (raw) {
    EGS_REQUIRE(K == 16 && sh_degree >= 0, "projection_fwd_raw: needs sh_0 [N,1,3] + sh_rest [N,15,3] and sh_degree >= 0");
  }
  const cudaStream_t st = (cudaStream_t)stream;
  return camera_model == kOrtho     ? ortho::launch_fwd(p, pc, vec4, st)
         : camera_model == kFisheye ? fisheye::launch_fwd(p, pc, vec4, st)
                                    : launch_projection_fwd(p, pc, vec4, st);
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
                               void* workspace = nullptr, int64_t workspace_bytes = 0, float* v_Ks = nullptr,
                               int depth_grad = 0, int camera_model = kPinhole) {
  const int raw = sh_rest != nullptr;
  EGS_REQUIRE(C >= 0 && N >= 0, "projection_bwd: negative sizes C=%d N=%d", C, N);
  EGS_REQUIRE(sh_degree <= 4, "projection_bwd: sh_degree %d > 4 is not supported", sh_degree);
  EGS_REQUIRE(sh_degree < 0 || K >= (sh_degree + 1) * (sh_degree + 1), "projection_bwd: K=%d too small for sh_degree=%d", K, sh_degree);
  EGS_REQUIRE(colors_per_camera == 0 || colors_per_camera == 1, "projection_bwd: colors_per_camera=%d must be 0 or 1",
              colors_per_camera);
  const bool kg = v_Ks != nullptr;              // intrinsics gradients: the egs::ksgrad kernels, 20-float partials
  const bool vg = kg || v_viewmats != nullptr;  // camera-gradient partials and a finalize launch
  if (kg) {
    EGS_REQUIRE(C <= 65535, "projection_bwd: C=%d exceeds 65535 cameras per call", C);
    EGS_REQUIRE(workspace != nullptr && workspace_bytes >= egs_projection_bwd_intrinsics_workspace_bytes(C, N),
                "projection_bwd: intrinsics gradients need %lld workspace bytes (got %lld)",
                (long long)egs_projection_bwd_intrinsics_workspace_bytes(C, N), (long long)workspace_bytes);
    if (N == 0 && C > 0) EGS_CUDA(cudaMemsetAsync(v_Ks, 0, sizeof(float) * 9 * (size_t)C, (cudaStream_t)stream));
    if (N == 0 && C > 0 && v_viewmats != nullptr)
      EGS_CUDA(cudaMemsetAsync(v_viewmats, 0, sizeof(float) * 16 * (size_t)C, (cudaStream_t)stream));
  } else if (vg) {
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
  const int partial_floats = kg ? kCamKsPartialFloats : kCamPartialFloats;
  if (vg) {
    p.cam_partials = static_cast<float*>(workspace);
    p.cam_counters = reinterpret_cast<int*>(p.cam_partials + (size_t)(C * vg_slots + C * vg_slices(vg_slots)) * partial_floats);
  }
  // viewmat_grad_finalize_kernel / intrinsics_grad_finalize_kernel, after either backward kernel
  auto finalize = [&]() -> int {
    if (C == 0) return 0;
    const int S = vg_slices(vg_slots);
    float* slices = p.cam_partials + (size_t)C * vg_slots * partial_floats;
    if (kg) {
      intrinsics_grad_finalize_kernel<<<dim3((unsigned)S, (unsigned)C), kVgFinalizeThreads, 0, (cudaStream_t)stream>>>(
          (int)vg_slots, p.cam_partials, slices, p.cam_counters, viewmats, v_viewmats, v_Ks);
      return check_launch("intrinsics_grad_finalize_kernel");
    }
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
  const bool pc = sh_degree >= 0 && colors_per_camera;  // per-camera SH coefficients [C,N,K,3]
  const cudaStream_t st = (cudaStream_t)stream;
  const int rc = camera_model == kOrtho     ? ortho::launch_bwd(p, kg, vg, pc, vec4, antialiased, st)
                 : camera_model == kFisheye ? fisheye::launch_bwd(p, kg, vg, pc, vec4, antialiased, st)
                 : depth_grad               ? depth::launch_projection_bwd(p, kg, vg, pc, vec4, antialiased, raw, st)
                                            : launch_projection_bwd(p, kg, vg, pc, vec4, antialiased, raw, st);
  return (rc != 0 || !vg) ? rc : finalize();
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

/* ---- gradients w.r.t. the intrinsics ---- */
extern "C" int64_t egs_projection_bwd_intrinsics_workspace_bytes(int32_t C, int32_t N) {
  if (C <= 0 || N < 0) return 0;
  const int64_t slots = vg_partial_slots(N);
  return (int64_t)C * (slots + vg_slices(slots)) * kCamKsPartialFloats * (int64_t)sizeof(float) +
         (int64_t)C * (int64_t)sizeof(int);
}

extern "C" int egs_projection_bwd_intrinsics(
    int32_t C, int32_t N, const float* means, const float* quats, const float* scales, const float* opacities,
    const float* sh_coeffs, int32_t K, int32_t sh_degree, int32_t colors_per_camera, const float* viewmats,
    const float* Ks, int32_t width, int32_t height, float eps2d, const int32_t* radii, const float* colors,
    const float* v_splats, const float* v_means2d_extra, float* v_means, float* v_quats, float* v_scales,
    float* v_opacities, float* v_sh_coeffs, float* absgrad, int32_t antialiased, float* v_viewmats, float* v_Ks,
    void* workspace, int64_t workspace_bytes, egs_stream_t stream) {
  EGS_REQUIRE(v_Ks != nullptr, "projection_bwd_intrinsics: v_Ks output is required");
  return projection_bwd_impl(C, N, means, quats, scales, antialiased ? opacities : nullptr, sh_coeffs, nullptr, K,
                             sh_degree, colors_per_camera, viewmats, Ks, width, height, eps2d, radii, colors, v_splats,
                             v_means2d_extra, v_means, v_quats, v_scales, v_opacities, v_sh_coeffs, nullptr, absgrad,
                             stream, antialiased ? 1 : 0, v_viewmats, workspace, workspace_bytes, v_Ks);
}

extern "C" int egs_projection_bwd_raw_intrinsics(
    int32_t C, int32_t N, const float* means, const float* quats, const float* log_scales, const float* logit_opacities,
    const float* sh_0, const float* sh_rest, int32_t sh_degree, const float* viewmats, const float* Ks, int32_t width,
    int32_t height, float eps2d, const int32_t* radii, const float* colors, const float* v_splats,
    const float* v_means2d_extra, float* v_means, float* v_quats, float* v_log_scales, float* v_logit_opacities,
    float* v_sh_0, float* v_sh_rest, float* absgrad, float* v_viewmats, float* v_Ks, void* workspace,
    int64_t workspace_bytes, egs_stream_t stream) {
  EGS_REQUIRE(v_Ks != nullptr, "projection_bwd_raw_intrinsics: v_Ks output is required");
  EGS_REQUIRE(sh_rest != nullptr && sh_0 != nullptr, "projection_bwd_raw: sh_0 and sh_rest are required");
  EGS_REQUIRE(reinterpret_cast<uintptr_t>(sh_0) % 16 == 0 && reinterpret_cast<uintptr_t>(sh_rest) % 16 == 0 &&
                  reinterpret_cast<uintptr_t>(v_sh_0) % 16 == 0 && reinterpret_cast<uintptr_t>(v_sh_rest) % 16 == 0,
              "projection_bwd_raw: sh_0 / sh_rest and their gradients must be 16-byte aligned");
  return projection_bwd_impl(C, N, means, quats, log_scales, logit_opacities, sh_0, sh_rest, 16, sh_degree, 0, viewmats,
                             Ks, width, height, eps2d, radii, colors, v_splats, v_means2d_extra, v_means, v_quats,
                             v_log_scales, v_logit_opacities, v_sh_0, v_sh_rest, absgrad, stream, 0, v_viewmats,
                             workspace, workspace_bytes, v_Ks);
}

/* ---- with the depth cotangent of the gradient records (render modes with expected depth) ---- */
extern "C" int egs_projection_bwd_depth(
    int32_t C, int32_t N, const float* means, const float* quats, const float* scales, const float* opacities,
    const float* sh_coeffs, int32_t K, int32_t sh_degree, int32_t colors_per_camera, const float* viewmats,
    const float* Ks, int32_t width, int32_t height, float eps2d, const int32_t* radii, const float* colors,
    const float* v_splats, const float* v_means2d_extra, float* v_means, float* v_quats, float* v_scales,
    float* v_opacities, float* v_sh_coeffs, float* absgrad, int32_t antialiased, float* v_viewmats, float* v_Ks,
    void* workspace, int64_t workspace_bytes, egs_stream_t stream) {
  return projection_bwd_impl(C, N, means, quats, scales, antialiased ? opacities : nullptr, sh_coeffs, nullptr, K,
                             sh_degree, colors_per_camera, viewmats, Ks, width, height, eps2d, radii, colors, v_splats,
                             v_means2d_extra, v_means, v_quats, v_scales, v_opacities, v_sh_coeffs, nullptr, absgrad,
                             stream, antialiased ? 1 : 0, v_viewmats, workspace, workspace_bytes, v_Ks, 1);
}

/* ---- orthographic and fisheye camera models ---- */
extern "C" int egs_projection_fwd_camera_model(
    int32_t camera_model, int32_t C, int32_t N, const float* means, const float* quats, const float* scales,
    const float* opacities, const float* sh_coeffs, int32_t K, int32_t sh_degree, int32_t colors_per_camera,
    const float* viewmats, const float* Ks, int32_t width, int32_t height, float eps2d, float near_plane, float far_plane,
    float radius_clip, int32_t tile_size, int32_t tile_width, int32_t tile_height, int32_t* radii, float* means2d,
    float* depths, float* conics, float* colors, int32_t* tiles_per_gauss, int32_t* tight_rects, float* splats,
    float* compensations, egs_stream_t stream) {
  EGS_REQUIRE(camera_model == kOrtho || camera_model == kFisheye,
              "projection_fwd_camera_model: camera_model=%d must be 1 (ortho) or 2 (fisheye)", camera_model);
  return projection_fwd_impl(C, N, means, quats, scales, opacities, sh_coeffs, nullptr, K, sh_degree, colors_per_camera,
                             viewmats, Ks, width, height, eps2d, near_plane, far_plane, radius_clip, tile_size,
                             tile_width, tile_height, radii, means2d, depths, conics, colors, tiles_per_gauss, tight_rects,
                             splats, stream, compensations, camera_model);
}

extern "C" int egs_projection_bwd_camera_model(
    int32_t camera_model, int32_t C, int32_t N, const float* means, const float* quats, const float* scales,
    const float* opacities, const float* sh_coeffs, int32_t K, int32_t sh_degree, int32_t colors_per_camera,
    const float* viewmats, const float* Ks, int32_t width, int32_t height, float eps2d, const int32_t* radii,
    const float* colors, const float* v_splats, const float* v_means2d_extra, float* v_means, float* v_quats,
    float* v_scales, float* v_opacities, float* v_sh_coeffs, float* absgrad, int32_t antialiased, float* v_viewmats,
    float* v_Ks, void* workspace, int64_t workspace_bytes, egs_stream_t stream) {
  EGS_REQUIRE(camera_model == kOrtho || camera_model == kFisheye,
              "projection_bwd_camera_model: camera_model=%d must be 1 (ortho) or 2 (fisheye)", camera_model);
  return projection_bwd_impl(C, N, means, quats, scales, antialiased ? opacities : nullptr, sh_coeffs, nullptr, K,
                             sh_degree, colors_per_camera, viewmats, Ks, width, height, eps2d, radii, colors, v_splats,
                             v_means2d_extra, v_means, v_quats, v_scales, v_opacities, v_sh_coeffs, nullptr, absgrad,
                             stream, antialiased ? 1 : 0, v_viewmats, workspace, workspace_bytes, v_Ks, 1, camera_model);
}
