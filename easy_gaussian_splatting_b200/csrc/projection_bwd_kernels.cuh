// The projection backward kernels (generic, K = 16, SH degree 4), compiled four times, each with two flags (and the
// four again with the depth flag below)
// (projection_kernels.cuh includes this file in egs and egs::percam, projection.cu includes it in egs::ksgrad and
// egs::ksgrad::percam):
// - kPerCameraSh: SH coefficients [N,K,3] shared by all cameras (or direct colours), or [C,N,K,3], one row per
//   (camera, Gaussian);
// - kKsGrad: the camera-gradient (VG) forms also reduce the intrinsics gradient, 4 more floats per partial.
// egs and egs::percam hold the kernels without intrinsics gradients, egs::ksgrad and egs::ksgrad::percam those with.
// Both flags are behind `if constexpr`, so the kernels of egs keep their names and compile exactly as without them.
// A third flag, kDepthGrad, passes the depth cotangent of gradient-record slot 11 (written by the depth blend) to
// project_bwd; projection.cu includes the file again under egs::depth with it set.  The forms without it read 0, so
// their registers and code are those of the kernels before the flag existed.
// kCameraModel: see projection_kernels.cuh.  The ortho and fisheye forms are compiled with kDepthGrad only: slot 11 is 0
// from every blend backward but the depth one, so one set of forms serves every render mode.
// (No include guard on purpose.)

// Camera-gradient floats per (camera, Gaussian) pair and per warp partial: 15 padded to 16 for the view matrices, with
// the intrinsics 15 + 4 padded to 20.
constexpr int kCamAccFloats = kKsGrad ? kCamGradFloats + kKsGradFloats : kCamGradFloats;
constexpr int kCamPartialStride = kKsGrad ? kCamKsPartialFloats : kCamPartialFloats;
// Near plane of the backward kernels' recomputation of the projection.  Visibility was decided by the forward pass, so
// the recomputation must not cull a pair the forward kept: the ortho and fisheye forms cull nothing on z (near_plane
// <= 0 lets z <= 0 through, fisheye theta up to pi).  The pinhole forms keep the 0 they have always been built with.
constexpr float kBwdNearPlane = kCameraModel == kPinhole ? 0.f : -INFINITY;

// One thread per Gaussian, looping over cameras: gradients summed over cameras stay in registers,
// so there are no atomics for any C.  Every output element is written exactly once (zeros for culled
// Gaussians and inactive SH bands), so the caller does not have to clear the gradient buffers.
// VG: also the view-matrix gradient partials (see store_cam_partial).  Every lane of a warp then runs the camera loop
// (the shuffles need all 32), lanes past N as if they saw nothing.
// Per-camera SH ([C,N,K,3]): camera c's coefficient row is loaded when camera c sees the Gaussian, and its gradient row
// is cleared and stored inside the camera loop; v_means still sums the SH-direction terms in camera order.
// kKsGrad (VG forms only): the partials also carry v_fx, v_fy, v_cx, v_cy.
template <bool VEC4, bool VG = false>
__global__ void __launch_bounds__(kProjBwdThreads) projection_bwd_kernel(const ProjBwdParams p) {
  static_assert(VG || !kKsGrad, "intrinsics gradients are reduced with the view-matrix gradient partials");
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

  const bool has_sh = kPerCameraSh || p.sh_degree >= 0;
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
    if constexpr (kPerCameraSh) {
#pragma unroll
      for (int i = 0; i < 48; ++i) vco[i] = 0.f;
    }
    float vcam[kCamAccFloats];
    if constexpr (VG) {
#pragma unroll
      for (int k = 0; k < kCamAccFloats; ++k) vcam[k] = 0.f;
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
      project_fwd<kCameraModel>(mean, quat, scale, *cam, p.width, p.height, p.eps2d, kBwdNearPlane, INFINITY, -1.f, st, o);
      // (culling thresholds are irrelevant here: visibility was decided by the forward pass; the
      //  off-screen test cannot fire differently because it only depends on the same values.)
      float v_comp = 0.f, w_opac = 1.f;
      if (p.antialiased) { v_comp = g1.y * __ldg(p.opacities + n); w_opac = o.comp; }
      if (o.radius > 0)
        project_bwd<kCameraModel>(st, scale, *cam, v_m2x, v_m2y, kDepthGrad ? g2.w : 0.f, g0.z, g0.w, g1.x, o, v_mean, v_quat, v_scale, v_comp, p.eps2d,
                    VG ? vcam : nullptr, mean, kKsGrad ? vcam + kCamGradFloats : nullptr);
      v_opac += g1.y * w_opac;
      v_rgb[0] = g1.z; v_rgb[1] = g1.w; v_rgb[2] = g2.x;
      if (has_sh) {
        if (kPerCameraSh) load_coeffs<VEC4>(p.sh + idx * p.K * 3, nb * 3, co);
        else if (!co_loaded) { load_coeffs<VEC4>(p.sh + (size_t)n * p.K * 3, nb * 3, co); co_loaded = true; }
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
    if (kPerCameraSh && in_range) store_coeff_grads<VEC4>(p.v_sh + idx * p.K * 3, p.K * 3, vco);
    if constexpr (VG)
      store_cam_partial(vcam, __ballot_sync(0xffffffffu, vis) != 0, cam_partial<kCamPartialStride>(p, c, warp), lane);
  }
  if (!in_range) return;

  p.v_means[3 * (size_t)n + 0] = v_mean[0]; p.v_means[3 * (size_t)n + 1] = v_mean[1]; p.v_means[3 * (size_t)n + 2] = v_mean[2];
  reinterpret_cast<float4*>(p.v_quats)[n] = make_float4(v_quat[0], v_quat[1], v_quat[2], v_quat[3]);
  p.v_scales[3 * (size_t)n + 0] = v_scale[0]; p.v_scales[3 * (size_t)n + 1] = v_scale[1]; p.v_scales[3 * (size_t)n + 2] = v_scale[2];
  p.v_opacities[n] = v_opac;
  if (kPerCameraSh) {
    // (gradient rows stored per camera above)
  } else if (has_sh) {
    store_coeff_grads<VEC4>(p.v_sh + (size_t)n * p.K * 3, p.K * 3, vco);
  } else if (!p.colors_per_camera) {
    p.v_sh[3 * (size_t)n + 0] = v_rgb_sum[0]; p.v_sh[3 * (size_t)n + 1] = v_rgb_sum[1]; p.v_sh[3 * (size_t)n + 2] = v_rgb_sum[2];
  }
}

// AA: rasterize_mode="antialiased" (a separate instantiation keeps the classic kernel at 128 registers).
// VG: also the view-matrix gradient partials (see store_cam_partial).  The camera loop then runs on every lane of a warp
// that has a seen Gaussian (the shuffles need all 32); lanes that see nothing only take part in the sums.
// Per-camera SH ([C,N,16,3]): the camera loop runs on every lane of such a warp as well.  For each camera the warp
// stages that camera's rows of the Gaussians it sees in co_tile, accumulates into vc_tile and stores all 32 gradient
// rows of the camera (zeros for rows it does not see) coalesced before moving on.
// kKsGrad (VG forms only): the partials also carry v_fx, v_fy, v_cx, v_cy.
// kDepthGrad: the per-camera form spills 16 bytes at 168 registers even without VG, so it runs 2 CTAs per SM as well.
// kFisheye: the classic VG form spills 32 bytes at 168 registers (the fisheye Jacobian's VJP), so it runs 2 as well.
template <bool AA, bool VG = false>
__global__ void EGS_PB_BOUNDS(((kPerCameraSh || kKsGrad || (kCameraModel == kFisheye && !AA)) && VG) || (kDepthGrad && kPerCameraSh)) projection_bwd_sh16_kernel(const ProjBwdParams p) {
  static_assert(VG || !kKsGrad, "intrinsics gradients are reduced with the view-matrix gradient partials");
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
        float4* d = reinterpret_cast<float4*>(cam_partial<kCamPartialStride>(p, c, warp));
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        d[0] = z; d[1] = z; d[2] = z; d[3] = z;
        if constexpr (kKsGrad) d[4] = z;
      }
  }

  // phase 1: coalesced load of the coefficient rows that are needed (per camera, below, for per-camera SH); zero the
  // gradient rows
  if (!kPerCameraSh && !p.raw) {
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
    if (!kPerCameraSh && p.sh_degree >= 1) load_rows_raw<kRowStride>(co_tile, p.sh, p.sh_rest, n_base, p.N, seen_mask, lane);
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
  constexpr bool kWarpLoop = VG || kPerCameraSh;  // the camera loop runs on every lane of the warp
  if (kWarpLoop ? seen_mask != 0 : seen) {
    const int nl = kWarpLoop ? (in_range ? n : n_base) : n;  // a lane past the range reads the warp's first Gaussian
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
      if (kWarpLoop && !in_range) nrad = 0;
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
      if constexpr (kPerCameraSh) stage_sh_rows(co_tile, p.sh, p.sh_degree, c, p.N, n_base, __ballot_sync(0xffffffffu, rad > 0), lane);
      float vcam[kCamAccFloats];
      if constexpr (VG) {
#pragma unroll
        for (int k = 0; k < kCamAccFloats; ++k) vcam[k] = 0.f;
      } else if constexpr (!kPerCameraSh) {
        if (!(rad > 0)) continue;
      }
      do {  // (VG, per-camera SH: lanes that do not see camera c skip to the warp's sum / row store below)
      if (kWarpLoop && !(rad > 0)) break;
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
        project_fwd<kCameraModel>(mean, quat, scale, *cam, p.width, p.height, p.eps2d, kBwdNearPlane, INFINITY, -1.f, st, o);
        if constexpr (AA) {
          float op = __ldg(p.opacities + n);
          if (p.raw) op = act_sigmoid(op);
          if (o.radius > 0)
            project_bwd<kCameraModel>(st, scale, *cam, v_m2x, v_m2y, kDepthGrad ? g2.w : 0.f, g0.z, g0.w, g1.x, o, v_mean, v_quat, v_scale, g1.y * op, p.eps2d,
                        VG ? vcam : nullptr, mean, kKsGrad ? vcam + kCamGradFloats : nullptr);
          v_opac += g1.y * o.comp;
        } else {
          if (o.radius > 0)
            project_bwd<kCameraModel>(st, scale, *cam, v_m2x, v_m2y, kDepthGrad ? g2.w : 0.f, g0.z, g0.w, g1.x, o, v_mean, v_quat, v_scale, 0.f, 0.f,
                        VG ? vcam : nullptr, mean, kKsGrad ? vcam + kCamGradFloats : nullptr);
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
      if constexpr (VG)
        store_cam_partial(vcam, __ballot_sync(0xffffffffu, rad > 0) != 0, cam_partial<kCamPartialStride>(p, c, warp), lane);
      if constexpr (kPerCameraSh) store_sh_grad_rows(vc_tile, p.v_sh, c, p.N, n_base, lane);
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
  if constexpr (kPerCameraSh) {
    if (seen_mask == 0)  // no camera sees the warp's Gaussians: zero rows for every camera (stored per camera otherwise)
      for (int c = 0; c < p.C; ++c) store_sh_grad_rows(vc_tile, p.v_sh, c, p.N, n_base, lane);
  }
  if (!kPerCameraSh && !p.raw) {
    float4* dst = reinterpret_cast<float4*>(p.v_sh) + (size_t)n_base * (kRowFloats / 4);
#pragma unroll
    for (int i = 0; i < kRowFloats / 4; ++i) {
      const int f = i * 32 + lane;
      const int row = f / 12, c4 = f - row * 12;
      if (n_base + row < p.N) dst[f] = *reinterpret_cast<const float4*>(vc_tile + row * kRowStride + c4 * 4);
    }
  } else if (!kPerCameraSh) {
    store_rows_raw<kRowStride>(vc_tile, p.v_sh, p.v_sh_rest, n_base, p.N, lane);
  }
  if (in_range) {
    p.v_means[3 * (size_t)n + 0] = v_mean[0]; p.v_means[3 * (size_t)n + 1] = v_mean[1]; p.v_means[3 * (size_t)n + 2] = v_mean[2];
    reinterpret_cast<float4*>(p.v_quats)[n] = make_float4(v_quat[0], v_quat[1], v_quat[2], v_quat[3]);
    p.v_scales[3 * (size_t)n + 0] = v_scale[0]; p.v_scales[3 * (size_t)n + 1] = v_scale[1]; p.v_scales[3 * (size_t)n + 2] = v_scale[2];
    p.v_opacities[n] = v_opac;
  }
}

// Backward, SH degree 4 (K >= 25), the structure of projection_bwd_sh16_kernel: the coefficient rows and the gradient
// rows of a warp's 32 Gaussians go through two shared-memory tiles (stage_sh4_rows / store_sh4_rows), every gradient
// element is written once (zeros for Gaussians or pairs no camera sees and for the bands past 4).  2 x 38.4 KB of tiles
// per block: 2 CTAs per SM.
template <bool AA, bool VG = false>
__global__ void __launch_bounds__(kPB2Threads, kSh4BwdMinCtas) projection_bwd_sh4_kernel(const ProjBwdParams p) {
  static_assert(VG || !kKsGrad, "intrinsics gradients are reduced with the view-matrix gradient partials");
  extern __shared__ __align__(16) float smem_pb[];
  __shared__ Camera cams[kMaxCamerasSmem];
  for (int c = threadIdx.x; c < p.C && c < kMaxCamerasSmem; c += kPB2Threads)
    load_camera(p.viewmats + (size_t)c * 16, p.Ks + (size_t)c * 9, cams[c]);
  if constexpr (VG) clear_cam_counters(p);
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* co_tile = smem_pb + (size_t)warp * kSh4TileFloats;                // coefficients
  float* vc_tile = smem_pb + (size_t)(kPB2Warps + warp) * kSh4TileFloats;  // gradient accumulation
  const int n_base = blockIdx.x * kPB2Threads + warp * 32;
  const int n = n_base + lane;
  const bool in_range = n < p.N;
  const int rows = min(32, p.N - n_base);
  const int K3 = p.K * 3;

  bool seen = false;
  if (in_range)
    for (int c = 0; c < p.C; ++c) seen = seen || (p.radii[(size_t)c * p.N + n] > 0);
  const uint32_t seen_mask = __ballot_sync(0xffffffffu, seen);
  if constexpr (VG) {
    if (seen_mask == 0)  // the warp sees nothing: zero partials for every camera
      for (int c = lane; c < p.C; c += 32) {
        float4* d = reinterpret_cast<float4*>(cam_partial<kCamPartialStride>(p, c, warp));
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        d[0] = z; d[1] = z; d[2] = z; d[3] = z;
        if constexpr (kKsGrad) d[4] = z;
      }
  }

  // phase 1: the shared coefficient rows that are needed (per camera, below, for per-camera SH); zero gradient rows
  if (!kPerCameraSh && seen_mask != 0) stage_sh4_rows(co_tile, p.sh, (size_t)n_base, rows, K3, seen_mask, lane);
  for (int f = lane; f < kSh4TileVec4; f += 32) reinterpret_cast<float4*>(vc_tile)[f] = make_float4(0.f, 0.f, 0.f, 0.f);
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
  constexpr bool kWarpLoop = VG || kPerCameraSh;  // the camera loop runs on every lane of the warp
  if (kWarpLoop ? seen_mask != 0 : seen) {
    const int nl = kWarpLoop ? (in_range ? n : n_base) : n;  // a lane past the range reads the warp's first Gaussian
    float mean[3], quat[4], scale[3];
    mean[0] = __ldg(p.means + 3 * (size_t)nl + 0);
    mean[1] = __ldg(p.means + 3 * (size_t)nl + 1);
    mean[2] = __ldg(p.means + 3 * (size_t)nl + 2);
    const float4 q4 = __ldg(reinterpret_cast<const float4*>(p.quats) + nl);
    quat[0] = q4.x; quat[1] = q4.y; quat[2] = q4.z; quat[3] = q4.w;
    scale[0] = __ldg(p.scales + 3 * (size_t)nl + 0);
    scale[1] = __ldg(p.scales + 3 * (size_t)nl + 1);
    scale[2] = __ldg(p.scales + 3 * (size_t)nl + 2);
    const float* co = co_tile + lane * kSh4RowFloats;
    float* vc = vc_tile + lane * kSh4RowFloats;
    // the records of camera c + 1 are requested before camera c is worked on, as in projection_bwd_sh16_kernel
    float4 ng0, ng1, ng2;
    float ncol[3];
    int nrad;
    auto fetch = [&](int c) {
      const size_t idx = (size_t)c * p.N + nl;
      nrad = p.radii[idx];
      if (kWarpLoop && !in_range) nrad = 0;
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
      if constexpr (kPerCameraSh) {
        const uint32_t cam_mask = __ballot_sync(0xffffffffu, rad > 0);
        if (cam_mask != 0) stage_sh4_rows(co_tile, p.sh, (size_t)c * p.N + n_base, rows, K3, cam_mask, lane);
      }
      float vcam[kCamAccFloats];
      if constexpr (VG) {
#pragma unroll
        for (int k = 0; k < kCamAccFloats; ++k) vcam[k] = 0.f;
      } else if constexpr (!kPerCameraSh) {
        if (!(rad > 0)) continue;
      }
      do {  // (VG, per-camera SH: lanes that do not see camera c skip to the warp's sum / row store below)
      if (kWarpLoop && !(rad > 0)) break;
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
        project_fwd<kCameraModel>(mean, quat, scale, *cam, p.width, p.height, p.eps2d, kBwdNearPlane, INFINITY, -1.f, st, o);
        if constexpr (AA) {
          if (o.radius > 0)
            project_bwd<kCameraModel>(st, scale, *cam, v_m2x, v_m2y, kDepthGrad ? g2.w : 0.f, g0.z, g0.w, g1.x, o, v_mean, v_quat, v_scale,
                        g1.y * __ldg(p.opacities + n), p.eps2d, VG ? vcam : nullptr, mean,
                        kKsGrad ? vcam + kCamGradFloats : nullptr);
          v_opac += g1.y * o.comp;
        } else {
          if (o.radius > 0)
            project_bwd<kCameraModel>(st, scale, *cam, v_m2x, v_m2y, kDepthGrad ? g2.w : 0.f, g0.z, g0.w, g1.x, o, v_mean, v_quat, v_scale, 0.f, 0.f,
                        VG ? vcam : nullptr, mean, kKsGrad ? vcam + kCamGradFloats : nullptr);
          v_opac += g1.y;
        }
      }
      const float v_rgb[3] = {g1.z, g1.w, g2.x};
      sh4_color_bwd(mean, *cam, co, col, v_rgb, vc, v_mean, VG ? vcam : nullptr);
      } while (0);
      if constexpr (VG)
        store_cam_partial(vcam, __ballot_sync(0xffffffffu, rad > 0) != 0, cam_partial<kCamPartialStride>(p, c, warp), lane);
      if constexpr (kPerCameraSh) store_sh4_rows(vc_tile, p.v_sh, (size_t)c * p.N + n_base, rows, K3, lane);
    }
  }
  __syncwarp();

  // phase 3: the gradient rows; small per-Gaussian outputs directly
  if constexpr (kPerCameraSh) {
    if (seen_mask == 0)  // no camera sees the warp's Gaussians: zero rows for every camera (stored per camera otherwise)
      for (int c = 0; c < p.C; ++c) store_sh4_rows(vc_tile, p.v_sh, (size_t)c * p.N + n_base, rows, K3, lane);
  } else {
    store_sh4_rows(vc_tile, p.v_sh, (size_t)n_base, rows, K3, lane);
  }
  if (in_range) {
    p.v_means[3 * (size_t)n + 0] = v_mean[0]; p.v_means[3 * (size_t)n + 1] = v_mean[1]; p.v_means[3 * (size_t)n + 2] = v_mean[2];
    reinterpret_cast<float4*>(p.v_quats)[n] = make_float4(v_quat[0], v_quat[1], v_quat[2], v_quat[3]);
    p.v_scales[3 * (size_t)n + 0] = v_scale[0]; p.v_scales[3 * (size_t)n + 1] = v_scale[1]; p.v_scales[3 * (size_t)n + 2] = v_scale[2];
    p.v_opacities[n] = v_opac;
  }
}
