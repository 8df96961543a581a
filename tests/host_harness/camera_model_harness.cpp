// TEST INFRASTRUCTURE.  project_fwd / project_bwd of csrc/egs_math.cuh for the orthographic and fisheye camera models,
// compiled with the HOST compiler (g++ -ffp-contract=off) and looped over the (camera, Gaussian) pairs on the CPU the
// way the egs::ortho / egs::fisheye projection kernels call them.  The forward is per pair (bit-exactness is checked
// against tests/camera_model_reference.py); the backward sums over cameras (v_means, quats, scales) and over Gaussians
// (camera gradients) in fp64: this checks the formulas, not the kernels' summation order.  Never loaded by the product.
#include <cstdint>
#include <cstring>
#include <cmath>
using std::isfinite;
#include "../../easy_gaussian_splatting_b200/csrc/egs_math.cuh"

using namespace egs;

template <int CM>
static void fwd(int C, int N, const float* means, const float* quats, const float* scales, const float* viewmats,
                const float* Ks, int W, int H, float eps2d, float near_plane, float far_plane, float radius_clip,
                int32_t* radii, float* means2d, float* depths, float* conics, float* comps) {
  for (int c = 0; c < C; ++c) {
    Camera cam;
    load_camera(viewmats + c * 16, Ks + c * 9, cam);
    for (int n = 0; n < N; ++n) {
      const size_t idx = (size_t)c * N + n;
      ProjState st;
      ProjOut o;
      project_fwd<CM>(means + 3 * n, quats + 4 * n, scales + 3 * n, cam, (float)W, (float)H, eps2d, near_plane, far_plane,
                      radius_clip, st, o);
      radii[idx] = o.radius;
      means2d[idx * 2] = o.m2x; means2d[idx * 2 + 1] = o.m2y;
      depths[idx] = o.depth;
      conics[idx * 3] = o.ca; conics[idx * 3 + 1] = o.cb; conics[idx * 3 + 2] = o.cc;
      comps[idx] = o.comp;
    }
  }
}

template <int CM>
static void bwd(int C, int N, const float* means, const float* quats, const float* scales, const float* viewmats,
                const float* Ks, int W, int H, float eps2d, const int32_t* radii, const float* v_means2d,
                const float* v_depths, const float* v_conics, const float* v_comps, float* v_means, float* v_quats,
                float* v_scales, float* v_viewmats, float* v_Ks) {
  constexpr int kAcc = kCamGradFloats + kKsGradFloats;
  double* acc_n = new double[(size_t)N * 10]();
  for (int c = 0; c < C; ++c) {
    Camera cam;
    load_camera(viewmats + c * 16, Ks + c * 9, cam);
    double acc[kAcc] = {0};
    for (int n = 0; n < N; ++n) {
      const size_t idx = (size_t)c * N + n;
      if (radii[idx] <= 0) continue;
      float vcam[kAcc] = {0};
      float v_mean[3] = {0, 0, 0}, v_quat[4] = {0, 0, 0, 0}, v_scale[3] = {0, 0, 0};
      ProjState st;
      ProjOut o;
      // the kernels' kBwdNearPlane: visibility is the forward's, the recomputation culls nothing on z
      project_fwd<CM>(means + 3 * n, quats + 4 * n, scales + 3 * n, cam, (float)W, (float)H, eps2d,
                      CM == kPinhole ? 0.f : -INFINITY, INFINITY, -1.f, st, o);
      if (o.radius > 0)
        project_bwd<CM>(st, scales + 3 * n, cam, v_means2d[idx * 2], v_means2d[idx * 2 + 1], v_depths[idx],
                        v_conics[idx * 3], v_conics[idx * 3 + 1], v_conics[idx * 3 + 2], o, v_mean, v_quat, v_scale,
                        v_comps ? v_comps[idx] : 0.f, eps2d, vcam, means + 3 * n, vcam + kCamGradFloats);
      for (int k = 0; k < 3; ++k) acc_n[(size_t)n * 10 + k] += v_mean[k];
      for (int k = 0; k < 4; ++k) acc_n[(size_t)n * 10 + 3 + k] += v_quat[k];
      for (int k = 0; k < 3; ++k) acc_n[(size_t)n * 10 + 7 + k] += v_scale[k];
      for (int k = 0; k < kAcc; ++k) acc[k] += vcam[k];
    }
    float sum[kCamGradFloats], vk[kKsGradFloats];
    for (int k = 0; k < kCamGradFloats; ++k) sum[k] = (float)acc[k];
    for (int k = 0; k < kKsGradFloats; ++k) vk[k] = (float)acc[kCamGradFloats + k];
    viewmat_grad_finalize(viewmats + c * 16, sum, v_viewmats + c * 16);
    ks_grad_finalize(vk, v_Ks + c * 9);
  }
  for (int n = 0; n < N; ++n) {
    for (int k = 0; k < 3; ++k) v_means[n * 3 + k] = (float)acc_n[(size_t)n * 10 + k];
    for (int k = 0; k < 4; ++k) v_quats[n * 4 + k] = (float)acc_n[(size_t)n * 10 + 3 + k];
    for (int k = 0; k < 3; ++k) v_scales[n * 3 + k] = (float)acc_n[(size_t)n * 10 + 7 + k];
  }
  delete[] acc_n;
}

// model: 0 pinhole, 1 ortho, 2 fisheye
extern "C" void hh_cm_fwd(int model, int C, int N, const float* means, const float* quats, const float* scales,
                          const float* viewmats, const float* Ks, int W, int H, float eps2d, float near_plane,
                          float far_plane, float radius_clip, int32_t* radii, float* means2d, float* depths,
                          float* conics, float* comps) {
  auto f = model == kOrtho ? fwd<kOrtho> : model == kFisheye ? fwd<kFisheye> : fwd<kPinhole>;
  f(C, N, means, quats, scales, viewmats, Ks, W, H, eps2d, near_plane, far_plane, radius_clip, radii, means2d, depths,
    conics, comps);
}

// v_comps nullable (antialiased mode).  -> v_means[N,3], v_quats[N,4], v_scales[N,3], v_viewmats[C,16], v_Ks[C,9]
extern "C" void hh_cm_bwd(int model, int C, int N, const float* means, const float* quats, const float* scales,
                          const float* viewmats, const float* Ks, int W, int H, float eps2d, const int32_t* radii,
                          const float* v_means2d, const float* v_depths, const float* v_conics, const float* v_comps,
                          float* v_means, float* v_quats, float* v_scales, float* v_viewmats, float* v_Ks) {
  auto f = model == kOrtho ? bwd<kOrtho> : model == kFisheye ? bwd<kFisheye> : bwd<kPinhole>;
  f(C, N, means, quats, scales, viewmats, Ks, W, H, eps2d, radii, v_means2d, v_depths, v_conics, v_comps, v_means,
    v_quats, v_scales, v_viewmats, v_Ks);
}

// theta / r (and g) of fisheye_theta_over_r for n pairs (r, z), r2 = r * r, q = 1 / (r2 + z * z)
extern "C" void hh_theta_over_r(int n, const float* r, const float* z, float* s, float* g) {
  for (int i = 0; i < n; ++i) {
    const float r2 = r[i] * r[i];
    fisheye_theta_over_r(r[i], r2, z[i], 1.0f / (r2 + z[i] * z[i]), s[i], g[i]);
  }
}
