// TEST INFRASTRUCTURE.  The degree-4 SH colour of csrc/egs_math.cuh (sh4_color_fwd, sh4_color_bwd) with the projection
// VJP (project_bwd with the camera and intrinsics accumulators, viewmat_grad_finalize, ks_grad_finalize), compiled with
// the HOST compiler (g++ -ffp-contract=off) and looped over the (camera, Gaussian) pairs on the CPU the way the
// projection_bwd_sh4_kernel instantiations do.  Sums over cameras and Gaussians run in fp64 here: this checks the
// formulas, not the kernels' summation order.  Never loaded by the product package.
#include <cstdint>
#include <cstring>
#include <cmath>
#include <vector>
using std::isfinite;
#include "../../easy_gaussian_splatting_b200/csrc/egs_math.cuh"

using namespace egs;

// sh[N or C*N, K, 3] (per_cam: one row per (camera, Gaussian)).  radii[C,N] from the forward pass.
// -> colors[C,N,3] (0 for culled pairs), v_sh (shape of sh; 0 past band 4 and for culled rows), v_means[N,3],
//    v_viewmats[C,16], v_Ks[C,9].  v_comps nullable (antialiased mode).
extern "C" void hh_sh4(int C, int N, const float* means, const float* quats, const float* scales, const float* sh, int K,
                       int per_cam, const float* viewmats, const float* Ks, int W, int H, float eps2d,
                       const int32_t* radii, const float* v_means2d, const float* v_conics, const float* v_colors,
                       const float* v_comps, float* colors, float* v_sh, float* v_means, float* v_viewmats, float* v_Ks) {
  constexpr int kAcc = kCamGradFloats + kKsGradFloats;
  const size_t rows = (size_t)(per_cam ? C : 1) * N;
  std::vector<double> vsh(rows * K * 3, 0.0), vmean((size_t)N * 3, 0.0);
  for (int c = 0; c < C; ++c) {
    Camera cam;
    load_camera(viewmats + c * 16, Ks + c * 9, cam);
    double acc[kAcc] = {0};
    for (int n = 0; n < N; ++n) {
      const size_t idx = (size_t)c * N + n;
      const size_t row = per_cam ? idx : (size_t)n;
      float* col = colors + idx * 3;
      col[0] = col[1] = col[2] = 0.f;
      if (radii[idx] <= 0) continue;
      const float* co = sh + row * K * 3;
      sh4_color_fwd(means + 3 * n, cam, co, col);
      float vcam[kAcc] = {0};
      float v_mean[3] = {0, 0, 0}, v_quat[4] = {0, 0, 0, 0}, v_scale[3] = {0, 0, 0};
      ProjState st;
      ProjOut o;
      project_fwd(means + 3 * n, quats + 4 * n, scales + 3 * n, cam, (float)W, (float)H, eps2d, 0.f, INFINITY, -1.f, st, o);
      if (o.radius > 0)
        project_bwd(st, scales + 3 * n, cam, v_means2d[idx * 2], v_means2d[idx * 2 + 1], 0.f, v_conics[idx * 3],
                    v_conics[idx * 3 + 1], v_conics[idx * 3 + 2], o, v_mean, v_quat, v_scale,
                    v_comps ? v_comps[idx] : 0.f, eps2d, vcam, means + 3 * n, vcam + kCamGradFloats);
      float vco[kSh4Bands * 3] = {0};
      sh4_color_bwd(means + 3 * n, cam, co, col, v_colors + idx * 3, vco, v_mean, vcam);
      for (int i = 0; i < kSh4Bands * 3; ++i) vsh[row * K * 3 + i] += vco[i];
      for (int k = 0; k < 3; ++k) vmean[(size_t)n * 3 + k] += v_mean[k];
      for (int k = 0; k < kAcc; ++k) acc[k] += vcam[k];
    }
    float vc[kCamGradFloats], vk[kKsGradFloats];
    for (int k = 0; k < kCamGradFloats; ++k) vc[k] = (float)acc[k];
    for (int k = 0; k < kKsGradFloats; ++k) vk[k] = (float)acc[kCamGradFloats + k];
    viewmat_grad_finalize(viewmats + c * 16, vc, v_viewmats + c * 16);
    ks_grad_finalize(vk, v_Ks + c * 9);
  }
  for (size_t i = 0; i < vsh.size(); ++i) v_sh[i] = (float)vsh[i];
  for (size_t i = 0; i < vmean.size(); ++i) v_means[i] = (float)vmean[i];
}
