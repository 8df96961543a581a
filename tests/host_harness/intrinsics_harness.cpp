// TEST INFRASTRUCTURE.  The intrinsics gradient of csrc/egs_math.cuh (project_bwd with v_K, ks_grad_finalize),
// compiled with the HOST compiler (g++ -ffp-contract=off) and looped over the (camera, Gaussian) pairs on the CPU the
// way the egs::ksgrad instantiations of the projection backward kernels do: each pair's camera gradient (view matrix
// and intrinsics) is accumulated into one array, as the kernels do.  The per-camera sum runs in fp64 here: this checks
// the formulas, not the kernels' summation order.  Never loaded by the product package.
#include <cstdint>
#include <cstring>
#include <cmath>
using std::isfinite;
#include "../../easy_gaussian_splatting_b200/csrc/egs_math.cuh"

using namespace egs;

// deg < 0: no SH colours.  v_comps nullable (antialiased mode).  -> v_Ks[C,9]
extern "C" void hh_intrinsics_grad(int C, int N, const float* means, const float* quats, const float* scales,
                                   const float* sh, int K, int deg, const float* viewmats, const float* Ks, int W, int H,
                                   float eps2d, const int32_t* radii, const float* colors, const float* v_means2d,
                                   const float* v_conics, const float* v_colors, const float* v_comps, float* v_Ks) {
  constexpr int kAcc = kCamGradFloats + kKsGradFloats;
  for (int c = 0; c < C; ++c) {
    Camera cam;
    load_camera(viewmats + c * 16, Ks + c * 9, cam);
    double acc[kAcc] = {0};
    for (int n = 0; n < N; ++n) {
      size_t idx = (size_t)c * N + n;
      if (radii[idx] <= 0) continue;
      float vcam[kAcc] = {0};
      float v_mean[3] = {0, 0, 0}, v_quat[4] = {0, 0, 0, 0}, v_scale[3] = {0, 0, 0};
      ProjState st;
      ProjOut o;
      project_fwd(means + 3 * n, quats + 4 * n, scales + 3 * n, cam, (float)W, (float)H, eps2d, 0.f, INFINITY, -1.f, st, o);
      if (o.radius > 0)
        project_bwd(st, scales + 3 * n, cam, v_means2d[idx * 2], v_means2d[idx * 2 + 1], 0.f, v_conics[idx * 3],
                    v_conics[idx * 3 + 1], v_conics[idx * 3 + 2], o, v_mean, v_quat, v_scale,
                    v_comps ? v_comps[idx] : 0.f, eps2d, vcam, means + 3 * n, vcam + kCamGradFloats);
      if (deg >= 0) {
        float co[48], vco[48];
        int nb = (deg + 1) * (deg + 1);
        for (int i = 0; i < 48; ++i) { co[i] = i < nb * 3 ? sh[(size_t)n * K * 3 + i] : 0.f; vco[i] = 0.f; }
        sh_color_bwd(deg, means + 3 * n, cam, co, colors + idx * 3, v_colors + idx * 3, vco, v_mean, vcam);
      }
      for (int k = 0; k < kAcc; ++k) acc[k] += vcam[k];
    }
    float vk[kKsGradFloats];
    for (int k = 0; k < kKsGradFloats; ++k) vk[k] = (float)acc[kCamGradFloats + k];
    ks_grad_finalize(vk, v_Ks + c * 9);
  }
}
