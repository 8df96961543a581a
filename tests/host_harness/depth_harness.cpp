// TEST INFRASTRUCTURE.  The depth cotangent of csrc/egs_math.cuh (project_bwd's v_depth, with the view-matrix and
// intrinsics gradients), compiled with the HOST compiler (g++ -ffp-contract=off) and looped over the (camera, Gaussian)
// pairs on the CPU the way the egs::depth::ksgrad instantiations of the projection backward kernels call it.  The sums
// over cameras (v_means) and over Gaussians (camera gradients) run in fp64 here: this checks the formulas, not the
// kernels' summation order.  Never loaded by the product package.
#include <cstdint>
#include <cstring>
#include <cmath>
using std::isfinite;
#include "../../easy_gaussian_splatting_b200/csrc/egs_math.cuh"

using namespace egs;

// v_comps nullable (antialiased mode).  -> v_means[N,3], v_viewmats[C,16], v_Ks[C,9]
extern "C" void hh_depth_grad(int C, int N, const float* means, const float* quats, const float* scales,
                              const float* viewmats, const float* Ks, int W, int H, float eps2d, const int32_t* radii,
                              const float* v_means2d, const float* v_depths, const float* v_conics,
                              const float* v_comps, float* v_means, float* v_viewmats, float* v_Ks) {
  constexpr int kAcc = kCamGradFloats + kKsGradFloats;
  double* vm_acc = new double[(size_t)N * 3]();
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
        project_bwd(st, scales + 3 * n, cam, v_means2d[idx * 2], v_means2d[idx * 2 + 1], v_depths[idx], v_conics[idx * 3],
                    v_conics[idx * 3 + 1], v_conics[idx * 3 + 2], o, v_mean, v_quat, v_scale,
                    v_comps ? v_comps[idx] : 0.f, eps2d, vcam, means + 3 * n, vcam + kCamGradFloats);
      for (int k = 0; k < 3; ++k) vm_acc[(size_t)n * 3 + k] += v_mean[k];
      for (int k = 0; k < kAcc; ++k) acc[k] += vcam[k];
    }
    float sum[kCamGradFloats], vk[kKsGradFloats];
    for (int k = 0; k < kCamGradFloats; ++k) sum[k] = (float)acc[k];
    for (int k = 0; k < kKsGradFloats; ++k) vk[k] = (float)acc[kCamGradFloats + k];
    viewmat_grad_finalize(viewmats + c * 16, sum, v_viewmats + c * 16);
    ks_grad_finalize(vk, v_Ks + c * 9);
  }
  for (size_t i = 0; i < (size_t)N * 3; ++i) v_means[i] = (float)vm_acc[i];
  delete[] vm_acc;
}
