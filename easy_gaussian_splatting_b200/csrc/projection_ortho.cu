// The projection kernels of the orthographic camera model (camera_model="ortho"): projection_kernels.cuh compiled again
// in egs::ortho with kCameraModel = kOrtho, the backward forms with the depth cotangent (kDepthGrad) for every render mode.
// A translation unit of its own, compiled with -fmad=false like projection.cu (the forward is bit-exact against the CPU
// reference), in parallel with the other units.  The ABI entries are in projection.cu.
#include "projection_common.cuh"

namespace egs {
namespace ortho {
constexpr int kCameraModel = kOrtho;
constexpr bool kPerCameraSh = false;
constexpr bool kKsGrad = false;
constexpr bool kDepthGrad = true;
#include "projection_kernels.cuh"

namespace percam {
constexpr bool kPerCameraSh = true;
#include "projection_kernels.cuh"
}  // namespace percam

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

int launch_fwd(const ProjFwdParams& p, bool pc, bool vec4, cudaStream_t stream) {
  return launch_projection_fwd(p, pc, vec4, stream);
}

int launch_bwd(const ProjBwdParams& p, bool kg, bool vg, bool pc, bool vec4, bool antialiased, cudaStream_t stream) {
  return launch_projection_bwd(p, kg, vg, pc, vec4, antialiased, false, stream);
}
}  // namespace ortho
}  // namespace egs
