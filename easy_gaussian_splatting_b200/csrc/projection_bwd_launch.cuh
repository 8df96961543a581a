// Picks and launches the projection backward kernel for a call: SH degree 4, the K = 16 staged rows (and raw mode), or
// the generic kernel; shared or per-camera coefficients; classic or antialiased; with camera-gradient partials (vg) and
// intrinsics (kg) or without.  projection.cu includes this file in egs and in egs::depth, so the unqualified and the
// percam:: / ksgrad:: names below are the kernels of that namespace.  The caller runs the finalize kernel when vg.
// (No include guard on purpose.)
static int launch_projection_bwd(const ProjBwdParams& p, bool kg, bool vg, bool pc, bool vec4, bool antialiased, bool raw,
                                 cudaStream_t stream) {
  if (p.sh_degree == 4) {  // (raw mode has K = 16 and cannot get here)
    constexpr int kSmem = 2 * kPB2Warps * kSh4TileFloats * (int)sizeof(float);
    auto kern = kg ? (pc ? (antialiased ? ksgrad::percam::projection_bwd_sh4_kernel<true, true>
                                        : ksgrad::percam::projection_bwd_sh4_kernel<false, true>)
                         : (antialiased ? ksgrad::projection_bwd_sh4_kernel<true, true>
                                        : ksgrad::projection_bwd_sh4_kernel<false, true>))
              : pc ? (vg ? (antialiased ? percam::projection_bwd_sh4_kernel<true, true> : percam::projection_bwd_sh4_kernel<false, true>)
                         : (antialiased ? percam::projection_bwd_sh4_kernel<true> : percam::projection_bwd_sh4_kernel<false>))
                   : vg ? (antialiased ? projection_bwd_sh4_kernel<true, true> : projection_bwd_sh4_kernel<false, true>)
                        : (antialiased ? projection_bwd_sh4_kernel<true> : projection_bwd_sh4_kernel<false>);
    const cudaError_t attr_rc = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
    if (attr_rc != cudaSuccess) return fail((int)attr_rc, "projection_bwd: shared memory opt-in failed: %s", cudaGetErrorString(attr_rc));
    kern<<<(unsigned)ceil_div(p.N, kPB2Threads), kPB2Threads, kSmem, stream>>>(p);
    return check_launch("projection_bwd_sh4_kernel");
  }
  if (raw || (vec4 && p.K == 16)) {
    // the reference's layout (K = 16): coalesced shared-memory staged rows
    constexpr int kSmem = 2 * kPB2Warps * 32 * kRowStride * (int)sizeof(float);
    auto kern = kg ? (pc ? (antialiased ? ksgrad::percam::projection_bwd_sh16_kernel<true, true>
                                        : ksgrad::percam::projection_bwd_sh16_kernel<false, true>)
                         : (antialiased ? ksgrad::projection_bwd_sh16_kernel<true, true>
                                        : ksgrad::projection_bwd_sh16_kernel<false, true>))
              : pc ? (vg ? (antialiased ? percam::projection_bwd_sh16_kernel<true, true> : percam::projection_bwd_sh16_kernel<false, true>)
                         : (antialiased ? percam::projection_bwd_sh16_kernel<true> : percam::projection_bwd_sh16_kernel<false>))
                   : vg ? (antialiased ? projection_bwd_sh16_kernel<true, true> : projection_bwd_sh16_kernel<false, true>)
                        : (antialiased ? projection_bwd_sh16_kernel<true> : projection_bwd_sh16_kernel<false>);
    const cudaError_t attr_rc =  // per-device attribute: set on every call (cheap), not once per process
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
    if (attr_rc != cudaSuccess) return fail((int)attr_rc, "projection_bwd: shared memory opt-in failed: %s", cudaGetErrorString(attr_rc));
    kern<<<(unsigned)ceil_div(p.N, kPB2Threads), kPB2Threads, kSmem, stream>>>(p);
    return check_launch("projection_bwd_sh16_kernel");
  }
  unsigned grid = (unsigned)ceil_div(p.N, kProjBwdThreads);
  if (kg) {
    auto kern = pc ? (vec4 ? ksgrad::percam::projection_bwd_kernel<true, true> : ksgrad::percam::projection_bwd_kernel<false, true>)
                   : (vec4 ? ksgrad::projection_bwd_kernel<true, true> : ksgrad::projection_bwd_kernel<false, true>);
    kern<<<grid, kProjBwdThreads, 0, stream>>>(p);
    return check_launch("projection_bwd_kernel");
  }
  if (pc) {
    auto kern = vg ? (vec4 ? percam::projection_bwd_kernel<true, true> : percam::projection_bwd_kernel<false, true>)
                   : (vec4 ? percam::projection_bwd_kernel<true> : percam::projection_bwd_kernel<false>);
    kern<<<grid, kProjBwdThreads, 0, stream>>>(p);
    return check_launch("projection_bwd_kernel");
  }
  // (through a pointer: a direct call would also find egs:: kernels of the same name by argument-dependent lookup)
  auto kern = vg ? (vec4 ? projection_bwd_kernel<true, true> : projection_bwd_kernel<false, true>)
                 : (vec4 ? projection_bwd_kernel<true> : projection_bwd_kernel<false>);
  kern<<<grid, kProjBwdThreads, 0, stream>>>(p);
  return check_launch("projection_bwd_kernel");
}
