// Picks and launches the projection forward kernel for a call: SH degree 4, the K = 16 staged rows (and raw mode), or
// the generic kernel; shared or per-camera coefficients.  Included by projection.cu in egs and by the camera-model
// translation units in egs::ortho / egs::fisheye, so the unqualified and percam:: names below are the kernels of that
// namespace.  (No include guard on purpose.)
static int launch_projection_fwd(const ProjFwdParams& p, bool pc, bool vec4, cudaStream_t stream) {
  if (p.sh_degree == 4) {
    const unsigned grid2 = (unsigned)(ceil_div(p.N, kPF2Threads) * p.C);
    auto kern = pc ? percam::projection_fwd_sh4_kernel : projection_fwd_sh4_kernel;
    kern<<<grid2, kPF2Threads, 0, stream>>>(p);
    return check_launch("projection_fwd_sh4_kernel");
  }
  if (p.raw || (vec4 && p.K == 16)) {
    const unsigned grid2 = (unsigned)(ceil_div(p.N, kPF2Threads) * p.C);
    auto kern = pc ? percam::projection_fwd_sh16_kernel : projection_fwd_sh16_kernel;
    kern<<<grid2, kPF2Threads, 0, stream>>>(p);
    return check_launch("projection_fwd_sh16_kernel");
  }
  const unsigned grid = (unsigned)(ceil_div(p.N, kProjThreads) * p.C);
  auto kern = pc ? (vec4 ? percam::projection_fwd_kernel<true> : percam::projection_fwd_kernel<false>)
                 : (vec4 ? projection_fwd_kernel<true> : projection_fwd_kernel<false>);
  kern<<<grid, kProjThreads, 0, stream>>>(p);
  return check_launch("projection_fwd_kernel");
}
