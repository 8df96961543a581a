/*
 * egs_raster.h — C ABI of the B200-native differentiable Gaussian rasterizer.
 *
 * This is the drop-in boundary for the ONE hot path of li199603/easy_gaussian_splatting:
 * the call `gsplat.rendering.rasterization(...)` at /root/reference/model/gaussian.py:353-367
 * (import at model/gaussian.py:8).  The reference has no FFI of its own — it is pure Python and
 * reaches CUDA through the third-party `gsplat` package — so every entry point below cites the
 * gsplat-1.0.0 operator whose role it takes behind that call (SURVEY.md §2.1 / §8a rows g1–g9)
 * and, where one exists, the reference line that consumes the result.
 *
 * Conventions
 *   - plain C, no torch / C++ types; all pointers are DEVICE pointers unless named `host_*`;
 *   - all arrays are dense, row-major, fp32 / int32 / int64 as named;
 *   - the library never allocates, frees or caches device memory and keeps no device state;
 *     work buffers are passed in (`*_workspace_bytes` tells how large);
 *   - every call is asynchronous on `stream` (a cudaStream_t) and re-entrant;
 *   - return value: 0 on success, otherwise a negative egs_status or a positive cudaError_t;
 *     `egs_last_error_string()` (thread local) explains the last failure.  Nothing throws.
 */
#ifndef EGS_RASTER_H_
#define EGS_RASTER_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EGS_ABI_VERSION 1

typedef void* egs_stream_t; /* cudaStream_t */

enum egs_status {
  EGS_OK = 0,
  EGS_ERR_INVALID_ARGUMENT = -1,
  EGS_ERR_WORKSPACE_TOO_SMALL = -2,
  EGS_ERR_UNSUPPORTED = -3,
};

/* Number of floats in one packed splat record / one packed gradient record (48 bytes, 16B aligned).
 * splat record : {x, y, conic_a, conic_b | conic_c, opacity, r, g | b, depth, 0, sigma_cut}
 *                sigma_cut = ln(255 * opacity) (+ margin): the largest sigma at which alpha can reach 1/255.  The
 *                blending kernels drop a Gaussian for a warp when min sigma over the warp's pixels exceeds it
 *                (+inf disables that culling; <= 0 = never visible)
 * grad  record : {v_x, v_y, v_conic_a, v_conic_b | v_conic_c, v_opacity, v_r, v_g | v_b, |v_x|, |v_y|, v_depth}
 *                v_depth: gradient w.r.t. the camera-space depth of slot 9, written by egs_rasterize_bwd_depth (0 from
 *                every other blend backward); egs_projection_bwd_depth routes it into v_means and v_viewmats */
#define EGS_SPLAT_FLOATS 12

int egs_abi_version(void);
const char* egs_last_error_string(void);
/* Kernels this library has enqueued since it was loaded (process-wide, monotonically increasing, counted at the
 * launch sites): the difference over a region is the number of the library's own kernel launches in it.  Used by
 * bench.py for `gpu_launches`; not part of the reference's interface (the reference has no such counter). */
int64_t egs_kernel_launch_count(void);

/* ---- g1 + g2 (+ the count half of g3): fused projection, SH colour, tile count ---------------
 * Replaces gsplat `fully_fused_projection` fwd, `spherical_harmonics` fwd, the Python glue
 * `dirs = means - inverse(viewmats)[:3,3]`, `clamp_min(rgb + 0.5, 0)` and the first launch of
 * `isect_tiles`, all reached from model/gaussian.py:353-367.
 *   means[N,3] quats[N,4](wxyz, unnormalised) scales[N,3] opacities[N]
 *   sh_coeffs: sh_degree >= 0 → SH coefficients (K >= (sh_degree+1)^2, sh_degree <= 4; the _raw entries take
 *              K = 16, so degree <= 3), [N,K,3] shared by all
 *              cameras (colors_per_camera = 0) or [C,N,K,3], one row per (camera, Gaussian) (colors_per_camera = 1);
 *              sh_degree <  0 → colours used as they are, [N,3] (colors_per_camera = 0)
 *              or [C,N,3] (colors_per_camera = 1)
 *   colors_per_camera must be 0 or 1 (rejected before any launch otherwise), here and in every entry below that
 *   takes it; the _raw entries have shared coefficients by construction
 *   viewmats[C,4,4] Ks[C,3,3]
 * outputs (culled entries are zero-filled, radii == 0):
 *   radii[C,N] i32, means2d[C,N,2], depths[C,N], conics[C,N,3], colors[C,N,3],
 *   tiles_per_gauss[C,N] i32 (gsplat's count: tiles of the 3-sigma square), splats[C,N,12] packed records (only
 *   visible entries are written),
 *   tight_rects[C,N,2] i32 (nullable; all egs_projection_fwd* entries): the TIGHT tile rectangle — the square
 *   intersected with the axis-aligned extent of {alpha >= 1/255} — that the blend kernels' own lists are built from
 *   (egs_isect_sorted), packed {x0 | y0 << 16, w | h << 16} in tiles; {0, 0} for culled entries and for Gaussians
 *   that reach no pixel.  Needs tile grids below 65536 tiles per side. */
int egs_projection_fwd(int32_t C, int32_t N, const float* means, const float* quats, const float* scales,
                       const float* opacities, const float* sh_coeffs, int32_t K, int32_t sh_degree,
                       int32_t colors_per_camera, const float* viewmats, const float* Ks, int32_t width,
                       int32_t height, float eps2d, float near_plane, float far_plane, float radius_clip,
                       int32_t tile_size, int32_t tile_width, int32_t tile_height, int32_t* radii,
                       float* means2d, float* depths, float* conics, float* colors, int32_t* tiles_per_gauss,
                       int32_t* tight_rects, float* splats, egs_stream_t stream);

/* ---- g8 + g9: fused SH backward + projection backward ------------------------------------------
 * Replaces gsplat `spherical_harmonics` bwd and `fully_fused_projection` bwd (summed over cameras).
 *   v_splats[C,N,12]: packed gradient records produced by egs_rasterize_bwd
 *   v_means2d_extra[C,N,2] (nullable): user gradient that arrived on meta["means2d"] itself
 * outputs (dense, written for every Gaussian): v_means[N,3], v_quats[N,4], v_scales[N,3],
 *   v_opacities[N], v_sh_coeffs (same shape as sh_coeffs; inactive bands and culled entries are 0; per-camera
 *   coefficients get one gradient row per (camera, Gaussian), not summed over cameras);
 *   absgrad[C,N,2] (nullable): the |v_x|,|v_y| slots of the gradient records as a dense tensor — what the
 *   reference reads as meta["means2d"].absgrad (model/gaussian.py:191). */
int egs_projection_bwd(int32_t C, int32_t N, const float* means, const float* quats, const float* scales,
                       const float* sh_coeffs, int32_t K, int32_t sh_degree, int32_t colors_per_camera,
                       const float* viewmats, const float* Ks, int32_t width, int32_t height, float eps2d,
                       const int32_t* radii, const float* colors, const float* v_splats,
                       const float* v_means2d_extra, float* v_means, float* v_quats, float* v_scales,
                       float* v_opacities, float* v_sh_coeffs, float* absgrad, egs_stream_t stream);

/* ---- §8f-4: rasterize_mode="antialiased" of the same two kernels ---------------------------------------------
 * gsplat 1.0.0 `fully_fused_projection(calc_compensations=True)` + the Python glue `opacities * compensations`
 * (the reference passes the default rasterize_mode="classic", model/gaussian.py:353-367; this is the other value the
 * call accepts).  compensation = sqrt(max(0, det(cov2d) / det(cov2d + eps2d I))) is written to compensations[C,N]
 * (0 for culled entries) and the splat records carry opacity * compensation.  The backward takes the activated
 * opacities[N] as well: v_opacities = sum_c v_record_opacity * compensation, and the compensation's gradient
 * v_record_opacity * opacity flows into the 2D covariance (gsplat's add_blur_vjp, 1e-6 guard included). */
int egs_projection_fwd_antialiased(int32_t C, int32_t N, const float* means, const float* quats, const float* scales,
                                   const float* opacities, const float* sh_coeffs, int32_t K, int32_t sh_degree,
                                   int32_t colors_per_camera, const float* viewmats, const float* Ks, int32_t width,
                                   int32_t height, float eps2d, float near_plane, float far_plane, float radius_clip,
                                   int32_t tile_size, int32_t tile_width, int32_t tile_height, int32_t* radii,
                                   float* means2d, float* depths, float* conics, float* colors,
                                   int32_t* tiles_per_gauss, int32_t* tight_rects, float* splats, float* compensations,
                                   egs_stream_t stream);
int egs_projection_bwd_antialiased(int32_t C, int32_t N, const float* means, const float* quats, const float* scales,
                                   const float* opacities, const float* sh_coeffs, int32_t K, int32_t sh_degree,
                                   int32_t colors_per_camera, const float* viewmats, const float* Ks, int32_t width,
                                   int32_t height, float eps2d, const int32_t* radii, const float* colors,
                                   const float* v_splats, const float* v_means2d_extra, float* v_means,
                                   float* v_quats, float* v_scales, float* v_opacities, float* v_sh_coeffs,
                                   float* absgrad, egs_stream_t stream);

/* ---- §8f-2: the same two kernels fed with the reference's RAW parameters ---------------------------------------
 * GaussianModel recomputes scales = exp(log_scales), opacities = sigmoid(logit_opacities) and
 * shs = cat(sh_0, sh_rest) on every access (/root/reference/model/gaussian.py:97-107); the cat alone moves
 * 384 B/Gaussian forward and again backward.  These entry points take log_scales[N,3], logit_opacities[N],
 * sh_0[N,1,3], sh_rest[N,15,3] and fold exp / sigmoid / cat and their VJPs into the kernels (torch's exact CUDA
 * formulas: expf(x), 1/(1+expf(-x))).  Outputs as above; gradients are w.r.t. the raw parameters. */
int egs_projection_fwd_raw(int32_t C, int32_t N, const float* means, const float* quats, const float* log_scales,
                           const float* logit_opacities, const float* sh_0, const float* sh_rest, int32_t sh_degree,
                           const float* viewmats, const float* Ks, int32_t width, int32_t height, float eps2d,
                           float near_plane, float far_plane, float radius_clip, int32_t tile_size,
                           int32_t tile_width, int32_t tile_height, int32_t* radii, float* means2d, float* depths,
                           float* conics, float* colors, int32_t* tiles_per_gauss, int32_t* tight_rects, float* splats,
                           egs_stream_t stream);
int egs_projection_bwd_raw(int32_t C, int32_t N, const float* means, const float* quats, const float* log_scales,
                           const float* logit_opacities, const float* sh_0, const float* sh_rest, int32_t sh_degree,
                           const float* viewmats, const float* Ks, int32_t width, int32_t height, float eps2d,
                           const int32_t* radii, const float* colors, const float* v_splats,
                           const float* v_means2d_extra, float* v_means, float* v_quats, float* v_log_scales,
                           float* v_logit_opacities, float* v_sh_0, float* v_sh_rest, float* absgrad,
                           egs_stream_t stream);

/* ---- gradients w.r.t. the view matrices (camera pose refinement) ------------------------------------------------
 * The backward entries above, plus v_viewmats[C,4,4]: the gradient of gsplat 1.0.0's `rasterization()` w.r.t.
 * viewmats, summed over the visible Gaussians of each camera.  Two paths: the projection (mean_c = R m + t,
 * cov_c = R Sigma R^T; top 3x4 block) and, with SH colours, the view directions m - campos with
 * campos = inverse(viewmat)[:3,3] (all four rows).  Deterministic: per camera, one partial per warp and a fixed-order
 * sum in a second, small kernel (no float atomics), so the same inputs give bit-identical v_viewmats.  Every other
 * output is bit-identical to the entry without viewmat gradients.
 *   workspace: egs_projection_bwd_viewmats_workspace_bytes(C, N) bytes of device memory, 16-byte aligned; no need to
 *   clear it.  One call at a time per workspace.
 * egs_projection_bwd_viewmats: egs_projection_bwd (antialiased = 0) or egs_projection_bwd_antialiased (antialiased =
 *   1: opacities[N] required; otherwise it may be NULL). */
int64_t egs_projection_bwd_viewmats_workspace_bytes(int32_t C, int32_t N);
int egs_projection_bwd_viewmats(int32_t C, int32_t N, const float* means, const float* quats, const float* scales,
                                const float* opacities, const float* sh_coeffs, int32_t K, int32_t sh_degree,
                                int32_t colors_per_camera, const float* viewmats, const float* Ks, int32_t width,
                                int32_t height, float eps2d, const int32_t* radii, const float* colors,
                                const float* v_splats, const float* v_means2d_extra, float* v_means, float* v_quats,
                                float* v_scales, float* v_opacities, float* v_sh_coeffs, float* absgrad,
                                int32_t antialiased, float* v_viewmats, void* workspace, int64_t workspace_bytes,
                                egs_stream_t stream);
int egs_projection_bwd_raw_viewmats(int32_t C, int32_t N, const float* means, const float* quats,
                                    const float* log_scales, const float* logit_opacities, const float* sh_0,
                                    const float* sh_rest, int32_t sh_degree, const float* viewmats, const float* Ks,
                                    int32_t width, int32_t height, float eps2d, const int32_t* radii,
                                    const float* colors, const float* v_splats, const float* v_means2d_extra,
                                    float* v_means, float* v_quats, float* v_log_scales, float* v_logit_opacities,
                                    float* v_sh_0, float* v_sh_rest, float* absgrad, float* v_viewmats,
                                    void* workspace, int64_t workspace_bytes, egs_stream_t stream);

/* ---- gradients w.r.t. the intrinsics (camera intrinsics refinement) ---------------------------------------------
 * The viewmat entries above with a required v_Ks[C,3,3] and a nullable v_viewmats[C,4,4].  gsplat 1.0.0 returns no
 * Ks gradient; this is the exact derivative of its projection, summed over the visible Gaussians of each camera:
 *   v_Ks[c] = [[v_fx, 0, v_cx], [0, v_fy, v_cy], [0, 0, 0]]
 * v_cx / v_cy sum the means2d cotangents (v_means2d_extra included); v_fx / v_fy also take the conic's and, in
 * antialiased mode, the compensation's cotangents through the Jacobian (J02 = -fx tx / z^2 does not depend on fx where
 * the fov clamp is active).  The skew and the last row are not read by the projection: 0.  Deterministic in the same
 * way as v_viewmats (one backward launch and one finalize launch, also when v_viewmats is requested), and every other
 * output is bit-identical to the entry without camera gradients.  C = 0 or N = 0: v_Ks (and v_viewmats) are zeros.
 *   workspace: egs_projection_bwd_intrinsics_workspace_bytes(C, N) bytes (wider partials than the viewmat entries'),
 *   16-byte aligned; no need to clear it.  One call at a time per workspace.
 * Rejected before any launch: v_Ks NULL, too small a workspace, C > 65535. */
int64_t egs_projection_bwd_intrinsics_workspace_bytes(int32_t C, int32_t N);
int egs_projection_bwd_intrinsics(int32_t C, int32_t N, const float* means, const float* quats, const float* scales,
                                  const float* opacities, const float* sh_coeffs, int32_t K, int32_t sh_degree,
                                  int32_t colors_per_camera, const float* viewmats, const float* Ks, int32_t width,
                                  int32_t height, float eps2d, const int32_t* radii, const float* colors,
                                  const float* v_splats, const float* v_means2d_extra, float* v_means, float* v_quats,
                                  float* v_scales, float* v_opacities, float* v_sh_coeffs, float* absgrad,
                                  int32_t antialiased, float* v_viewmats, float* v_Ks, void* workspace,
                                  int64_t workspace_bytes, egs_stream_t stream);
int egs_projection_bwd_raw_intrinsics(int32_t C, int32_t N, const float* means, const float* quats,
                                      const float* log_scales, const float* logit_opacities, const float* sh_0,
                                      const float* sh_rest, int32_t sh_degree, const float* viewmats, const float* Ks,
                                      int32_t width, int32_t height, float eps2d, const int32_t* radii,
                                      const float* colors, const float* v_splats, const float* v_means2d_extra,
                                      float* v_means, float* v_quats, float* v_log_scales, float* v_logit_opacities,
                                      float* v_sh_0, float* v_sh_rest, float* absgrad, float* v_viewmats, float* v_Ks,
                                      void* workspace, int64_t workspace_bytes, egs_stream_t stream);

/* ---- the depth cotangent (render modes with expected depth) ---------------------------------------------------------
 * The backward entries above also take slot 11 of the gradient records (v_depth, written by egs_rasterize_bwd_depth) as
 * the gradient w.r.t. the camera-space depth z = R[2,:] m + t[2] of each visible (camera, Gaussian): it adds
 * v_depth * R[2,:] to v_means and, when v_viewmats is requested, v_depth * (m, 1) to row 2 of v_viewmats.  v_Ks does not
 * depend on it (z does not depend on K).  One entry for every form: antialiased as in egs_projection_bwd_viewmats;
 * v_viewmats and v_Ks both nullable, with egs_projection_bwd_intrinsics_workspace_bytes(C, N) bytes of workspace when
 * v_Ks is given, egs_projection_bwd_viewmats_workspace_bytes(C, N) when only v_viewmats is, none otherwise.  The entries
 * above read v_depth as 0; their kernels are compiled separately from these. */
int egs_projection_bwd_depth(int32_t C, int32_t N, const float* means, const float* quats, const float* scales,
                             const float* opacities, const float* sh_coeffs, int32_t K, int32_t sh_degree,
                             int32_t colors_per_camera, const float* viewmats, const float* Ks, int32_t width,
                             int32_t height, float eps2d, const int32_t* radii, const float* colors,
                             const float* v_splats, const float* v_means2d_extra, float* v_means, float* v_quats,
                             float* v_scales, float* v_opacities, float* v_sh_coeffs, float* absgrad,
                             int32_t antialiased, float* v_viewmats, float* v_Ks, void* workspace,
                             int64_t workspace_bytes, egs_stream_t stream);

/* ---- orthographic and fisheye camera models ----------------------------------------------------------------------------
 * The projection of the entries above for another camera model; pinhole calls keep the entries above.
 *   camera_model = 1 (ortho):   means2d = (fx x + cx, fy y + cy), J = [[fx, 0, 0], [0, fy, 0]];
 *   camera_model = 2 (fisheye): equidistant, r = sqrt(x^2 + y^2), theta = atan2(r, z),
 *                               means2d = (fx x theta / r + cx, fy y theta / r + cy), J its exact Jacobian;
 * (x, y, z) the camera-space mean.  Neither has the pinhole fov clamp; culling, the eps2d blur, radius, compensation and
 * depths (camera-space z) are the pinhole ones.  Any other camera_model is rejected before any launch.
 * egs_projection_fwd_camera_model: egs_projection_fwd, or egs_projection_fwd_antialiased when compensations is not NULL.
 * egs_projection_bwd_camera_model: egs_projection_bwd_depth for the camera model (slot 11 of the gradient records is
 *   always read; it is 0 from every blend backward but the depth one), same nullable v_viewmats / v_Ks and workspace.
 *   v_Ks[c] = [[v_fx, 0, v_cx], [0, v_fy, v_cy], [0, 0, 0]] with v_fx = (v_m2x (m2x - cx) + sum_j v_J0j J0j) / fx. */
int egs_projection_fwd_camera_model(int32_t camera_model, int32_t C, int32_t N, const float* means, const float* quats,
                                    const float* scales, const float* opacities, const float* sh_coeffs, int32_t K,
                                    int32_t sh_degree, int32_t colors_per_camera, const float* viewmats, const float* Ks,
                                    int32_t width, int32_t height, float eps2d, float near_plane, float far_plane,
                                    float radius_clip, int32_t tile_size, int32_t tile_width, int32_t tile_height,
                                    int32_t* radii, float* means2d, float* depths, float* conics, float* colors,
                                    int32_t* tiles_per_gauss, int32_t* tight_rects, float* splats, float* compensations,
                                    egs_stream_t stream);
int egs_projection_bwd_camera_model(int32_t camera_model, int32_t C, int32_t N, const float* means, const float* quats,
                                    const float* scales, const float* opacities, const float* sh_coeffs, int32_t K,
                                    int32_t sh_degree, int32_t colors_per_camera, const float* viewmats, const float* Ks,
                                    int32_t width, int32_t height, float eps2d, const int32_t* radii, const float* colors,
                                    const float* v_splats, const float* v_means2d_extra, float* v_means, float* v_quats,
                                    float* v_scales, float* v_opacities, float* v_sh_coeffs, float* absgrad,
                                    int32_t antialiased, float* v_viewmats, float* v_Ks, void* workspace,
                                    int64_t workspace_bytes, egs_stream_t stream);

/* ---- g3: exclusive scan of tiles_per_gauss, then key emission -------------------------------------
 * Replaces `torch.cumsum` + the second launch of gsplat `isect_tiles`.
 * egs_exclusive_scan: out[i] = sum_{j<i} in[j] (int64), *total = sum of all (device int64). */
int64_t egs_exclusive_scan_workspace_bytes(int64_t n);
int egs_exclusive_scan(int64_t n, const int32_t* in, int64_t* out, int64_t* total, void* workspace,
                       int64_t workspace_bytes, egs_stream_t stream);

/* key = cam << (32 + tile_n_bits) | tile << 32 | bits(depth);  value = c*N + n.
 * Emission order: flat (c,n) order, tiles row-major inside a Gaussian (SURVEY.md A-3). */
int egs_isect_emit(int32_t C, int32_t N, const float* means2d, const int32_t* radii, const float* depths,
                   const int64_t* cum_tiles_excl, int32_t tile_size, int32_t tile_width, int32_t tile_height,
                   int32_t tile_n_bits, int64_t n_isects, int64_t* isect_ids, int32_t* flatten_ids,
                   egs_stream_t stream);

/* ---- g4: stable LSD onesweep radix sort of (u64 key, u32 value) pairs ----------------------------
 * Replaces `cub::DeviceRadixSort::SortPairs` inside gsplat `isect_tiles`.  Sorts on key bits
 * [0, end_bit) in ceil(end_bit / 8) passes, ping-ponging between (keys_a, vals_a) and
 * (keys_b, vals_b); input is taken from the `a` buffers.  Returns in *result_in_b (HOST int)
 * whether the sorted data ended in the `b` buffers. */
int64_t egs_radix_sort_workspace_bytes(int64_t n, int32_t end_bit);
int egs_radix_sort_pairs_u64_u32(int64_t n, uint64_t* keys_a, uint32_t* vals_a, uint64_t* keys_b,
                                 uint32_t* vals_b, int32_t end_bit, void* workspace, int64_t workspace_bytes,
                                 int32_t* host_result_in_b, egs_stream_t stream);

/* Same sort for 32-bit keys (used by the fast binning path below). */
int egs_radix_sort_pairs_u32_u32(int64_t n, uint32_t* keys_a, uint32_t* vals_a, uint32_t* keys_b, uint32_t* vals_b,
                                 int32_t end_bit, void* workspace, int64_t workspace_bytes,
                                 int32_t* host_result_in_b, egs_stream_t stream);

/* ---- g3-g5 fast path: identical sorted (isect_ids, flatten_ids, isect_offsets), ~3x less traffic ----------
 * A stable sort on cam|tile|depth keys equals (1) a stable sort of the VISIBLE entries of all cameras on depth
 * (ties keep flat-index order), (2) emitting their tiles in that order, (3) a stable sort of the emitted pairs on
 * the (cam,tile) index alone — which also separates the cameras, so level 1 needs no camera bits.
 *   egs_isect_visible_keys : compacts visible entries (tiles_per_gauss > 0) into level-1 pairs
 *                            keys1 = bits(depth) (u32), vals1 = flat index; totals[4] = {n_vis, n_isects, 0, 0} (device)
 *   (sort keys1/vals1 with egs_radix_sort_pairs_u32_u32 on bits [0, 32))
 *   egs_exclusive_scan_gather : out[i] = sum_{j<i} src[gather[j]]  (tile counts in depth order)
 *   egs_isect_emit_sorted  : warp-cooperative emission of tile_keys = cam*n_tiles + tile (u32), flat_vals
 *   (sort tile_keys/flat_vals with egs_radix_sort_pairs_u32_u32 on bits [0, ceil(log2(C*n_tiles))))
 *   egs_isect_finalize     : derives the tile offsets and/or rebuilds the 64-bit isect_ids (either output
 *                            pointer may be NULL: the Python side materialises isect_ids lazily, on first access) */
/* Sync-free form of the route (what rasterization() runs): after egs_isect_visible_keys has left the level-1 pairs
 * and the counts on the device, ONE call enqueues everything else — level-1 sort, tile-count scan + emission (one
 * launch, chained across thread blocks by decoupled look-back), level-2 sort, tile offsets — for a CAPACITY of intersections chosen by the caller (e.g. from the previous call), every
 * kernel reading the live counts from `stats` on the device.  No host round trip is needed to size anything.
 *   stats[4] (device int64): [0] n_vis, [1] n_isects as left by egs_isect_visible_keys (inputs); [2] receives the
 *            longest tile list.  If n_isects > capacity the outputs hold a truncated, memory-safe but meaningless
 *            binning: the caller reads stats back, and calls again with a sufficient capacity.
 *   keys1 / vals1: the level-1 pairs (clobbered).  tile_keys / flatten_ids [capacity]: sorted (camera, tile) keys and
 *            flat indices, the first n_isects valid.  offsets [C * n_tiles + 1]: tile offsets plus a SENTINEL entry
 *            holding n_isects, which egs_rasterize_* read when they are given a negative n_isects.
 *   tile_order [C * n_tiles] (nullable): the flat tile indices sorted by list length, longest first — the launch
 *            order for egs_rasterize_* (their tile_order argument).
 *   tight_rects: NULL gives gsplat's lists bit for bit (rectangles from means2d / radii).  TIGHT lists —
 *            tight_rects = that output of egs_projection_fwd*: every Gaussian is listed only in the tiles of its
 *            classic rectangle that hold a pixel it can reach with alpha >= 1/255 (the rectangle intersected with
 *            the axis-aligned extent of sigma <= sigma_cut).  The blend kernels produce the same pixels and gradients
 *            from them (a dropped entry has alpha < 1/255 at every pixel of its tile); a third fewer entries to
 *            sort, stage and cull.  stats[1] is rewritten with the emitted total. */
int64_t egs_isect_sorted_workspace_bytes(int32_t C, int32_t N, int32_t n_tiles, int64_t capacity);
int egs_isect_sorted(int32_t C, int32_t N, const int32_t* tight_rects, const float* means2d,
                     const int32_t* radii, uint32_t* keys1, uint32_t* vals1, int64_t* stats, int32_t tile_size, int32_t tile_width,
                     int32_t tile_height, int64_t capacity, void* workspace, int64_t workspace_bytes,
                     uint32_t* tile_keys, uint32_t* flatten_ids, int32_t* offsets, int32_t* tile_order,
                     egs_stream_t stream);
int64_t egs_isect_scan_workspace_bytes(int64_t n);
int egs_isect_visible_keys(int32_t C, int32_t N, const int32_t* tiles_per_gauss, const float* depths, uint32_t* keys1,
                           uint32_t* vals1, int64_t* totals, void* workspace, int64_t workspace_bytes,
                           egs_stream_t stream);
int egs_exclusive_scan_gather(int64_t n, const int32_t* src, const uint32_t* gather, int64_t* out, int64_t* total,
                              void* workspace, int64_t workspace_bytes, egs_stream_t stream);
int egs_isect_emit_sorted(int32_t C, int32_t N, int64_t n_vis, const uint32_t* order, const int64_t* cum_excl,
                          const float* means2d, const int32_t* radii, int32_t tile_size, int32_t tile_width,
                          int32_t tile_height, int64_t n_isects, uint32_t* tile_keys, uint32_t* flat_vals,
                          egs_stream_t stream);
int egs_isect_finalize(int64_t n_isects, const uint32_t* tile_keys_sorted, const uint32_t* flat_sorted,
                       const float* depths, int32_t C, int32_t n_tiles, int32_t tile_n_bits, int64_t* isect_ids,
                       int32_t* offsets, egs_stream_t stream);

/* ---- g5: tile offsets -------------------------------------------------------------------------------
 * Replaces gsplat `isect_offset_encode`.  offsets[C*n_tiles] i32 (fully written, also for n = 0). */
int egs_isect_offset_encode(int64_t n_isects, const int64_t* isect_ids_sorted, int32_t C, int32_t n_tiles,
                            int32_t tile_n_bits, int32_t* offsets, egs_stream_t stream);

/* ---- g6: alpha blending forward ----------------------------------------------------------------------
 * Replaces gsplat `rasterize_to_pixels` fwd (3 colour channels, tile_size 16).
 *   backgrounds[C,3] nullable.  outputs: render_colors[C,H,W,3], render_alphas[C,H,W,1],
 *   last_ids[C,H,W] i32 (index into the sorted intersection list of the last blended Gaussian).
 *   n_isects (all egs_rasterize_* entries): the list length, or a NEGATIVE number -capacity when only the device
 *   knows it: tile_offsets then has C * n_tiles + 1 entries, the last one holding the live length (egs_isect_sorted
 *   writes it), and capacity bounds it (sizes the segment launch / the checkpoint buffer).
 *   tile_order (nullable, egs_rasterize_fwd / _fwd_checkpointed / _bwd / _bwd_segmented): a permutation of the
 *   C * n_tiles flat tile indices; thread block b works on tile tile_order[b].  egs_isect_sorted emits one that puts
 *   the longest lists first, so that the end of a launch is made of the cheapest tiles (the GPU runs thread blocks
 *   roughly in index order).  Results do not depend on it. */
int egs_rasterize_fwd(int32_t C, int32_t N, int64_t n_isects, const float* splats, const int32_t* tile_offsets,
                      const int32_t* flatten_ids, const float* backgrounds, int32_t width, int32_t height,
                      int32_t tile_width, int32_t tile_height, float* render_colors, float* render_alphas,
                      int32_t* last_ids, const int32_t* tile_order, egs_stream_t stream);

/* Instrumented variant used only by bench.py / tests for the roofline model: additionally adds the
 * number of evaluated and accepted (pixel, Gaussian) pairs (P_eval, P_acc of SURVEY.md §8d) to
 * pair_counters[0..1] (device uint64, zeroed by the caller). */
int egs_rasterize_fwd_count(int32_t C, int32_t N, int64_t n_isects, const float* splats,
                            const int32_t* tile_offsets, const int32_t* flatten_ids, const float* backgrounds,
                            int32_t width, int32_t height, int32_t tile_width, int32_t tile_height,
                            float* render_colors, float* render_alphas, int32_t* last_ids,
                            uint64_t* pair_counters, egs_stream_t stream);

/* ---- g7: alpha blending backward ----------------------------------------------------------------------
 * Replaces gsplat `rasterize_to_pixels` bwd incl. absgrad (model/gaussian.py:191 reads it).
 * v_splats[C,N,12] must be zero-filled by the caller; gradients are accumulated with
 * warp-reduced global reductions. */
int egs_rasterize_bwd(int32_t C, int32_t N, int64_t n_isects, const float* splats, const int32_t* tile_offsets,
                      const int32_t* flatten_ids, const float* backgrounds, int32_t width, int32_t height,
                      int32_t tile_width, int32_t tile_height, const float* render_alphas,
                      const int32_t* last_ids, const float* v_render_colors, const float* v_render_alphas,
                      float* v_splats, const int32_t* tile_order, egs_stream_t stream);

/* ---- g6 / g7 with the depth as a fourth channel (gsplat's render_mode "ED" / "RGB+ED") ------------------------------
 * egs_rasterize_fwd / _bwd with one more blended channel: the camera-space depth of splat-record slot 9, background 0.
 * egs_rasterize_fwd_depth: render_colors[C,H,W,4] = {r, g, b, accumulated depth}; backgrounds[C,3] (nullable) apply to
 *   r, g, b only.  render_alphas and last_ids, and the r, g, b channels, are bit-identical to egs_rasterize_fwd's.
 * egs_rasterize_bwd_depth: v_render_colors[C,H,W,4].  The depth channel enters v_alpha like a colour channel, and
 *   sum fac * v_depth_channel is added into slot 11 (v_depth) of the gradient records.  With a zero depth cotangent,
 *   slots 0-10 equal egs_rasterize_bwd's.
 * Neither has a segmented / checkpointed form: long lists are replayed in one piece. */
int egs_rasterize_fwd_depth(int32_t C, int32_t N, int64_t n_isects, const float* splats, const int32_t* tile_offsets,
                            const int32_t* flatten_ids, const float* backgrounds, int32_t width, int32_t height,
                            int32_t tile_width, int32_t tile_height, float* render_colors, float* render_alphas,
                            int32_t* last_ids, const int32_t* tile_order, egs_stream_t stream);
int egs_rasterize_bwd_depth(int32_t C, int32_t N, int64_t n_isects, const float* splats, const int32_t* tile_offsets,
                            const int32_t* flatten_ids, const float* backgrounds, int32_t width, int32_t height,
                            int32_t tile_width, int32_t tile_height, const float* render_alphas,
                            const int32_t* last_ids, const float* v_render_colors, const float* v_render_alphas,
                            float* v_splats, const int32_t* tile_order, egs_stream_t stream);

/* ---- g7 on long lists: segmented replay ---------------------------------------------------------------------------
 * A tile whose list has thousands of entries (object-centric scenes: a few hundred tiles hold the whole object) makes
 * the backward pass a serial walk of one warp per tile half.  The checkpointed forward stores the per-pixel state
 * {T, r, g, b} after every `segment` entries of a list (segment: a multiple of 64; checkpoints: caller-allocated,
 * egs_rasterize_checkpoint_bytes(n_isects, segment) bytes, need not be cleared); the segmented backward then replays
 * every segment with its own warp (an extra launch over the checkpoint slots), starting from the checkpoint and
 * from "final colour minus colour in front" for what lies behind.  Only lists of at least seg_min_len entries
 * (raised to segment + 1 if smaller) are treated this way; shorter lists are replayed in one piece as by
 * egs_rasterize_bwd, so ordinary tiles pay nothing.  Results equal egs_rasterize_fwd / _bwd up to fp32 summation
 * order; segment = 0 is exactly those two calls. */
int64_t egs_rasterize_checkpoint_bytes(int64_t n_isects, int32_t segment);
int egs_rasterize_fwd_checkpointed(int32_t C, int32_t N, int64_t n_isects, const float* splats,
                                   const int32_t* tile_offsets, const int32_t* flatten_ids, const float* backgrounds,
                                   int32_t width, int32_t height, int32_t tile_width, int32_t tile_height,
                                   float* render_colors, float* render_alphas, int32_t* last_ids, float* checkpoints,
                                   int32_t segment, int32_t seg_min_len, const int32_t* tile_order, egs_stream_t stream);
int egs_rasterize_bwd_segmented(int32_t C, int32_t N, int64_t n_isects, const float* splats,
                                const int32_t* tile_offsets, const int32_t* flatten_ids, const float* backgrounds,
                                int32_t width, int32_t height, int32_t tile_width, int32_t tile_height,
                                const float* render_colors, const float* render_alphas, const int32_t* last_ids,
                                const float* v_render_colors, const float* v_render_alphas, const float* checkpoints,
                                int32_t segment, int32_t seg_min_len, float* v_splats, const int32_t* tile_order,
                                egs_stream_t stream);

/* ---- g6 / g7 with colours of any number of channels ("features") ---------------------------------------------------
 * gsplat 1.0.0 `rasterize_to_pixels` with colors[..., D], D >= 1 (rasterization() with sh_degree=None and [N,D] or
 * [C,N,D] colours).  The splat records still carry the geometry (their r, g, b slots are not read); the colours come
 * from a separate row array:
 *   features [rows, feat_stride] fp32, row = flat id - cam * N (shared_rows = 1: one [N, .] array for all cameras) or
 *            the flat id (shared_rows = 0: [C*N, .]).  A call reads channels [c0, c0 + CH) of every row it blends, so
 *            feat_stride >= c0 + CH: pad the rows with zero channels up to the chunk width.  CH is one of 1, 2, 4, 8, 16,
 *            32; features, feat_stride and c0 must be aligned to min(CH, 4) floats (rows are copied in 4 / 8 / 16-byte
 *            pieces).  0 <= c0 < D.
 *   A call covers channels [c0, c0 + min(CH, D - c0)) of the [C,H,W,D] images; colours wider than 32 channels take one
 *   call per chunk on the same binning result.  CH <= 8 reproduces egs_rasterize_fwd's render_alphas and last_ids bit
 *   for bit; CH = 16 / 32 blend one pixel per lane and their transmittance can differ from that in the last bits
 *   (measured: alphas within 2.4e-7).  Take render_alphas / last_ids from one chunk and pass those to every backward
 *   chunk of the call.
 *   backgrounds[C,D] (nullable): the call adds T_final * backgrounds[cam, c0 + k].
 * egs_rasterize_fwd_features: render_colors[C,H,W,D] (channels of this chunk written); render_alphas, last_ids as in
 *   egs_rasterize_fwd, both nullable (chunks after the first need not write them again).
 * egs_rasterize_bwd_features: render_alphas / last_ids from the forward; v_render_colors[C,H,W,D];
 *   v_render_alphas (nullable: pass it to exactly one chunk of a call; the others get NULL).  Adds (RED.ADD) into
 *   caller-zeroed buffers: the geometry slots of v_splats[C,N,12] (v_x, v_y, v_conic, v_opacity, |v_x|, |v_y|; the
 *   v_r, v_g, v_b slots are left alone, so egs_projection_bwd* consume the records unchanged) and, when v_features is
 *   given, v_features [rows, feat_stride] (same layout as features; only the chunk's real channels).  With several
 *   chunks the geometry slots, |v_x| and |v_y| included, sum over the chunks.
 * No segmented replay: long lists are replayed in one piece. */
int egs_rasterize_fwd_features(int32_t C, int32_t N, int64_t n_isects, const float* splats, const int32_t* tile_offsets,
                               const int32_t* flatten_ids, const float* features, int32_t feat_stride,
                               int32_t shared_rows, int32_t D, int32_t c0, int32_t CH, const float* backgrounds,
                               int32_t width, int32_t height, int32_t tile_width, int32_t tile_height,
                               float* render_colors, float* render_alphas, int32_t* last_ids, const int32_t* tile_order,
                               egs_stream_t stream);
int egs_rasterize_bwd_features(int32_t C, int32_t N, int64_t n_isects, const float* splats, const int32_t* tile_offsets,
                               const int32_t* flatten_ids, const float* features, int32_t feat_stride,
                               int32_t shared_rows, int32_t D, int32_t c0, int32_t CH, const float* backgrounds,
                               int32_t width, int32_t height, int32_t tile_width, int32_t tile_height,
                               const float* render_alphas, const int32_t* last_ids, const float* v_render_colors,
                               const float* v_render_alphas, float* v_splats, float* v_features,
                               const int32_t* tile_order, egs_stream_t stream);

/* ---- §8f-1: fused, sync-free densification statistics (C-aware) ----------------------------------------
 * Replaces GaussianModel.update_statistics, /root/reference/model/gaussian.py:188-197, applied once
 * per camera: visible = radii > 0; max_radii = max(max_radii, radii / max_hw);
 * grad_norm_accum += |absgrad|_2 * max_hw; collecting_counts += 1.
 *   radii[C,N] i32, absgrad[C,N,2] (the tensor tagged on meta["means2d"].absgrad), stats [N] f32. */
int egs_densify_stats_update(int32_t C, int32_t N, const int32_t* radii, const float* absgrad, float max_hw,
                             float* max_radii, float* grad_norm_accum, float* collecting_counts,
                             egs_stream_t stream);

/* ---- §8f-3: fused Adam over up to 8 parameter groups ---------------------------------------------------------
 * Replaces torch.optim.Adam for the reference's six groups (/root/reference/model/gaussian.py:389-412,
 * train.py:156-157): default Adam (no weight decay, no amsgrad), one launch, 28 B/element.
 * params/grads/exp_avg/exp_avg_sq: HOST arrays of n_groups DEVICE pointers; numels, lrs: HOST arrays; step >= 1. */
int egs_fused_adam(int32_t n_groups, float* const* params, const float* const* grads, float* const* exp_avg,
                   float* const* exp_avg_sq, const int64_t* numels, const float* lrs, float beta1, float beta2,
                   float eps, int64_t step, egs_stream_t stream);

/* ---- §8e: gradient exchange as a two-shot all-reduce over NVLink peer memory -------------------------------------
 * Every rank's flat fp32 bucket is mapped into every peer (symmetric memory); peer_buffers_dev: DEVICE array of
 * `world` device pointers, entry p = rank p's bucket as mapped on this GPU.  Both exchanges of the view-sharded step
 * (SURVEY.md section 8e) go in ONE launch: the first n_sum_floats of the bucket are SUMmed over the ranks (parameter
 * gradients, then the grad_norm_accum / collecting_counts rows of the step's densify statistics,
 * model/gaussian.py:196-197), the n_max_floats behind them take the MAXimum (the max_radii row, gaussian.py:194; values
 * must be >= 0: the NVLS variant compares their bit patterns as unsigned integers).  Both counts are multiples of 4;
 * n_max_floats = 0 is a plain SUM all-reduce.
 * Rank r reduces slice r over all buckets in rank order (peer loads) and writes it into every bucket (peer stores):
 * in place, bit-identical on all replicas.  The caller brackets the call with inter-rank barriers
 * (all buckets complete before, all slices written after); world = 1 is a no-op. */
int egs_allreduce_f32_peer(int32_t world, int32_t rank, const void* peer_buffers_dev, int64_t n_sum_floats,
                           int64_t n_max_floats, egs_stream_t stream);
/* The same exchange through the NVSwitch (NVLS): multicast_ptr is the multicast mapping of the symmetric bucket;
 * rank r pulls the in-switch reduction of slice r (multimem.ld_reduce) and broadcasts it back (multimem.st). */
int egs_allreduce_f32_multimem(int32_t world, int32_t rank, void* multicast_ptr, int64_t n_sum_floats,
                               int64_t n_max_floats, egs_stream_t stream);

/* ---- measurement utility (bench.py only) -----------------------------------------------------------------
 * Dependent-FMA throughput probe: the FP32-SIMT roofline denominator for the blending kernels
 * (BASELINE.md §3).  blocks x 256 threads x iters x 32 FMAs; *host_flops (HOST double) = flops issued. */
int egs_probe_fp32_fma(int32_t blocks, int32_t iters, float* out, double* host_flops, egs_stream_t stream);

/* ---- §8f-4: fused L1 + SSIM photometric loss (LossComputer, /root/reference/model/gaussian.py:415-453) ----------
 * x = mask * gt + (1 - mask) * render; l1 = mean |x - gt|; ssim_loss = 1 - SSIM(gt, x) with torchmetrics'
 * StructuralSimilarityIndexMeasure(data_range=1.0) defaults (11-tap Gaussian window, sigma 1.5, k1 .01, k2 .03,
 * reflect pad + crop == valid window over the unpadded image); total = (1 - lambda) l1 + lambda ssim_loss.
 *   render, gt [C,H,W,3] (the layout rasterization() returns), mask [C,H,W] (nullable = all zeros), H, W >= 11
 *   egs_l1_ssim_fwd: sums[C,2] (double, zeroed by the caller) += {sum |x - gt|, sum of the SSIM map};
 *                    maps (nullable: no gradient wanted) = 3 planes [C,3,H-10,W-10] (channel planar, internal to
 *                    this pair of calls) of SSIM partial derivatives
 *   egs_l1_ssim_bwd: v_render[C,H,W,3] = v_total[c] * d total_c / d render  (v_total: DEVICE array [C]) */
int egs_l1_ssim_fwd(int32_t C, int32_t H, int32_t W, const float* render, const float* gt, const float* mask,
                    float* maps, double* sums, egs_stream_t stream);
int egs_l1_ssim_bwd(int32_t C, int32_t H, int32_t W, const float* render, const float* gt, const float* mask,
                    const float* maps, float lambda_ssim, const float* v_total, float* v_render, egs_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* EGS_RASTER_H_ */
