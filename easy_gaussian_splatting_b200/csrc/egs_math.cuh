// Per-element math of the projection / SH stages, shared by the CUDA kernels and by the
// host-side test harness (tests/ compile this header with the host compiler to check the
// formulas against the oracle without a GPU; the product never runs it on the CPU).
//
// BIT-EXACTNESS CONTRACT: project_fwd() performs exactly the sequence of IEEE-754 fp32
// round-to-nearest operations documented as "CANONICAL OP ORDER" in oracle/gsplat_oracle.py.
// Translation units including this header for that purpose must be compiled with FMA
// contraction OFF (nvcc -fmad=false, gcc -ffp-contract=off) and without fast-math, so that
// radii, tile counts and depth key bits are identical to the oracle's.
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define EGS_HD __host__ __device__ __forceinline__
#else
#define EGS_HD inline
#endif

namespace egs {

struct Camera {
  float r[9];       // world->camera rotation, row major
  float t[3];       // translation
  float fx, fy, cx, cy;
  float campos[3];  // camera centre in world coordinates = -R^-1 t
};

// Build the per-camera constants from a row-major [4,4] view matrix and [3,3] K.
// campos uses the general 3x3 inverse (adjugate), matching torch.inverse(viewmat)[:3,3]
// up to rounding also for non-rigid view matrices.
EGS_HD void load_camera(const float* V, const float* K, Camera& c) {
  c.r[0] = V[0]; c.r[1] = V[1]; c.r[2] = V[2];  c.t[0] = V[3];
  c.r[3] = V[4]; c.r[4] = V[5]; c.r[5] = V[6];  c.t[1] = V[7];
  c.r[6] = V[8]; c.r[7] = V[9]; c.r[8] = V[10]; c.t[2] = V[11];
  c.fx = K[0]; c.cx = K[2]; c.fy = K[4]; c.cy = K[5];
  const float* r = c.r;
  float a00 = r[4] * r[8] - r[5] * r[7];
  float a01 = r[2] * r[7] - r[1] * r[8];
  float a02 = r[1] * r[5] - r[2] * r[4];
  float a10 = r[5] * r[6] - r[3] * r[8];
  float a11 = r[0] * r[8] - r[2] * r[6];
  float a12 = r[2] * r[3] - r[0] * r[5];
  float a20 = r[3] * r[7] - r[4] * r[6];
  float a21 = r[1] * r[6] - r[0] * r[7];
  float a22 = r[0] * r[4] - r[1] * r[3];
  float det = r[0] * a00 + r[1] * a10 + r[2] * a20;
  float id = 1.0f / det;
  c.campos[0] = -(a00 * c.t[0] + a01 * c.t[1] + a02 * c.t[2]) * id;
  c.campos[1] = -(a10 * c.t[0] + a11 * c.t[1] + a12 * c.t[2]) * id;
  c.campos[2] = -(a20 * c.t[0] + a21 * c.t[1] + a22 * c.t[2]) * id;
}

// wxyz (unnormalised) -> row-major rotation; also returns the normalised quaternion and 1/|q|.
EGS_HD void quat_to_rotmat(const float q[4], float R[9], float qn[4], float& inv_norm) {
  float w = q[0], x = q[1], y = q[2], z = q[3];
  float s = ((w * w + x * x) + y * y) + z * z;
  float inv = 1.0f / sqrtf(s);
  w = w * inv; x = x * inv; y = y * inv; z = z * inv;
  qn[0] = w; qn[1] = x; qn[2] = y; qn[3] = z;
  inv_norm = inv;
  float x2 = x * x, y2 = y * y, z2 = z * z;
  float xy = x * y, xz = x * z, yz = y * z;
  float wx = w * x, wy = w * y, wz = w * z;
  R[0] = 1.0f - 2.0f * (y2 + z2);
  R[1] = 2.0f * (xy - wz);
  R[2] = 2.0f * (xz + wy);
  R[3] = 2.0f * (xy + wz);
  R[4] = 1.0f - 2.0f * (x2 + z2);
  R[5] = 2.0f * (yz - wx);
  R[6] = 2.0f * (xz - wy);
  R[7] = 2.0f * (yz + wx);
  R[8] = 1.0f - 2.0f * (x2 + y2);
}

// Everything the backward pass needs to re-derive from the forward pass.
struct ProjState {
  float R[9], qn[4], inv_norm;
  float M[9];                 // R * diag(scale)
  float S[6];                 // world covariance (00,01,02,11,12,22)
  float x, y, z;              // camera-space mean
  float k[6];                 // camera-space covariance (00,01,02,11,12,22)
  float rz, rz2, tx, ty;
  float J00, J02, J11, J12;
  float a, b, d, det;         // blurred 2D covariance and its determinant
  float det_orig;             // determinant before the eps2d blur (antialiased mode: compensation factor)
  bool clamp_x, clamp_y;      // fov clamp active
  float J01, J10;             // kOrtho / kFisheye: the rest of the 2x3 Jacobian (0 for kOrtho)
  float fs, fg, fq, r2;       // kFisheye: theta / r, g (fisheye_theta_over_r), 1 / (r^2 + z^2), r^2 = x^2 + y^2
};

// ---- camera models -------------------------------------------------------------------------------------------------
// The camera enters the projection only through (x, y, z, Sigma_cam) -> (means2d, cov2d = J Sigma_cam J^T) and its VJP;
// project_fwd / project_bwd take the model as a template argument, kPinhole by default.
//   kPinhole: means2d = (fx x / z + cx, fy y / z + cy), gsplat's persp_proj J with the 1.3 x fov clamp (the code below
//             the model switch is the one every pinhole kernel has always compiled).
//   kOrtho:   means2d = (fx x + cx, fy y + cy), J = [[fx, 0, 0], [0, fy, 0]], no clamp.
//   kFisheye: equidistant, r = sqrt(x^2 + y^2), theta = atan2(r, z): means2d = (fx x theta / r + cx, fy y theta / r + cy),
//             J the exact Jacobian of means2d (gsplat's fisheye_proj J), no clamp.
// Culling (near / far on z, eps2d blur, radius, off-screen test) and the compensation are the same for all three.
constexpr int kPinhole = 0, kOrtho = 1, kFisheye = 2;

// atan(sqrt(u)) / sqrt(u) and (1 / (1 + u) - atan(sqrt(u)) / sqrt(u)) / u on u in [0, 1]: fp32 polynomials fitted by
// scripts/fit_fisheye_theta.py (0.86 and 2.6 ulp there), evaluated by Horner from the highest term, mul then add.
EGS_HD float fisheye_poly_p(float u) {
  float p = 0.0010774789843708277f;
  p = p * u + -0.007134431507438421f;
  p = p * u + 0.022145025432109833f;
  p = p * u + -0.044218774884939194f;
  p = p * u + 0.0670754536986351f;
  p = p * u + -0.0879582092165947f;
  p = p * u + 0.11054043471813202f;
  p = p * u + -0.142791748046875f;
  p = p * u + 0.1999961882829666f;
  p = p * u + -0.33333325386047363f;
  p = p * u + 1.0f;
  return p;
}

EGS_HD float fisheye_poly_h(float u) {
  float p = -0.015319157391786575f;
  p = p * u + 0.09921801835298538f;
  p = p * u + -0.29700547456741333f;
  p = p * u + 0.5588876008987427f;
  p = p * u + -0.7710589170455933f;
  p = p * u + 0.876106321811676f;
  p = p * u + -0.9004436731338501f;
  p = p * u + 0.8879852890968323f;
  p = p * u + -0.8571013808250427f;
  p = p * u + 0.7999998927116394f;
  p = p * u + -0.6666666865348816f;
  return p;
}

// a * b = p + e exactly: Dekker's product with Veltkamp's split (round to nearest, no FMA, |a|, |b| < 1e34)
EGS_HD void two_prod(float a, float b, float& p, float& e) {
  const float ca = 4097.0f * a, cb = 4097.0f * b;
  const float ah = ca - (ca - a), bh = cb - (cb - b);
  const float al = a - ah, bl = b - bh;
  p = a * b;
  e = ((ah * bh - p) + ah * bl + al * bh) + al * bl;
}

// s = theta / r with theta = atan2(r, z) in [0, pi], and g = (1 / r) ds/dr = (z q - s) / r^2, q = 1 / (r^2 + z^2), for
// r = sqrt(r2) >= 0.  Built only from +, x, / (no atan2f, whose device and host results differ), so that a CPU
// reference reproduces it bit for bit.  CANONICAL OP ORDER, four ranges of theta (r > z in all but the first):
//   r <= z     (theta <= pi/4):           u = r2 / (z * z), s = P(u) / z,  g = H(u) / ((z * z) * z)
//   z >= r / 2 (theta <= atan 2):         t = (r - z) / (r + z), d = (pi/4)_lo + t * P(t * t), hi = (pi/4)_hi
//   r > -z     (theta < 3pi/4):           t = z / r,             d = (pi/2)_lo - t * P(t * t), hi = (pi/2)_hi
//   otherwise  (theta >= 3pi/4):          t = r / (-z),          d = pi_lo - t * P(t * t),     hi = pi_hi
//   then s = (d + hi) / r corrected by the remainder of the division as written below, g = (z * q - s) / r2
//   (_hi + _lo is the fp32 split of the constant).  The second range keeps |atan t| below 0.42 theta, so that its
//   error stays small against theta.  Measured error of s against fp64: 1.6 ulp at most over [0, pi).
// The first range does not use r at all: s and g are exact limits at r = 0 (s = 1/z) and keep full precision for any
// r / z (g by its own polynomial; the direct formula cancels there).  r = 0 with z <= 0 gives non-finite values, which
// the projection culls.
EGS_HD void fisheye_theta_over_r(float r, float r2, float z, float q, float& s, float& g) {
  if (r <= z) {
    const float u = r2 / (z * z);
    s = fisheye_poly_p(u) / z;
    g = fisheye_poly_h(u) / ((z * z) * z);
    return;
  }
  const bool low = z >= 0.5f * r, mid = r > -z;
  const float t = low ? (r - z) / (r + z) : mid ? z / r : r / (-z);
  const float u = t * t;
  const float at = t * fisheye_poly_p(u);
  const float hi = low ? 0.7853981852531433f : mid ? 1.5707963705062866f : 3.1415927410125732f;
  const float d = low ? -2.1855694143368964e-08f + at : (mid ? -4.371138828673793e-08f : -8.742277657347586e-08f) - at;
  // theta = th + tl exactly (|d| < hi), s0 = th / r, and the remainder th + tl - s0 r of that division (s0 r = p + e
  // exactly, th - p exact) corrects it: neither the rounding of theta nor that of the division reaches s
  const float th = d + hi;
  const float tl = d - (th - hi);
  const float s0 = th / r;
  float p, e;
  two_prod(s0, r, p, e);
  s = s0 + (((th - p) - e) + tl) / r;
  g = (z * q - s) / r2;
}

struct ProjOut {
  float m2x, m2y, depth, ca, cb, cc;
  float lambda_max;           // largest eigenvalue of the blurred 2D covariance (clamped like the radius)
  float comp;                 // sqrt(max(0, det_orig / det_blur)): opacity compensation of rasterize_mode="antialiased"
  int32_t radius;             // 0 = culled
};

// Returns true when the Gaussian is visible.  st is filled as far as the computation went.  CM: the camera model.
template <int CM = kPinhole>
EGS_HD bool project_fwd(const float mean[3], const float quat[4], const float scale[3], const Camera& cam,
                        float width, float height, float eps2d, float near_plane, float far_plane,
                        float radius_clip, ProjState& st, ProjOut& o) {
  o.m2x = 0.f; o.m2y = 0.f; o.depth = 0.f; o.ca = 0.f; o.cb = 0.f; o.cc = 0.f; o.radius = 0; o.lambda_max = 0.f; o.comp = 0.f;
  quat_to_rotmat(quat, st.R, st.qn, st.inv_norm);
  const float* R = st.R;
  float* M = st.M;
  M[0] = R[0] * scale[0]; M[1] = R[1] * scale[1]; M[2] = R[2] * scale[2];
  M[3] = R[3] * scale[0]; M[4] = R[4] * scale[1]; M[5] = R[5] * scale[2];
  M[6] = R[6] * scale[0]; M[7] = R[7] * scale[1]; M[8] = R[8] * scale[2];
  float c00 = (M[0] * M[0] + M[1] * M[1]) + M[2] * M[2];
  float c01 = (M[0] * M[3] + M[1] * M[4]) + M[2] * M[5];
  float c02 = (M[0] * M[6] + M[1] * M[7]) + M[2] * M[8];
  float c11 = (M[3] * M[3] + M[4] * M[4]) + M[5] * M[5];
  float c12 = (M[3] * M[6] + M[4] * M[7]) + M[5] * M[8];
  float c22 = (M[6] * M[6] + M[7] * M[7]) + M[8] * M[8];
  st.S[0] = c00; st.S[1] = c01; st.S[2] = c02; st.S[3] = c11; st.S[4] = c12; st.S[5] = c22;
  const float* W = cam.r;
  float x = ((W[0] * mean[0] + W[1] * mean[1]) + W[2] * mean[2]) + cam.t[0];
  float y = ((W[3] * mean[0] + W[4] * mean[1]) + W[5] * mean[2]) + cam.t[1];
  float z = ((W[6] * mean[0] + W[7] * mean[1]) + W[8] * mean[2]) + cam.t[2];
  st.x = x; st.y = y; st.z = z;
  if (!(z >= near_plane && z <= far_plane)) return false;
  // A = W * Sigma ; Sc = A * W^T
  float Sm[9] = {c00, c01, c02, c01, c11, c12, c02, c12, c22};
  float A[9];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j)
      A[i * 3 + j] = (W[i * 3 + 0] * Sm[0 * 3 + j] + W[i * 3 + 1] * Sm[1 * 3 + j]) + W[i * 3 + 2] * Sm[2 * 3 + j];
#define EGS_SC(i, j) ((A[i * 3 + 0] * W[j * 3 + 0] + A[i * 3 + 1] * W[j * 3 + 1]) + A[i * 3 + 2] * W[j * 3 + 2])
  float k00 = EGS_SC(0, 0), k01 = EGS_SC(0, 1), k02 = EGS_SC(0, 2);
  float k11 = EGS_SC(1, 1), k12 = EGS_SC(1, 2), k22 = EGS_SC(2, 2);
#undef EGS_SC
  st.k[0] = k00; st.k[1] = k01; st.k[2] = k02; st.k[3] = k11; st.k[4] = k12; st.k[5] = k22;
  float fx = cam.fx, fy = cam.fy;
  float a, b, d, m2x, m2y;
  if constexpr (CM == kPinhole) {
  float tan_fovx = (0.5f * width) / fx;
  float tan_fovy = (0.5f * height) / fy;
  float lim_x = 1.3f * tan_fovx;
  float lim_y = 1.3f * tan_fovy;
  float rz = 1.0f / z;
  float rz2 = rz * rz;
  float xr = x * rz, yr = y * rz;
  float tx = z * fminf(lim_x, fmaxf(-lim_x, xr));
  float ty = z * fminf(lim_y, fmaxf(-lim_y, yr));
  st.clamp_x = !(xr <= lim_x && xr >= -lim_x);
  st.clamp_y = !(yr <= lim_y && yr >= -lim_y);
  float J00 = fx * rz;
  float J02 = -((fx * tx) * rz2);
  float J11 = fy * rz;
  float J12 = -((fy * ty) * rz2);
  st.rz = rz; st.rz2 = rz2; st.tx = tx; st.ty = ty;
  st.J00 = J00; st.J02 = J02; st.J11 = J11; st.J12 = J12;
  float B00 = J00 * k00 + J02 * k02;
  float B01 = J00 * k01 + J02 * k12;
  float B02 = J00 * k02 + J02 * k22;
  float B11 = J11 * k11 + J12 * k12;
  float B12 = J11 * k12 + J12 * k22;
  a = B00 * J00 + B02 * J02;
  b = B01 * J11 + B02 * J12;
  d = B11 * J11 + B12 * J12;
  m2x = (fx * x) * rz + cam.cx;
  m2y = (fy * y) * rz + cam.cy;
  } else if constexpr (CM == kOrtho) {
    // CANONICAL: cov2d = (fx k00 fx, fx k01 fy, fy k11 fy) in that order; means2d = fx x + cx
    st.J00 = fx; st.J01 = 0.f; st.J02 = 0.f; st.J10 = 0.f; st.J11 = fy; st.J12 = 0.f;
    a = (fx * k00) * fx;
    b = (fx * k01) * fy;
    d = (fy * k11) * fy;
    m2x = fx * x + cam.cx;
    m2y = fy * y + cam.cy;
  } else {
    static_assert(CM == kFisheye, "unknown camera model");
    // CANONICAL: r2 = x*x + y*y, r = sqrt(r2), q = 1 / (r2 + z*z), (s, g) = fisheye_theta_over_r, then
    // J0. = fx (s + (x*x) g, (x*y) g, -(x q)), J1. = fy ((x*y) g, s + (y*y) g, -(y q)) (fx times the bracket),
    // B = J Sc row by row, B_ij = (J_i0 k0j + J_i1 k1j) + J_i2 k2j, cov2d_ij = (B_i0 J_j0 + B_i1 J_j1) + B_i2 J_j2,
    // means2d = (fx x) s + cx
    const float xx = x * x, yy = y * y;
    const float r2 = xx + yy;
    const float r = sqrtf(r2);
    const float q = 1.0f / (r2 + z * z);
    float s, g;
    fisheye_theta_over_r(r, r2, z, q, s, g);
    const float xyg = (x * y) * g;
    const float J00 = fx * (s + xx * g), J01 = fx * xyg, J02 = -(fx * (x * q));
    const float J10 = fy * xyg, J11 = fy * (s + yy * g), J12 = -(fy * (y * q));
    st.J00 = J00; st.J01 = J01; st.J02 = J02; st.J10 = J10; st.J11 = J11; st.J12 = J12;
    st.fs = s; st.fg = g; st.fq = q; st.r2 = r2;
    const float B00 = (J00 * k00 + J01 * k01) + J02 * k02;
    const float B01 = (J00 * k01 + J01 * k11) + J02 * k12;
    const float B02 = (J00 * k02 + J01 * k12) + J02 * k22;
    const float B10 = (J10 * k00 + J11 * k01) + J12 * k02;
    const float B11 = (J10 * k01 + J11 * k11) + J12 * k12;
    const float B12 = (J10 * k02 + J11 * k12) + J12 * k22;
    a = (B00 * J00 + B01 * J01) + B02 * J02;
    b = (B00 * J10 + B01 * J11) + B02 * J12;
    d = (B10 * J10 + B11 * J11) + B12 * J12;
    m2x = (fx * x) * s + cam.cx;
    m2y = (fy * y) * s + cam.cy;
  }
  const float det_orig = a * d - b * b;
  a = a + eps2d;
  d = d + eps2d;
  float det = a * d - b * b;
  st.a = a; st.b = b; st.d = d; st.det = det; st.det_orig = det_orig;
  if (!(det > 0.f)) return false;
  float mid = 0.5f * (a + d);
  float v1 = mid + sqrtf(fmaxf(mid * mid - det, 0.01f));
  float radius = ceilf(3.0f * sqrtf(v1));
  if (!(radius > radius_clip)) return false;
  if (m2x + radius <= 0.f || m2x - radius >= width || m2y + radius <= 0.f || m2y - radius >= height) return false;
  if (!(isfinite(radius) && isfinite(m2x) && isfinite(m2y))) return false;
  float inv_det = 1.0f / det;
  o.ca = d * inv_det;
  o.cb = -(b * inv_det);
  o.cc = a * inv_det;
  o.m2x = m2x; o.m2y = m2y; o.depth = z;
  o.lambda_max = v1;
  o.comp = sqrtf(fmaxf(0.f, det_orig / det));
  o.radius = (int32_t)fminf(radius, 2147483520.0f);
  return true;
}

// Largest sigma at which alpha = min(.999, o exp(-sigma)) can still reach 1/255: ln(255 o), with a small
// margin that keeps every use of it conservative under fp32 rounding.  <= 0 means never visible.  The
// blending kernels drop a Gaussian for a whole warp when the minimum of sigma over the warp's pixel
// rectangle exceeds this value.
EGS_HD float sigma_cutoff(float opacity) {
  const float t = 255.0f * opacity;
  if (!(t > 1.0f)) return -1.0f;
  return logf(t) * 1.001f + 2e-3f;  // margin >> fp32 cancellation error of sigma for strongly anisotropic conics
}

// Tile rectangle of a visible Gaussian: min inclusive, max exclusive (SURVEY.md A-3).
// Divisions by the power-of-two tile size are exact, so this is bit-reproducible.
EGS_HD void tile_rect(float m2x, float m2y, int32_t radius, float tile_size, int32_t tile_w, int32_t tile_h,
                      int32_t& xmin, int32_t& ymin, int32_t& xmax, int32_t& ymax) {
  float tx = m2x / tile_size, ty = m2y / tile_size, tr = (float)radius / tile_size;
  float fw = (float)tile_w, fh = (float)tile_h;
  xmin = (int32_t)fminf(fmaxf(floorf(tx - tr), 0.f), fw);
  ymin = (int32_t)fminf(fmaxf(floorf(ty - tr), 0.f), fh);
  xmax = (int32_t)fminf(fmaxf(ceilf(tx + tr), 0.f), fw);
  ymax = (int32_t)fminf(fmaxf(ceilf(ty + tr), 0.f), fh);
}

// Tight tile rectangle of a visible Gaussian for the BLEND kernels' lists: the classic rectangle above (3-sigma square
// of the major axis, gsplat's rule, which the meta lists must reproduce bit for bit) intersected with the axis-aligned
// extent of {alpha >= 1/255} = {sigma <= sigma_cut}: |dx| <= sqrt(2 sigma_cut cov_xx), cov = conic^-1.  Tiles outside
// it hold no pixel the Gaussian can reach, so the blend kernels need not see it there: 36 % fewer list entries on the
// 1 M-Gaussian benchmark scene (scripts/analysis/tight_rects.py), i.e. 36 % less to sort, stage and cull, for the same
// pixels and gradients.  Margins: sigma_cut itself is ln(255 o) * 1.001 + 2e-3, the extents get another 0.1 % +
// 0.05 px, and an ill-conditioned conic (determinant lost to cancellation) keeps the classic rectangle.
// In: the classic rectangle; out: the tight one (empty when the Gaussian can never reach 1/255).
EGS_HD void tighten_tile_rect(float m2x, float m2y, float ca, float cb, float cc, float sigma_cut, float tile_size,
                              int32_t& x0, int32_t& y0, int32_t& x1, int32_t& y1) {
  if (!(sigma_cut > 0.f)) { x1 = x0; y1 = y0; return; }
  const float det = ca * cc - cb * cb;
  if (!(det > 1e-4f * ca * cc) || !(det > 0.f)) return;
  const float k = 2.0f * sigma_cut / det;
  const float hx = sqrtf(k * cc) * 1.001f + 0.05f, hy = sqrtf(k * ca) * 1.001f + 0.05f;
  if (!(hx < 1e8f) || !(hy < 1e8f)) return;
  // pixel centres p + 0.5 within [m - h, m + h]  ->  tiles floor(p / tile_size), max exclusive
  const float inv = 1.0f / tile_size;
  const float tx0 = floorf(ceilf(m2x - hx - 0.5f) * inv), tx1 = floorf(floorf(m2x + hx - 0.5f) * inv) + 1.0f;
  const float ty0 = floorf(ceilf(m2y - hy - 0.5f) * inv), ty1 = floorf(floorf(m2y + hy - 0.5f) * inv) + 1.0f;
  const int32_t ix0 = (int32_t)fminf(fmaxf(tx0, -1e9f), 1e9f), ix1 = (int32_t)fminf(fmaxf(tx1, -1e9f), 1e9f);
  const int32_t iy0 = (int32_t)fminf(fmaxf(ty0, -1e9f), 1e9f), iy1 = (int32_t)fminf(fmaxf(ty1, -1e9f), 1e9f);
  x0 = x0 > ix0 ? x0 : ix0;
  x1 = x1 < ix1 ? x1 : ix1;
  y0 = y0 > iy0 ? y0 : iy0;
  y1 = y1 < iy1 ? y1 : iy1;
  if (x1 < x0) x1 = x0;
  if (y1 < y0) y1 = y0;
}

// A tile rectangle in 8 bytes, as the projection kernel hands the tight rectangles to the binning route:
// {x0 | y0 << 16, w | h << 16}; tile grids stay below 65536 tiles per side (the entry points check).
EGS_HD void pack_tile_rect(int32_t x0, int32_t y0, int32_t x1, int32_t y1, int32_t& origin, int32_t& extent) {
  const int32_t w = x1 - x0, h = y1 - y0;
  const bool empty = w <= 0 || h <= 0;
  origin = empty ? 0 : (x0 | (y0 << 16));
  extent = empty ? 0 : (w | (h << 16));
}

// Camera gradient of one (camera, Gaussian) pair, 15 floats: v_R[9] (row major) and v_t[3] of the view matrix's
// top 3x4 block, then v_campos[3], the gradient w.r.t. the camera centre the SH directions are taken from.
constexpr int kCamGradFloats = 15;
// Intrinsics gradient of one (camera, Gaussian) pair, 4 floats: v_fx, v_fy, v_cx, v_cy.
constexpr int kKsGradFloats = 4;

// VJP of project_fwd for a visible Gaussian (SURVEY.md A-8).  Accumulates (+=) into
// v_mean[3], v_quat[4], v_scale[3].
// v_cam (nullable, with the Gaussian's world-space mean): also accumulates v_R and v_t (entries 0..11 of the camera
// gradient above) through mean_c = R m + t and cov_c = R Sigma R^T.  A literal nullptr compiles the block out.
// v_K (nullable): also accumulates the intrinsics gradient above through means2d and the Jacobian J (which carries the
// conic's and the compensation's cotangents).  A literal nullptr compiles the block out.
// CM: the camera model of the project_fwd that filled st.  For kOrtho and kFisheye, v_K holds
// v_fx = (v_m2x (m2x - cx) + sum_j vJ_0j J_0j) / fx (likewise v_fy), v_cx = v_m2x, v_cy = v_m2y.
template <int CM = kPinhole>
EGS_HD void project_bwd(const ProjState& st, const float scale[3], const Camera& cam, float v_m2x, float v_m2y,
                        float v_depth, float v_ca, float v_cb, float v_cc, const ProjOut& o, float v_mean[3],
                        float v_quat[4], float v_scale[3], float v_comp = 0.f, float eps2d = 0.f,
                        float* v_cam = nullptr, const float* mean = nullptr, float* v_K = nullptr) {
  // conic = inverse(cov2d'):  V = -Q * G * Q with G = [[v_ca, v_cb/2],[v_cb/2, v_cc]]
  float q00 = o.ca, q01 = o.cb, q11 = o.cc;
  float g00 = v_ca, g01 = 0.5f * v_cb, g11 = v_cc;
  float h00 = q00 * g00 + q01 * g01, h01 = q00 * g01 + q01 * g11;
  float h10 = q01 * g00 + q11 * g01, h11 = q01 * g01 + q11 * g11;
  float V00 = -(h00 * q00 + h01 * q01);
  float V01 = -(h00 * q01 + h01 * q11);
  float V11 = -(h10 * q01 + h11 * q11);
  if (v_comp != 0.f) {  // (a literal 0 in the classic instantiations: the block is compiled out)
    // antialiased mode: comp^2 = det_orig / det_blur, so d comp^2 / d cov2d = ((1 - comp^2) conic - eps2d det(conic) I)
    // (gsplat 1.0.0 add_blur_vjp, including its 1e-6 guard on the division by comp)
    const float vs = v_comp * 0.5f / (o.comp + 1e-6f);
    const float om = 1.0f - o.comp * o.comp;
    const float detc = q00 * q11 - q01 * q01;
    V00 += vs * (om * q00 - eps2d * detc);
    V01 += vs * (om * q01);
    V11 += vs * (om * q11 - eps2d * detc);
  }
  // cov2d = J Sc J^T ;  v_Sc = J^T V J ; v_J = 2 V J Sc
  const float* k = st.k;
  float vx, vy, vz;
  float vk00, vk01, vk02, vk10, vk11, vk12, vk20, vk21, vk22;
  if constexpr (CM == kPinhole) {
  float J00 = st.J00, J02 = st.J02, J11 = st.J11, J12 = st.J12;
  // VJ (2x3) = V * J
  float VJ00 = V00 * J00, VJ01 = V01 * J11, VJ02 = V00 * J02 + V01 * J12;
  float VJ10 = V01 * J00, VJ11 = V11 * J11, VJ12 = V01 * J02 + V11 * J12;
  // v_Sc (3x3 symmetric, full matrix gradient) = J^T (V J)
  vk00 = J00 * VJ00; vk01 = J00 * VJ01; vk02 = J00 * VJ02;
  vk10 = J11 * VJ10; vk11 = J11 * VJ11; vk12 = J11 * VJ12;
  vk20 = J02 * VJ00 + J12 * VJ10; vk21 = J02 * VJ01 + J12 * VJ11; vk22 = J02 * VJ02 + J12 * VJ12;
  // v_J = 2 * (V J) Sc   (only the 4 structurally non-zero entries are needed)
  float vJ00 = 2.f * (VJ00 * k[0] + VJ01 * k[1] + VJ02 * k[2]);
  float vJ02 = 2.f * (VJ00 * k[2] + VJ01 * k[4] + VJ02 * k[5]);
  float vJ11 = 2.f * (VJ10 * k[1] + VJ11 * k[3] + VJ12 * k[4]);
  float vJ12 = 2.f * (VJ10 * k[2] + VJ11 * k[4] + VJ12 * k[5]);
  float fx = cam.fx, fy = cam.fy, rz = st.rz, rz2 = st.rz2, rz3 = st.rz2 * st.rz;
  float x = st.x, y = st.y;
  if (v_K != nullptr) {
    // mean2d = (fx x rz + cx, fy y rz + cy); J00 = fx rz; J02 = -fx tx rz^2 depends on fx only while the fov clamp is
    // off (clamped, fx tx = z * 1.3 * 0.5 * width does not); likewise for y
    float vfx = v_m2x * x * rz + vJ00 * rz;
    float vfy = v_m2y * y * rz + vJ11 * rz;
    if (!st.clamp_x) vfx -= vJ02 * st.tx * rz2;
    if (!st.clamp_y) vfy -= vJ12 * st.ty * rz2;
    v_K[0] += vfx;
    v_K[1] += vfy;
    v_K[2] += v_m2x;
    v_K[3] += v_m2y;
  }
  // mean2d = (fx x rz + cx, fy y rz + cy); depth = z
  vx = fx * rz * v_m2x;
  vy = fy * rz * v_m2y;
  vz = -(fx * x * v_m2x + fy * y * v_m2y) * rz2 + v_depth;
  // J00 = fx rz ; J11 = fy rz
  vz += -fx * rz2 * vJ00 - fy * rz2 * vJ11;
  // J02 = -fx tx rz^2 with tx = x (unclamped) or z*lim (clamped)
  if (!st.clamp_x) { vx += -fx * rz2 * vJ02; vz += 2.f * fx * st.tx * rz3 * vJ02; }
  else             { vz += fx * st.tx * rz3 * vJ02; }
  if (!st.clamp_y) { vy += -fy * rz2 * vJ12; vz += 2.f * fy * st.ty * rz3 * vJ12; }
  else             { vz += fy * st.ty * rz3 * vJ12; }
  } else {
    // full 2x3 J (kOrtho: only J00 = fx and J11 = fy, the zeros are literals and compile out)
    const bool ortho = CM == kOrtho;
    const float J00 = st.J00, J11 = st.J11;
    const float J01 = ortho ? 0.f : st.J01, J02 = ortho ? 0.f : st.J02;
    const float J10 = ortho ? 0.f : st.J10, J12 = ortho ? 0.f : st.J12;
    const float VJ00 = V00 * J00 + V01 * J10, VJ01 = V00 * J01 + V01 * J11, VJ02 = V00 * J02 + V01 * J12;
    const float VJ10 = V01 * J00 + V11 * J10, VJ11 = V01 * J01 + V11 * J11, VJ12 = V01 * J02 + V11 * J12;
    vk00 = J00 * VJ00 + J10 * VJ10; vk01 = J00 * VJ01 + J10 * VJ11; vk02 = J00 * VJ02 + J10 * VJ12;
    vk10 = J01 * VJ00 + J11 * VJ10; vk11 = J01 * VJ01 + J11 * VJ11; vk12 = J01 * VJ02 + J11 * VJ12;
    vk20 = J02 * VJ00 + J12 * VJ10; vk21 = J02 * VJ01 + J12 * VJ11; vk22 = J02 * VJ02 + J12 * VJ12;
    // v_J = 2 (V J) Sc, all six entries
    const float vJ00 = 2.f * (VJ00 * k[0] + VJ01 * k[1] + VJ02 * k[2]);
    const float vJ01 = 2.f * (VJ00 * k[1] + VJ01 * k[3] + VJ02 * k[4]);
    const float vJ02 = 2.f * (VJ00 * k[2] + VJ01 * k[4] + VJ02 * k[5]);
    const float vJ10 = 2.f * (VJ10 * k[0] + VJ11 * k[1] + VJ12 * k[2]);
    const float vJ11 = 2.f * (VJ10 * k[1] + VJ11 * k[3] + VJ12 * k[4]);
    const float vJ12 = 2.f * (VJ10 * k[2] + VJ11 * k[4] + VJ12 * k[5]);
    const float fx = cam.fx, fy = cam.fy, x = st.x, y = st.y;
    if constexpr (CM == kOrtho) {
      // mean2d = (fx x + cx, fy y + cy), J constant in (x, y, z); depth = z
      if (v_K != nullptr) {
        v_K[0] += v_m2x * x + vJ00;
        v_K[1] += v_m2y * y + vJ11;
        v_K[2] += v_m2x;
        v_K[3] += v_m2y;
      }
      vx = fx * v_m2x;
      vy = fy * v_m2y;
      vz = v_depth;
    } else {
      // J is the Jacobian of mean2d, so mean2d contributes J^T v_m2.  With s = theta / r, g = (1/r) ds/dr,
      // q = 1 / (r^2 + z^2) and G = (1/r) dg/dr = (-2 z q^2 - 3 g) / r^2:  ds/d(x, y, z) = (x g, y g, -q),
      // dg/d(x, y, z) = (x G, y G, 2 q^2), dq/d(x, y, z) = -2 q^2 (x, y, z).  sum_ij vJ_ij J_ij is
      //   Phi = A0 (s + x^2 g) + A1 x y g + A2 (s + y^2 g) - (B0 x + B1 y) q
      // with A0 = fx vJ00, A1 = fx vJ01 + fy vJ10, A2 = fy vJ11, B0 = fx vJ02, B1 = fy vJ12, and its gradient is
      //   dPhi/dx = g ((3 A0 + A2) x + A1 y) + x Qf G - B0 q + 2 q^2 x L
      //   dPhi/dy = g ((A0 + 3 A2) y + A1 x) + y Qf G - B1 q + 2 q^2 y L
      //   dPhi/dz = -q (A0 + A2) + 2 q^2 Qf + 2 z q^2 L,    Qf = A0 x^2 + A1 x y + A2 y^2, L = B0 x + B1 y.
      // Qf G is evaluated as (-2 z q^2 - 3 g) (Qf / r^2): Qf / r^2 is bounded, and the cancellation in the bracket
      // is then scaled by |x| <= r, so no term loses precision as r -> 0 (r = 0: Qf / r^2 = 0).
      const float s = st.fs, g = st.fg, q = st.fq, r2 = st.r2, z = st.z;
      if (v_K != nullptr) {
        v_K[0] += v_m2x * (x * s) + ((vJ00 * (s + (x * x) * g) + vJ01 * ((x * y) * g)) - vJ02 * (x * q));
        v_K[1] += v_m2y * (y * s) + ((vJ10 * ((x * y) * g) + vJ11 * (s + (y * y) * g)) - vJ12 * (y * q));
        v_K[2] += v_m2x;
        v_K[3] += v_m2y;
      }
      const float A0 = fx * vJ00, A1 = fx * vJ01 + fy * vJ10, A2 = fy * vJ11, B0 = fx * vJ02, B1 = fy * vJ12;
      const float Qf = A0 * (x * x) + A1 * (x * y) + A2 * (y * y);
      const float L = B0 * x + B1 * y;
      const float q2 = q * q;
      const float QG = (-2.f * z * q2 - 3.f * g) * (r2 > 0.f ? Qf / r2 : 0.f);
      vx = J00 * v_m2x + J10 * v_m2y + g * ((3.f * A0 + A2) * x + A1 * y) + x * QG - B0 * q + 2.f * q2 * x * L;
      vy = J01 * v_m2x + J11 * v_m2y + g * ((A0 + 3.f * A2) * y + A1 * x) + y * QG - B1 * q + 2.f * q2 * y * L;
      vz = J02 * v_m2x + J12 * v_m2y + v_depth - q * (A0 + A2) + 2.f * q2 * Qf + 2.f * z * q2 * L;
    }
  }
  // camera -> world
  const float* W = cam.r;
  v_mean[0] += W[0] * vx + W[3] * vy + W[6] * vz;
  v_mean[1] += W[1] * vx + W[4] * vy + W[7] * vz;
  v_mean[2] += W[2] * vx + W[5] * vy + W[8] * vz;
  // v_Sigma = W^T v_Sc W
  float vkm[9] = {vk00, vk01, vk02, vk10, vk11, vk12, vk20, vk21, vk22};
  if (v_cam != nullptr) {
    // mean_c = W m + t: v_W += v_mean_c m^T, v_t += v_mean_c
    const float vc[3] = {vx, vy, vz};
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
      for (int j = 0; j < 3; ++j) v_cam[i * 3 + j] += vc[i] * mean[j];
      v_cam[9 + i] += vc[i];
    }
    // cov_c = W Sigma W^T: v_W += (v_Sc + v_Sc^T) W Sigma
    const float* S = st.S;
    const float Sm[9] = {S[0], S[1], S[2], S[1], S[3], S[4], S[2], S[4], S[5]};
    float WS[9];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j)
        WS[i * 3 + j] = W[i * 3 + 0] * Sm[0 * 3 + j] + W[i * 3 + 1] * Sm[1 * 3 + j] + W[i * 3 + 2] * Sm[2 * 3 + j];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j)
        v_cam[i * 3 + j] += (vkm[i * 3 + 0] + vkm[0 * 3 + i]) * WS[0 * 3 + j] +
                            (vkm[i * 3 + 1] + vkm[1 * 3 + i]) * WS[1 * 3 + j] +
                            (vkm[i * 3 + 2] + vkm[2 * 3 + i]) * WS[2 * 3 + j];
  }
  float Tm[9];  // Tm = vSc * W
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j)
      Tm[i * 3 + j] = vkm[i * 3 + 0] * W[0 * 3 + j] + vkm[i * 3 + 1] * W[1 * 3 + j] + vkm[i * 3 + 2] * W[2 * 3 + j];
  float vS[9];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j)
      vS[i * 3 + j] = W[0 * 3 + i] * Tm[0 * 3 + j] + W[1 * 3 + i] * Tm[1 * 3 + j] + W[2 * 3 + i] * Tm[2 * 3 + j];
  // Sigma = M M^T : v_M = (vS + vS^T) M
  const float* M = st.M;
  float vM[9];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j)
      vM[i * 3 + j] = (vS[i * 3 + 0] + vS[0 * 3 + i]) * M[0 * 3 + j] + (vS[i * 3 + 1] + vS[1 * 3 + i]) * M[1 * 3 + j] +
                      (vS[i * 3 + 2] + vS[2 * 3 + i]) * M[2 * 3 + j];
  // M = R diag(s)
  const float* R = st.R;
  float vR[9];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) vR[i * 3 + j] = vM[i * 3 + j] * scale[j];
  v_scale[0] += R[0] * vM[0] + R[3] * vM[3] + R[6] * vM[6];
  v_scale[1] += R[1] * vM[1] + R[4] * vM[4] + R[7] * vM[7];
  v_scale[2] += R[2] * vM[2] + R[5] * vM[5] + R[8] * vM[8];
  // rotation -> normalised quaternion -> raw quaternion
  float w = st.qn[0], qx = st.qn[1], qy = st.qn[2], qz = st.qn[3];
  float vqw = 2.f * (qx * (vR[7] - vR[5]) + qy * (vR[2] - vR[6]) + qz * (vR[3] - vR[1]));
  float vqx = 2.f * (-2.f * qx * (vR[4] + vR[8]) + qy * (vR[1] + vR[3]) + qz * (vR[2] + vR[6]) + w * (vR[7] - vR[5]));
  float vqy = 2.f * (qx * (vR[1] + vR[3]) - 2.f * qy * (vR[0] + vR[8]) + qz * (vR[5] + vR[7]) + w * (vR[2] - vR[6]));
  float vqz = 2.f * (qx * (vR[2] + vR[6]) + qy * (vR[5] + vR[7]) - 2.f * qz * (vR[0] + vR[4]) + w * (vR[3] - vR[1]));
  float dotp = vqw * w + vqx * qx + vqy * qy + vqz * qz;
  v_quat[0] += (vqw - dotp * w) * st.inv_norm;
  v_quat[1] += (vqx - dotp * qx) * st.inv_norm;
  v_quat[2] += (vqy - dotp * qy) * st.inv_norm;
  v_quat[3] += (vqz - dotp * qz) * st.inv_norm;
}

// ---- spherical harmonics, degrees 0..3 (SURVEY.md A-2) -----------------------------------------

#define EGS_SH_C0 0.2820947917738781f
#define EGS_SH_C1 0.48860251190292f

// basis values for a normalised direction
EGS_HD void sh_basis(int degree, float x, float y, float z, float Y[16]) {
  Y[0] = EGS_SH_C0;
  if (degree < 1) return;
  Y[1] = -EGS_SH_C1 * y; Y[2] = EGS_SH_C1 * z; Y[3] = -EGS_SH_C1 * x;
  if (degree < 2) return;
  float z2 = z * z;
  float fTmp0B = -1.092548430592079f * z;
  float fC1 = x * x - y * y;
  float fS1 = 2.f * x * y;
  Y[4] = 0.5462742152960395f * fS1;
  Y[5] = fTmp0B * y;
  Y[6] = 0.9461746957575601f * z2 - 0.3153915652525201f;
  Y[7] = fTmp0B * x;
  Y[8] = 0.5462742152960395f * fC1;
  if (degree < 3) return;
  float fTmp0C = -2.285228997322329f * z2 + 0.4570457994644658f;
  float fTmp1B = 1.445305721320277f * z;
  float fC2 = x * fC1 - y * fS1;
  float fS2 = x * fS1 + y * fC1;
  Y[9] = -0.5900435899266435f * fS2;
  Y[10] = fTmp1B * fS1;
  Y[11] = fTmp0C * y;
  Y[12] = z * (1.865881662950577f * z2 - 1.119528997770346f);
  Y[13] = fTmp0C * x;
  Y[14] = fTmp1B * fC1;
  Y[15] = -0.5900435899266435f * fC2;
}

// d(sum_k g[k] * Y_k)/d(x,y,z) for a normalised direction; g[k] = sum_ch coeff[k][ch] * v_rgb[ch]
EGS_HD void sh_basis_vjp(int degree, float x, float y, float z, const float g[16], float& vx, float& vy, float& vz) {
  vx = 0.f; vy = 0.f; vz = 0.f;
  if (degree < 1) return;
  vx += -EGS_SH_C1 * g[3]; vy += -EGS_SH_C1 * g[1]; vz += EGS_SH_C1 * g[2];
  if (degree < 2) return;
  float z2 = z * z;
  float fTmp0B = -1.092548430592079f * z;
  float fC1 = x * x - y * y;
  float fS1 = 2.f * x * y;
  const float k2 = 0.5462742152960395f;
  vx += g[4] * (k2 * 2.f * y) + g[7] * fTmp0B + g[8] * (k2 * 2.f * x);
  vy += g[4] * (k2 * 2.f * x) + g[5] * fTmp0B - g[8] * (k2 * 2.f * y);
  vz += g[5] * (-1.092548430592079f * y) + g[6] * (2.f * 0.9461746957575601f * z) + g[7] * (-1.092548430592079f * x);
  if (degree < 3) return;
  float fTmp0C = -2.285228997322329f * z2 + 0.4570457994644658f;
  float fTmp1B = 1.445305721320277f * z;
  const float k3 = 0.5900435899266435f;
  const float dTmp0C = -2.f * 2.285228997322329f * z;  // d fTmp0C / dz
  vx += g[9] * (-k3 * 3.f * fS1) + g[10] * (fTmp1B * 2.f * y) + g[13] * fTmp0C + g[14] * (fTmp1B * 2.f * x) +
        g[15] * (-k3 * 3.f * fC1);
  vy += g[9] * (-k3 * 3.f * fC1) + g[10] * (fTmp1B * 2.f * x) + g[11] * fTmp0C - g[14] * (fTmp1B * 2.f * y) +
        g[15] * (k3 * 3.f * fS1);
  vz += g[10] * (1.445305721320277f * fS1) + g[11] * (dTmp0C * y) +
        g[12] * (3.f * 1.865881662950577f * z2 - 1.119528997770346f) + g[13] * (dTmp0C * x) +
        g[14] * (1.445305721320277f * fC1);
}

// SH colour of one Gaussian for one camera: rgb = max(sum_k Y_k(dir) c_k + 0.5, 0), dir = mean - campos
// (the gsplat glue `dirs = means - camtoworlds[:3,3]`, `clamp_min(colors + 0.5, 0)`).
// co holds the first (degree+1)^2 coefficient rows, [k][channel].
EGS_HD void sh_color_fwd(int degree, const float mean[3], const Camera& cam, const float (&co)[48], float rgb[3]) {
  const int nb = (degree + 1) * (degree + 1);
  float dx = mean[0] - cam.campos[0], dy = mean[1] - cam.campos[1], dz = mean[2] - cam.campos[2];
  float inorm = 1.0f / sqrtf(dx * dx + dy * dy + dz * dz);
  float Y[16];
  sh_basis(degree, dx * inorm, dy * inorm, dz * inorm, Y);
  float r = 0.f, g = 0.f, b = 0.f;
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    if (k < nb) {
      r += Y[k] * co[3 * k + 0];
      g += Y[k] * co[3 * k + 1];
      b += Y[k] * co[3 * k + 2];
    }
  }
  rgb[0] = fmaxf(r + 0.5f, 0.f);
  rgb[1] = fmaxf(g + 0.5f, 0.f);
  rgb[2] = fmaxf(b + 0.5f, 0.f);
}

// VJP of sh_color_fwd.  rgb_stored is the forward output (gradient passes where it is > 0).
// Accumulates (+=) into vco[48] and v_mean[3].  v_cam (nullable): dir = mean - campos, so the direction gradient is
// also subtracted from v_campos (entries 12..14 of the camera gradient, see project_bwd).
EGS_HD void sh_color_bwd(int degree, const float mean[3], const Camera& cam, const float (&co)[48],
                         const float rgb_stored[3], const float v_rgb_in[3], float (&vco)[48], float v_mean[3],
                         float* v_cam = nullptr) {
  const int nb = (degree + 1) * (degree + 1);
  float v_rgb[3];
  v_rgb[0] = (rgb_stored[0] > 0.f) ? v_rgb_in[0] : 0.f;
  v_rgb[1] = (rgb_stored[1] > 0.f) ? v_rgb_in[1] : 0.f;
  v_rgb[2] = (rgb_stored[2] > 0.f) ? v_rgb_in[2] : 0.f;
  float dx = mean[0] - cam.campos[0], dy = mean[1] - cam.campos[1], dz = mean[2] - cam.campos[2];
  float inorm = 1.0f / sqrtf(dx * dx + dy * dy + dz * dz);
  float x = dx * inorm, y = dy * inorm, z = dz * inorm;
  float Y[16];
  sh_basis(degree, x, y, z, Y);
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    if (k < nb) {
      vco[3 * k + 0] += Y[k] * v_rgb[0];
      vco[3 * k + 1] += Y[k] * v_rgb[1];
      vco[3 * k + 2] += Y[k] * v_rgb[2];
    }
  }
  if (degree >= 1) {
    float g[16];
#pragma unroll
    for (int k = 0; k < 16; ++k)
      g[k] = (k < nb) ? (co[3 * k + 0] * v_rgb[0] + co[3 * k + 1] * v_rgb[1] + co[3 * k + 2] * v_rgb[2]) : 0.f;
    float vx, vy, vz;
    sh_basis_vjp(degree, x, y, z, g, vx, vy, vz);
    float dp = vx * x + vy * y + vz * z;
    const float d0 = (vx - dp * x) * inorm, d1 = (vy - dp * y) * inorm, d2 = (vz - dp * z) * inorm;
    v_mean[0] += d0;
    v_mean[1] += d1;
    v_mean[2] += d2;
    if (v_cam != nullptr) { v_cam[12] -= d0; v_cam[13] -= d1; v_cam[14] -= d2; }
  }
}

// ---- spherical harmonics, degree 4: 25 bands ------------------------------------------------------
// Bands 0..3 are sh_basis / sh_basis_vjp / sh_color_fwd / sh_color_bwd at degree 3, term for term and in the same
// order, and band 4 is added after them: with zero band-4 coefficients the results equal degree 3's bit for bit.
// Band 4 is the real SH basis of the lower bands' convention (sqrt(2) Re / Im of Y_4^|m| with the Condon-Shortley
// phase, m = -4..4), written with fCm / fSm = Re / Im (x + iy)^(m+1) as in sh_basis.
constexpr int kSh4Bands = 25;

EGS_HD void sh_basis4(float x, float y, float z, float Y[kSh4Bands]) {
  sh_basis(3, x, y, z, Y);
  float z2 = z * z;
  float fC1 = x * x - y * y;
  float fS1 = 2.f * x * y;
  float fC2 = x * fC1 - y * fS1;
  float fS2 = x * fS1 + y * fC1;
  float fC3 = x * fC2 - y * fS2;
  float fS3 = x * fS2 + y * fC2;
  float fTmp0D = 3.31161143515146f * z2 - 0.47308734787878f;
  float fTmp1C = z * (-4.683325804901025f * z2 + 2.007139630671868f);
  float fTmp2B = -1.770130769779931f * z;
  Y[16] = 0.6258357354491763f * fS3;
  Y[17] = fTmp2B * fS2;
  Y[18] = fTmp0D * fS1;
  Y[19] = fTmp1C * y;
  Y[20] = 1.984313483298443f * z * Y[12] - 1.006230589874905f * Y[6];
  Y[21] = fTmp1C * x;
  Y[22] = fTmp0D * fC1;
  Y[23] = fTmp2B * fC2;
  Y[24] = 0.6258357354491763f * fC3;
}

// d(sum_k g[k] * Y_k)/d(x,y,z) of sh_basis4.  d(fCm, fSm)/dx = (m+1) (fC(m-1), fS(m-1)), d/dy = (m+1) (-fS(m-1), fC(m-1)).
EGS_HD void sh_basis4_vjp(float x, float y, float z, const float g[kSh4Bands], float& vx, float& vy, float& vz) {
  sh_basis_vjp(3, x, y, z, g, vx, vy, vz);
  float z2 = z * z;
  float fC1 = x * x - y * y;
  float fS1 = 2.f * x * y;
  float fC2 = x * fC1 - y * fS1;
  float fS2 = x * fS1 + y * fC1;
  float fTmp0D = 3.31161143515146f * z2 - 0.47308734787878f;
  float fTmp1C = z * (-4.683325804901025f * z2 + 2.007139630671868f);
  float fTmp2B = -1.770130769779931f * z;
  const float k4 = 0.6258357354491763f;
  const float dTmp1C = -3.f * 4.683325804901025f * z2 + 2.007139630671868f;  // d fTmp1C / dz
  // d Y20 / dz with Y6 = 0.946.. z^2 - 0.315.. and Y12 = z (1.865.. z^2 - 1.119..)
  const float dY20 = 1.984313483298443f * (z * (3.f * 1.865881662950577f * z2 - 1.119528997770346f) +
                                           z * (1.865881662950577f * z2 - 1.119528997770346f)) -
                     1.006230589874905f * (2.f * 0.9461746957575601f * z);
  vx += g[16] * (k4 * 4.f * fS2) + g[17] * (fTmp2B * 3.f * fS1) + g[18] * (fTmp0D * 2.f * y) + g[21] * fTmp1C +
        g[22] * (fTmp0D * 2.f * x) + g[23] * (fTmp2B * 3.f * fC1) + g[24] * (k4 * 4.f * fC2);
  vy += g[16] * (k4 * 4.f * fC2) + g[17] * (fTmp2B * 3.f * fC1) + g[18] * (fTmp0D * 2.f * x) + g[19] * fTmp1C -
        g[22] * (fTmp0D * 2.f * y) - g[23] * (fTmp2B * 3.f * fS1) - g[24] * (k4 * 4.f * fS2);
  vz += g[17] * (-1.770130769779931f * fS2) + g[18] * (2.f * 3.31161143515146f * z * fS1) + g[19] * (dTmp1C * y) +
        g[20] * dY20 + g[21] * (dTmp1C * x) + g[22] * (2.f * 3.31161143515146f * z * fC1) +
        g[23] * (-1.770130769779931f * fC2);
}

// sh_color_fwd at degree 4.  co: the first 25 coefficient rows, [k][channel] (75 floats; shared memory in the kernels).
EGS_HD void sh4_color_fwd(const float mean[3], const Camera& cam, const float* co, float rgb[3]) {
  float dx = mean[0] - cam.campos[0], dy = mean[1] - cam.campos[1], dz = mean[2] - cam.campos[2];
  float inorm = 1.0f / sqrtf(dx * dx + dy * dy + dz * dz);
  float Y[kSh4Bands];
  sh_basis4(dx * inorm, dy * inorm, dz * inorm, Y);
  float r = 0.f, g = 0.f, b = 0.f;
#pragma unroll
  for (int k = 0; k < kSh4Bands; ++k) {
    r += Y[k] * co[3 * k + 0];
    g += Y[k] * co[3 * k + 1];
    b += Y[k] * co[3 * k + 2];
  }
  rgb[0] = fmaxf(r + 0.5f, 0.f);
  rgb[1] = fmaxf(g + 0.5f, 0.f);
  rgb[2] = fmaxf(b + 0.5f, 0.f);
}

// sh_color_bwd at degree 4: accumulates (+=) into vco (75 floats) and v_mean[3]; v_cam (nullable) as in sh_color_bwd.
EGS_HD void sh4_color_bwd(const float mean[3], const Camera& cam, const float* co, const float rgb_stored[3],
                          const float v_rgb_in[3], float* vco, float v_mean[3], float* v_cam = nullptr) {
  float v_rgb[3];
  v_rgb[0] = (rgb_stored[0] > 0.f) ? v_rgb_in[0] : 0.f;
  v_rgb[1] = (rgb_stored[1] > 0.f) ? v_rgb_in[1] : 0.f;
  v_rgb[2] = (rgb_stored[2] > 0.f) ? v_rgb_in[2] : 0.f;
  float dx = mean[0] - cam.campos[0], dy = mean[1] - cam.campos[1], dz = mean[2] - cam.campos[2];
  float inorm = 1.0f / sqrtf(dx * dx + dy * dy + dz * dz);
  float x = dx * inorm, y = dy * inorm, z = dz * inorm;
  float Y[kSh4Bands], g[kSh4Bands];
  sh_basis4(x, y, z, Y);
#pragma unroll
  for (int k = 0; k < kSh4Bands; ++k) {
    vco[3 * k + 0] += Y[k] * v_rgb[0];
    vco[3 * k + 1] += Y[k] * v_rgb[1];
    vco[3 * k + 2] += Y[k] * v_rgb[2];
    g[k] = co[3 * k + 0] * v_rgb[0] + co[3 * k + 1] * v_rgb[1] + co[3 * k + 2] * v_rgb[2];
  }
  float vx, vy, vz;
  sh_basis4_vjp(x, y, z, g, vx, vy, vz);
  float dp = vx * x + vy * y + vz * z;
  const float d0 = (vx - dp * x) * inorm, d1 = (vy - dp * y) * inorm, d2 = (vz - dp * z) * inorm;
  v_mean[0] += d0;
  v_mean[1] += d1;
  v_mean[2] += d2;
  if (v_cam != nullptr) { v_cam[12] -= d0; v_cam[13] -= d1; v_cam[14] -= d2; }
}

// The [4,4] gradient of one view matrix V from its camera gradient summed over the Gaussians (v_R, v_t, g = v_campos,
// see project_bwd).  campos = inv(V)[:3,3] with inv(V) = [[A, c], [0, 1]] (A = R^-1 by the same adjugate as
// load_camera, c = campos), and the VJP of a matrix inverse is -inv(V)^T G inv(V)^T with g in column 3 of G:
//   v_V = [[v_R, v_t], [0, 0]] - [[(A^T g) c^T, A^T g], [(c.g) c^T, c.g]]
// The bottom row is not zero when the SH directions carry a gradient, as in gsplat.
EGS_HD void viewmat_grad_finalize(const float* V, const float vcam[kCamGradFloats], float out[16]) {
  const float r[9] = {V[0], V[1], V[2], V[4], V[5], V[6], V[8], V[9], V[10]};
  const float t[3] = {V[3], V[7], V[11]};
  float a[9];
  a[0] = r[4] * r[8] - r[5] * r[7];
  a[1] = r[2] * r[7] - r[1] * r[8];
  a[2] = r[1] * r[5] - r[2] * r[4];
  a[3] = r[5] * r[6] - r[3] * r[8];
  a[4] = r[0] * r[8] - r[2] * r[6];
  a[5] = r[2] * r[3] - r[0] * r[5];
  a[6] = r[3] * r[7] - r[4] * r[6];
  a[7] = r[1] * r[6] - r[0] * r[7];
  a[8] = r[0] * r[4] - r[1] * r[3];
  const float det = r[0] * a[0] + r[1] * a[3] + r[2] * a[6];
  const float id = 1.0f / det;
  float c[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) c[i] = -(a[i * 3 + 0] * t[0] + a[i * 3 + 1] * t[1] + a[i * 3 + 2] * t[2]) * id;
  const float* g = vcam + 12;
  float Atg[3];  // A^T g, A = a * id
#pragma unroll
  for (int i = 0; i < 3; ++i) Atg[i] = (a[0 * 3 + i] * g[0] + a[1 * 3 + i] * g[1] + a[2 * 3 + i] * g[2]) * id;
  const float cg = c[0] * g[0] + c[1] * g[1] + c[2] * g[2];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
#pragma unroll
    for (int j = 0; j < 3; ++j) out[i * 4 + j] = vcam[i * 3 + j] - Atg[i] * c[j];
    out[i * 4 + 3] = vcam[9 + i] - Atg[i];
    out[12 + i] = -(cg * c[i]);
  }
  out[15] = -cg;
}

// The [3,3] gradient of one K from its intrinsics gradient summed over the Gaussians (v_fx, v_fy, v_cx, v_cy, see
// project_bwd).  The projection reads no other entry, so the skew and the last row get 0.
EGS_HD void ks_grad_finalize(const float vk[kKsGradFloats], float out[9]) {
  out[0] = vk[0]; out[1] = 0.f;   out[2] = vk[2];
  out[3] = 0.f;   out[4] = vk[1]; out[5] = vk[3];
  out[6] = 0.f;   out[7] = 0.f;   out[8] = 0.f;
}

}  // namespace egs
