// g6 / g7: alpha blending forward and backward (takes the place of gsplat's
// rasterize_to_pixels fwd/bwd).  FP32 SIMT + MUFU bound (SURVEY.md §8d); no dense contraction, so
// no tensor cores.
//
// Work decomposition.  One CTA (2 warps) per 16x16 pixel tile; each WARP owns a 16x8 pixel half of
// the tile and runs on its own (there is no block-level barrier in either kernel); each lane owns a
// 2x2 pixel block, so shared-memory reads, loop overhead, the separable parts of the quadratic form
// and — in the backward pass — the warp reduction are amortised over 4 pixels.
//
// Staging + exact culling.  A warp walks the tile's depth-sorted intersection list in batches of 64
// packed 48-byte splat records, copied with cp.async (LDGSTS.128 x3 per record, double buffered, the
// flatten ids of the batch after next prefetched into registers).  The binning that produced the list
// is deliberately coarse (3-sigma bounding SQUARE of the major axis vs 16x16 tiles — it has to be, to
// stay bit-identical with gsplat's lists), so before a batch is blended every lane tests its two records
// against the warp's pixel rectangle: the minimum of sigma over the rectangle (closed form: centre
// inside, else the best point of the four edges) is compared with sigma_cut = ln(255 o), beyond which
// alpha < 1/255 for every pixel of the warp.  Survivors are compacted, in order, into a slot list
// (ballot + popc); the blend loop only visits survivors.  On the 1M-Gaussian benchmark scene ~47 % of the
// (tile, Gaussian) pairs fail this test.  Results are unchanged: a culled Gaussian contributes to no pixel.
//
// Loops over a batch are WARP-UNIFORM (finished pixels are predicated off, a vote at the top of the
// body is the reconvergence point).  A per-lane break/continue lets the lanes of a warp drift apart
// under independent thread scheduling: measured with ncu on the first version of the forward kernel,
// 1.9 active threads per instruction and a 20x slowdown (profiles/r1a_*).
//
// Packed fp32.  Both kernels are issue bound (ncu: 80 % issue-active, FMA pipe 40 % before this change), so in
// the 2x2 layout the two pixels of a row share FADD2 / FMUL2 / FFMA2 instructions (sm_100) and the per-pixel
// updates are branch free: a pixel that does not take part blends with weight 0.
//
// Backward: per-pixel back-to-front replay from the warp's own last blended index; the 11 (12 with depth) per-Gaussian
// partial gradients are summed over the lane's 4 pixels in registers, then over the warp through a 1.6 KB
// shared-memory scratch (11 conflict-free row stores, 4 LDS.128 + a packed add tree per lane, one shuffle), and
// 11 lanes issue one coalesced RED.ADD.F32 into the packed 48-byte gradient record of the Gaussian.
#include <stdlib.h>

#include "egs_common.cuh"

namespace egs {

constexpr int kTileSize = 16;
// Resident CTAs per SM the compiler must leave room for (register cap = 65536 / (threads * this)); tuning knobs,
// overridable at build time for A/B runs (scripts/build_variant.py).
#ifdef EGS_FWD_MIN_CTAS
#define EGS_FWD_BOUNDS(T) __launch_bounds__(T, EGS_FWD_MIN_CTAS)
#else
#define EGS_FWD_BOUNDS(T) __launch_bounds__(T)
#endif
#ifdef EGS_BWD_MIN_CTAS
#define EGS_BWD_BOUNDS(T) __launch_bounds__(T, EGS_BWD_MIN_CTAS)
#else
#define EGS_BWD_BOUNDS(T) __launch_bounds__(T)
#endif
// A lane owns PX x PY pixels, a warp 8 x 4 lanes = (8 PX) x (4 PY) pixels.  <2,2>: 2 warps of 16x8 pixels per
// tile — the RGB kernels and the feature kernels up to 8 channels.  <1,1>: 8 warps of 8x4 pixels per tile, one
// pixel per lane — the 16- and 32-channel feature kernels, whose per-lane colour state would not fit 4 pixels.
template <int PX, int PY>
struct Geo {
  static constexpr int NP = PX * PY;
  static constexpr int kWarpW = 8 * PX, kWarpH = 4 * PY;
  static constexpr int kWarpsX = kTileSize / kWarpW, kWarpsY = kTileSize / kWarpH;
  static constexpr int kWarps = kWarpsX * kWarpsY;
  static constexpr int kThreads = 32 * kWarps;
  // records staged per warp per batch: 2 per lane for the 2-warp layout, 1 per lane for the 8-warp layout
  // (keeps the CTA's static shared memory under 48 KB)
  static constexpr int RPL = kWarps <= 2 ? 2 : 1;
  static constexpr int kBatch = 32 * RPL;
};
constexpr float kAlphaMin = 1.0f / 255.0f;
constexpr float kAlphaMax = 0.999f;
constexpr float kTMin = 1e-4f;
constexpr float kNegLog2e = -1.4426950408889634f;
constexpr int kGradValues = 11;  // floats of the packed gradient record that the backward blend produces
constexpr int kRedStride = 36;   // words per row of the backward kernel's warp-sum scratch (32 lanes + 4: conflict-free LDS.128)

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ex2 of an argument that is already scaled by -log2(e) (flush-to-zero: anything that small is rejected)
__device__ __forceinline__ float fast_ex2(float x) {
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x));
  return e;
}
// 1/x as a single MUFU.RCP (the operands here are never denormal: 1 - alpha >= 1e-3, opacity >= 1/255, conic
// diagonals of visible splats; the fast-division intrinsic would add 4 range-fixup instructions around it)
__device__ __forceinline__ float fast_rcp(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ void sts_f32(uint32_t addr, float v) {
  asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
// predicated RED.ADD.F32 on a known-global address (no branch, no reconvergence barrier around it)
__device__ __forceinline__ void red_add_f32_if(int flag, float* gptr, float v) {
  asm volatile("{ .reg .pred p; setp.ne.s32 p, %0, 0; @p red.global.add.f32 [%1], %2; }" ::"r"(flag), "l"(gptr), "f"(v) : "memory");
}
// Stops ptxas from re-deriving a loop-invariant value inside the loop (it otherwise rematerialises
// the pixel-centre coordinates with I2FP + FADD in every iteration to save two registers).
__device__ __forceinline__ float opaque(float x) {
  asm volatile("" : "+f"(x));
  return x;
}

// Per-warp shared memory: raw double-buffered batches, their flatten ids, and the survivor slot list.
template <int kBatch>
struct WarpStage {
  float4 rec[2][kBatch * 3];
  int id[2][kBatch];
  int list[kBatch];
};

struct WarpView {
  int cam, x0, y0;               // first pixel of this lane's block
  int range_start, range_end;    // the tile's slice of the sorted intersection list
  float2 npx2, npy2;             // minus the pixel centres of the block's first / last column, first / last row
  float rx_lo, rx_hi, ry_lo, ry_hi;  // pixel-centre rectangle of the warp
};

// The block's tile: the given flat tile index (cam * tile_h + ty) * tile_w + tx when tile_id >= 0 (the segment launch
// of the backward pass maps blocks to list segments), else tile_order[block] when tile_order is given (longest lists
// first, egs_isect_sorted), else the block's position in the (tile_w, tile_h, C) grid.
template <class G>
__device__ __forceinline__ WarpView warp_setup(int tile_w, int tile_h, int64_t n_isects,
                                               const int32_t* __restrict__ tile_offsets, int n_tiles_total,
                                               const int32_t* __restrict__ tile_order, int tile_id = -1) {
  constexpr int PX = G::kWarpW / 8, PY = G::kWarpH / 4;
  WarpView v;
  if (tile_id < 0 && tile_order != nullptr)
    tile_id = tile_order[(blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x];
  int bx = blockIdx.x, by = blockIdx.y;
  v.cam = blockIdx.z;
  if (tile_id < 0) {
    tile_id = (v.cam * tile_h + by) * tile_w + bx;
  } else {
    v.cam = tile_id / (tile_w * tile_h);
    const int rem = tile_id - v.cam * (tile_w * tile_h);
    by = rem / tile_w;
    bx = rem - by * tile_w;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int wx = warp % G::kWarpsX, wy = warp / G::kWarpsX;
  const int wx0 = bx * kTileSize + wx * G::kWarpW, wy0 = by * kTileSize + wy * G::kWarpH;
  v.x0 = wx0 + (lane & 7) * PX;
  v.y0 = wy0 + (lane >> 3) * PY;
  v.range_start = tile_offsets[tile_id];
  // n_isects < 0: the offsets carry a sentinel entry behind the last tile (the live list length, written on the
  // device by egs_isect_sorted); otherwise the last tile ends at n_isects
  v.range_end = (tile_id == n_tiles_total - 1 && n_isects >= 0) ? (int)n_isects : tile_offsets[tile_id + 1];
  float pxf[PX], pyf[PY];
#pragma unroll
  for (int i = 0; i < PX; ++i) pxf[i] = opaque((float)(v.x0 + i) + 0.5f);
#pragma unroll
  for (int i = 0; i < PY; ++i) pyf[i] = opaque((float)(v.y0 + i) + 0.5f);
  v.npx2 = make_float2(-pxf[0], -pxf[PX - 1]);
  v.npy2 = make_float2(-pyf[0], -pyf[PY - 1]);
  const float rx_lo = (float)wx0 + 0.5f, ry_lo = (float)wy0 + 0.5f;
  v.rx_lo = opaque(rx_lo);
  v.rx_hi = opaque(rx_lo + (float)(G::kWarpW - 1));
  v.ry_lo = opaque(ry_lo);
  v.ry_hi = opaque(ry_lo + (float)(G::kWarpH - 1));
  return v;
}

// Can alpha reach 1/255 anywhere in the rectangle?  min over the rectangle of
// sigma(d) = 0.5 (a dx^2 + c dy^2) + b dx dy  (d = pixel - mean) against sigma_cut.
__device__ __forceinline__ bool splat_touches_rect(const float4 g0, const float4 g1, float sigma_cut, float rx_lo,
                                                   float rx_hi, float ry_lo, float ry_hi) {
  if (!(sigma_cut > 0.f)) return false;
  const float a = g0.z, b = g0.w, c = g1.x;
  const float dxl = rx_lo - g0.x, dxh = rx_hi - g0.x, dyl = ry_lo - g0.y, dyh = ry_hi - g0.y;
  if (dxl <= 0.f && dxh >= 0.f && dyl <= 0.f && dyh >= 0.f) return true;  // centre inside
  const float nb_c = -b * fast_rcp(c), nb_a = -b * fast_rcp(a);
  float best;
  {
    const float dy = fminf(fmaxf(nb_c * dxl, dyl), dyh);
    best = 0.5f * (a * dxl * dxl + c * dy * dy) + b * dxl * dy;
  }
  {
    const float dy = fminf(fmaxf(nb_c * dxh, dyl), dyh);
    best = fminf(best, 0.5f * (a * dxh * dxh + c * dy * dy) + b * dxh * dy);
  }
  {
    const float dx = fminf(fmaxf(nb_a * dyl, dxl), dxh);
    best = fminf(best, 0.5f * (a * dx * dx + c * dyl * dyl) + b * dx * dyl);
  }
  {
    const float dx = fminf(fmaxf(nb_a * dyh, dxl), dxh);
    best = fminf(best, 0.5f * (a * dx * dx + c * dyh * dyh) + b * dx * dyh);
  }
  return best <= sigma_cut;  // NaN (degenerate conic) compares false -> culled; such a splat has NaN alpha anyway
}

// Tests this lane's RPL records of raw batch `buf` (record slots lane, lane+32, ...), writes the survivor
// slots, in order, to st.list and returns the number of survivors (warp-uniform).
template <int RPL>
__device__ __forceinline__ int cull_and_compact(WarpStage<32 * RPL>& st, int buf, int batch_size, int lane,
                                                const WarpView& wv) {
  bool keep[RPL];
#pragma unroll
  for (int r = 0; r < RPL; ++r) {
    const int slot = r * 32 + lane;
    keep[r] = false;
    if (slot < batch_size) {
      const float4 g0 = st.rec[buf][slot * 3 + 0];
      const float4 g1 = st.rec[buf][slot * 3 + 1];
      const float cut = st.rec[buf][slot * 3 + 2].w;
      keep[r] = splat_touches_rect(g0, g1, cut, wv.rx_lo, wv.rx_hi, wv.ry_lo, wv.ry_hi);
    }
  }
  const uint32_t lt = (1u << lane) - 1u;
  int base = 0;
#pragma unroll
  for (int r = 0; r < RPL; ++r) {
    const uint32_t m = __ballot_sync(0xffffffffu, keep[r]);
    if (keep[r]) st.list[base + __popc(m & lt)] = r * 32 + lane;
    base += __popc(m);
  }
  __syncwarp();
  return base;
}

// The staging pipeline of all four blend kernels.  Walks the sorted list entries first, first + 1, ..., end - 1 (front
// to back) or, with BACK, first, first - 1, ..., end + 1, in batches of kBatch records; the walk must hold at least one
// entry.  The flatten ids of the batch after next are prefetched into registers, each record is copied with three
// 16-byte cp.async (double buffered), and extra(buf, slot, id) may issue one more copy per record into the same group
// (the feature kernels' colour row).  KEEP_IDS also stores the batch's flatten ids in st.id.  Once a batch has landed
// it is culled against the warp's rectangle and body(b, ns, base) runs on batch b: st.rec[b & 1] holds its records,
// st.list[0, ns) the surviving slots in walk order, and slot s is sorted entry base + s (front to back) or base - s
// (back to front).  The walk ends when body returns true.
template <bool BACK, bool KEEP_IDS, int RPL, class Extra, class Body>
__device__ __forceinline__ void stage_batches(WarpStage<32 * RPL>& st, const float4* __restrict__ splats,
                                              const int32_t* __restrict__ flatten_ids, int first, int end, int lane,
                                              const WarpView& wv, Extra&& extra, Body&& body) {
  constexpr int kBatch = 32 * RPL;
  const int nb = ((BACK ? first - end : end - first) + kBatch - 1) / kBatch;
  // the callers guarantee it; without the hint the loop below gets a second entry test and the kernels more registers
  __builtin_assume(nb > 0);
  auto load_ids = [&](int b, int (&ids)[RPL]) {
#pragma unroll
    for (int r = 0; r < RPL; ++r) {
      const int k = b * kBatch + r * 32 + lane;
      const int idx = BACK ? first - k : first + k;
      ids[r] = (BACK ? idx > end : idx < end) ? __ldg(flatten_ids + idx) : -1;  // b >= nb: past the end
    }
  };
  auto issue = [&](int buf, const int (&ids)[RPL]) {
#pragma unroll
    for (int r = 0; r < RPL; ++r) {
      const int slot = r * 32 + lane;
      if (ids[r] >= 0) {
        const float4* src = splats + (size_t)ids[r] * 3;
        float4* dst = &st.rec[buf][slot * 3];
        cp_async16(dst + 0, src + 0);
        cp_async16(dst + 1, src + 1);
        cp_async16(dst + 2, src + 2);
        extra(buf, slot, ids[r]);
      }
      if constexpr (KEEP_IDS) st.id[buf][slot] = ids[r];
    }
    cp_async_commit();
  };

  int ids[RPL];
  load_ids(0, ids);
  issue(0, ids);
  load_ids(1, ids);
  for (int b = 0; b < nb; ++b) {
    if (b + 1 < nb) {
      issue((b + 1) & 1, ids);
      load_ids(b + 2, ids);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncwarp();  // batch b has landed for every lane of this warp
    const int base = BACK ? first - b * kBatch : first + b * kBatch;
    const int batch_size = min(kBatch, BACK ? base - end : end - base);
    const int ns = cull_and_compact<RPL>(st, b & 1, batch_size, lane, wv);
    if (body(b, ns, base)) {
      cp_async_wait<0>();  // the next batch may still be in flight
      return;
    }
    __syncwarp();  // every lane is done with buffer b&1, its ids and the list before they are overwritten
  }
}

// q = -log2(e) * sigma and ov = opacity * 2^q (before the 0.999 clamp) at the lane's pixels, with dx / dy = mean - pixel
// centre per column / row.  Packed FADD2 / FMUL2 / FFMA2 in the <2,2> layout (sm_100: the two pixels of a row share one
// instruction; the kernels are issue bound, not FMA-pipe bound, profiles/r1g, so halving the issue slots of the
// arithmetic is what counts), the same sequence one pixel at a time in <1,1>.  Every kernel evaluates alphas here, so
// their alphas agree bit for bit.
template <int P>
__device__ __forceinline__ void splat_eval(const float4 g0, const float4 g1, const float2 npx2, const float2 npy2,
                                           float (&dx)[P], float (&dy)[P], float (&q)[P * P], float (&ov)[P * P]) {
  // q(dx,dy) = -log2(e) * sigma, separable parts shared by the rows / columns of the pixel block
  const float la = (0.5f * kNegLog2e) * g0.z, lc = (0.5f * kNegLog2e) * g1.x, lb = kNegLog2e * g0.w;
  if constexpr (P == 2) {
    const float2 dx2 = __fadd2_rn(make_float2(g0.x, g0.x), npx2);
    const float2 dy2 = __fadd2_rn(make_float2(g0.y, g0.y), npy2);
    const float2 qx = __fmul2_rn(__fmul2_rn(dx2, make_float2(la, la)), dx2);
    const float2 bx = __fmul2_rn(dx2, make_float2(lb, lb));
    const float2 qy = __fmul2_rn(__fmul2_rn(dy2, make_float2(lc, lc)), dy2);
    const float2 o2 = make_float2(g1.y, g1.y);
    const float2 q0 = __ffma2_rn(bx, make_float2(dy2.x, dy2.x), __fadd2_rn(qx, make_float2(qy.x, qy.x)));
    const float2 q1 = __ffma2_rn(bx, make_float2(dy2.y, dy2.y), __fadd2_rn(qx, make_float2(qy.y, qy.y)));
    const float2 a0 = __fmul2_rn(o2, make_float2(fast_ex2(q0.x), fast_ex2(q0.y)));
    const float2 a1 = __fmul2_rn(o2, make_float2(fast_ex2(q1.x), fast_ex2(q1.y)));
    dx[0] = dx2.x; dx[1] = dx2.y; dy[0] = dy2.x; dy[1] = dy2.y;
    q[0] = q0.x; q[1] = q0.y; q[2] = q1.x; q[3] = q1.y;
    ov[0] = a0.x; ov[1] = a0.y; ov[2] = a1.x; ov[3] = a1.y;
  } else {
    static_assert(P == 1, "the blend kernels use the <2,2> and <1,1> layouts");
    dx[0] = __fadd_rn(g0.x, npx2.x);
    dy[0] = __fadd_rn(g0.y, npy2.x);
    const float qx = __fmul_rn(__fmul_rn(dx[0], la), dx[0]), bx = __fmul_rn(dx[0], lb);
    const float qy = __fmul_rn(__fmul_rn(dy[0], lc), dy[0]);
    q[0] = __fmaf_rn(bx, dy[0], __fadd_rn(qx, qy));
    ov[0] = __fmul_rn(g1.y, fast_ex2(q[0]));
  }
}

// Warp sum of up to 16 per-lane values and one RED per value, the tail of both backward kernels.  Every lane stores its
// values v[0, n) to the rows of its warp's scratch (row k = value k, row stride kRedStride words: conflict free;
// red_st = this lane's column), then lane 2k+p adds half p of row k (`row`: 4 LDS.128, a packed add tree), one shuffle
// joins the halves and the lanes with `flag` set (lane 2k, k < n) issue the RED of their row's total to `dst`.
// ~40 issue slots against ~90 for the 16-slot shuffle reduce-scatter (32 selects + 16 SHFL + 16 FADD) — the kernels
// are issue bound.
template <int N>
__device__ __forceinline__ void warp_sum_red(const float (&v)[N], int n, uint32_t red_st, const float4* row, int flag,
                                             float* dst) {
  __syncwarp();  // the previous round's (or survivor's) row reads are complete
#pragma unroll
  for (int k = 0; k < N; ++k)
    if (k < n) sts_f32(red_st + k * kRedStride * 4, v[k]);
  __syncwarp();
  // rows past n hold stale data; no lane issues them
  const float4 r0 = row[0], r1 = row[1], r2 = row[2], r3 = row[3];
  float2 s0 = __fadd2_rn(make_float2(r0.x, r0.y), make_float2(r0.z, r0.w));
  float2 s1 = __fadd2_rn(make_float2(r1.x, r1.y), make_float2(r1.z, r1.w));
  float2 s2 = __fadd2_rn(make_float2(r2.x, r2.y), make_float2(r2.z, r2.w));
  float2 s3 = __fadd2_rn(make_float2(r3.x, r3.y), make_float2(r3.z, r3.w));
  s0 = __fadd2_rn(__fadd2_rn(s0, s1), __fadd2_rn(s2, s3));
  float total = s0.x + s0.y;
  total += __shfl_xor_sync(0xffffffffu, total, 1);
  red_add_f32_if(flag, dst, total);
}

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
// DEPTH: a fourth channel, the camera-space depth of record slot 9, blended like r, g, b with background 0 (render_colors
// then has 4 floats per pixel); never with COUNT or checkpoints.
template <bool COUNT, bool DEPTH = false>
__global__ void EGS_FWD_BOUNDS((Geo<2, 2>::kThreads)) rasterize_fwd_kernel(
    int64_t n_isects, const float4* __restrict__ splats, const int32_t* __restrict__ tile_offsets,
    const int32_t* __restrict__ flatten_ids, const float* __restrict__ backgrounds, int width, int height, int tile_w,
    int tile_h, int n_tiles_total, float* __restrict__ render_colors, float* __restrict__ render_alphas,
    int32_t* __restrict__ last_ids, unsigned long long* __restrict__ pair_counters, float4* __restrict__ ckpt,
    int ckpt_k, int seg_min_len,
    // nullable: block b handles tile tile_order[b] (longest lists first, egs_isect_sorted) instead of the tile at its grid position
    const int32_t* __restrict__ tile_order) {
  using G = Geo<2, 2>;
  constexpr int NP = G::NP;
  constexpr int RPL = G::RPL, kBatch = G::kBatch;
  __shared__ __align__(16) WarpStage<kBatch> stage[G::kWarps];
  const int lane = threadIdx.x & 31;
  WarpStage<kBatch>& st = stage[threadIdx.x >> 5];
  const WarpView wv = warp_setup<G>(tile_w, tile_h, n_isects, tile_offsets, n_tiles_total, tile_order);
  // T[j] > 0: transmittance of a live pixel; T[j] < 0: pixel finished, |T[j]| is its final transmittance
  // (the "done" flag lives in the sign bit, so liveness is one more FSETP in the accept test).
  float T[NP], cr[NP], cg[NP], cb[NP], cd[NP];
  int last[NP], term[NP];
  bool all_done = true;
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    const bool inside = (wv.x0 + (j % 2)) < width && (wv.y0 + (j / 2)) < height;
    T[j] = inside ? 1.0f : -1.0f; cr[j] = 0.f; cg[j] = 0.f; cb[j] = 0.f; last[j] = 0; term[j] = -1;
    if constexpr (DEPTH) cd[j] = 0.f;
    all_done = all_done && !inside;
  }
  unsigned int n_acc = 0;

  if (wv.range_end > wv.range_start && !__all_sync(0xffffffffu, all_done)) {
    stage_batches<false, false, RPL>(
        st, splats, flatten_ids, wv.range_start, wv.range_end, lane, wv, [](int, int, int) {},
        [&](int b, int ns, int batch_start) {
          const float4* s = st.rec[b & 1];
          // Two survivors per trip: their alphas do not depend on the running transmittance, so both are evaluated
          // up front (independent LDS / FMA / MUFU chains = twice the ILP for a warp that walks a long list alone),
          // then blended in order.  The vote at the top is the warp-uniform exit and the reconvergence point.
          for (int t = 0; t < ns; t += 2) {
            if (__all_sync(0xffffffffu, all_done)) break;
            const bool has_b = t + 1 < ns;  // warp-uniform
            const int cur_a = st.list[t], cur_b = st.list[has_b ? t + 1 : t];
            float4 g0[2], g1[2];
            float cbl[2], dep[2], alpha[2][NP], q[2][NP];
            g0[0] = s[cur_a * 3 + 0]; g1[0] = s[cur_a * 3 + 1]; cbl[0] = s[cur_a * 3 + 2].x;
            g0[1] = s[cur_b * 3 + 0]; g1[1] = s[cur_b * 3 + 1]; cbl[1] = s[cur_b * 3 + 2].x;
            if constexpr (DEPTH) { dep[0] = s[cur_a * 3 + 2].y; dep[1] = s[cur_b * 3 + 2].y; }
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              float dx[2], dy[2];
              splat_eval<2>(g0[e], g1[e], wv.npx2, wv.npy2, dx, dy, q[e], alpha[e]);
#pragma unroll
              for (int j = 0; j < NP; ++j) alpha[e][j] = fminf(kAlphaMax, alpha[e][j]);
            }
            float tmax = -1.0f;
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              if (e == 0 || has_b) {
                const int cur = e == 0 ? cur_a : cur_b;
                // branch-free, two pixels (one row of the lane's block) per packed instruction: a rejected or
                // finished pixel blends with weight 0 (exact: c + g * 0 = c) and keeps its T
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                  const int j0 = 2 * r, j1 = 2 * r + 1;
                  const float2 a2 = make_float2(alpha[e][j0], alpha[e][j1]);
                  const float2 T2 = make_float2(T[j0], T[j1]);
                  const float2 nT = __fmul2_rn(T2, __ffma2_rn(a2, make_float2(-1.f, -1.f), make_float2(1.f, 1.f)));
                  float2 w = __fmul2_rn(a2, T2);
                  const bool acc0 = T[j0] > 0.f && q[e][j0] <= 0.f && alpha[e][j0] >= kAlphaMin;
                  const bool acc1 = T[j1] > 0.f && q[e][j1] <= 0.f && alpha[e][j1] >= kAlphaMin;
                  const bool bl0 = acc0 && nT.x > kTMin, bl1 = acc1 && nT.y > kTMin;
                  w.x = bl0 ? w.x : 0.f;
                  w.y = bl1 ? w.y : 0.f;
                  if (acc0) T[j0] = bl0 ? nT.x : -T[j0];  // not blended: finished, sign flags it
                  if (acc1) T[j1] = bl1 ? nT.y : -T[j1];
                  if (bl0) last[j0] = batch_start + cur;
                  if (bl1) last[j1] = batch_start + cur;
                  if (COUNT) {
                    if (acc0 && !bl0) term[j0] = batch_start + cur;
                    if (acc1 && !bl1) term[j1] = batch_start + cur;
                    n_acc += (bl0 ? 1u : 0u) + (bl1 ? 1u : 0u);
                  }
                  const float2 c_r = __ffma2_rn(make_float2(g1[e].z, g1[e].z), w, make_float2(cr[j0], cr[j1]));
                  const float2 c_g = __ffma2_rn(make_float2(g1[e].w, g1[e].w), w, make_float2(cg[j0], cg[j1]));
                  const float2 c_b = __ffma2_rn(make_float2(cbl[e], cbl[e]), w, make_float2(cb[j0], cb[j1]));
                  cr[j0] = c_r.x; cr[j1] = c_r.y; cg[j0] = c_g.x; cg[j1] = c_g.y; cb[j0] = c_b.x; cb[j1] = c_b.y;
                  if constexpr (DEPTH) {
                    const float2 c_d = __ffma2_rn(make_float2(dep[e], dep[e]), w, make_float2(cd[j0], cd[j1]));
                    cd[j0] = c_d.x; cd[j1] = c_d.y;
                  }
                }
              }
            }
#pragma unroll
            for (int j = 0; j < NP; ++j) tmax = fmaxf(tmax, T[j]);
            all_done = !(tmax > 0.f);
          }
          if (__all_sync(0xffffffffu, all_done)) return true;  // this warp needs nothing further down the list
          // Per-pixel state after every ckpt_k entries of a long list: lets the backward pass start its back-to-front
          // replay at any of these boundaries, one warp per segment (see rasterize_bwd_kernel).  Slot numbering
          // floor(start / K) + k is collision free across tiles because their list ranges are disjoint and ordered.
          const int done_local = (b + 1) * kBatch;
          if (!DEPTH && ckpt != nullptr && wv.range_end - wv.range_start >= seg_min_len && done_local % ckpt_k == 0 &&
              done_local < wv.range_end - wv.range_start) {
            const size_t slot = (size_t)(wv.range_start / ckpt_k + done_local / ckpt_k);
            float4* dst = ckpt + ((slot * G::kWarps + (threadIdx.x >> 5)) * NP) * 32 + lane;
#pragma unroll
            for (int j = 0; j < NP; ++j) dst[j * 32] = make_float4(T[j], cr[j], cg[j], cb[j]);
          }
          return false;
        });
  }

  float bgr = 0.f, bgg = 0.f, bgb = 0.f;
  if (backgrounds != nullptr) {
    bgr = backgrounds[wv.cam * 3 + 0]; bgg = backgrounds[wv.cam * 3 + 1]; bgb = backgrounds[wv.cam * 3 + 2];
  }
  unsigned int n_eval = 0;
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    const int x = wv.x0 + (j % 2), y = wv.y0 + (j / 2);
    if (x < width && y < height) {
      const size_t pix = ((size_t)wv.cam * height + y) * width + x;
      const float Tf = fabsf(T[j]);
      constexpr int PS = DEPTH ? 4 : 3;  // floats per pixel of render_colors
      render_colors[pix * PS + 0] = fmaf(Tf, bgr, cr[j]);
      render_colors[pix * PS + 1] = fmaf(Tf, bgg, cg[j]);
      render_colors[pix * PS + 2] = fmaf(Tf, bgb, cb[j]);
      if constexpr (DEPTH) render_colors[pix * PS + 3] = cd[j];
      render_alphas[pix] = 1.0f - Tf;
      last_ids[pix] = last[j];
      // P_eval in the reference's sense: list entries up to and including the terminating one
      if (COUNT) n_eval += (unsigned)((term[j] >= 0 ? term[j] + 1 : wv.range_end) - wv.range_start);
    }
  }
  if (COUNT) {
    for (int d = 16; d > 0; d >>= 1) {
      n_eval += __shfl_xor_sync(0xffffffffu, n_eval, d);
      n_acc += __shfl_xor_sync(0xffffffffu, n_acc, d);
    }
    if (lane == 0) {
      atomicAdd(pair_counters + 0, (unsigned long long)n_eval);
      atomicAdd(pair_counters + 1, (unsigned long long)n_acc);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------------
// DEPTH: the backward of the DEPTH forward.  v_render_colors has 4 floats per pixel; the depth channel (background 0)
// enters v_alpha through depth * v_d, and sum fac * v_d is reduced as a twelfth value into gradient-record slot 11
// (v_depth).  No segmented replay.
template <bool DEPTH = false>
__global__ void EGS_BWD_BOUNDS((Geo<2, 2>::kThreads)) rasterize_bwd_kernel(
    int64_t n_isects, const float4* __restrict__ splats, const int32_t* __restrict__ tile_offsets,
    const int32_t* __restrict__ flatten_ids, const float* __restrict__ backgrounds, int width, int height, int tile_w,
    int tile_h, int n_tiles_total, const float* __restrict__ render_alphas,
    const int32_t* __restrict__ last_ids, const float* __restrict__ v_render_colors,
    const float* __restrict__ v_render_alphas, float* __restrict__ v_splats,
    // Segmented replay of long lists (ckpt != nullptr): the forward pass left the per-pixel state after every ckpt_k
    // entries of a list, so a list of L entries is replayed by ceil(L / ckpt_k) independent warps per tile half.
    // seg_launch = 0: blocks are tiles and replay the LAST segment their warp needs (from the warp's last blended
    // entry down to the segment boundary below it, initial state = the final image, as without segments);
    // seg_launch = 1: blocks are checkpoint slots and replay the full segment that ends at their checkpoint.
    // Only lists of at least seg_min_len (> ckpt_k) entries are replayed in segments; shorter ones as one piece.
    const float* __restrict__ render_colors, const float4* __restrict__ ckpt, int ckpt_k, int seg_min_len, int seg_launch,
    const int32_t* __restrict__ tile_order /* nullable, tile launch only: see the forward kernel */) {
  using G = Geo<2, 2>;
  constexpr int NP = G::NP;
  constexpr int RPL = G::RPL, kBatch = G::kBatch;
  constexpr int NV = DEPTH ? kGradValues + 1 : kGradValues;  // values reduced per Gaussian
  constexpr int PS = DEPTH ? 4 : 3;                           // floats per pixel of v_render_colors
  __shared__ __align__(16) WarpStage<kBatch> stage[G::kWarps];
  __shared__ __align__(16) float red_all[G::kWarps][NV * kRedStride];
  const int lane = threadIdx.x & 31;
  WarpStage<kBatch>& st = stage[threadIdx.x >> 5];
  float* red = red_all[threadIdx.x >> 5];
  int seg_tile = -1, seg_k = 0;
  if (seg_launch) {
    // slot j = blockIdx.x + 1 belongs to the last tile whose list starts before entry j * K (empty tiles share
    // their successor's start, so the last one is the tile that really holds that entry)
    const int64_t bound = ((int64_t)blockIdx.x + 1) * ckpt_k;
    int lo_t = 0, hi_t = n_tiles_total - 1;
    while (lo_t < hi_t) {
      const int mid = (lo_t + hi_t + 1) >> 1;
      if ((int64_t)tile_offsets[mid] < bound) lo_t = mid; else hi_t = mid - 1;
    }
    seg_tile = lo_t;
    seg_k = (int)(blockIdx.x + 1) - tile_offsets[seg_tile] / ckpt_k;
  }
  const WarpView wv = warp_setup<G>(tile_w, tile_h, n_isects, tile_offsets, n_tiles_total, tile_order, seg_tile);
  {
    const int len = wv.range_end - wv.range_start;
    if (len <= 0) return;  // block-uniform
    if (seg_launch && (len < seg_min_len || seg_k < 1 || (int64_t)seg_k * ckpt_k >= len)) return;  // block-uniform: slot not in use
  }

  // per-pixel replay state.  nbt_ = tfv - bdot with bdot = sum over the Gaussians behind of fac * (rgb . v_colour),
  // which is all the backward pass needs of the colour accumulated behind, and
  // tfv = T_final * (v_alpha_out - bg . v_colour).
  float T[NP], nbt_[NP], vcr[NP], vcg[NP], vcb[NP], vcd[NP];
  int bin_final[NP];
  int my_last = -1;
  float bgr = 0.f, bgg = 0.f, bgb = 0.f;
  if (backgrounds != nullptr) {
    bgr = backgrounds[wv.cam * 3 + 0]; bgg = backgrounds[wv.cam * 3 + 1]; bgb = backgrounds[wv.cam * 3 + 2];
  }
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    const int x = wv.x0 + (j % 2), y = wv.y0 + (j / 2);
    T[j] = 1.f; nbt_[j] = 0.f; vcr[j] = 0.f; vcg[j] = 0.f; vcb[j] = 0.f;
    if constexpr (DEPTH) vcd[j] = 0.f;
    bin_final[j] = -1;  // pixels outside the image never match any index
    if (x < width && y < height) {
      const size_t pix = ((size_t)wv.cam * height + y) * width + x;
      const float T_final = 1.0f - render_alphas[pix];
      T[j] = T_final;
      bin_final[j] = last_ids[pix];
      vcr[j] = v_render_colors[pix * PS + 0];
      vcg[j] = v_render_colors[pix * PS + 1];
      vcb[j] = v_render_colors[pix * PS + 2];
      if constexpr (DEPTH) vcd[j] = v_render_colors[pix * PS + 3];
      nbt_[j] = T_final * (v_render_alphas[pix] - (bgr * vcr[j] + bgg * vcg[j] + bgb * vcb[j]));
    }
    my_last = max(my_last, bin_final[j]);
  }
  // nothing behind the last blended Gaussian of any pixel of the warp can receive gradient
  const int warp_last = __reduce_max_sync(0xffffffffu, my_last);
  int end_idx = min(wv.range_end - 1, warp_last);
  if (end_idx < wv.range_start) return;  // warp-uniform
  int lo_idx = wv.range_start;  // the replay walks end_idx, end_idx - 1, ..., lo_idx
  if (!DEPTH && ckpt != nullptr && wv.range_end - wv.range_start >= seg_min_len) {
    const int last_seg = (end_idx - wv.range_start) / ckpt_k;  // segment that holds the warp's last blended entry
    if (!seg_launch) {
      lo_idx = wv.range_start + last_seg * ckpt_k;
    } else {
      if (seg_k > last_seg) return;  // warp-uniform: nothing of this warp reaches into or beyond this segment
      end_idx = wv.range_start + seg_k * ckpt_k - 1;
      lo_idx = end_idx + 1 - ckpt_k;
      // state after entry end_idx: transmittance and colour accumulated in front of the boundary (the forward
      // checkpoint); what lies behind it is the final colour minus that
      const size_t slot = (size_t)(wv.range_start / ckpt_k + seg_k);
      const float4* src = ckpt + ((slot * G::kWarps + (threadIdx.x >> 5)) * NP) * 32 + lane;
#pragma unroll
      for (int j = 0; j < NP; ++j) {
        const int x = wv.x0 + (j % 2), y = wv.y0 + (j / 2);
        if (x < width && y < height) {
          const size_t pix = ((size_t)wv.cam * height + y) * width + x;
          const float4 ck = src[j * 32];
          const float T_final = T[j];
          const float br = render_colors[pix * 3 + 0] - T_final * bgr - ck.y;
          const float bgn = render_colors[pix * 3 + 1] - T_final * bgg - ck.z;
          const float bb = render_colors[pix * 3 + 2] - T_final * bgb - ck.w;
          nbt_[j] -= br * vcr[j] + bgn * vcg[j] + bb * vcb[j];
          T[j] = fabsf(ck.x);
        }
      }
    }
  } else if (seg_launch) {
    return;
  }

  // Addresses of the warp-sum scratch and of the gradient slot this lane reduces, pinned in registers: ptxas
  // otherwise re-derives them from %tid / the CTA's shared window for every survivor (~12 of the loop's ~200
  // instructions).
  const int out_slot = lane >> 1;
  int red_flag = ((lane & 1) == 0 && out_slot < NV) ? 1 : 0;
  asm volatile("" : "+r"(red_flag));
  uint32_t red_st = (uint32_t)__cvta_generic_to_shared(red + lane);
  asm volatile("" : "+r"(red_st));
  const float4* row = reinterpret_cast<const float4*>(red + min(out_slot, NV - 1) * kRedStride + (lane & 1) * 16);
  float* out_base = v_splats + min(out_slot, NV - 1);
  asm volatile("" : "+l"(out_base));

  stage_batches<true, true, RPL>(
      st, splats, flatten_ids, end_idx, lo_idx - 1, lane, wv, [](int, int, int) {},
      [&](int b, int ns, int batch_end) {  // batch_end: sorted index held in slot 0 (the one furthest back)
        const float4* s = st.rec[b & 1];
        const int* sid = st.id[b & 1];
        int slot = st.list[0];
        for (int t = 0; t < ns; ++t) {  // warp-uniform bounds
          const int cur = slot;
          slot = st.list[min(t + 1, kBatch - 1)];
          const int idx = batch_end - cur;
          const float4 g0 = s[cur * 3 + 0];  // x, y, conic_a, conic_b
          const float4 g1 = s[cur * 3 + 1];  // conic_c, opacity, r, g
          const float cbl = s[cur * 3 + 2].x;
          float dep = 0.f;
          if constexpr (DEPTH) dep = s[cur * 3 + 2].y;
          const float inv_o = fast_rcp(g1.y);
          // Packed fp32 (FADD2 / FMUL2 / FFMA2): the two pixels of a row of the lane's block share one instruction,
          // and the replay is branch free — a pixel that does not take part gets alpha = 0 and ov = 0, which makes
          // every one of its contributions an exact zero and leaves its running state untouched.
          float dx[2], dy[2], q[NP], ov[NP];
          splat_eval<2>(g0, g1, wv.npx2, wv.npy2, dx, dy, q, ov);
          const float2 dx2 = make_float2(dx[0], dx[1]);
          bool valid[NP];
          bool any_valid = false;
#pragma unroll
          for (int j = 0; j < NP; ++j) {
            valid[j] = idx <= bin_final[j] && q[j] <= 0.f && ov[j] >= kAlphaMin;  // min(.999, ov) >= 1/255 <=> ov >= 1/255
            any_valid = any_valid || valid[j];
          }
          if (!__any_sync(0xffffffffu, any_valid)) continue;  // warp-uniform
          float2 s_gx = make_float2(0.f, 0.f), s_gy = s_gx, s_xx = s_gx, s_xy = s_gx, s_yy = s_gx, s_w = s_gx, s_r = s_gx,
                 s_g = s_gx, s_b = s_gx, s_ax = s_gx, s_ay = s_gx, s_d = s_gx;
#pragma unroll
          for (int r = 0; r < 2; ++r) {
            const int j0 = 2 * r, j1 = 2 * r + 1;
            const float2 dyb = make_float2(dy[r], dy[r]);
            float2 ae, oe;  // alpha and ov of the pixels that take part, 0 for the others
            // ov of the pixels that take part, 0 for the others; everything downstream is then an exact no-op for
            // a pixel that does not take part: alpha = 0, 1 - alpha = 1, MUFU.RCP(1) = 1 exactly
            // (scripts/probes/rcp_one.cu), so T * 1 = T needs no select
            const float ovx = valid[j0] ? ov[j0] : 0.f, ovy = valid[j1] ? ov[j1] : 0.f;
            ae.x = fminf(kAlphaMax, ovx);
            ae.y = fminf(kAlphaMax, ovy);
            oe.x = ovx <= kAlphaMax ? ovx : 0.f;  // clamp inactive: alpha depends on sigma, opacity
            oe.y = ovy <= kAlphaMax ? ovy : 0.f;
            const float2 om = __ffma2_rn(ae, make_float2(-1.f, -1.f), make_float2(1.f, 1.f));
            const float2 ra = make_float2(fast_rcp(om.x), fast_rcp(om.y));
            const float2 Tf = __fmul2_rn(make_float2(T[j0], T[j1]), ra);  // transmittance in front of this Gaussian
            T[j0] = Tf.x; T[j1] = Tf.y;
            const float2 fac = __fmul2_rn(ae, Tf);
            const float2 vr2 = make_float2(vcr[j0], vcr[j1]), vg2 = make_float2(vcg[j0], vcg[j1]), vb2 = make_float2(vcb[j0], vcb[j1]);
            s_r = __ffma2_rn(fac, vr2, s_r);
            s_g = __ffma2_rn(fac, vg2, s_g);
            s_b = __ffma2_rn(fac, vb2, s_b);
            float2 cdot = __ffma2_rn(make_float2(cbl, cbl), vb2,
                                     __ffma2_rn(make_float2(g1.w, g1.w), vg2, __fmul2_rn(make_float2(g1.z, g1.z), vr2)));
            if constexpr (DEPTH) {
              const float2 vd2 = make_float2(vcd[j0], vcd[j1]);
              s_d = __ffma2_rn(fac, vd2, s_d);
              cdot = __ffma2_rn(make_float2(dep, dep), vd2, cdot);
            }
            // nbt = tfv - bdot (kept negated so that v_alpha is one FMUL2 + one FFMA2)
            const float2 nbt = make_float2(nbt_[j0], nbt_[j1]);
            const float2 v_alpha = __ffma2_rn(Tf, cdot, __fmul2_rn(ra, nbt));
            const float2 nfac = make_float2(-fac.x, -fac.y);
            const float2 nbt_new = __ffma2_rn(cdot, nfac, nbt);
            nbt_[j0] = nbt_new.x; nbt_[j1] = nbt_new.y;
            const float2 w = __fmul2_rn(oe, v_alpha);  // = opacity * d(alpha)/d(opacity) * v_alpha = -v_sigma
            const float2 nw = make_float2(-w.x, -w.y);
            const float2 sx = __fmul2_rn(nw, dx2), sy = __fmul2_rn(nw, dyb);
            s_xx = __ffma2_rn(sx, dx2, s_xx);
            s_xy = __ffma2_rn(sx, dyb, s_xy);
            s_yy = __ffma2_rn(sy, dyb, s_yy);
            const float2 gx = __ffma2_rn(make_float2(g0.w, g0.w), sy, __fmul2_rn(make_float2(g0.z, g0.z), sx));
            const float2 gy = __ffma2_rn(make_float2(g1.x, g1.x), sy, __fmul2_rn(make_float2(g0.w, g0.w), sx));
            s_gx = __fadd2_rn(s_gx, gx);
            s_gy = __fadd2_rn(s_gy, gy);
            s_ax = __fadd2_rn(s_ax, make_float2(fabsf(gx.x), fabsf(gx.y)));
            s_ay = __fadd2_rn(s_ay, make_float2(fabsf(gy.x), fabsf(gy.y)));
            s_w = __fadd2_rn(s_w, w);
          }
          // v[2], v[3], v[4] are the sums of sx*dx, sx*dy, sy*dy (the 0.5 of the conic gradient is applied once, after
          // the per-lane sum); v[5] the sum of ov * v_alpha (the 1/opacity is applied after the per-lane sum).
          float v[NV];
          v[0] = s_gx.x + s_gx.y; v[1] = s_gy.x + s_gy.y; v[2] = s_xx.x + s_xx.y; v[3] = s_xy.x + s_xy.y;
          v[4] = s_yy.x + s_yy.y; v[5] = s_w.x + s_w.y; v[6] = s_r.x + s_r.y; v[7] = s_g.x + s_g.y;
          v[8] = s_b.x + s_b.y; v[9] = s_ax.x + s_ax.y; v[10] = s_ay.x + s_ay.y;
          if constexpr (DEPTH) v[11] = s_d.x + s_d.y;
          v[2] *= 0.5f; v[4] *= 0.5f; v[5] *= inv_o;
          warp_sum_red(v, NV, red_st, row, red_flag, out_base + (size_t)sid[cur] * EGS_SPLAT_FLOATS);
        }
        return false;
      });
}

// ------------------------------------------------------------------------------------------------
// colours with any number of channels ("features")
// ------------------------------------------------------------------------------------------------
// The same blend as above with CH colour channels per launch, read from a separate fp32 row array instead of the r, g, b
// slots of the splat record (which these kernels do not read).  Row of a list entry: flat id - cam * N when one [N, .]
// array serves every camera, the flat id for a [C * N, .] array.  A launch covers channels [c0, c0 + CH) of the rows;
// wider colours are several launches on the same binning result.  The prologue (warp_setup), the staging and culling
// (stage_batches), the alpha evaluation (splat_eval), the accept / finish tests and the warp-sum tail (warp_sum_red) are
// the RGB kernels'; in the <2,2> layout (CH <= 8) alphas and last_ids come out bit-identical to them, while the <1,1>
// layout's transmittance differs in the last bits (measured on a B200: alphas within 2.4e-7).
// Pixel layout: CH <= 8 keeps the RGB kernels' <2,2> layout (4 pixels per lane, 4 CH colour registers); CH = 16 / 32
// use <1,1> (one pixel per lane, 8 warps per tile), which keeps the per-lane colour state at CH registers.  Long lists
// are always replayed in one piece (no checkpoints).
constexpr int kFeatRedRows = 16;  // values per warp-sum round of the feature backward (two lanes per value)

template <int CH>
struct FeatGeo {
  static constexpr int P = CH <= 8 ? 2 : 1;
  using G = Geo<P, P>;
};

// Per-warp shared memory of the feature kernels (dynamic: up to ~111 KB per CTA at CH = 32): the RGB staging plus the
// colour rows of both batches.  The backward kernel places its warp-sum scratch behind the array of these.
template <int kBatch, int CH>
struct FeatStage {
  WarpStage<kBatch> w;
  float feat[2][kBatch * CH];
};

template <int BYTES>
__device__ __forceinline__ void cp_async_ca(void* smem, const void* gmem) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"(s), "l"(gmem), "n"(BYTES) : "memory");
}

// One colour row of CH floats: 4- or 8-byte copies for CH = 1 / 2, 16-byte copies from CH = 4 on (the entries check
// that features, feat_stride and c0 are aligned for that).
template <int CH>
__device__ __forceinline__ void cp_async_row(float* dst, const float* src) {
  if constexpr (CH == 1) {
    cp_async_ca<4>(dst, src);
  } else if constexpr (CH == 2) {
    cp_async_ca<8>(dst, src);
  } else {
#pragma unroll
    for (int i = 0; i < CH; i += 4) cp_async16(dst + i, src + i);
  }
}

template <int CH>
__device__ __forceinline__ void load_row(float (&f)[CH], const float* src) {
  if constexpr (CH >= 4) {
#pragma unroll
    for (int i = 0; i < CH; i += 4) {
      const float4 t = *reinterpret_cast<const float4*>(src + i);
      f[i] = t.x; f[i + 1] = t.y; f[i + 2] = t.z; f[i + 3] = t.w;
    }
  } else {
#pragma unroll
    for (int i = 0; i < CH; ++i) f[i] = src[i];
  }
}

template <int CH>
__global__ void __launch_bounds__(FeatGeo<CH>::G::kThreads) rasterize_fwd_features_kernel(
    int64_t n_isects, const float4* __restrict__ splats, const int32_t* __restrict__ tile_offsets,
    const int32_t* __restrict__ flatten_ids, const float* __restrict__ features, int feat_stride, int row_cam_stride,
    int D, int c0, const float* __restrict__ backgrounds, int width, int height, int tile_w, int tile_h,
    int n_tiles_total, float* __restrict__ render_colors, float* __restrict__ render_alphas,
    int32_t* __restrict__ last_ids, const int32_t* __restrict__ tile_order) {
  constexpr int P = FeatGeo<CH>::P;
  using G = typename FeatGeo<CH>::G;
  constexpr int NP = G::NP, RPL = G::RPL, kBatch = G::kBatch;
  extern __shared__ __align__(16) unsigned char feat_smem[];
  FeatStage<kBatch, CH>& fs = reinterpret_cast<FeatStage<kBatch, CH>*>(feat_smem)[threadIdx.x >> 5];
  WarpStage<kBatch>& st = fs.w;
  const int lane = threadIdx.x & 31;
  const WarpView wv = warp_setup<G>(tile_w, tile_h, n_isects, tile_offsets, n_tiles_total, tile_order);
  const int64_t row_off = (int64_t)wv.cam * row_cam_stride;

  // T as in the RGB kernel: > 0 live, < 0 finished with final transmittance |T|
  float T[NP], col[NP][CH];
  int last[NP];
  bool all_done = true;
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    const bool inside = (wv.x0 + (j % P)) < width && (wv.y0 + (j / P)) < height;
    T[j] = inside ? 1.0f : -1.0f;
    last[j] = 0;
#pragma unroll
    for (int k = 0; k < CH; ++k) col[j][k] = 0.f;
    all_done = all_done && !inside;
  }

  if (wv.range_end > wv.range_start && !__all_sync(0xffffffffu, all_done)) {
    stage_batches<false, false, RPL>(
        st, splats, flatten_ids, wv.range_start, wv.range_end, lane, wv,
        [&](int buf, int slot, int id) {
          cp_async_row<CH>(&fs.feat[buf][slot * CH], features + ((int64_t)id - row_off) * feat_stride + c0);
        },
        [&](int b, int ns, int batch_start) {
          const float4* s = st.rec[b & 1];
          for (int t = 0; t < ns; ++t) {
            if (__all_sync(0xffffffffu, all_done)) break;  // warp-uniform exit and reconvergence point
            const int cur = st.list[t];
            float dx[P], dy[P], q[NP], ov[NP];
            splat_eval<P>(s[cur * 3 + 0], s[cur * 3 + 1], wv.npx2, wv.npy2, dx, dy, q, ov);
            float f[CH];
            load_row<CH>(f, &fs.feat[b & 1][cur * CH]);
            float tmax = -1.0f;
#pragma unroll
            for (int j = 0; j < NP; ++j) {
              // branch free: a rejected or finished pixel blends with weight 0 and keeps its T (as the RGB kernel)
              const float alpha = fminf(kAlphaMax, ov[j]);
              const float nT = __fmul_rn(T[j], __fmaf_rn(alpha, -1.f, 1.f));
              const bool acc = T[j] > 0.f && q[j] <= 0.f && alpha >= kAlphaMin;
              const bool bl = acc && nT > kTMin;
              const float w = bl ? __fmul_rn(alpha, T[j]) : 0.f;
              if (acc) T[j] = bl ? nT : -T[j];
              if (bl) last[j] = batch_start + cur;
#pragma unroll
              for (int k = 0; k < CH; ++k) col[j][k] = __fmaf_rn(f[k], w, col[j][k]);
              tmax = fmaxf(tmax, T[j]);
            }
            all_done = !(tmax > 0.f);
          }
          return __all_sync(0xffffffffu, all_done);
        });
  }

  const int nc = min(CH, D - c0);
  float bg[CH];
#pragma unroll
  for (int k = 0; k < CH; ++k) bg[k] = (backgrounds != nullptr && k < nc) ? backgrounds[(size_t)wv.cam * D + c0 + k] : 0.f;
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    const int x = wv.x0 + (j % P), y = wv.y0 + (j / P);
    if (x < width && y < height) {
      const size_t pix = ((size_t)wv.cam * height + y) * width + x;
      const float Tf = fabsf(T[j]);
      float* out = render_colors + pix * D + c0;
#pragma unroll
      for (int k = 0; k < CH; ++k)
        if (k < nc) out[k] = fmaf(Tf, bg[k], col[j][k]);
      if (render_alphas != nullptr) render_alphas[pix] = 1.0f - Tf;
      if (last_ids != nullptr) last_ids[pix] = last[j];
    }
  }
}

template <int CH>
__global__ void __launch_bounds__(FeatGeo<CH>::G::kThreads) rasterize_bwd_features_kernel(
    int64_t n_isects, const float4* __restrict__ splats, const int32_t* __restrict__ tile_offsets,
    const int32_t* __restrict__ flatten_ids, const float* __restrict__ features, int feat_stride, int row_cam_stride,
    int D, int c0, const float* __restrict__ backgrounds, int width, int height, int tile_w, int tile_h,
    int n_tiles_total, const float* __restrict__ render_alphas, const int32_t* __restrict__ last_ids,
    const float* __restrict__ v_render_colors, const float* __restrict__ v_render_alphas, float* __restrict__ v_splats,
    float* __restrict__ v_features, const int32_t* __restrict__ tile_order) {
  constexpr int P = FeatGeo<CH>::P;
  using G = typename FeatGeo<CH>::G;
  constexpr int NP = G::NP, RPL = G::RPL, kBatch = G::kBatch;
  constexpr int kValues = 8 + CH;  // v_x, v_y, v_conic (3), v_opacity, |v_x|, |v_y|, then the CH colour partials
  constexpr int kRounds = (kValues + kFeatRedRows - 1) / kFeatRedRows;
  extern __shared__ __align__(16) unsigned char feat_smem[];
  FeatStage<kBatch, CH>* stages = reinterpret_cast<FeatStage<kBatch, CH>*>(feat_smem);
  FeatStage<kBatch, CH>& fs = stages[threadIdx.x >> 5];
  WarpStage<kBatch>& st = fs.w;
  float* red = reinterpret_cast<float*>(stages + G::kWarps) + (threadIdx.x >> 5) * (kFeatRedRows * kRedStride);
  const int lane = threadIdx.x & 31;
  const WarpView wv = warp_setup<G>(tile_w, tile_h, n_isects, tile_offsets, n_tiles_total, tile_order);
  if (wv.range_end - wv.range_start <= 0) return;  // block-uniform
  const int64_t row_off = (int64_t)wv.cam * row_cam_stride;

  // replay state as in the RGB kernel: nbt_ = T_final * (v_alpha_out - bg . v_colour) - (colour behind) . v_colour,
  // over this chunk's channels; v_alpha_out only where the caller passes it (one chunk of a call)
  const int nc = min(CH, D - c0);
  float bg[CH];
#pragma unroll
  for (int k = 0; k < CH; ++k) bg[k] = (backgrounds != nullptr && k < nc) ? backgrounds[(size_t)wv.cam * D + c0 + k] : 0.f;
  float T[NP], nbt_[NP], vc[NP][CH];
  int bin_final[NP];
  int my_last = -1;
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    const int x = wv.x0 + (j % P), y = wv.y0 + (j / P);
    T[j] = 1.f; nbt_[j] = 0.f; bin_final[j] = -1;
#pragma unroll
    for (int k = 0; k < CH; ++k) vc[j][k] = 0.f;
    if (x < width && y < height) {
      const size_t pix = ((size_t)wv.cam * height + y) * width + x;
      const float T_final = 1.0f - render_alphas[pix];
      T[j] = T_final;
      bin_final[j] = last_ids[pix];
      float bdot = 0.f;
#pragma unroll
      for (int k = 0; k < CH; ++k) {
        if (k < nc) vc[j][k] = v_render_colors[pix * D + c0 + k];
        bdot = fmaf(bg[k], vc[j][k], bdot);
      }
      nbt_[j] = T_final * ((v_render_alphas != nullptr ? v_render_alphas[pix] : 0.f) - bdot);
    }
    my_last = max(my_last, bin_final[j]);
  }
  const int warp_last = __reduce_max_sync(0xffffffffu, my_last);
  const int end_idx = min(wv.range_end - 1, warp_last);
  if (end_idx < wv.range_start) return;  // warp-uniform

  // Warp sum in rounds of 16 values: lane 2k+p adds half p of row k, lane 2k issues the RED of value 16 r + k.
  // Value v < 8 goes to the gradient record (slots 0-5, then |v_x|, |v_y| in slots 9, 10; the r, g, b slots stay 0),
  // value 8 + c to v_features (only the chunk's nc real channels, and only when v_features is given).
  const int out_slot = lane >> 1;
  const uint32_t red_st = (uint32_t)__cvta_generic_to_shared(red + lane);
  const float4* row = reinterpret_cast<const float4*>(red + out_slot * kRedStride + (lane & 1) * 16);
  int rec_off[kRounds], red_flag[kRounds];
#pragma unroll
  for (int r = 0; r < kRounds; ++r) {
    const int v = r * kFeatRedRows + out_slot;
    const bool is_feat = v >= 8;
    red_flag[r] = ((lane & 1) == 0 && v < kValues && (!is_feat || (v - 8 < nc && v_features != nullptr))) ? 1 : 0;
    rec_off[r] = is_feat ? c0 + (v - 8) : (v < 6 ? v : v + 3);
  }

  stage_batches<true, true, RPL>(
      st, splats, flatten_ids, end_idx, wv.range_start - 1, lane, wv,
      [&](int buf, int slot, int id) {
        cp_async_row<CH>(&fs.feat[buf][slot * CH], features + ((int64_t)id - row_off) * feat_stride + c0);
      },
      [&](int b, int ns, int batch_end) {
        const float4* s = st.rec[b & 1];
        const int* sid = st.id[b & 1];
        for (int t = 0; t < ns; ++t) {  // warp-uniform bounds
          const int cur = st.list[t];
          const int idx = batch_end - cur;
          const float4 g0 = s[cur * 3 + 0];
          const float4 g1 = s[cur * 3 + 1];
          float dx[P], dy[P], q[NP], ov[NP];
          splat_eval<P>(g0, g1, wv.npx2, wv.npy2, dx, dy, q, ov);
          bool valid[NP];
          bool any_valid = false;
#pragma unroll
          for (int j = 0; j < NP; ++j) {
            valid[j] = idx <= bin_final[j] && q[j] <= 0.f && ov[j] >= kAlphaMin;
            any_valid = any_valid || valid[j];
          }
          if (!__any_sync(0xffffffffu, any_valid)) continue;  // warp-uniform
          float f[CH];
          load_row<CH>(f, &fs.feat[b & 1][cur * CH]);
          const float inv_o = fast_rcp(g1.y);
          // branch free as the RGB kernel: a pixel that does not take part has ov = 0, hence alpha = 0, 1 - alpha = 1,
          // MUFU.RCP(1) = 1, and contributes exact zeros
          float v[8], fac[NP];
#pragma unroll
          for (int k = 0; k < 8; ++k) v[k] = 0.f;
#pragma unroll
          for (int j = 0; j < NP; ++j) {
            const float ddx = dx[j % P], ddy = dy[j / P];
            const float ovj = valid[j] ? ov[j] : 0.f;
            const float ae = fminf(kAlphaMax, ovj);
            const float oe = ovj <= kAlphaMax ? ovj : 0.f;  // clamp inactive: alpha depends on sigma and opacity
            const float ra = fast_rcp(fmaf(ae, -1.f, 1.f));
            T[j] *= ra;  // transmittance in front of this Gaussian
            fac[j] = ae * T[j];
            float cdot = 0.f;
#pragma unroll
            for (int k = 0; k < CH; ++k) cdot = fmaf(f[k], vc[j][k], cdot);
            const float v_alpha = fmaf(T[j], cdot, ra * nbt_[j]);
            nbt_[j] = fmaf(cdot, -fac[j], nbt_[j]);
            const float w = oe * v_alpha;  // = -v_sigma
            const float sx = -w * ddx, sy = -w * ddy;
            v[2] = fmaf(sx, ddx, v[2]);
            v[3] = fmaf(sx, ddy, v[3]);
            v[4] = fmaf(sy, ddy, v[4]);
            const float gx = fmaf(g0.w, sy, g0.z * sx);
            const float gy = fmaf(g1.x, sy, g0.w * sx);
            v[0] += gx;
            v[1] += gy;
            v[6] += fabsf(gx);
            v[7] += fabsf(gy);
            v[5] += w;
          }
          v[2] *= 0.5f; v[4] *= 0.5f; v[5] *= inv_o;
          const int64_t fid = sid[cur];
#pragma unroll
          for (int r = 0; r < kRounds; ++r) {
            float rv[kFeatRedRows];  // the round's values: geometry partials, then colour partials
#pragma unroll
            for (int i = 0; i < kFeatRedRows; ++i) {
              const int vi = r * kFeatRedRows + i;
              rv[i] = 0.f;
              if (vi < 8) {
                rv[i] = v[vi];
              } else if (vi < kValues) {
#pragma unroll
                for (int j = 0; j < NP; ++j) rv[i] = fmaf(fac[j], vc[j][vi - 8], rv[i]);
              }
            }
            const bool feat_slot = r * kFeatRedRows + out_slot >= 8;
            float* dst = feat_slot ? v_features + (fid - row_off) * feat_stride + rec_off[r]
                                   : v_splats + fid * EGS_SPLAT_FLOATS + rec_off[r];
            warp_sum_red(rv, min(kFeatRedRows, kValues - r * kFeatRedRows), red_st, row, red_flag[r], dst);
          }
        }
        return false;
      });
}

}  // namespace egs

using namespace egs;

static int check_raster_args(const char* who, int32_t C, int64_t n_isects, int32_t width, int32_t height,
                             int32_t tile_width, int32_t tile_height) {
  EGS_REQUIRE(C >= 0 && C <= 65535, "%s: C=%d out of [0,65535]", who, C);
  EGS_REQUIRE(width >= 1 && height >= 1, "%s: width/height must be >= 1", who);
  EGS_REQUIRE(tile_width == (width + kTileSize - 1) / kTileSize && tile_height == (height + kTileSize - 1) / kTileSize,
              "%s: tile grid %dx%d does not match %dx%d pixels at tile_size 16", who, tile_width, tile_height, width, height);
  EGS_REQUIRE(tile_height <= 65535, "%s: tile_height=%d exceeds the grid limit", who, tile_height);
  EGS_REQUIRE(n_isects > -0x7fffffffLL && n_isects < 0x7fffffffLL, "%s: n_isects=%lld out of int32 range", who, (long long)n_isects);
  EGS_REQUIRE((int64_t)C * tile_width * tile_height < 0x7fffffffLL, "%s: too many tiles", who);
  return 0;
}

// The RGB kernels handle every tile in the <2,2> layout.  A second launch with the 8-warps-per-tile <1,1> layout for very long
// lists was measured twice (round 1: object scene, 4 views per call: forward 0.48 -> 0.42 ms, backward 0.59 -> 0.72 ms;
// round 2, one view per call: 1.224 -> 1.225 ms per view, gpurun_out/r2c_knobs.log) and is no longer built: the busy
// tiles of an object scene are bound by their serial walk, and eight warps that each cull the whole list do 1.5 x the
// instructions of two.

template <bool COUNT, bool DEPTH = false>
static int launch_fwd(int32_t C, int64_t n_isects, const float* splats, const int32_t* tile_offsets,
                      const int32_t* flatten_ids, const float* backgrounds, int32_t width, int32_t height,
                      int32_t tile_width, int32_t tile_height, float* render_colors, float* render_alphas,
                      int32_t* last_ids, uint64_t* pair_counters, const int32_t* tile_order, egs_stream_t stream,
                      float* checkpoints = nullptr, int32_t segment = 0, int32_t seg_min_len = 0) {
  dim3 grid(tile_width, tile_height, C);
  const int n_tiles = C * tile_width * tile_height;
  float4* ck = segment > 0 ? reinterpret_cast<float4*>(checkpoints) : nullptr;
  const float4* sp = reinterpret_cast<const float4*>(splats);
  unsigned long long* pc = reinterpret_cast<unsigned long long*>(pair_counters);
  cudaStream_t st = (cudaStream_t)stream;
  rasterize_fwd_kernel<COUNT, DEPTH><<<grid, Geo<2, 2>::kThreads, 0, st>>>(
      n_isects, sp, tile_offsets, flatten_ids, backgrounds, width, height, tile_width, tile_height, n_tiles,
      render_colors, render_alphas, last_ids, pc, ck, segment, seg_min_len > segment ? seg_min_len : segment + 1,
      tile_order);
  return check_launch("rasterize_fwd_kernel");
}

extern "C" int egs_rasterize_fwd(int32_t C, int32_t N, int64_t n_isects, const float* splats,
                                 const int32_t* tile_offsets, const int32_t* flatten_ids, const float* backgrounds,
                                 int32_t width, int32_t height, int32_t tile_width, int32_t tile_height,
                                 float* render_colors, float* render_alphas, int32_t* last_ids,
                                 const int32_t* tile_order, egs_stream_t stream) {
  (void)N;
  if (int rc = check_raster_args("rasterize_fwd", C, n_isects, width, height, tile_width, tile_height)) return rc;
  if (C == 0) return 0;
  return launch_fwd<false>(C, n_isects, splats, tile_offsets, flatten_ids, backgrounds, width, height, tile_width,
                           tile_height, render_colors, render_alphas, last_ids, nullptr, tile_order, stream);
}

// Instrumented variant for the roofline model: also accumulates P_eval and P_acc (SURVEY.md §8d, in the
// reference algorithm's sense: culled list entries count as evaluated) into pair_counters[2] (device,
// uint64, caller-zeroed).  Not used on the product path.
extern "C" int egs_rasterize_fwd_count(int32_t C, int32_t N, int64_t n_isects, const float* splats,
                                       const int32_t* tile_offsets, const int32_t* flatten_ids,
                                       const float* backgrounds, int32_t width, int32_t height, int32_t tile_width,
                                       int32_t tile_height, float* render_colors, float* render_alphas,
                                       int32_t* last_ids, uint64_t* pair_counters, egs_stream_t stream) {
  (void)N;
  if (int rc = check_raster_args("rasterize_fwd_count", C, n_isects, width, height, tile_width, tile_height)) return rc;
  if (C == 0) return 0;
  return launch_fwd<true>(C, n_isects, splats, tile_offsets, flatten_ids, backgrounds, width, height, tile_width,
                          tile_height, render_colors, render_alphas, last_ids, pair_counters, nullptr, stream);
}

static int segment_ok(const char* who, int32_t segment) {
  EGS_REQUIRE(segment == 0 || (segment >= 64 && segment % 64 == 0), "%s: segment=%d must be 0 or a multiple of 64", who, segment);
  return 0;
}

extern "C" int64_t egs_rasterize_checkpoint_bytes(int64_t n_isects, int32_t segment) {
  if (n_isects < 0) n_isects = -n_isects;  // sentinel mode: the capacity
  if (segment <= 0) return 0;
  // slots 0 .. n_isects / segment, each: 2 warps x 4 pixels x 32 lanes x float4
  return (n_isects / segment + 2) * (int64_t)(Geo<2, 2>::kWarps * Geo<2, 2>::NP * 32 * sizeof(float4));
}

extern "C" int egs_rasterize_fwd_checkpointed(int32_t C, int32_t N, int64_t n_isects, const float* splats,
                                              const int32_t* tile_offsets, const int32_t* flatten_ids,
                                              const float* backgrounds, int32_t width, int32_t height,
                                              int32_t tile_width, int32_t tile_height, float* render_colors,
                                              float* render_alphas, int32_t* last_ids, float* checkpoints,
                                              int32_t segment, int32_t seg_min_len, const int32_t* tile_order,
                                              egs_stream_t stream) {
  (void)N;
  if (int rc = check_raster_args("rasterize_fwd_checkpointed", C, n_isects, width, height, tile_width, tile_height)) return rc;
  if (int rc = segment_ok("rasterize_fwd_checkpointed", segment)) return rc;
  EGS_REQUIRE(segment == 0 || checkpoints != nullptr, "rasterize_fwd_checkpointed: checkpoints buffer is required");
  if (C == 0) return 0;
  return launch_fwd<false>(C, n_isects, splats, tile_offsets, flatten_ids, backgrounds, width, height, tile_width,
                           tile_height, render_colors, render_alphas, last_ids, nullptr, tile_order, stream, checkpoints,
                           segment, seg_min_len);
}

template <bool DEPTH = false>
static int launch_bwd(int32_t C, int64_t n_isects, const float* splats, const int32_t* tile_offsets,
                      const int32_t* flatten_ids, const float* backgrounds, int32_t width, int32_t height,
                      int32_t tile_width, int32_t tile_height, const float* render_alphas, const int32_t* last_ids,
                      const float* v_render_colors, const float* v_render_alphas, float* v_splats,
                      const float* render_colors, const float* checkpoints, int32_t segment, int32_t seg_min_len,
                      const int32_t* tile_order, egs_stream_t stream) {
  seg_min_len = seg_min_len > segment ? seg_min_len : segment + 1;
  dim3 grid(tile_width, tile_height, C);
  const int n_tiles = C * tile_width * tile_height;
  const float4* sp = reinterpret_cast<const float4*>(splats);
  const float4* ck = segment > 0 ? reinterpret_cast<const float4*>(checkpoints) : nullptr;
  cudaStream_t st = (cudaStream_t)stream;
  // the segment launch goes first: its warps all have full segments to replay, the tile launch then fills in
  const int64_t n_slots = ck != nullptr ? (n_isects < 0 ? -n_isects : n_isects) / segment : 0;
  if (n_slots > 0)
    rasterize_bwd_kernel<DEPTH><<<(unsigned)n_slots, Geo<2, 2>::kThreads, 0, st>>>(
        n_isects, sp, tile_offsets, flatten_ids, backgrounds, width, height, tile_width, tile_height, n_tiles,
        render_alphas, last_ids, v_render_colors, v_render_alphas, v_splats, render_colors, ck, segment, seg_min_len, 1, nullptr);
  rasterize_bwd_kernel<DEPTH><<<grid, Geo<2, 2>::kThreads, 0, st>>>(
      n_isects, sp, tile_offsets, flatten_ids, backgrounds, width, height, tile_width, tile_height, n_tiles,
      render_alphas, last_ids, v_render_colors, v_render_alphas, v_splats, render_colors, ck, segment, seg_min_len, 0, tile_order);
  return check_launch("rasterize_bwd_kernel", 1 + (n_slots > 0 ? 1 : 0));
}

extern "C" int egs_rasterize_bwd(int32_t C, int32_t N, int64_t n_isects, const float* splats,
                                 const int32_t* tile_offsets, const int32_t* flatten_ids, const float* backgrounds,
                                 int32_t width, int32_t height, int32_t tile_width, int32_t tile_height,
                                 const float* render_alphas, const int32_t* last_ids, const float* v_render_colors,
                                 const float* v_render_alphas, float* v_splats, const int32_t* tile_order,
                                 egs_stream_t stream) {
  (void)N;
  if (int rc = check_raster_args("rasterize_bwd", C, n_isects, width, height, tile_width, tile_height)) return rc;
  if (C == 0 || n_isects == 0) return 0;
  return launch_bwd(C, n_isects, splats, tile_offsets, flatten_ids, backgrounds, width, height, tile_width, tile_height,
                    render_alphas, last_ids, v_render_colors, v_render_alphas, v_splats, nullptr, nullptr, 0, 0, tile_order,
                    stream);
}

extern "C" int egs_rasterize_bwd_segmented(int32_t C, int32_t N, int64_t n_isects, const float* splats,
                                           const int32_t* tile_offsets, const int32_t* flatten_ids,
                                           const float* backgrounds, int32_t width, int32_t height, int32_t tile_width,
                                           int32_t tile_height, const float* render_colors, const float* render_alphas,
                                           const int32_t* last_ids, const float* v_render_colors,
                                           const float* v_render_alphas, const float* checkpoints, int32_t segment,
                                           int32_t seg_min_len, float* v_splats, const int32_t* tile_order,
                                           egs_stream_t stream) {
  (void)N;
  if (int rc = check_raster_args("rasterize_bwd_segmented", C, n_isects, width, height, tile_width, tile_height)) return rc;
  if (int rc = segment_ok("rasterize_bwd_segmented", segment)) return rc;
  EGS_REQUIRE(segment == 0 || (checkpoints != nullptr && render_colors != nullptr),
              "rasterize_bwd_segmented: checkpoints and render_colors are required");
  if (C == 0 || n_isects == 0) return 0;
  return launch_bwd(C, n_isects, splats, tile_offsets, flatten_ids, backgrounds, width, height, tile_width, tile_height,
                    render_alphas, last_ids, v_render_colors, v_render_alphas, v_splats, render_colors, checkpoints,
                    segment, seg_min_len, tile_order, stream);
}

// ---- RGB plus expected depth: the DEPTH forms, 4 floats per pixel, no checkpoints --------------------------------------
extern "C" int egs_rasterize_fwd_depth(int32_t C, int32_t N, int64_t n_isects, const float* splats,
                                       const int32_t* tile_offsets, const int32_t* flatten_ids, const float* backgrounds,
                                       int32_t width, int32_t height, int32_t tile_width, int32_t tile_height,
                                       float* render_colors, float* render_alphas, int32_t* last_ids,
                                       const int32_t* tile_order, egs_stream_t stream) {
  (void)N;
  if (int rc = check_raster_args("rasterize_fwd_depth", C, n_isects, width, height, tile_width, tile_height)) return rc;
  if (C == 0) return 0;
  return launch_fwd<false, true>(C, n_isects, splats, tile_offsets, flatten_ids, backgrounds, width, height, tile_width,
                                 tile_height, render_colors, render_alphas, last_ids, nullptr, tile_order, stream);
}

extern "C" int egs_rasterize_bwd_depth(int32_t C, int32_t N, int64_t n_isects, const float* splats,
                                       const int32_t* tile_offsets, const int32_t* flatten_ids, const float* backgrounds,
                                       int32_t width, int32_t height, int32_t tile_width, int32_t tile_height,
                                       const float* render_alphas, const int32_t* last_ids,
                                       const float* v_render_colors, const float* v_render_alphas, float* v_splats,
                                       const int32_t* tile_order, egs_stream_t stream) {
  (void)N;
  if (int rc = check_raster_args("rasterize_bwd_depth", C, n_isects, width, height, tile_width, tile_height)) return rc;
  if (C == 0 || n_isects == 0) return 0;
  return launch_bwd<true>(C, n_isects, splats, tile_offsets, flatten_ids, backgrounds, width, height, tile_width,
                          tile_height, render_alphas, last_ids, v_render_colors, v_render_alphas, v_splats, nullptr,
                          nullptr, 0, 0, tile_order, stream);
}

// ---- colours with any number of channels -------------------------------------------------------------------------
static int check_feature_args(const char* who, int32_t N, const float* features, int32_t feat_stride,
                              int32_t shared_rows, int32_t D, int32_t c0, int32_t CH) {
  EGS_REQUIRE(CH == 1 || CH == 2 || CH == 4 || CH == 8 || CH == 16 || CH == 32,
              "%s: CH=%d is not an instantiated chunk width (1, 2, 4, 8, 16, 32)", who, CH);
  EGS_REQUIRE(D >= 1, "%s: D=%d must be >= 1", who, D);
  EGS_REQUIRE(c0 >= 0 && c0 < D, "%s: c0=%d out of [0, D=%d)", who, c0, D);
  EGS_REQUIRE(shared_rows == 0 || shared_rows == 1, "%s: shared_rows must be 0 or 1", who);
  EGS_REQUIRE(N >= 0, "%s: N=%d must be >= 0", who, N);
  EGS_REQUIRE(features != nullptr, "%s: features is required", who);
  EGS_REQUIRE(feat_stride >= c0 + CH, "%s: feat_stride=%d < c0 + CH = %d (rows are read CH floats wide)", who,
              feat_stride, c0 + CH);
  const int align = CH < 4 ? CH : 4;  // floats per cp.async copy of a row
  EGS_REQUIRE(feat_stride % align == 0 && c0 % align == 0 && (uintptr_t)features % (4 * align) == 0,
              "%s: CH=%d reads %d-byte pieces: feat_stride=%d, c0=%d and the features pointer must be aligned to them",
              who, CH, 4 * align, feat_stride, c0);
  return 0;
}

template <int CH>
static size_t feature_smem_bytes(bool backward) {
  using G = typename FeatGeo<CH>::G;
  return G::kWarps * (sizeof(FeatStage<G::kBatch, CH>) + (backward ? kFeatRedRows * kRedStride * sizeof(float) : 0));
}

template <int CH>
static int launch_fwd_features(int32_t C, int32_t N, int64_t n_isects, const float* splats, const int32_t* tile_offsets,
                               const int32_t* flatten_ids, const float* features, int32_t feat_stride,
                               int32_t shared_rows, int32_t D, int32_t c0, const float* backgrounds, int32_t width,
                               int32_t height, int32_t tile_width, int32_t tile_height, float* render_colors,
                               float* render_alphas, int32_t* last_ids, const int32_t* tile_order, cudaStream_t st) {
  const size_t smem = feature_smem_bytes<CH>(false);
  EGS_CUDA(cudaFuncSetAttribute(rasterize_fwd_features_kernel<CH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid(tile_width, tile_height, C);
  rasterize_fwd_features_kernel<CH><<<grid, FeatGeo<CH>::G::kThreads, smem, st>>>(
      n_isects, reinterpret_cast<const float4*>(splats), tile_offsets, flatten_ids, features, feat_stride,
      shared_rows ? N : 0, D, c0, backgrounds, width, height, tile_width, tile_height, C * tile_width * tile_height,
      render_colors, render_alphas, last_ids, tile_order);
  return check_launch("rasterize_fwd_features_kernel");
}

template <int CH>
static int launch_bwd_features(int32_t C, int32_t N, int64_t n_isects, const float* splats, const int32_t* tile_offsets,
                               const int32_t* flatten_ids, const float* features, int32_t feat_stride,
                               int32_t shared_rows, int32_t D, int32_t c0, const float* backgrounds, int32_t width,
                               int32_t height, int32_t tile_width, int32_t tile_height, const float* render_alphas,
                               const int32_t* last_ids, const float* v_render_colors, const float* v_render_alphas,
                               float* v_splats, float* v_features, const int32_t* tile_order, cudaStream_t st) {
  const size_t smem = feature_smem_bytes<CH>(true);
  EGS_CUDA(cudaFuncSetAttribute(rasterize_bwd_features_kernel<CH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid(tile_width, tile_height, C);
  rasterize_bwd_features_kernel<CH><<<grid, FeatGeo<CH>::G::kThreads, smem, st>>>(
      n_isects, reinterpret_cast<const float4*>(splats), tile_offsets, flatten_ids, features, feat_stride,
      shared_rows ? N : 0, D, c0, backgrounds, width, height, tile_width, tile_height, C * tile_width * tile_height,
      render_alphas, last_ids, v_render_colors, v_render_alphas, v_splats, v_features, tile_order);
  return check_launch("rasterize_bwd_features_kernel");
}

#define EGS_FEATURE_DISPATCH(LAUNCH, ...)        \
  switch (CH) {                                  \
    case 1: return LAUNCH<1>(__VA_ARGS__);       \
    case 2: return LAUNCH<2>(__VA_ARGS__);       \
    case 4: return LAUNCH<4>(__VA_ARGS__);       \
    case 8: return LAUNCH<8>(__VA_ARGS__);       \
    case 16: return LAUNCH<16>(__VA_ARGS__);     \
    default: return LAUNCH<32>(__VA_ARGS__);     \
  }

extern "C" int egs_rasterize_fwd_features(int32_t C, int32_t N, int64_t n_isects, const float* splats,
                                          const int32_t* tile_offsets, const int32_t* flatten_ids,
                                          const float* features, int32_t feat_stride, int32_t shared_rows, int32_t D,
                                          int32_t c0, int32_t CH, const float* backgrounds, int32_t width,
                                          int32_t height, int32_t tile_width, int32_t tile_height,
                                          float* render_colors, float* render_alphas, int32_t* last_ids,
                                          const int32_t* tile_order, egs_stream_t stream) {
  if (int rc = check_raster_args("rasterize_fwd_features", C, n_isects, width, height, tile_width, tile_height)) return rc;
  if (int rc = check_feature_args("rasterize_fwd_features", N, features, feat_stride, shared_rows, D, c0, CH)) return rc;
  EGS_REQUIRE(render_colors != nullptr, "rasterize_fwd_features: render_colors is required");
  if (C == 0) return 0;
  EGS_FEATURE_DISPATCH(launch_fwd_features, C, N, n_isects, splats, tile_offsets, flatten_ids, features, feat_stride,
                       shared_rows, D, c0, backgrounds, width, height, tile_width, tile_height, render_colors,
                       render_alphas, last_ids, tile_order, (cudaStream_t)stream)
}

extern "C" int egs_rasterize_bwd_features(int32_t C, int32_t N, int64_t n_isects, const float* splats,
                                          const int32_t* tile_offsets, const int32_t* flatten_ids,
                                          const float* features, int32_t feat_stride, int32_t shared_rows, int32_t D,
                                          int32_t c0, int32_t CH, const float* backgrounds, int32_t width,
                                          int32_t height, int32_t tile_width, int32_t tile_height,
                                          const float* render_alphas, const int32_t* last_ids,
                                          const float* v_render_colors, const float* v_render_alphas, float* v_splats,
                                          float* v_features, const int32_t* tile_order, egs_stream_t stream) {
  if (int rc = check_raster_args("rasterize_bwd_features", C, n_isects, width, height, tile_width, tile_height)) return rc;
  if (int rc = check_feature_args("rasterize_bwd_features", N, features, feat_stride, shared_rows, D, c0, CH)) return rc;
  if (C == 0 || n_isects == 0) return 0;
  EGS_FEATURE_DISPATCH(launch_bwd_features, C, N, n_isects, splats, tile_offsets, flatten_ids, features, feat_stride,
                       shared_rows, D, c0, backgrounds, width, height, tile_width, tile_height, render_alphas, last_ids,
                       v_render_colors, v_render_alphas, v_splats, v_features, tile_order, (cudaStream_t)stream)
}
