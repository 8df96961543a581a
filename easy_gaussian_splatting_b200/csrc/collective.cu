// Gradient exchange of the view-sharded training step (SURVEY.md §8e) as a hand-written two-shot all-reduce over
// NVLink peer memory: every rank's flat gradient bucket lives in symmetric memory (the same virtual layout on every
// GPU, each mapped into every peer), rank r sums slice r of all buckets with peer LOADS and writes the result back
// into every bucket with peer STORES.  Each GPU moves (R-1)/R of the bucket in and out once — the NVSwitch gives
// every pair full bandwidth, so this is the traffic floor of an all-reduce — and the sum is taken in rank order by
// exactly one GPU per element, so all replicas receive bit-identical gradients.  The two inter-rank barriers around
// the kernel are the caller's (torch symmetric-memory signal pads, stream ordered).
#include "egs_common.cuh"

namespace egs {

constexpr int kArThreads = 256;
constexpr int kArMaxWorld = 16;
// float4s a thread of the NVLS kernel keeps in flight per trip / resident CTAs per SM the grid is capped at
// (build-time A/B knobs, scripts/build_variant.py)
#ifndef EGS_AR_UNROLL
#define EGS_AR_UNROLL 2
#endif
#ifndef EGS_AR_CTAS_PER_SM
#define EGS_AR_CTAS_PER_SM 8
#endif
// Two ranges are used.  With room for fewer than 8, ptxas (CUDA 12.9) copies the kernel argument to a stack frame for
// the loop over the ranges, and the two-shot kernels for 5-8 GPUs need up to 44 more registers.
constexpr int kArMaxRanges = 8;

// The float4 ranges one launch reduces, each cut into `world` slices of which this rank owns one: the SUM range carries
// the gradients (and the two accumulator rows of the densify statistics), the MAX range behind it the max_radii row.
struct ArRanges {
  int n;
  int64_t off4[kArMaxRanges];  // first float4 of the range
  int64_t n4[kArMaxRanges];    // float4s in the range
  int is_max[kArMaxRanges];
};

template <int WORLD>
__global__ void __launch_bounds__(kArThreads) allreduce_two_shot_kernel(float* const* __restrict__ bufs, int rank,
                                                                        const ArRanges rg) {
  float4* b[WORLD];
#pragma unroll
  for (int p = 0; p < WORLD; ++p) b[p] = reinterpret_cast<float4*>(bufs[p]);
  const int64_t stride = (int64_t)gridDim.x * kArThreads;
  for (int r = 0; r < rg.n; ++r) {
    const int64_t per = (rg.n4[r] + WORLD - 1) / WORLD;
    const int64_t lo = rg.off4[r] + (int64_t)rank * per, hi = min(rg.off4[r] + rg.n4[r], lo + per);
    const bool sum = rg.is_max[r] == 0;
    for (int64_t i = lo + (int64_t)blockIdx.x * kArThreads + threadIdx.x; i < hi; i += 2 * stride) {
      const int64_t i1 = i + stride;
      const bool two = i1 < hi;
      float4 v0[WORLD], v1[WORLD];
#pragma unroll
      for (int p = 0; p < WORLD; ++p) {  // every peer load of the trip in flight before the first add
        v0[p] = b[p][i];
        v1[p] = two ? b[p][i1] : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      float4 a0 = v0[0], a1 = v1[0];
#pragma unroll
      for (int p = 1; p < WORLD; ++p) {  // fixed rank order: deterministic, identical on every replica
        a0.x = sum ? a0.x + v0[p].x : fmaxf(a0.x, v0[p].x); a0.y = sum ? a0.y + v0[p].y : fmaxf(a0.y, v0[p].y);
        a0.z = sum ? a0.z + v0[p].z : fmaxf(a0.z, v0[p].z); a0.w = sum ? a0.w + v0[p].w : fmaxf(a0.w, v0[p].w);
        a1.x = sum ? a1.x + v1[p].x : fmaxf(a1.x, v1[p].x); a1.y = sum ? a1.y + v1[p].y : fmaxf(a1.y, v1[p].y);
        a1.z = sum ? a1.z + v1[p].z : fmaxf(a1.z, v1[p].z); a1.w = sum ? a1.w + v1[p].w : fmaxf(a1.w, v1[p].w);
      }
#pragma unroll
      for (int p = 0; p < WORLD; ++p) {
        b[p][i] = a0;
        if (two) b[p][i1] = a1;
      }
    }
  }
}

// MAX of non-negative floats == MAX of their bit patterns as unsigned integers, which is what the switch offers
// (multimem.ld_reduce has .add for f32 but .min/.max only for integer and 16-bit float types).
__device__ __forceinline__ void multimem_max_u32x4(uint32_t* p) {
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    uint32_t v;
    asm volatile("multimem.ld_reduce.relaxed.sys.global.max.u32 %0, [%1];" : "=r"(v) : "l"(p + k) : "memory");
    asm volatile("multimem.st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p + k), "r"(v) : "memory");
  }
}

// Same exchange through the NVSwitch's multicast / in-switch reduction (NVLS): one multimem.ld_reduce pulls the SUM
// of an element over all replicas (the switch reads every GPU's copy and adds in flight), one multimem.st pushes it
// back to all of them.  Per GPU only 1/R of the bucket crosses its own link in each direction.
__global__ void __launch_bounds__(kArThreads) allreduce_multimem_kernel(float* __restrict__ mc, int world, int rank,
                                                                        const ArRanges rg) {
  const int64_t stride = (int64_t)gridDim.x * kArThreads;
  float4* m4 = reinterpret_cast<float4*>(mc);
  for (int r = 0; r < rg.n; ++r) {
    const int64_t per = (rg.n4[r] + world - 1) / world;
    const int64_t lo = rg.off4[r] + (int64_t)rank * per, hi = min(rg.off4[r] + rg.n4[r], lo + per);
    if (rg.is_max[r]) {  // a few MB at most: scalar u32 ops
      for (int64_t i = lo + (int64_t)blockIdx.x * kArThreads + threadIdx.x; i < hi; i += stride)
        multimem_max_u32x4(reinterpret_cast<uint32_t*>(mc) + 4 * i);
      continue;
    }
    constexpr int U = EGS_AR_UNROLL;
    for (int64_t i = lo + (int64_t)blockIdx.x * kArThreads + threadIdx.x; i < hi; i += U * stride) {
      float4 v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {  // every in-switch reduction of the trip in flight before the first store
        const int64_t iu = i + u * stride;
        v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (iu < hi)
          asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
                       : "=f"(v[u].x), "=f"(v[u].y), "=f"(v[u].z), "=f"(v[u].w) : "l"(m4 + iu) : "memory");
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t iu = i + u * stride;
        if (iu < hi)
          asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(m4 + iu), "f"(v[u].x), "f"(v[u].y), "f"(v[u].z), "f"(v[u].w) : "memory");
      }
    }
  }
}

// [0, n_sum) summed, [n_sum, n_sum + n_max) maximised
static int make_ranges(const char* who, int64_t n_sum_floats, int64_t n_max_floats, ArRanges& rg, int64_t& total4) {
  const int64_t offsets[2] = {0, n_sum_floats}, lengths[2] = {n_sum_floats, n_max_floats};
  rg.n = 0;
  total4 = 0;
  for (int r = 0; r < 2; ++r) {
    EGS_REQUIRE(offsets[r] >= 0 && lengths[r] >= 0 && offsets[r] % 4 == 0 && lengths[r] % 4 == 0,
                "%s: range %d (offset %lld, length %lld floats) must be non-negative multiples of 4", who, r,
                (long long)offsets[r], (long long)lengths[r]);
    if (lengths[r] == 0) continue;
    rg.off4[rg.n] = offsets[r] / 4;
    rg.n4[rg.n] = lengths[r] / 4;
    rg.is_max[rg.n] = r == 1;
    total4 += rg.n4[rg.n];
    ++rg.n;
  }
  return 0;
}

static unsigned ar_blocks(int64_t total4, int world) {
  int64_t blocks = ceil_div(ceil_div(total4, world), 2 * kArThreads);
  if (blocks < 1) blocks = 1;
  if (blocks > 148 * EGS_AR_CTAS_PER_SM) blocks = 148 * EGS_AR_CTAS_PER_SM;
  return (unsigned)blocks;
}

}  // namespace egs

using namespace egs;

extern "C" int egs_allreduce_f32_multimem(int32_t world, int32_t rank, void* multicast_ptr, int64_t n_sum_floats,
                                          int64_t n_max_floats, egs_stream_t stream) {
  EGS_REQUIRE(world >= 1 && rank >= 0 && rank < world, "allreduce_multimem: bad world=%d rank=%d", world, rank);
  EGS_REQUIRE(multicast_ptr != nullptr, "allreduce_multimem: multicast pointer is required");
  ArRanges rg;
  int64_t total4 = 0;
  if (int rc = make_ranges("allreduce_multimem", n_sum_floats, n_max_floats, rg, total4)) return rc;
  if (total4 == 0 || world == 1) return 0;
  allreduce_multimem_kernel<<<ar_blocks(total4, world), kArThreads, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<float*>(multicast_ptr), world, rank, rg);
  return check_launch("allreduce_multimem_kernel");
}

extern "C" int egs_allreduce_f32_peer(int32_t world, int32_t rank, const void* peer_buffers_dev, int64_t n_sum_floats,
                                      int64_t n_max_floats, egs_stream_t stream) {
  EGS_REQUIRE(world >= 1 && world <= kArMaxWorld && rank >= 0 && rank < world, "allreduce_peer: bad world=%d rank=%d", world, rank);
  EGS_REQUIRE(peer_buffers_dev != nullptr, "allreduce_peer: peer buffer table is required");
  ArRanges rg;
  int64_t total4 = 0;
  if (int rc = make_ranges("allreduce_peer", n_sum_floats, n_max_floats, rg, total4)) return rc;
  if (total4 == 0 || world == 1) return 0;
  float* const* bufs = reinterpret_cast<float* const*>(peer_buffers_dev);
  const unsigned grid = ar_blocks(total4, world);
  cudaStream_t st = (cudaStream_t)stream;
  switch (world) {
    case 2: allreduce_two_shot_kernel<2><<<grid, kArThreads, 0, st>>>(bufs, rank, rg); break;
    case 3: allreduce_two_shot_kernel<3><<<grid, kArThreads, 0, st>>>(bufs, rank, rg); break;
    case 4: allreduce_two_shot_kernel<4><<<grid, kArThreads, 0, st>>>(bufs, rank, rg); break;
    case 5: allreduce_two_shot_kernel<5><<<grid, kArThreads, 0, st>>>(bufs, rank, rg); break;
    case 6: allreduce_two_shot_kernel<6><<<grid, kArThreads, 0, st>>>(bufs, rank, rg); break;
    case 7: allreduce_two_shot_kernel<7><<<grid, kArThreads, 0, st>>>(bufs, rank, rg); break;
    case 8: allreduce_two_shot_kernel<8><<<grid, kArThreads, 0, st>>>(bufs, rank, rg); break;
    default: return fail(EGS_ERR_UNSUPPORTED, "allreduce_peer: world=%d is not instantiated (2..8)", world);
  }
  return check_launch("allreduce_two_shot_kernel");
}
