// mbarrier + TMA bulk-copy (cp.async.bulk) primitives for the feature-streaming kernels.
//
// The donor feature maps are [B, C, N] planes of fp32, or of bf16 held as raw 16-bit values
// (autocast-trained donors; converted exactly to fp32 in registers by feat_f32).  A producer warp
// streams [CH channels x T pixels] stages into a shared-memory ring with 1-D bulk async copies
// (one per channel row, completion counted on an mbarrier); consumer warps read the stage from
// shared memory.  Rows whose start is only element-aligned (HRNet: N = 155*155 is odd) are
// fetched as the enclosing 16-byte-aligned span and indexed with a per-row shift of
// 0..FeatElem<FT>::G-1 elements (0..3 fp32, 0..7 bf16), so the same pipeline serves every plane
// size.  The span never leaves the 16-byte granules that hold valid bytes of the tensor.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace rhseg {

// Feature element types: float, or uint16_t = the bit pattern of a bf16 value.  G = elements per 16-byte granule.
template <typename FT> struct FeatElem;
template <> struct FeatElem<float> { static constexpr int G = 4, LOG2_G = 2, LOG2_SIZE = 2; };
template <> struct FeatElem<uint16_t> { static constexpr int G = 8, LOG2_G = 3, LOG2_SIZE = 1; };

__device__ __forceinline__ float feat_f32(float v) { return v; }
__device__ __forceinline__ float feat_f32(uint16_t v) { return __uint_as_float((uint32_t)v << 16); }  // exact
__device__ __forceinline__ float bf16_lo(uint32_t w) { return __uint_as_float(w << 16); }       // element 2i of a pair
__device__ __forceinline__ float bf16_hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }  // element 2i+1
// fp32 pair -> two bf16 (round to nearest even, cvt.rn.bf16x2.f32); `lo` goes to the lower address
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ uint16_t to_bf16_bits(float v) { return __bfloat16_as_ushort(__float2bfloat16_rn(v)); }

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// Barriers of an NS-stage ring: full[i] = bars[i] completes on `producers` arrivals (plus the copied bytes), empty[i] =
// bars[NS + i] on `consumer_warps` arrivals.  Called by the whole CTA.
template <int NS>
__device__ __forceinline__ void ring_bars_init(uint64_t* bars, uint32_t producers, uint32_t consumer_warps) {
  if (threadIdx.x == 0) {
    for (int i = 0; i < NS; ++i) {
      mbar_init(smem_u32(&bars[i]), producers);
      mbar_init(smem_u32(&bars[NS + i]), consumer_warps);
    }
    mbar_fence_init();
  }
  __syncthreads();
}
// L2 policy for read-once streams: do not let 300-400 MB of features evict the small tensors
// (logits, targets, probabilities) that the following kernels re-read.
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
// 1-D bulk async copy global -> shared, completion (bytes) signalled on `bar`.
// dst / src 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
      ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(policy)
      : "memory");
}
// named barrier among the consumer warps only (the producer warp never joins)
__device__ __forceinline__ void consumer_sync(int nthreads) {
  asm volatile("bar.sync 1, %0;" ::"r"(nthreads) : "memory");
}

// shift (elements) of the 16-byte-aligned span that contains element `e` of a tensor whose base
// pointer sits `a0` elements past a 16-byte boundary
template <typename FT = float>
__device__ __forceinline__ int row_shift(long e, int a0) { return (int)((e + a0) & (FeatElem<FT>::G - 1)); }
// a0 of a feature tensor (host side)
template <typename FT>
inline int base_shift(const void* p) {
  return (int)((reinterpret_cast<uintptr_t>(p) >> FeatElem<FT>::LOG2_SIZE) & (FeatElem<FT>::G - 1));
}

// Pipeline shape: NCW consumer warps + NPW producer warps, CH channel rows per stage, NS stages.
// One elected lane per producer warp issues the row copies of its share of a stage (measured:
// a single issuing lane sustains ~1 copy / 90 cycles, faster than 16 lanes issuing one each).
template <int NCW_, int CH_, int NS_, int NPW_ = 1>
struct PipeCfg {
  static constexpr int NCW = NCW_;
  static constexpr int NPW = NPW_;
  static constexpr int CONSUMERS = NCW_ * 32;
  static constexpr int THREADS = CONSUMERS + NPW_ * 32;
  static constexpr int CH = CH_;
  static constexpr int NS = NS_;
};

// Issues the row copies r = first, first+step, ... < ccnt of one stage (rows N elements apart,
// starting at element e0 of `base`) and arrives on `bar` with the byte count.  Single thread.
template <typename FT>
__device__ __forceinline__ void issue_stage_rows(const FT* base, long e0, int N, int t_act, int ccnt, int first,
                                                 int step, int a0, uint32_t dst_row0, uint32_t row_pitch_bytes,
                                                 uint32_t bar, uint64_t pol) {
  constexpr int G = FeatElem<FT>::G, LOG2_G = FeatElem<FT>::LOG2_G;
  uint32_t total = 0;
  for (int r = first; r < ccnt; r += step) {
    const long e = e0 + (long)r * N;
    const int sh = row_shift<FT>(e, a0);
    const uint32_t bytes = (uint32_t)(((sh + t_act + G - 1) >> LOG2_G) << 4);
    bulk_g2s(dst_row0 + (uint32_t)r * row_pitch_bytes, base + (e - sh), bytes, bar, pol);
    total += bytes;
  }
  mbar_arrive_expect_tx(bar, total);
}

}  // namespace rhseg
