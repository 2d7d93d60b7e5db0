// 1x1-conv backward of the head for channels-last features (RHSEG_FEATS_NHWC), fp32 and bf16: dfeats written
// channels-last, the same fp64 sums S / s as conv_bwd_kernel.  DESIGN.md 3.8.
//
//   dfeats[b,n,c] = sum_k w[b,k,c] dz[b,k,n]      S[b,k,c] = sum_n dz[b,k,n] feats[b,n,c]      s[b,k] = sum_n dz[b,k,n]
//
// In NHWC a run of pixels is one contiguous block of memory, all channels included.  Work unit = (sample, tile of TP
// pixels); the producer warp streams the tile's [TP x C] block with ONE 1-D bulk copy into a shared-memory ring.
// Consumer thread (pl, cg) owns the 16-byte channel group cg (4 fp32 / 8 bf16 channels) and the pixels pl, pl + PL, ...
// of each tile: per pixel one 128-bit shared load, K loads of dz (the same address for the threads of a pixel lane: L1
// broadcasts), the K x group products summed over pixels in registers (no shuffles), and one 16-byte store of dfeats.
// The per-thread sums are reduced over the PL pixel lanes in shared memory and leave the CTA as fp64 atomics when the
// sample changes (and every FLUSH_UNITS units).  dfeats takes the per-element k order of conv_bwd_kernel (a = 0, then
// fmaf over k ascending, K = 3 padded to 4), so it equals the NCHW kernel's bit for bit.
#include <algorithm>
#include "conv_bwd_kernel.cuh"
#include "feats_nhwc.cuh"

namespace rhseg {

constexpr int BWD_NHWC_MAX_CONS = 256;         // consumer threads at most (plus one producer warp)
constexpr int BWD_NHWC_STAGE_BYTES = 24 << 10;  // target size of a ring stage
constexpr int BWD_NHWC_NS = 4;

__device__ __forceinline__ void st_group(float* p, const float (&o)[4]) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(o[0]), "f"(o[1]), "f"(o[2]), "f"(o[3])
               : "memory");
}
__device__ __forceinline__ void st_group(uint16_t* p, const float (&o)[8]) {  // rounded to nearest even here, once
  asm volatile("st.global.L1::no_allocate.v4.b32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(pack_bf16x2(o[0], o[1])),
               "r"(pack_bf16x2(o[2], o[3])), "r"(pack_bf16x2(o[4], o[5])), "r"(pack_bf16x2(o[6], o[7]))
               : "memory");
}

template <typename FT, int K>
__global__ void __launch_bounds__(BWD_NHWC_MAX_CONS + 32)
conv_bwd_nhwc_kernel(const FT* __restrict__ feats, const float* __restrict__ dz, const float* __restrict__ eff_w, int C,
                     int N, int TP, int n_tiles, long units_total, int PL, int NG, int w_shared, FT* __restrict__ dfeats,
                     double* __restrict__ S, double* __restrict__ s, ParamTail pt) {
  pdl_wait();
  constexpr int VC = 16 / (int)sizeof(FT);  // channels of a 16-byte group
  constexpr int KC = (K == 3) ? 4 : K;      // as conv_bwd_kernel: dfeats sums over the zero-padded fourth channel
  constexpr int NS = BWD_NHWC_NS;
  constexpr int FLUSH_UNITS = 64;
  const int ncons = blockDim.x - 32;
  const int ncw = ncons >> 5;
  const size_t stage_elems = (size_t)TP * C;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);                 // full[NS], empty[NS]
  FT* ring = reinterpret_cast<FT*>(smem_raw + 128);                       // [NS][TP][C]
  float* red = reinterpret_cast<float*>(ring + (size_t)NS * stage_elems);  // [ncons][VC + 1]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long u_begin = units_total * blockIdx.x / gridDim.x;
  const long u_end = units_total * (blockIdx.x + 1) / gridDim.x;
  ring_bars_init<NS>(bars, 1, ncw);

  if (warp >= ncw) {
    // ------------------------------ producer ------------------------------
    if (lane == 0) {
      const uint64_t pol = l2_evict_first_policy();
      int slot = 0;
      uint32_t phase = 1;
      for (long u = u_begin; u < u_end; ++u) {
        mbar_wait(smem_u32(&bars[NS + slot]), phase);
        const int b = (int)(u / n_tiles);
        const int p0 = (int)(u - (long)b * n_tiles) * TP;
        const uint32_t bytes = (uint32_t)(min(TP, N - p0) * (size_t)C * sizeof(FT));
        bulk_g2s(smem_u32(ring + (size_t)slot * stage_elems), feats + ((size_t)b * N + p0) * C, bytes,
                 smem_u32(&bars[slot]), pol);
        mbar_arrive_expect_tx(smem_u32(&bars[slot]), bytes);
        if (++slot == NS) { slot = 0; phase ^= 1u; }
      }
    }
    return;
  }

  // -------------------------------- consumers --------------------------------
  const int pl = tid / NG, cg = tid - pl * NG;
  const bool active = pl < PL;
  const int c0 = cg * VC;
  float w[KC][VC], sacc[K][VC], s_acc[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    s_acc[k] = 0.f;
#pragma unroll
    for (int v = 0; v < VC; ++v) sacc[k][v] = 0.f;
  }
  int cur_b = -1, since_flush = 0;

  // per-thread sums -> reduced over the pixel lanes in shared memory -> fp64 atomics (all consumer threads take part)
  auto flush = [&](int fb) {
    float* r = red + (size_t)tid * (VC + 1);
#pragma unroll
    for (int k = 0; k < K; ++k) {
      consumer_sync(ncons);
#pragma unroll
      for (int v = 0; v < VC; ++v) r[v] = sacc[k][v];
      r[VC] = s_acc[k];
      consumer_sync(ncons);
      for (int c = tid; c < C; c += ncons) {
        const int g = c / VC, v = c - g * VC;
        double a = 0.0;
        for (int q = 0; q < PL; ++q) a += (double)red[(size_t)(q * NG + g) * (VC + 1) + v];
        atomicAdd(&S[((size_t)fb * K + k) * C + c], a);
      }
      if (tid == 0) {  // every channel group of a pixel lane summed the same dz: group 0 reports it
        double a = 0.0;
        for (int q = 0; q < PL; ++q) a += (double)red[(size_t)(q * NG) * (VC + 1) + VC];
        atomicAdd(&s[fb * K + k], a);
      }
      s_acc[k] = 0.f;
#pragma unroll
      for (int v = 0; v < VC; ++v) sacc[k][v] = 0.f;
    }
    since_flush = 0;
  };

  int slot = 0;
  uint32_t phase = 0;
  for (long u = u_begin; u < u_end; ++u) {
    const int b = (int)(u / n_tiles);
    const int p0 = (int)(u - (long)b * n_tiles) * TP;
    const int t_act = min(TP, N - p0);
    if (b != cur_b || since_flush >= FLUSH_UNITS) {  // uniform over the CTA
      if (cur_b >= 0) flush(cur_b);
      if (b != cur_b) {
        const float* wb = eff_w + (size_t)(w_shared ? 0 : b) * K * C;
#pragma unroll
        for (int k = 0; k < KC; ++k)
#pragma unroll
          for (int v = 0; v < VC; ++v) w[k][v] = (active && k < K) ? __ldg(wb + (size_t)k * C + c0 + v) : 0.f;
        cur_b = b;
      }
    }
    ++since_flush;
    mbar_wait(smem_u32(&bars[slot]), phase);
    if (active) {
      const FT* stg = ring + (size_t)slot * stage_elems + c0;
      const float* dzb = dz + (size_t)b * K * N + p0;
      FT* dfb = dfeats ? dfeats + ((size_t)b * N + p0) * C + c0 : nullptr;
#pragma unroll 2
      for (int p = pl; p < t_act; p += PL) {
        float f[VC];
        chunk_f32(lds128(stg + (size_t)p * C), f, FT{});
        float g[KC];
#pragma unroll
        for (int k = 0; k < KC; ++k) g[k] = k < K ? __ldg(dzb + (size_t)k * N + p) : 0.f;
#pragma unroll
        for (int k = 0; k < K; ++k) {
          s_acc[k] += g[k];
#pragma unroll
          for (int v = 0; v < VC; ++v) sacc[k][v] = fmaf(g[k], f[v], sacc[k][v]);
        }
        if (dfb) {
          float o[VC];
#pragma unroll
          for (int v = 0; v < VC; ++v) {
            float a = 0.f;
#pragma unroll
            for (int k = 0; k < KC; ++k) a = fmaf(w[k][v], g[k], a);
            o[v] = a;
          }
          st_group(dfb + (size_t)p * C, o);
        }
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(smem_u32(&bars[NS + slot]));
    if (++slot == NS) { slot = 0; phase ^= 1u; }
  }
  if (cur_b >= 0) flush(cur_b);
  if (pt.ticket != nullptr) level0_param_tail<K>(pt, S, s, C, ncons);
}

template <typename FT, int K>
static int launch_conv_bwd_nhwc(const FT* feats, const float* dz, const float* eff_w, int B, int C, int N, FT* dfeats,
                                double* S, double* s, int sm_count, cudaStream_t st, int w_shared, const ParamTail& pt) {
  constexpr int VC = 16 / (int)sizeof(FT);
  const int NG = C / VC;
  if (NG > BWD_NHWC_MAX_CONS) return RHSEG_ERR_UNSUPPORTED;
  const int PL = BWD_NHWC_MAX_CONS / NG;
  const int ncons = (PL * NG + 31) / 32 * 32;
  const size_t pix_bytes = (size_t)C * sizeof(FT);
  const int TP = std::max<int>(PL, (int)(BWD_NHWC_STAGE_BYTES / pix_bytes) / PL * PL);
  const size_t smem = 128 + (size_t)BWD_NHWC_NS * TP * pix_bytes + (size_t)ncons * (VC + 1) * sizeof(float);
  auto kern = conv_bwd_nhwc_kernel<FT, K>;
  int per_sm = 0;
  RHSEG_CUDA(cached_launch_prep(reinterpret_cast<const void*>(kern), ncons + 32, smem, smem, &per_sm));
  if (per_sm < 1) return RHSEG_ERR_UNSUPPORTED;
  const int n_tiles = (N + TP - 1) / TP;
  const long units_total = (long)B * n_tiles;
  const long grid = std::max<long>(1, std::min<long>((long)sm_count * per_sm, units_total));
  launch_pdl(kern, dim3((unsigned)grid), dim3(ncons + 32), smem, st, feats, dz, eff_w, C, N, TP, n_tiles, units_total, PL, NG,
             w_shared, dfeats, S, s, pt);
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}

template <typename FT>
int conv_bwd_nhwc(int K, const FT* feats, const float* dz, const float* eff_w, int B, int C, int N, FT* dfeats, double* S,
                  double* s, int sm_count, cudaStream_t st, int w_shared, const ParamTail& pt) {
  RHSEG_DISPATCH_K(K, {
    return launch_conv_bwd_nhwc<FT, KK>(feats, dz, eff_w, B, C, N, dfeats, S, s, sm_count, st, w_shared, pt);
  });
  return RHSEG_OK;
}
template int conv_bwd_nhwc<float>(int, const float*, const float*, const float*, int, int, int, float*, double*, double*, int,
                                  cudaStream_t, int, const ParamTail&);
template int conv_bwd_nhwc<uint16_t>(int, const uint16_t*, const float*, const float*, int, int, int, uint16_t*, double*,
                                     double*, int, cudaStream_t, int, const ParamTail&);

}  // namespace rhseg
