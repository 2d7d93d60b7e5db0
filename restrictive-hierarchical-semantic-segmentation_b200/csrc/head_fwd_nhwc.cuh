// Fused 1x1 conv (+ activation) of the head forward for channels-last features, templated on the feature element type
// (float, or uint16_t = bf16 bits): included by head_fwd_nhwc.cu (fp32) and head_fwd_nhwc_bf16.cu (bf16).
//
// Same work decomposition as head_fwd_kernel (unit = sample, pixel tile of T pixels, channel stage of CH = 8 channels;
// the unit space split evenly over one resident wave), same arithmetic: a logit starts at the bias and takes one fmaf
// per channel in ascending order, so logits and probabilities equal the NCHW kernel's bit for bit.  The split, the
// cursor, the weight staging and the epilogue are head_fwd_kernel.cuh's.  What differs is the stage: the producer
// copies a [T pixels x 8 channels] box of the [C, N, B] tensor map (pixel rows of 32 bytes fp32, swizzled, or 16 bytes
// bf16), and consumer thread tid owns the pixels j*NCONS + tid, reading each pixel's 8 channels with one or two 128-bit
// shared loads.  Where the NCHW kernel gives a thread 4 consecutive pixels (16-byte rows, XCHG), the finished logits
// pass through shared memory to that ownership before the epilogue, so that the per-thread probability sums (psum, the
// FiLM pool of the next level) add the same pixels in the same order.  DESIGN.md 3.8.
#pragma once
#include <algorithm>
#include "feats_nhwc.cuh"
#include "head_common.cuh"
#include "head_fwd_kernel.cuh"

namespace rhseg {

constexpr int NHWC_CH = 8;  // channels per stage

template <typename FT, int K, int J, int MODE, typename CFG, bool XCHG>
__global__ void __launch_bounds__(CFG::THREADS)
head_fwd_nhwc_kernel(const __grid_constant__ CUtensorMap fmap, const float* __restrict__ eff_w,
                     const float* __restrict__ eff_b, const float* __restrict__ prev_probs,
                     const int32_t* __restrict__ table, int C, int N, int K_prev, int n_tiles, int n_stages,
                     long units_total, int w_shared, float* __restrict__ logits, float* __restrict__ probs,
                     double* __restrict__ psum) {
  pdl_wait();
  constexpr int KP = pad_k(K);
  constexpr int NCONS = CFG::CONSUMERS;
  constexpr int T = NCONS * J;
  constexpr int CH = NHWC_CH;
  constexpr int IB = CH * (int)sizeof(FT);  // bytes of a pixel row of the stage: 32 (swizzled) or 16
  constexpr int BOX = T < 256 ? T : 256;     // tensor-map boxes hold at most 256 pixels
  constexpr int NBOX = T / BOX;
  constexpr int STAGE = T * IB;
  constexpr int NS = CFG::NS;
  // epilogue ownership: 4 consecutive pixels (XCHG, as head_fwd_kernel with VEC = 4) or the pixels j*NCONS + tid
  static_assert(!XCHG || J == 4, "the exchange regroups 4 pixels per thread");
  static_assert(T % BOX == 0 && (IB == 16 || IB == 32), "stage shape");
  extern __shared__ __align__(128) unsigned char smem_raw[];
  // [bars 128 B] ... [ring: NS stages, 1024-byte aligned (swizzle atom)] [w_t C x KP] [red NCW x K] [xbuf T]
  const uint32_t raw_u32 = smem_u32(smem_raw);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);
  unsigned char* ring = smem_raw + (((raw_u32 + 128 + 1023) & ~1023u) - raw_u32);
  float* w_t = reinterpret_cast<float*>(ring + (size_t)NS * STAGE);
  float* red = w_t + (size_t)C * KP;
  float* xbuf = red + CFG::NCW * K;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  long u_begin, u_end;
  fwd_units<MODE>(units_total, n_stages, u_begin, u_end);
  ring_bars_init<NS>(bars, CFG::NPW, CFG::NCW);
  FwdCursor at(u_begin, n_tiles, n_stages);

  if (warp >= CFG::NCW) {
    // ------------------------------ producers ------------------------------
    if (lane == 0) {
      const int pw = warp - CFG::NCW;
      int slot = 0;
      uint32_t phase = 1;
      for (long u = u_begin; u < u_end; ++u) {
        mbar_wait(smem_u32(&bars[NS + slot]), phase);
        const int p0 = at.tile * T;
        uint32_t bytes = 0;
        for (int i = pw; i < NBOX; i += CFG::NPW) {
          if (p0 + i * BOX >= N) break;  // boxes wholly past the plane: nothing of them is read
          tma_load_3d(smem_u32(ring + (size_t)slot * STAGE + i * BOX * IB), &fmap, at.stage * CH, p0 + i * BOX, at.b,
                      smem_u32(&bars[slot]));
          bytes += BOX * IB;
        }
        mbar_arrive_expect_tx(smem_u32(&bars[slot]), bytes);
        if (++slot == NS) { slot = 0; phase ^= 1u; }
        at.advance();
      }
    }
    return;
  }

  // -------------------------------- consumers --------------------------------
  LevelInfo li;
  if constexpr (MODE != MODE_CONV_ONLY) li = load_level_info<K>(MODE == RHSEG_ACT_GROUPED ? table : nullptr);
  int cur_b = -1;
  float bias[K], ps[K], acc[K][J];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    bias[k] = 0.f;
    ps[k] = 0.f;
#pragma unroll
    for (int j = 0; j < J; ++j) acc[k][j] = 0.f;
  }
  bool from_stage0 = false;
  int slot = 0;
  uint32_t phase = 0;
  for (long u = u_begin; u < u_end; ++u) {
    const int p0 = at.tile * T;
    const int t_act = min(T, N - p0);
    if (at.stage == 0 || u == u_begin)  // first unit of this tile in this CTA (uniform)
      from_stage0 = fwd_tile_begin<K, J, MODE, CFG>(at, tid, cur_b, eff_w, eff_b, C, w_shared, w_t, red, psum, bias, ps, acc);

    const int c0 = at.stage * CH;
    const int ccnt = min(CH, C - c0);
    const float* wrow = w_t + (size_t)c0 * KP;
    mbar_wait(smem_u32(&bars[slot]), phase);
    const unsigned char* st = ring + (size_t)slot * STAGE;
    float f[J][CH];
#pragma unroll
    for (int j = 0; j < J; ++j) {
      const int r = j * NCONS + tid;
      if constexpr (IB == 32) {
        const int x = (r >> 2) & 1;  // 32-byte swizzle: chunk q of row r sits at chunk q ^ x
        chunk_f32(lds128(st + r * 32 + (x << 4)), &f[j][0], FT{});
        chunk_f32(lds128(st + r * 32 + ((x ^ 1) << 4)), &f[j][4], FT{});
      } else {
        chunk_f32(lds128(st + r * 16), &f[j][0], FT{});
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(smem_u32(&bars[NS + slot]));

    auto channel = [&](int cc) {
      float w[KP];
      ld_wvec<KP>(wrow + cc * KP, w);
#pragma unroll
      for (int j = 0; j < J; ++j)
#pragma unroll
        for (int k = 0; k < K; ++k) acc[k][j] = fmaf(w[k], f[j][cc], acc[k][j]);
    };
    if (ccnt == CH) {
#pragma unroll
      for (int cc = 0; cc < CH; ++cc) channel(cc);
    } else {  // last stage of a C that is not a multiple of 8 (C*esz is a multiple of 16: 4 fp32 channels left)
#pragma unroll
      for (int cc = 0; cc < CH; ++cc)
        if (cc < ccnt) channel(cc);
    }

    if (at.stage == n_stages - 1 || u == u_end - 1) {  // last unit of this tile in this CTA: epilogue
      if constexpr (XCHG) {  // regroup: 4 consecutive pixels per thread
        float e[K][4];
#pragma unroll
        for (int k = 0; k < K; ++k) {
          consumer_sync(NCONS);
#pragma unroll
          for (int j = 0; j < J; ++j) xbuf[j * NCONS + tid] = acc[k][j];
          consumer_sync(NCONS);
          const float4 t = *reinterpret_cast<const float4*>(xbuf + 4 * tid);
          e[k][0] = t.x; e[k][1] = t.y; e[k][2] = t.z; e[k][3] = t.w;
        }
        fwd_epilogue<K, 1, 4, MODE, NCONS>(e, at, tid, from_stage0, li, N, p0, t_act, K_prev, prev_probs, logits, probs, ps);
      } else {
        fwd_epilogue<K, J, 1, MODE, NCONS>(acc, at, tid, from_stage0, li, N, p0, t_act, K_prev, prev_probs, logits, probs, ps);
      }
    }
    if (++slot == NS) { slot = 0; phase ^= 1u; }
    at.advance();
  }
  fwd_flush_psum<K, MODE, CFG>(cur_b, ps, red, psum);
}

template <typename FT, int K, int J, int MODE, typename CFG, bool XCHG>
static int launch_fwd_nhwc(const FT* feats, const float* eff_w, const float* eff_b, const float* prev_probs,
                           const int32_t* table, int B, int C, int N, int K_prev, float* logits, float* probs,
                           double* psum, cudaStream_t st, bool out_prezeroed, int w_shared) {
  constexpr int KP = pad_k(K);
  constexpr int T = CFG::CONSUMERS * J;
  constexpr int IB = NHWC_CH * (int)sizeof(FT);
  const size_t smem = 1024 + 128 + (size_t)CFG::NS * T * IB + ((size_t)C * KP + CFG::NCW * K + (XCHG ? T : 0)) * sizeof(float);
  auto kern = head_fwd_nhwc_kernel<FT, K, J, MODE, CFG, XCHG>;
  CUtensorMap map;
  int rc = encode_feats_map<FT>(&map, feats, B, C, N, NHWC_CH, T < 256 ? T : 256);
  if (rc != RHSEG_OK) return rc;
  FwdGrid g;
  rc = fwd_grid<MODE>(reinterpret_cast<const void*>(kern), CFG::THREADS, smem, B, C, N, K, T, NHWC_CH, logits, out_prezeroed,
                      st, g);
  if (rc != RHSEG_OK) return rc;
  launch_pdl(kern, dim3((unsigned)g.ctas), dim3(CFG::THREADS), smem, st, map, eff_w, eff_b, prev_probs, table, C, N, K_prev,
             g.n_tiles, g.n_stages, g.units_total, w_shared, logits, probs, psum);
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}

// Ring shapes.  Each mirrors the NCHW kernel's for the same plane (FwdCfgV4 / FwdCfgS1: consumers, producers, tile
// size, about the same shared memory), so that both kernels get the same resident wave and split the pixel tiles
// between CTAs alike: the psum of a level then adds the same pixels per thread and per CTA.
using FwdNhwcCfgV4 = FwdCfgV4;                   // T = 1024 px: 3 stages of 32 KB (fp32) / 16 KB (bf16)
using FwdNhwcCfgS1 = PipeCfg<4, NHWC_CH, 8, 2>;  // T = 128*J px: 8 stages of 8 KB (fp32, J = 2) / 8 KB (bf16, J = 4)

// z_lo == nullptr: conv + activation at feature resolution; otherwise the low-res conv of an upsampled head into z_lo
// [B,K,Nf].  The tile shape follows what the NCHW path picks for the same plane.
template <typename FT>
int level_conv_nhwc(const FT* feats, const float* eff_w, const float* eff_b, const float* prev_probs, const int32_t* table,
                    int B, int C, int Nf, int K, int K_prev, int act_mode, float* z_lo, bool zlo_zeroed, float* logits,
                    float* probs, double* psum, int w_shared, cudaStream_t st) {
  constexpr int J1 = s1_j<FT>();
  if (z_lo == nullptr) {
    const bool v4 = Nf % FeatElem<FT>::G == 0 && rows_vec4(logits, Nf) && rows_vec4(probs, Nf) &&
                    (!prev_probs || rows_vec4(prev_probs, Nf));
    RHSEG_DISPATCH_K(K, {
      if (v4) {
        if (act_mode == RHSEG_ACT_SIGMOID)
          return launch_fwd_nhwc<FT, KK, 4, RHSEG_ACT_SIGMOID, FwdNhwcCfgV4, true>(feats, eff_w, eff_b, prev_probs, table, B, C,
                                                                                  Nf, K_prev, logits, probs, psum, st, false,
                                                                                  w_shared);
        if (act_mode == RHSEG_ACT_GROUPED)
          return launch_fwd_nhwc<FT, KK, 4, RHSEG_ACT_GROUPED, FwdNhwcCfgV4, true>(feats, eff_w, eff_b, prev_probs, table, B, C,
                                                                                  Nf, K_prev, logits, probs, psum, st, false,
                                                                                  w_shared);
        return launch_fwd_nhwc<FT, KK, 4, RHSEG_ACT_ZEROS, FwdNhwcCfgV4, true>(feats, eff_w, eff_b, prev_probs, table, B, C, Nf,
                                                                              K_prev, logits, probs, psum, st, false, w_shared);
      }
      if (act_mode == RHSEG_ACT_SIGMOID)
        return launch_fwd_nhwc<FT, KK, J1, RHSEG_ACT_SIGMOID, FwdNhwcCfgS1, false>(feats, eff_w, eff_b, prev_probs, table, B, C,
                                                                                  Nf, K_prev, logits, probs, psum, st, false,
                                                                                  w_shared);
      if (act_mode == RHSEG_ACT_GROUPED)
        return launch_fwd_nhwc<FT, KK, J1, RHSEG_ACT_GROUPED, FwdNhwcCfgS1, false>(feats, eff_w, eff_b, prev_probs, table, B, C,
                                                                                  Nf, K_prev, logits, probs, psum, st, false,
                                                                                  w_shared);
      return launch_fwd_nhwc<FT, KK, J1, RHSEG_ACT_ZEROS, FwdNhwcCfgS1, false>(feats, eff_w, eff_b, prev_probs, table, B, C, Nf,
                                                                              K_prev, logits, probs, psum, st, false, w_shared);
    });
  }
  RHSEG_DISPATCH_K(K, {
    return launch_fwd_nhwc<FT, KK, J1, MODE_CONV_ONLY, FwdNhwcCfgS1, false>(feats, eff_w, eff_b, nullptr, nullptr, B, C, Nf,
                                                                           K_prev, z_lo, nullptr, nullptr, st, zlo_zeroed,
                                                                           w_shared);
  });
  return RHSEG_OK;
}

}  // namespace rhseg
