// Fused 1x1 conv (+ activation) of the head forward for channels-last features, templated on the feature element type
// (float, or uint16_t = bf16 bits): included by head_fwd_nhwc.cu (fp32) and head_fwd_nhwc_bf16.cu (bf16).
//
// Same work decomposition as head_fwd_kernel (unit = sample, pixel tile of T pixels, channel stage of CH = 8 channels;
// the unit space split evenly over one resident wave), same arithmetic: a logit starts at the bias and takes one fmaf
// per channel in ascending order, so logits and probabilities equal the NCHW kernel's bit for bit.  What differs is the
// stage: the producer copies a [T pixels x 8 channels] box of the [C, N, B] tensor map (pixel rows of 32 bytes fp32,
// swizzled, or 16 bytes bf16), and consumer thread tid owns the pixels j*NCONS + tid, reading each pixel's 8 channels
// with one or two 128-bit shared loads.  Where the NCHW kernel gives a thread 4 consecutive pixels (16-byte rows,
// XCHG), the finished logits pass through shared memory to that ownership before the epilogue, so that the per-thread
// probability sums (psum, the FiLM pool of the next level) add the same pixels in the same order.  DESIGN.md 3.8.
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
  constexpr int VE = XCHG ? 4 : 1;
  constexpr int JE = XCHG ? 1 : J;
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
  if constexpr (MODE == MODE_CONV_ONLY) {
    u_begin = units_total * blockIdx.x / gridDim.x;
    u_end = units_total * (blockIdx.x + 1) / gridDim.x;
  } else {
    const long tiles_total = units_total / n_stages;
    u_begin = (tiles_total * blockIdx.x / gridDim.x) * n_stages;
    u_end = (tiles_total * (blockIdx.x + 1) / gridDim.x) * n_stages;
  }
  if (tid == 0) {
    for (int i = 0; i < NS; ++i) {
      mbar_init(smem_u32(&bars[i]), CFG::NPW);
      mbar_init(smem_u32(&bars[NS + i]), CFG::NCW);
    }
    mbar_fence_init();
  }
  __syncthreads();

  int stage, tile, b;
  {
    const long tile_lin = u_begin / n_stages;
    stage = (int)(u_begin - tile_lin * n_stages);
    b = (int)(tile_lin / n_tiles);
    tile = (int)(tile_lin - (long)b * n_tiles);
  }
  auto advance = [&]() {
    if (++stage == n_stages) {
      stage = 0;
      if (++tile == n_tiles) { tile = 0; ++b; }
    }
  };

  if (warp >= CFG::NCW) {
    // ------------------------------ producers ------------------------------
    if (lane == 0) {
      const int pw = warp - CFG::NCW;
      int slot = 0;
      uint32_t phase = 1;
      for (long u = u_begin; u < u_end; ++u) {
        mbar_wait(smem_u32(&bars[NS + slot]), phase);
        const int p0 = tile * T;
        uint32_t bytes = 0;
        for (int i = pw; i < NBOX; i += CFG::NPW) {
          if (p0 + i * BOX >= N) break;  // boxes wholly past the plane: nothing of them is read
          tma_load_3d(smem_u32(ring + (size_t)slot * STAGE + i * BOX * IB), &fmap, stage * CH, p0 + i * BOX, b,
                      smem_u32(&bars[slot]));
          bytes += BOX * IB;
        }
        mbar_arrive_expect_tx(smem_u32(&bars[slot]), bytes);
        if (++slot == NS) { slot = 0; phase ^= 1u; }
        advance();
      }
    }
    return;
  }

  // -------------------------------- consumers --------------------------------
  auto csync = [] { consumer_sync(NCONS); };
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
    const int p0 = tile * T;
    const int t_act = min(T, N - p0);
    if (stage == 0 || u == u_begin) {
      if (b != cur_b) {
        if constexpr (MODE != MODE_CONV_ONLY) {
          if (cur_b >= 0) {
            block_psum<K, CFG::NCW>(ps, psum + (size_t)cur_b * K, red, csync);
#pragma unroll
            for (int k = 0; k < K; ++k) ps[k] = 0.f;
          }
        }
        csync();
        const float* wsrc = w_shared ? eff_w : eff_w + (size_t)b * K * C;
        for (int k = 0; k < K; ++k)
          for (int c = tid; c < C; c += NCONS) w_t[c * KP + k] = wsrc[(size_t)k * C + c];
        if constexpr (KP > K)
          for (int k = K; k < KP; ++k)
            for (int c = tid; c < C; c += NCONS) w_t[c * KP + k] = 0.f;
#pragma unroll
        for (int k = 0; k < K; ++k) bias[k] = eff_b[(w_shared ? 0 : b * K) + k];
        cur_b = b;
        csync();
      }
      from_stage0 = stage == 0;
#pragma unroll
      for (int k = 0; k < K; ++k)
#pragma unroll
        for (int j = 0; j < J; ++j) acc[k][j] = from_stage0 ? bias[k] : 0.f;
    }

    const int c0 = stage * CH;
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
      if constexpr (KP == 4) {
        const float4 t = *reinterpret_cast<const float4*>(wrow + cc * KP);
        w[0] = t.x; w[1] = t.y; w[2] = t.z; w[3] = t.w;
      } else if constexpr (KP == 8) {
        const float4 t0 = *reinterpret_cast<const float4*>(wrow + cc * KP);
        const float4 t1 = *reinterpret_cast<const float4*>(wrow + cc * KP + 4);
        w[0] = t0.x; w[1] = t0.y; w[2] = t0.z; w[3] = t0.w; w[4] = t1.x; w[5] = t1.y; w[6] = t1.z; w[7] = t1.w;
      } else if constexpr (KP == 2) {
        const float2 t = *reinterpret_cast<const float2*>(wrow + cc * KP);
        w[0] = t.x; w[1] = t.y;
      } else {
        w[0] = wrow[cc];
      }
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

    if (stage == n_stages - 1 || u == u_end - 1) {  // last unit of this tile in this CTA: epilogue
      float e[K][JE * VE];
      if constexpr (XCHG) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
          csync();
#pragma unroll
          for (int j = 0; j < J; ++j) xbuf[j * NCONS + tid] = acc[k][j];
          csync();
          const float4 t = *reinterpret_cast<const float4*>(xbuf + 4 * tid);
          e[k][0] = t.x; e[k][1] = t.y; e[k][2] = t.z; e[k][3] = t.w;
        }
      } else {
#pragma unroll
        for (int k = 0; k < K; ++k)
#pragma unroll
          for (int j = 0; j < J; ++j) e[k][j] = acc[k][j];
      }
      constexpr int PE = JE * VE;
      int lp[JE];
      bool ok[JE];
#pragma unroll
      for (int j = 0; j < JE; ++j) {
        lp[j] = (j * NCONS + tid) * VE;
        ok[j] = lp[j] < t_act;
      }
      float* zb = logits + (size_t)b * K * N + p0;
      if constexpr (MODE == MODE_CONV_ONLY) {
        const bool complete = from_stage0 && stage == n_stages - 1;
#pragma unroll
        for (int j = 0; j < JE; ++j) {
          if (!ok[j]) continue;
#pragma unroll
          for (int k = 0; k < K; ++k) {
            float* dst = zb + (size_t)k * N + lp[j];
            if (complete) *dst = e[k][j];
            else atomicAdd(dst, e[k][j]);
          }
        }
      } else {
        float pp[K][PE];
        if constexpr (MODE == RHSEG_ACT_GROUPED) {
          const float* pb = prev_probs + (size_t)b * K_prev * N + p0;
#pragma unroll
          for (int k = 0; k < K; ++k) {
            if ((li.start_mask >> k) & 1) {
#pragma unroll
              for (int j = 0; j < JE; ++j) {
                Vec<VE> t;
                if (ok[j]) t = ld_cached<VE>(pb + (size_t)li.parent[k] * N + lp[j]);
                else {
#pragma unroll
                  for (int v = 0; v < VE; ++v) t.v[v] = 0.f;
                }
#pragma unroll
                for (int v = 0; v < VE; ++v) pp[k][j * VE + v] = t.v[v];
              }
            } else {
#pragma unroll
              for (int p = 0; p < PE; ++p) pp[k][p] = pp[k > 0 ? k - 1 : 0][p];
            }
          }
        }
        float prob[K][PE];
        activate<K, PE, MODE>(e, pp, li.start_mask, prob);
        float* pb_out = probs + (size_t)b * K * N + p0;
#pragma unroll
        for (int k = 0; k < K; ++k) {
#pragma unroll
          for (int j = 0; j < JE; ++j) {
            if (!ok[j]) continue;
            Vec<VE> zo, po;
#pragma unroll
            for (int v = 0; v < VE; ++v) {
              zo.v[v] = e[k][j * VE + v];
              po.v[v] = prob[k][j * VE + v];
              ps[k] += po.v[v];
            }
            *reinterpret_cast<Vec<VE>*>(zb + (size_t)k * N + lp[j]) = zo;
            *reinterpret_cast<Vec<VE>*>(pb_out + (size_t)k * N + lp[j]) = po;
          }
        }
      }
    }
    if (++slot == NS) { slot = 0; phase ^= 1u; }
    advance();
  }
  if constexpr (MODE != MODE_CONV_ONLY) {
    if (cur_b >= 0) block_psum<K, CFG::NCW>(ps, psum + (size_t)cur_b * K, red, csync);
  }
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
  int per_sm = 0;
  RHSEG_CUDA(cached_launch_prep(reinterpret_cast<const void*>(kern), CFG::THREADS, smem, smem, &per_sm));
  if (per_sm < 1) return RHSEG_ERR_UNSUPPORTED;
  CUtensorMap map;
  const int rc = encode_feats_map<FT>(&map, feats, B, C, N, NHWC_CH, T < 256 ? T : 256);
  if (rc != RHSEG_OK) return rc;
  const int n_tiles = (N + T - 1) / T;
  const int n_stages = (C + NHWC_CH - 1) / NHWC_CH;
  const long tiles_total = (long)B * n_tiles;
  const long units_total = tiles_total * n_stages;
  long grid = (long)device_sm_count() * per_sm;
  grid = std::min<long>(grid, tiles_total);
  if (grid < 1) grid = 1;
  if (MODE == MODE_CONV_ONLY && grid > 1 && !out_prezeroed)
    RHSEG_CUDA(cudaMemsetAsync(logits, 0, sizeof(float) * (size_t)B * K * N, st));
  launch_pdl(kern, dim3((unsigned)grid), dim3(CFG::THREADS), smem, st, map, eff_w, eff_b, prev_probs, table, C, N, K_prev,
             n_tiles, n_stages, units_total, w_shared, logits, probs, psum);
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}

// Ring shapes.  Each mirrors the NCHW kernel's for the same plane (FwdCfgV4 / FwdCfgS1: consumers, producers, tile
// size, about the same shared memory), so that both kernels get the same resident wave and split the pixel tiles
// between CTAs alike: the psum of a level then adds the same pixels per thread and per CTA.
using FwdNhwcCfgV4 = FwdCfgV4;               // T = 1024 px: 3 stages of 32 KB (fp32) / 16 KB (bf16)
using FwdNhwcCfgS1 = PipeCfg<4, NHWC_CH, 8, 2>;  // T = 128*J px: 8 stages of 8 KB (fp32, J = 2) / 8 KB (bf16, J = 4)
template <typename FT> constexpr int fwd_nhwc_s1_j() { return sizeof(FT) == 4 ? 2 : 4; }

template <typename FT, int K, int MODE>
static int fwd_fullres_nhwc(bool v4, const FT* feats, const float* eff_w, const float* eff_b, const float* prev_probs,
                            const int32_t* table, int B, int C, int N, int K_prev, float* logits, float* probs, double* psum,
                            cudaStream_t st, int w_shared) {
  if (v4)
    return launch_fwd_nhwc<FT, K, 4, MODE, FwdNhwcCfgV4, true>(feats, eff_w, eff_b, prev_probs, table, B, C, N, K_prev, logits,
                                                               probs, psum, st, false, w_shared);
  return launch_fwd_nhwc<FT, K, fwd_nhwc_s1_j<FT>(), MODE, FwdNhwcCfgS1, false>(feats, eff_w, eff_b, prev_probs, table, B, C,
                                                                                N, K_prev, logits, probs, psum, st, false,
                                                                                w_shared);
}

// Level conv for NHWC features: z_lo == nullptr, conv + activation at feature resolution; otherwise the low-res conv of
// an upsampled head into z_lo [B,K,Nf].  The tile shape follows what the NCHW path picks for the same plane.
template <typename FT>
int level_conv_nhwc_impl(const FT* feats, const float* eff_w, const float* eff_b, const float* prev_probs,
                         const int32_t* table, int B, int C, int Nf, int K, int K_prev, int act_mode, float* z_lo,
                         bool zlo_zeroed, float* logits, float* probs, double* psum, int w_shared, cudaStream_t st) {
  if (z_lo == nullptr) {
    const bool v4 = Nf % FeatElem<FT>::G == 0 && rows_vec4(logits, Nf) && rows_vec4(probs, Nf) &&
                    (!prev_probs || rows_vec4(prev_probs, Nf));
    RHSEG_DISPATCH_K(K, {
      if (act_mode == RHSEG_ACT_SIGMOID)
        return fwd_fullres_nhwc<FT, KK, RHSEG_ACT_SIGMOID>(v4, feats, eff_w, eff_b, prev_probs, table, B, C, Nf, K_prev, logits,
                                                           probs, psum, st, w_shared);
      if (act_mode == RHSEG_ACT_GROUPED)
        return fwd_fullres_nhwc<FT, KK, RHSEG_ACT_GROUPED>(v4, feats, eff_w, eff_b, prev_probs, table, B, C, Nf, K_prev, logits,
                                                           probs, psum, st, w_shared);
      return fwd_fullres_nhwc<FT, KK, RHSEG_ACT_ZEROS>(v4, feats, eff_w, eff_b, prev_probs, table, B, C, Nf, K_prev, logits,
                                                       probs, psum, st, w_shared);
    });
  }
  RHSEG_DISPATCH_K(K, {
    return launch_fwd_nhwc<FT, KK, fwd_nhwc_s1_j<FT>(), MODE_CONV_ONLY, FwdNhwcCfgS1, false>(
        feats, eff_w, eff_b, nullptr, nullptr, B, C, Nf, K_prev, z_lo, nullptr, nullptr, st, zlo_zeroed, w_shared);
  });
  return RHSEG_OK;
}

}  // namespace rhseg
