// 1x1-conv backward of the head (dfeats + fp64 weight-gradient sums), templated on the feature element type (float,
// or uint16_t = bf16 bits): included by head_bwd.cu (fp32 instances) and head_bwd_bf16.cu (bf16 instances), so that
// the two sets compile in parallel.
#pragma once
#include <algorithm>
#include <cstdlib>
#include "common.cuh"
#include "pipeline.cuh"

namespace rhseg {

// dfeats store, streaming: fp32 as is, bf16 rounded to nearest even (pairs with cvt.rn.bf16x2.f32)
template <int VEC>
__device__ __forceinline__ void st_feats(float* p, const Vec<VEC>& r) { st_stream<VEC>(p, r); }
template <int VEC>
__device__ __forceinline__ void st_feats(uint16_t* p, const Vec<VEC>& r) {
  if constexpr (VEC == 4) {
    asm volatile("st.global.L1::no_allocate.v2.b32 [%0], {%1,%2};"
                 :: "l"(p), "r"(pack_bf16x2(r.v[0], r.v[1])), "r"(pack_bf16x2(r.v[2], r.v[3])) : "memory");
  } else {
    static_assert(VEC == 1, "bf16 stores: 1 or 4 elements");
    asm volatile("st.global.L1::no_allocate.b16 [%0], %1;" :: "l"(p), "h"(to_bf16_bits(r.v[0])) : "memory");
  }
}

// ------------------------------------------------------------------------------------
// 1x1 conv backward at feature resolution: TMA-fed, warp-specialised, persistent.
//
//   dfeats[b,c,n] = sum_k w[b,k,c] dz[b,k,n]            (pure write stream, registers -> global)
//   S[b,k,c]      = sum_n dz[b,k,n] feats[b,c,n]        (read stream + reduction)
//
// Work unit = (sample, channel stage of PIPE_CH channels, pixel tile), flattened in that order
// and split EVENLY over one resident wave of CTAs.  The producer warp streams the feature
// stage of each unit into the shared-memory ring (pipeline.cuh).  A consumer thread owns J
// vectors of VEC pixels: it re-loads dz for the tile (small, L2-resident) into registers,
// writes dfeats for the stage's channels, and forms K partial dot products per channel that
// are reduced across the warp with the transposed recursive-halving shuffle pattern
// (KP-1 + 5-log2(KP) shuffles).  The per-channel sums of the current (sample, stage) segment
// stay in registers across tiles and leave the warp as fp64 atomics when the segment ends.
// ------------------------------------------------------------------------------------

// Level WITHOUT FiLM (level 0): its parameter gradients are plain sums over the batch, d_head_w = sum_b S_b and
// d_head_b = sum_b s_b.  With a ticket, the last CTA of the conv backward forms them (a few thousand L2 loads) instead of
// a second kernel at the very end of the step.  Levels with FiLM take rhseg_head_param_grads.
struct ParamTail {
  unsigned* ticket;  // device counter, zero on entry, left zero; nullptr = no tail
  int B;
  float* d_head_w;
  float* d_head_b;
};

// called by the nthr consumer threads of every CTA once its share of S / s has been added
template <int K>
__device__ __forceinline__ void level0_param_tail(const ParamTail& pt, const double* __restrict__ S,
                                                  const double* __restrict__ s, int C, int nthr) {
  __shared__ int last_cta;
  const int tid = threadIdx.x;
  __threadfence();
  consumer_sync(nthr);
  if (tid == 0) last_cta = (atomicAdd(pt.ticket, 1u) == gridDim.x - 1) ? 1 : 0;
  consumer_sync(nthr);
  if (last_cta) {
    __threadfence();
    for (int i = tid; i < K * C; i += nthr) {
      double a = 0.0;
      for (int bb = 0; bb < pt.B; ++bb) a += __ldcg(S + (size_t)bb * K * C + i);  // accumulated by other CTAs: read at L2
      pt.d_head_w[i] = (float)a;
    }
    if (tid < K) {
      double a = 0.0;
      for (int bb = 0; bb < pt.B; ++bb) a += __ldcg(s + bb * K + tid);
      pt.d_head_b[tid] = (float)a;
    }
    if (tid == 0) *pt.ticket = 0u;  // ready for the next launch / graph replay
  }
}

// min-blocks 1 (0 = unspecified) for the scalar-row instances other than K = 2 / K = 4: left alone, ptxas squeezes them to
// 96 registers (+ spills) for a second CTA per SM that the shared-memory ring rules out anyway -- K = 3: 121 vs 112 us in
// the step.  K = 4 (140 registers unprompted) and K = 2 measured no better with the hint and keep ptxas' own choice.
template <typename FT, int K, int VEC, int J, typename CFG>
__global__ void __launch_bounds__(CFG::THREADS, ((VEC == 1 && K != 2 && K != 4) ? 1 : 0))
conv_bwd_kernel(const FT* __restrict__ feats, const float* __restrict__ dz, const float* __restrict__ eff_w,
                int C, int N, int n_tiles, int n_stages, int group, long units_total, int a0, int w_shared,
                FT* __restrict__ dfeats, double* __restrict__ S, double* __restrict__ s, ParamTail pt) {
  pdl_wait();
  constexpr int KP = pad_k(K);
  // Register arrays and inner loops run over KC channels.  K = 3 computes on its zero-padded fourth channel (dz loads as
  // 0, the weight table is zero-padded already): ptxas schedules the K = 3 instance at 96 registers with little load
  // batching (111 us per HRNet launch against 96 us for K = 4 and K = 2); with four channels it IS the K = 4 schedule.
  constexpr int KC = (K == 3) ? 4 : K;
  constexpr int P = J * VEC;
  constexpr int NCONS = CFG::CONSUMERS;
  constexpr int T = NCONS * P;
  constexpr int G = FeatElem<FT>::G;
  constexpr int ROWP = T + G;  // row pitch: a multiple of 16 bytes
  constexpr int CH = CFG::CH;
  constexpr int NS = CFG::NS;
  constexpr int FLUSH_TILES = 64;  // fp32 running sums are handed to fp64 at least this often
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);  // full[NS], empty[NS]
  FT* ring = reinterpret_cast<FT*>(smem_raw + 128);        // [NS][CH][ROWP]
  float* w_all = reinterpret_cast<float*>(ring + (size_t)NS * CH * ROWP);  // [NCW][CH][KP] per-warp weights of the current stage
  static_assert(2 * NS * 8 <= 128, "barrier block");
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long u_begin = units_total * blockIdx.x / gridDim.x;
  const long u_end = units_total * (blockIdx.x + 1) / gridDim.x;
  ring_bars_init<NS>(bars, CFG::NPW, CFG::NCW);

  // Unit order: sample b -> GROUP of `group` consecutive pixel tiles -> channel stage -> tile of the group.
  // group >= n_tiles is the plain order (b, stage, tile).  Large planes x large batches (UNet 1024^2, batch 8..64) use
  // small groups: dz of a tile is read once per channel stage, and in the plain order those re-reads are a whole plane
  // apart -- 16 MB per sample, hundreds of MB over the CTAs in flight, i.e. from DRAM (+23 % traffic); inside a group
  // they are `group` tiles apart and hit L2.  Decoded once, then advanced incrementally.
  int stage, tile, b, g_first, g_cnt;
  {
    const long upb = (long)n_stages * n_tiles;  // units per sample
    b = (int)(u_begin / upb);
    const long r = u_begin - (long)b * upb;
    const long fgu = (long)n_stages * group;    // units of a full group
    const int gi = (int)(r / fgu);
    g_first = gi * group;
    g_cnt = min(group, n_tiles - g_first);
    const long r2 = r - (long)gi * fgu;
    stage = (int)(r2 / g_cnt);
    tile = g_first + (int)(r2 - (long)stage * g_cnt);
  }
  auto step_unit = [&](int& tile_, int& stage_, int& b_, int& gf_, int& gc_) {
    if (++tile_ == gf_ + gc_) {            // the group's tiles are done for this stage
      if (++stage_ == n_stages) {          // ... and for every stage: next group
        stage_ = 0;
        gf_ += gc_;
        if (gf_ == n_tiles) { gf_ = 0; ++b_; }
        gc_ = min(group, n_tiles - gf_);
      }
      tile_ = gf_;
    }
  };
  auto advance = [&]() { step_unit(tile, stage, b, g_first, g_cnt); };

  if (warp >= CFG::NCW) {
    // ------------------------------ producers ------------------------------
    if (lane == 0) {
      const int pw = warp - CFG::NCW;
      const uint64_t pol = l2_evict_first_policy();
      int slot = 0;
      uint32_t phase = 1;
      for (long u = u_begin; u < u_end; ++u) {
        mbar_wait(smem_u32(&bars[NS + slot]), phase);
        const int p0 = tile * T;
        const int c0 = stage * CH;
        issue_stage_rows(feats, ((long)b * C + c0) * N + p0, N, min(T, N - p0), min(CH, C - c0), pw, CFG::NPW, a0,
                         smem_u32(ring + (size_t)slot * CH * ROWP), ROWP * sizeof(FT), smem_u32(&bars[slot]), pol);
        if (++slot == NS) { slot = 0; phase ^= 1u; }
        advance();
      }
    }
    return;
  }

  // -------------------------------- consumers --------------------------------
  const bool writer = transposed_writer<KP>(lane);
  const int my_k = transposed_index<KP>(lane);
  const int sN = N & (G - 1);
  float* w_s = w_all + (size_t)warp * CH * KP;
  float sacc[CH];  // writer lanes: running sum over pixels of dz[my_k] * feats[c0 + cc]
  float s_acc = 0.f;
#pragma unroll
  for (int cc = 0; cc < CH; ++cc) sacc[cc] = 0.f;
  long cur_seg = -1;
  int seg_b = 0, seg_c0 = 0, seg_cnt = 0, tiles_since_flush = 0;

  auto flush = [&]() {  // per warp, no CTA-wide sync needed: every warp owns its partial sums
    if (writer && my_k < K) {
#pragma unroll
      for (int cc = 0; cc < CH; ++cc)
        if (cc < seg_cnt) atomicAdd(&S[((size_t)seg_b * K + my_k) * C + seg_c0 + cc], (double)sacc[cc]);
      if (seg_c0 == 0) atomicAdd(&s[seg_b * K + my_k], (double)s_acc);
    }
#pragma unroll
    for (int cc = 0; cc < CH; ++cc) sacc[cc] = 0.f;
    s_acc = 0.f;
    tiles_since_flush = 0;
  };

  float g_next[KC][P];
  auto load_dz = [&](int bb, int tt) {
    const int q0 = tt * T;
    const int q_act = min(T, N - q0);
#pragma unroll
    for (int j = 0; j < J; ++j) {
      const int l = (j * NCONS + tid) * VEC;
#pragma unroll
      for (int k = 0; k < KC; ++k) {
        Vec<VEC> t;
        if (k < K && l < q_act) t = ld_cached<VEC>(dz + ((size_t)bb * K + k) * N + q0 + l);
        else {
#pragma unroll
          for (int v = 0; v < VEC; ++v) t.v[v] = 0.f;
        }
#pragma unroll
        for (int v = 0; v < VEC; ++v) g_next[k][j * VEC + v] = t.v[v];
      }
    }
  };
  if (u_begin < u_end) load_dz(b, tile);
  int slot = 0;
  uint32_t phase = 0;
  for (long u = u_begin; u < u_end; ++u) {
    const long seg = ((long)b * n_tiles + g_first) * n_stages + stage;  // (sample, tile group, channel stage)
    const int p0 = tile * T;
    const int t_act = min(T, N - p0);
    const int c0 = stage * CH;
    const int ccnt = min(CH, C - c0);
    if (seg != cur_seg || tiles_since_flush >= FLUSH_TILES) {
      if (cur_seg >= 0) flush();
      if (seg != cur_seg) {  // effective weights of the stage's channels -> this warp's table [CH][KP]
        __syncwarp();
        for (int e = lane; e < CH * KP; e += 32) {
          const int cc = e / KP, k = e - cc * KP;
          w_s[e] = (cc < ccnt && k < K) ? __ldg(eff_w + ((size_t)(w_shared ? 0 : b) * K + k) * C + c0 + cc) : 0.f;
        }
        __syncwarp();
      }
      cur_seg = seg; seg_b = b; seg_c0 = c0; seg_cnt = ccnt;
    }
    ++tiles_since_flush;

    // dz of this tile was prefetched during the previous unit; fetch the NEXT unit's dz now so
    // that its L2 latency hides behind this unit's barrier wait and math
    int lp[J];
    bool ok[J];
    float g[KC][P];
#pragma unroll
    for (int j = 0; j < J; ++j) {
      lp[j] = (j * NCONS + tid) * VEC;
      ok[j] = lp[j] < t_act;
#pragma unroll
      for (int k = 0; k < KC; ++k)
#pragma unroll
        for (int v = 0; v < VEC; ++v) g[k][j * VEC + v] = g_next[k][j * VEC + v];
    }
    if (u + 1 < u_end) {
      int nt = tile, ns_ = stage, nb = b, ngf = g_first, ngc = g_cnt;
      step_unit(nt, ns_, nb, ngf, ngc);
      load_dz(nb, nt);
    }

    // shift of stage row cc is (sh0 + cc*sN) & (G-1): only G distinct values, indexed by cc & (G-1)
    int off[G];
    int sh0 = 0;
#pragma unroll
    for (int q = 0; q < G; ++q) off[q] = 0;
    if constexpr (VEC == 1) {
      sh0 = row_shift<FT>(((long)b * C + c0) * N + p0, a0);
#pragma unroll
      for (int q = 0; q < G; ++q) off[q] = ((sh0 + q * sN) & (G - 1)) + tid;
    }
    FT* dfb = dfeats ? dfeats + ((size_t)b * C + c0) * N + p0 : nullptr;
    mbar_wait(smem_u32(&bars[slot]), phase);
    const FT* stage_base = ring + (size_t)slot * CH * ROWP;

    // `part` for pixels beyond the tile's end is harmless: their dz registers are zero
    auto channel = [&](int cc, int offv, float& acc_out) {
      const FT* row = stage_base + cc * ROWP;
      float w[KP];
      ld_wvec<KP>(w_s + cc * KP, w);
      float part[KP];
#pragma unroll
      for (int k = 0; k < KP; ++k) part[k] = 0.f;
#pragma unroll
      for (int j = 0; j < J; ++j) {
        float f[VEC];
        if constexpr (VEC == 4 && sizeof(FT) == 4) {
          const float4 t = *reinterpret_cast<const float4*>(row + lp[j]);
          f[0] = t.x; f[1] = t.y; f[2] = t.z; f[3] = t.w;
        } else if constexpr (VEC == 4) {
          const uint2 t = *reinterpret_cast<const uint2*>(row + lp[j]);
          f[0] = bf16_lo(t.x); f[1] = bf16_hi(t.x); f[2] = bf16_lo(t.y); f[3] = bf16_hi(t.y);
        } else {
          f[0] = feat_f32(row[offv + j * NCONS]);
        }
#pragma unroll
        for (int k = 0; k < KC; ++k)
#pragma unroll
          for (int v = 0; v < VEC; ++v) {
            // NaN-safe masking: stale shared memory past the tile end may hold any bit pattern
            const float fv = ok[j] ? f[v] : 0.f;
            part[k] = fmaf(g[k][j * VEC + v], fv, part[k]);
          }
        if (dfb && ok[j]) {
          Vec<VEC> o;
#pragma unroll
          for (int v = 0; v < VEC; ++v) {
            float a = 0.f;
#pragma unroll
            for (int k = 0; k < KC; ++k) a = fmaf(w[k], g[k][j * VEC + v], a);
            o.v[v] = a;
          }
          st_feats<VEC>(dfb + (size_t)cc * N + lp[j], o);  // bf16: rounded to nearest even here, once
        }
      }
      warp_reduce_transposed<KP>(part, lane);
      acc_out += part[0];
    };
    if (ccnt == CH) {
#pragma unroll
      for (int cc = 0; cc < CH; ++cc) channel(cc, off[cc & (G - 1)], sacc[cc]);
    } else {
#pragma unroll
      for (int cc = 0; cc < CH; ++cc)
        if (cc < ccnt) channel(cc, ((sh0 + cc * sN) & (G - 1)) + tid, sacc[cc]);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(smem_u32(&bars[NS + slot]));

    if (c0 == 0) {  // s[b][k] = sum_n dz: only the first channel stage contributes
      float sred[KP];
#pragma unroll
      for (int k = 0; k < KP; ++k) {
        sred[k] = 0.f;
        if (k < K) {
#pragma unroll
          for (int p = 0; p < P; ++p) sred[k] += g[k][p];
        }
      }
      warp_reduce_transposed<KP>(sred, lane);
      s_acc += sred[0];
    }
    if (++slot == NS) { slot = 0; phase ^= 1u; }
    advance();
  }
  if (cur_seg >= 0) flush();
  if (pt.ticket != nullptr) level0_param_tail<K>(pt, S, s, C, NCONS);
}

template <typename FT, int K, int VEC, int J, typename CFG>
static int launch_conv_bwd(const FT* feats, const float* dz, const float* eff_w, int B, int C, int N,
                           FT* dfeats, double* S, double* s, int sm_count, cudaStream_t st, int w_shared,
                           const ParamTail& pt) {
  constexpr int KP = pad_k(K);
  constexpr int T = CFG::CONSUMERS * J * VEC;
  const size_t smem = 128 + (size_t)CFG::NS * CFG::CH * (T + FeatElem<FT>::G) * sizeof(FT) + (size_t)CFG::NCW * CFG::CH * KP * sizeof(float);
  auto kern = conv_bwd_kernel<FT, K, VEC, J, CFG>;
  int per_sm = 0;
  RHSEG_CUDA(cached_launch_prep(reinterpret_cast<const void*>(kern), CFG::THREADS, smem, smem, &per_sm));
  if (per_sm < 1) return RHSEG_ERR_UNSUPPORTED;
  const int n_tiles = (N + T - 1) / T;
  const int n_stages = (C + CFG::CH - 1) / CFG::CH;
  const long units_total = (long)B * n_stages * n_tiles;
  // tile groups (see the kernel): only when dz no longer sits in L2 between two channel stages
  static int tune_group = -1;
  if (tune_group < 0) { const char* e = getenv("RHSEG_TUNE_BWD_GROUP"); tune_group = e ? atoi(e) : 0; }
  int group = n_tiles;
  if (tune_group > 0) group = std::min(n_tiles, tune_group);
  // measured, UNet tl 1024^2 batch 8 (dz = 134 MB), step in ms: plain 2.930 | groups of 2: 2.791 | 4: 2.656 | 6: 2.685 |
  // 8: 2.773 | 12: 2.908 | 16: 2.923; 620^2 batch 4 (dz = 25 MB, L2-resident anyway): plain 0.5507 | 4: 0.5557 | 8: 0.5519
  else if ((size_t)B * K * N * sizeof(float) > ((size_t)40 << 20) && n_stages > 1) group = std::min(n_tiles, 4);
  const long grid = std::max<long>(1, std::min<long>((long)sm_count * per_sm, units_total));
  const int a0 = base_shift<FT>(feats);
  launch_pdl(kern, dim3((unsigned)grid), dim3(CFG::THREADS), smem, st, feats, dz, eff_w, C, N, n_tiles, n_stages, group, units_total, a0, w_shared, dfeats, S, s, pt);
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}

using BwdCfgV4 = PipeCfg<8, 8, 3>;  // 8 consumer warps x float4 -> T = 1024 px, 4 KB row copies, 33 KB stages
using BwdCfgS1 = PipeCfg<8, 16, 2>;  // scalar rows: T = 256*J px, 66 KB stages (dz reused over 16 channels)

// Conv backward of NCHW features and dfeats [B,C,N], K dispatch and ring shapes included.  Instances: fp32 in
// head_bwd.cu, bf16 (feats / dfeats = bf16 bit patterns, 2-byte aligned) in head_bwd_bf16.cu.
template <typename FT>
int conv_bwd_nchw(int K, const FT* feats, const float* dz, const float* eff_w, int B, int C, int N, FT* dfeats, double* S,
                  double* s, int sm_count, cudaStream_t st, int w_shared, const ParamTail& pt) {
  const bool v4 = (N % FeatElem<FT>::G == 0) &&
                  (((reinterpret_cast<uintptr_t>(feats) | reinterpret_cast<uintptr_t>(dz) | reinterpret_cast<uintptr_t>(dfeats)) & 15u) == 0);
  RHSEG_DISPATCH_K(K, {
    if (v4) return launch_conv_bwd<FT, KK, 4, 1, BwdCfgV4>(feats, dz, eff_w, B, C, N, dfeats, S, s, sm_count, st, w_shared, pt);
    return launch_conv_bwd<FT, KK, 1, (KK <= 4 ? 4 : 2), BwdCfgS1>(feats, dz, eff_w, B, C, N, dfeats, S, s, sm_count, st, w_shared,
                                                                   pt);
  });
  return RHSEG_OK;
}

// conv backward of channels-last features and dfeats [B,N,C] (head_bwd_nhwc.cu): K dispatch included
template <typename FT>
int conv_bwd_nhwc(int K, const FT* feats, const float* dz, const float* eff_w, int B, int C, int N, FT* dfeats, double* S,
                  double* s, int sm_count, cudaStream_t st, int w_shared, const ParamTail& pt);

}  // namespace rhseg
