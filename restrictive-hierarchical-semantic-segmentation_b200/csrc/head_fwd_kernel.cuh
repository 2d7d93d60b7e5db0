// Fused 1x1 conv (+ activation) of the head forward, templated on the feature element type (float, or uint16_t =
// bf16 bits): included by head_fwd.cu (fp32 instances) and head_fwd_bf16.cu (bf16 instances), so that the two sets
// compile in parallel.  The work split, the per-sample weight staging and the epilogue are shared with the
// channels-last kernel (head_fwd_nhwc.cuh).
#pragma once
#include <algorithm>
#include "common.cuh"
#include "pipeline.cuh"
#include "head_common.cuh"

namespace rhseg {

// ------------------------------------------------------------------------------------
// Fused 1x1 conv (+ activation): TMA-fed, warp-specialised, persistent.
//
//   producer warp : streams [PIPE_CH channels x T pixels] stages of the feature planes into a
//                   shared-memory ring with 1-D bulk async copies (pipeline.cuh)
//   4 consumer warps: each thread owns J vectors of VEC pixels of the tile, accumulates
//                   K logits over the stages (weights [C][KP] in shared memory, one broadcast
//                   vector load per channel), then runs the activation epilogue
//
// Work unit = (sample, pixel tile, channel stage); the unit space is split EVENLY over one
// resident wave of CTAs.  MODE 0-2 (fused activation) splits on tile boundaries; MODE 3 (conv
// only, HRNet low-res pass, few pixels x many channels) splits anywhere: a tile shared by two
// CTAs is finished with fp32 atomics into the zero-initialised output (at most two partial
// sums per pixel, so the result does not depend on arrival order).
// ------------------------------------------------------------------------------------
constexpr int MODE_CONV_ONLY = 3;

// this CTA's units [u_begin, u_end)
template <int MODE>
__device__ __forceinline__ void fwd_units(long units_total, int n_stages, long& u_begin, long& u_end) {
  if constexpr (MODE == MODE_CONV_ONLY) {
    u_begin = units_total * blockIdx.x / gridDim.x;
    u_end = units_total * (blockIdx.x + 1) / gridDim.x;
  } else {
    const long tiles_total = units_total / n_stages;
    u_begin = (tiles_total * blockIdx.x / gridDim.x) * n_stages;
    u_end = (tiles_total * (blockIdx.x + 1) / gridDim.x) * n_stages;
  }
}

// unit u = (b * n_tiles + tile) * n_stages + stage; decoded once, then advanced incrementally
struct FwdCursor {
  int n_tiles, n_stages;
  int stage, tile, b;
  __device__ __forceinline__ FwdCursor(long u, int n_tiles_, int n_stages_) : n_tiles(n_tiles_), n_stages(n_stages_) {
    const long tile_lin = u / n_stages;
    stage = (int)(u - tile_lin * n_stages);
    b = (int)(tile_lin / n_tiles);
    tile = (int)(tile_lin - (long)b * n_tiles);
  }
  __device__ __forceinline__ void advance() {
    if (++stage == n_stages) {
      stage = 0;
      if (++tile == n_tiles) { tile = 0; ++b; }
    }
  }
};

// consumers: the FiLM pool sums of sample cur_b leave the CTA (one fp64 atomic per channel)
template <int K, int MODE, typename CFG>
__device__ __forceinline__ void fwd_flush_psum(int cur_b, float (&ps)[K], float* red, double* psum) {
  if constexpr (MODE != MODE_CONV_ONLY) {
    if (cur_b >= 0) {
      block_psum<K, CFG::NCW>(ps, psum + (size_t)cur_b * K, red, [] { consumer_sync(CFG::CONSUMERS); });
#pragma unroll
      for (int k = 0; k < K; ++k) ps[k] = 0.f;
    }
  }
}

// consumers, first unit of a tile in this CTA (uniform).  On a sample change the pool sums of the previous sample are
// flushed and the sample's effective weights [C][KP] (zero-padded) and biases are staged.  The logits start at the bias
// when the tile starts here at channel 0, else at 0 (the CTA that owns the tile's first stages adds the bias).  Returns
// whether the tile starts at channel 0.
template <int K, int P, int MODE, typename CFG>
__device__ __forceinline__ bool fwd_tile_begin(const FwdCursor& at, int tid, int& cur_b, const float* eff_w,
                                               const float* eff_b, int C, int w_shared, float* w_t, float* red, double* psum,
                                               float (&bias)[K], float (&ps)[K], float (&acc)[K][P]) {
  constexpr int KP = pad_k(K);
  constexpr int NCONS = CFG::CONSUMERS;
  const int b = at.b;
  if (b != cur_b) {
    fwd_flush_psum<K, MODE, CFG>(cur_b, ps, red, psum);
    consumer_sync(NCONS);
    const float* wsrc = w_shared ? eff_w : eff_w + (size_t)b * K * C;  // level 0: the head's own [K,C] weights
    for (int k = 0; k < K; ++k)
      for (int c = tid; c < C; c += NCONS) w_t[c * KP + k] = wsrc[(size_t)k * C + c];
    if constexpr (KP > K)
      for (int k = K; k < KP; ++k)
        for (int c = tid; c < C; c += NCONS) w_t[c * KP + k] = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) bias[k] = eff_b[(w_shared ? 0 : b * K) + k];
    cur_b = b;
    consumer_sync(NCONS);
  }
  const bool from_stage0 = at.stage == 0;
#pragma unroll
  for (int k = 0; k < K; ++k)
#pragma unroll
    for (int p = 0; p < P; ++p) acc[k][p] = from_stage0 ? bias[k] : 0.f;
  return from_stage0;
}

// Epilogue of the last unit of a tile in this CTA (at).  z = the tile's logits in the thread's pixel ownership: JE runs
// of VE consecutive pixels, run j starting at tile pixel (j * NCONS + tid) * VE.  MODE_CONV_ONLY stores them if this CTA
// summed all of the tile's stages, else adds them atomically.  Modes 0-2 apply the activation, store logits and
// probabilities, and add the probabilities to the thread's pool sums ps.
template <int K, int JE, int VE, int MODE, int NCONS>
__device__ __forceinline__ void fwd_epilogue(const float (&z)[K][JE * VE], const FwdCursor& at, int tid, bool from_stage0,
                                             const LevelInfo& li, int N, int p0, int t_act, int K_prev,
                                             const float* prev_probs, float* logits, float* probs, float (&ps)[K]) {
  constexpr int PE = JE * VE;
  const int b = at.b;
  int lp[JE];
  bool ok[JE];
#pragma unroll
  for (int j = 0; j < JE; ++j) {
    lp[j] = (j * NCONS + tid) * VE;
    ok[j] = lp[j] < t_act;
  }
  float* zb = logits + (size_t)b * K * N + p0;
  if constexpr (MODE == MODE_CONV_ONLY) {
    const bool complete = from_stage0 && at.stage == at.n_stages - 1;
#pragma unroll
    for (int j = 0; j < JE; ++j) {
      if (!ok[j]) continue;
#pragma unroll
      for (int k = 0; k < K; ++k) {
        float* dst = zb + (size_t)k * N + lp[j];
        if (complete) {
          Vec<VE> o;
#pragma unroll
          for (int v = 0; v < VE; ++v) o.v[v] = z[k][j * VE + v];
          *reinterpret_cast<Vec<VE>*>(dst) = o;
        } else {
#pragma unroll
          for (int v = 0; v < VE; ++v) atomicAdd(dst + v, z[k][j * VE + v]);
        }
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
    activate<K, PE, MODE>(z, pp, li.start_mask, prob);
    float* pb_out = probs + (size_t)b * K * N + p0;
#pragma unroll
    for (int k = 0; k < K; ++k) {
#pragma unroll
      for (int j = 0; j < JE; ++j) {
        if (!ok[j]) continue;
        Vec<VE> zo, po;
#pragma unroll
        for (int v = 0; v < VE; ++v) {
          zo.v[v] = z[k][j * VE + v];
          po.v[v] = prob[k][j * VE + v];
          ps[k] += po.v[v];
        }
        *reinterpret_cast<Vec<VE>*>(zb + (size_t)k * N + lp[j]) = zo;
        *reinterpret_cast<Vec<VE>*>(pb_out + (size_t)k * N + lp[j]) = po;
      }
    }
  }
}

template <typename FT, int K, int VEC, int J, int MODE, typename CFG>
__global__ void __launch_bounds__(CFG::THREADS)
head_fwd_kernel(const FT* __restrict__ feats, const float* __restrict__ eff_w,
                const float* __restrict__ eff_b, const float* __restrict__ prev_probs,
                const int32_t* __restrict__ table, int C, int N, int K_prev, int n_tiles, int n_stages,
                long units_total, int a0, int w_shared, float* __restrict__ logits, float* __restrict__ probs,
                double* __restrict__ psum) {
  pdl_wait();
  constexpr int KP = pad_k(K);
  constexpr int P = J * VEC;
  constexpr int NCONS = CFG::CONSUMERS;
  constexpr int T = NCONS * P;
  constexpr int G = FeatElem<FT>::G;
  constexpr int ROWP = T + G;  // row pitch: a multiple of 16 bytes
  constexpr int CH = CFG::CH;
  constexpr int NS = CFG::NS;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);            // full[NS], empty[NS]  (2*NS*8 bytes, padded to 128)
  FT* ring = reinterpret_cast<FT*>(smem_raw + 128);                  // [NS][CH][ROWP]
  float* w_t = reinterpret_cast<float*>(ring + (size_t)NS * CH * ROWP);  // [C][KP]
  float* red = w_t + (size_t)C * KP;                                 // [NCW][K]
  static_assert(2 * NS * 8 <= 128, "barrier block");
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  long u_begin, u_end;
  fwd_units<MODE>(units_total, n_stages, u_begin, u_end);
  ring_bars_init<NS>(bars, CFG::NPW, CFG::NCW);
  FwdCursor at(u_begin, n_tiles, n_stages);

  if (warp >= CFG::NCW) {
    // ------------------------------ producers ------------------------------
    if (lane == 0) {
      const int pw = warp - CFG::NCW;
      const uint64_t pol = l2_evict_first_policy();
      int slot = 0;
      uint32_t phase = 1;  // parity of the "slot is free" wait; flips every NS units
      for (long u = u_begin; u < u_end; ++u) {
        mbar_wait(smem_u32(&bars[NS + slot]), phase);
        const int p0 = at.tile * T;
        const int c0 = at.stage * CH;
        issue_stage_rows(feats, ((long)at.b * C + c0) * N + p0, N, min(T, N - p0), min(CH, C - c0), pw, CFG::NPW, a0,
                         smem_u32(ring + (size_t)slot * CH * ROWP), ROWP * sizeof(FT), smem_u32(&bars[slot]), pol);
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
  float bias[K], ps[K], acc[K][P];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    bias[k] = 0.f;
    ps[k] = 0.f;
#pragma unroll
    for (int p = 0; p < P; ++p) acc[k][p] = 0.f;
  }
  const int sN = N & (G - 1);
  bool from_stage0 = false;
  int slot = 0;
  uint32_t phase = 0;
  for (long u = u_begin; u < u_end; ++u) {
    const int p0 = at.tile * T;
    const int t_act = min(T, N - p0);
    if (at.stage == 0 || u == u_begin)  // first unit of this tile in this CTA (uniform)
      from_stage0 = fwd_tile_begin<K, P, MODE, CFG>(at, tid, cur_b, eff_w, eff_b, C, w_shared, w_t, red, psum, bias, ps, acc);

    const int c0 = at.stage * CH;
    const int ccnt = min(CH, C - c0);
    // shift of stage row cc is (sh0 + cc*sN) & (G-1): only G distinct values, indexed by cc & (G-1)
    int off[G];
    int sh0 = 0;
#pragma unroll
    for (int q = 0; q < G; ++q) off[q] = 0;
    if constexpr (VEC == 1) {
      sh0 = row_shift<FT>(((long)at.b * C + c0) * N + p0, a0);
#pragma unroll
      for (int q = 0; q < G; ++q) off[q] = ((sh0 + q * sN) & (G - 1)) + tid;
    }
    const float* wrow = w_t + (size_t)c0 * KP;
    mbar_wait(smem_u32(&bars[slot]), phase);
    const FT* stage_base = ring + (size_t)slot * CH * ROWP;

    auto channel = [&](int cc, int offv) {
      const FT* row = stage_base + cc * ROWP;
      float w[KP];
      ld_wvec<KP>(wrow + cc * KP, w);
#pragma unroll
      for (int j = 0; j < J; ++j) {
        float f[VEC];
        if constexpr (VEC == 4 && sizeof(FT) == 4) {
          const float4 t = *reinterpret_cast<const float4*>(row + (j * NCONS + tid) * 4);
          f[0] = t.x; f[1] = t.y; f[2] = t.z; f[3] = t.w;
        } else if constexpr (VEC == 4) {
          const uint2 t = *reinterpret_cast<const uint2*>(row + (j * NCONS + tid) * 4);
          f[0] = bf16_lo(t.x); f[1] = bf16_hi(t.x); f[2] = bf16_lo(t.y); f[3] = bf16_hi(t.y);
        } else {
          f[0] = feat_f32(row[offv + j * NCONS]);
        }
#pragma unroll
        for (int k = 0; k < K; ++k)
#pragma unroll
          for (int v = 0; v < VEC; ++v) acc[k][j * VEC + v] = fmaf(w[k], f[v], acc[k][j * VEC + v]);
      }
    };
    if (ccnt == CH) {  // full stage: branch-free, loads can be batched ahead of the FMAs
#pragma unroll
      for (int cc = 0; cc < CH; ++cc) channel(cc, off[cc & (G - 1)]);
    } else {
      for (int cc = 0; cc < ccnt; ++cc) channel(cc, ((sh0 + cc * sN) & (G - 1)) + tid);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(smem_u32(&bars[NS + slot]));

    if (at.stage == n_stages - 1 || u == u_end - 1)  // last unit of this tile in this CTA: epilogue
      fwd_epilogue<K, J, VEC, MODE, NCONS>(acc, at, tid, from_stage0, li, N, p0, t_act, K_prev, prev_probs, logits, probs, ps);
    if (++slot == NS) { slot = 0; phase ^= 1u; }
    at.advance();
  }
  fwd_flush_psum<K, MODE, CFG>(cur_b, ps, red, psum);
}

// Launch geometry shared by the forward launchers: one resident wave of CTAs, at most one per pixel tile (every CTA
// owns >= n_stages units: a split tile has <= 2 owners).  MODE_CONV_ONLY finishes split tiles with atomics, so its
// output is zero-filled here unless the caller did that already.
struct FwdGrid {
  int n_tiles, n_stages;
  long units_total, ctas;
};

template <int MODE>
static int fwd_grid(const void* kern, int threads, size_t smem, int B, int C, int N, int K, int T, int CH, float* out,
                    bool out_prezeroed, cudaStream_t st, FwdGrid& g) {
  int per_sm = 0;
  RHSEG_CUDA(cached_launch_prep(kern, threads, smem, smem, &per_sm));
  if (per_sm < 1) return RHSEG_ERR_UNSUPPORTED;
  g.n_tiles = (N + T - 1) / T;
  g.n_stages = (C + CH - 1) / CH;
  const long tiles_total = (long)B * g.n_tiles;
  g.units_total = tiles_total * g.n_stages;
  g.ctas = std::max<long>(1, std::min<long>((long)device_sm_count() * per_sm, tiles_total));
  if (MODE == MODE_CONV_ONLY && g.ctas > 1 && !out_prezeroed)
    RHSEG_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * (size_t)B * K * N, st));
  return RHSEG_OK;
}

template <typename FT, int K, int VEC, int J, int MODE, typename CFG>
static int launch_fwd(const FT* feats, const float* eff_w, const float* eff_b, const float* prev_probs,
                      const int32_t* table, int B, int C, int N, int K_prev, float* logits, float* probs,
                      double* psum, cudaStream_t st, bool out_prezeroed, int w_shared) {
  constexpr int KP = pad_k(K);
  constexpr int T = CFG::CONSUMERS * J * VEC;
  const size_t smem = 128 + (size_t)CFG::NS * CFG::CH * (T + FeatElem<FT>::G) * sizeof(FT) + ((size_t)C * KP + CFG::NCW * K) * sizeof(float);
  auto kern = head_fwd_kernel<FT, K, VEC, J, MODE, CFG>;
  FwdGrid g;
  const int rc = fwd_grid<MODE>(reinterpret_cast<const void*>(kern), CFG::THREADS, smem, B, C, N, K, T, CFG::CH, logits,
                                out_prezeroed, st, g);
  if (rc != RHSEG_OK) return rc;
  const int a0 = base_shift<FT>(feats);
  launch_pdl(kern, dim3((unsigned)g.ctas), dim3(CFG::THREADS), smem, st, feats, eff_w, eff_b, prev_probs, table, C, N, K_prev,
             g.n_tiles, g.n_stages, g.units_total, a0, w_shared, logits, probs, psum);
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}

// 16-byte vector rows: the plane pitch and the base are multiples of 16 bytes (every row then starts on a granule)
template <typename T>
static bool rows_vec4(const T* p, int N) {
  return (N % (16 / (int)sizeof(T)) == 0) && ((reinterpret_cast<uintptr_t>(p) & 15u) == 0);
}

// pipeline shapes (see DESIGN.md "conv kernels"): vec4 rows = full-resolution donors (UNet);
// scalar rows = planes whose pitch is not a multiple of 16 bytes (HRNet 155x155)
using FwdCfgV4 = PipeCfg<8, 8, 3>;      // 8 consumer warps x float4 -> T = 1024 px, 4 KB row copies (bf16: 2 KB)
using FwdCfgS1 = PipeCfg<4, 16, 4, 2>;  // scalar rows, T = 128*J px, two producer warps (1 KB row copies)
// pixels per thread on scalar rows (both layouts): fp32 T = 256 px; bf16 T = 512 px, which keeps the NCHW row copies at
// 1 KB (DESIGN.md 3.7)
template <typename FT> constexpr int s1_j() { return sizeof(FT) == 4 ? 2 : 4; }

template <typename FT>
int level_conv_nchw(const FT* feats, const float* eff_w, const float* eff_b, const float* prev_probs, const int32_t* table,
                    int B, int C, int Nf, int K, int K_prev, int act_mode, float* z_lo, bool zlo_zeroed, float* logits,
                    float* probs, double* psum, int w_shared, cudaStream_t st) {
  constexpr int J1 = s1_j<FT>();
  if (z_lo == nullptr) {
    const bool v4 = rows_vec4(feats, Nf) && rows_vec4(logits, Nf) && rows_vec4(probs, Nf) &&
                    (!prev_probs || rows_vec4(prev_probs, Nf));
    RHSEG_DISPATCH_K(K, {
      if (v4) {
        if (act_mode == RHSEG_ACT_SIGMOID)
          return launch_fwd<FT, KK, 4, 1, RHSEG_ACT_SIGMOID, FwdCfgV4>(feats, eff_w, eff_b, prev_probs, table, B, C, Nf, K_prev,
                                                                      logits, probs, psum, st, false, w_shared);
        if (act_mode == RHSEG_ACT_GROUPED)
          return launch_fwd<FT, KK, 4, 1, RHSEG_ACT_GROUPED, FwdCfgV4>(feats, eff_w, eff_b, prev_probs, table, B, C, Nf, K_prev,
                                                                      logits, probs, psum, st, false, w_shared);
        return launch_fwd<FT, KK, 4, 1, RHSEG_ACT_ZEROS, FwdCfgV4>(feats, eff_w, eff_b, prev_probs, table, B, C, Nf, K_prev,
                                                                  logits, probs, psum, st, false, w_shared);
      }
      if (act_mode == RHSEG_ACT_SIGMOID)
        return launch_fwd<FT, KK, 1, J1, RHSEG_ACT_SIGMOID, FwdCfgS1>(feats, eff_w, eff_b, prev_probs, table, B, C, Nf, K_prev,
                                                                     logits, probs, psum, st, false, w_shared);
      if (act_mode == RHSEG_ACT_GROUPED)
        return launch_fwd<FT, KK, 1, J1, RHSEG_ACT_GROUPED, FwdCfgS1>(feats, eff_w, eff_b, prev_probs, table, B, C, Nf, K_prev,
                                                                     logits, probs, psum, st, false, w_shared);
      return launch_fwd<FT, KK, 1, J1, RHSEG_ACT_ZEROS, FwdCfgS1>(feats, eff_w, eff_b, prev_probs, table, B, C, Nf, K_prev,
                                                                 logits, probs, psum, st, false, w_shared);
    });
  }
  const bool v4 = rows_vec4(feats, Nf) && rows_vec4(z_lo, Nf);
  RHSEG_DISPATCH_K(K, {
    if (v4)
      return launch_fwd<FT, KK, 4, 1, MODE_CONV_ONLY, FwdCfgV4>(feats, eff_w, eff_b, nullptr, nullptr, B, C, Nf, K_prev, z_lo,
                                                               nullptr, nullptr, st, zlo_zeroed, w_shared);
    return launch_fwd<FT, KK, 1, J1, MODE_CONV_ONLY, FwdCfgS1>(feats, eff_w, eff_b, nullptr, nullptr, B, C, Nf, K_prev, z_lo,
                                                              nullptr, nullptr, st, zlo_zeroed, w_shared);
  });
  return RHSEG_OK;
}

}  // namespace rhseg
