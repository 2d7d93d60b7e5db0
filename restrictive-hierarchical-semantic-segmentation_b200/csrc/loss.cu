// Hierarchical loss: one statistics pass (CE + Dice sums per sample and class), a tiny
// finalize kernel (scalars + closed-form backward coefficients) and one gradient pass.
// Reference semantics: Metrics/losses.py:16-134 (SoftDiceLoss, CrossEntropyLoss) and
// :150-177 (hierarchical_consistency_loss).
#include <math.h>
#include "common.cuh"
#include "logits_io.cuh"

namespace rhseg {

__device__ __forceinline__ bool vec_ok_ptr(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ------------------------------------------------------------------------------------
// statistics pass.  grid = (chunks, B); each thread handles ITER vectors of VEC pixels.
// per (b, c): [0] sum_m t*lp  [1] |m|  [2] sum_m p*t  [3] sum_m p  [4] sum_m t
// LT: logit element type (float, or uint16_t = bf16 bits, widened at the load: logits_io.cuh)
// ------------------------------------------------------------------------------------
template <int K, int VEC, int ITER, int THREADS, bool LOGITS, typename LT = float>
__global__ void __launch_bounds__(THREADS)
loss_stats_kernel(const LT* __restrict__ outs, const float* __restrict__ targets, long t_bstride,
                  long t_cstride, long N, double* __restrict__ stats) {
  pdl_wait();
  constexpr int NWARP = THREADS / 32;
  constexpr int NS = RHSEG_NSTAT;
  __shared__ float red[NWARP][K * NS];
  const int b = blockIdx.y, tid = threadIdx.x;
  float a[K][NS];
#pragma unroll
  for (int k = 0; k < K; ++k)
#pragma unroll
    for (int j = 0; j < NS; ++j) a[k][j] = 0.f;

  const LT* ob = outs + (size_t)b * K * N;
  const float* tb = targets + (size_t)b * t_bstride;
  const long chunk0 = (long)blockIdx.x * (THREADS * VEC * ITER);
#pragma unroll
  for (int it = 0; it < ITER; ++it) {
    const long px = chunk0 + (long)it * THREADS * VEC + (long)tid * VEC;
    if (px >= N) continue;
    float z[K][VEC], t[K][VEC];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const Vec<VEC> zv = ld_cached<VEC>(ob + (size_t)k * N + px);
      const Vec<VEC> tv = ld_cached<VEC>(tb + (size_t)k * t_cstride + px);
#pragma unroll
      for (int v = 0; v < VEC; ++v) { z[k][v] = zv.v[v]; t[k][v] = tv.v[v]; }
    }
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      float p[K], lp[K];
      if constexpr (LOGITS) {
        float zz[K], mx, sum;
#pragma unroll
        for (int k = 0; k < K; ++k) zz[k] = z[k][v];
        fast_softmax<K>(zz, p, mx, sum);
        const float lse = __logf(sum);
#pragma unroll
        for (int k = 0; k < K; ++k) lp[k] = (zz[k] - mx) - lse;
      } else {
#pragma unroll
        for (int k = 0; k < K; ++k) { p[k] = z[k][v]; lp[k] = z[k][v]; }
      }
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const float tk = t[k][v];
        if (tk != -1.0f) {
          a[k][0] = fmaf(tk, lp[k], a[k][0]);
          a[k][1] += 1.0f;
          a[k][2] = fmaf(p[k], tk, a[k][2]);
          a[k][3] += p[k];
          a[k][4] += tk;
        }
      }
    }
  }
  const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
  for (int k = 0; k < K; ++k)
#pragma unroll
    for (int j = 0; j < NS; ++j) {
      const float v = warp_sum(a[k][j]);
      if (lane == 0) red[warp][k * NS + j] = v;
    }
  __syncthreads();
  if (tid < K * NS) {
    double acc = 0.0;
#pragma unroll
    for (int w = 0; w < NWARP; ++w) acc += (double)red[w][tid];
    atomicAdd(&stats[(size_t)b * K * NS + tid], acc);
  }
}

// ------------------------------------------------------------------------------------
// finalize: one CTA.  out4 = {CE, Dice, #valid dice samples, #non-NaN CE samples};
// coef[b][c] = {dCE/dS0, dDice/dS2, dDice/dS3}.
// ------------------------------------------------------------------------------------
__device__ void finalize_level(const double* __restrict__ stats, const float* __restrict__ weights, int B, int K,
                               double smooth, float* __restrict__ out4, float* __restrict__ coef, double (*sh)[256]) {
  constexpr int NS = RHSEG_NSTAT;
  const int tid = threadIdx.x;
  double ce_sum = 0.0, dice_sum = 0.0, n_dice = 0.0, n_ce = 0.0;
  for (int b = tid; b < B; b += blockDim.x) {
    const double* st = stats + (size_t)b * K * NS;
    // CE (losses.py:107-116): sum_c -(w_c * S0 / cnt) / K ; any empty class mask -> NaN -> 1.0
    double ce = 0.0, I = 0.0, U = 0.0;
    bool ce_nan = false;
    for (int c = 0; c < K; ++c) {
      const double w = (double)weights[c];
      const double cnt = st[c * NS + 1];
      if (cnt == 0.0) ce_nan = true;
      else ce += -(w * st[c * NS + 0]) / cnt;
      I += w * st[c * NS + 2];
      U += w * st[c * NS + 3] + w * st[c * NS + 4];
    }
    ce = ce / (double)K;
    if (ce != ce) ce_nan = true;
    if (ce_nan) ce = 1.0; else n_ce += 1.0;
    ce_sum += ce;
    // Dice (losses.py:40-41, :64): 1 - (2I + smooth) / (U + smooth); NaN samples are dropped
    const double num = 2.0 * I + smooth, den = U + smooth;
    const double dl = 1.0 - num / den;
    const bool dice_ok = !(dl != dl);
    if (dice_ok) { dice_sum += dl; n_dice += 1.0; }
    for (int c = 0; c < K; ++c) {
      const double w = (double)weights[c];
      const double cnt = st[c * NS + 1];
      float* cf = coef + ((size_t)b * K + c) * 3;
      cf[0] = ce_nan ? 0.f : (float)(-w / (cnt * (double)K * (double)B));
      // per-sample derivatives; the 1/n_valid factor is applied below once n_valid is known
      cf[1] = dice_ok ? (float)(w * (-2.0 / den)) : 0.f;
      cf[2] = dice_ok ? (float)(w * (num / (den * den))) : 0.f;
    }
  }
  __syncthreads();
  sh[0][tid] = ce_sum; sh[1][tid] = dice_sum; sh[2][tid] = n_dice; sh[3][tid] = n_ce;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (tid < o) {
#pragma unroll
      for (int j = 0; j < 4; ++j) sh[j][tid] += sh[j][tid + o];
    }
    __syncthreads();
  }
  const double nv = sh[2][0];
  if (tid == 0) {
    out4[0] = (float)(sh[0][0] / (double)B);
    out4[1] = nv > 0.0 ? (float)(sh[1][0] / nv) : 0.f;
    out4[2] = (float)nv;
    out4[3] = (float)sh[3][0];
  }
  const float inv_nv = nv > 0.0 ? (float)(1.0 / nv) : 0.f;
  for (int i = tid; i < B * K; i += blockDim.x) {
    coef[(size_t)i * 3 + 1] *= inv_nv;
    coef[(size_t)i * 3 + 2] *= inv_nv;
  }
  __syncthreads();
}

__global__ void __launch_bounds__(256)
loss_finalize_kernel(const double* __restrict__ stats, const float* __restrict__ weights, int B, int K,
                     double smooth, float* __restrict__ out4, float* __restrict__ coef) {
  pdl_wait();
  __shared__ double sh[4][256];
  finalize_level(stats, weights, B, K, smooth, out4, coef, sh);
}

// All levels of one training step in one launch (see rhseg_step_finalize).
struct StepLevels {
  int n_levels;
  int K[RHSEG_MAX_LEVELS];
  int G[RHSEG_MAX_LEVELS];
  int child[RHSEG_MAX_LEVELS];
};

// Per-sample CE / Dice terms of one (level, sample): shared by both finalize kernels' fast path.
struct SampleLoss {
  double ce, dice;
  bool ce_nan, dice_ok;
};
__device__ __forceinline__ SampleLoss sample_loss(const double* __restrict__ st, const float* __restrict__ weights,
                                                  int K, int B, double smooth, float* __restrict__ cf) {
  constexpr int NS = RHSEG_NSTAT;
  SampleLoss r;
  double ce = 0.0, I = 0.0, U = 0.0;
  bool ce_nan = false;
  // fixed trip count + predicate: all loads of the sample are issued together (this kernel is pure latency)
  double sv[RHSEG_KERNEL_MAX_K][NS], wv[RHSEG_KERNEL_MAX_K];
#pragma unroll
  for (int c = 0; c < RHSEG_KERNEL_MAX_K; ++c) {
    wv[c] = c < K ? (double)weights[c] : 0.0;
#pragma unroll
    for (int j = 0; j < NS; ++j) sv[c][j] = c < K ? st[c * NS + j] : 1.0;
  }
#pragma unroll
  for (int c = 0; c < RHSEG_KERNEL_MAX_K; ++c) {
    if (c < K) {
      if (sv[c][1] == 0.0) ce_nan = true;
      else ce += fast_div(-(wv[c] * sv[c][0]), sv[c][1]);
      I += wv[c] * sv[c][2];
      U += wv[c] * sv[c][3] + wv[c] * sv[c][4];
    }
  }
  ce = fast_div(ce, (double)K);
  if (ce != ce) ce_nan = true;
  const double num = 2.0 * I + smooth, den = U + smooth;
  const double inv_den = fast_div(1.0, den);
  const double dl = 1.0 - num * inv_den;
  r.ce_nan = ce_nan;
  r.ce = ce_nan ? 1.0 : ce;
  r.dice_ok = !(dl != dl);
  r.dice = r.dice_ok ? dl : 0.0;
#pragma unroll
  for (int c = 0; c < RHSEG_KERNEL_MAX_K; ++c) {
    if (c < K) {
      cf[c * 3 + 0] = ce_nan ? 0.f : (float)fast_div(-wv[c], sv[c][1] * (double)K * (double)B);
      cf[c * 3 + 1] = r.dice_ok ? (float)(wv[c] * (-2.0 * inv_den)) : 0.f;   // scaled by 1/n_valid afterwards
      cf[c * 3 + 2] = r.dice_ok ? (float)(wv[c] * (num * inv_den * inv_den)) : 0.f;
    }
  }
  return r;
}

// All levels of a step in one launch, ONE barrier.  The kernel sits on the critical path between the last forward kernel
// and the first gradient kernel and is pure latency, so it is laid out to have a single dependent chain:
//   every thread derives the workspace offsets it needs itself (<= 8 integer steps, no shared table, no barrier);
//   thread <-> (level, sample): per-sample CE / Dice + backward coefficients kept in registers, its four sums into a
//     shared slot; concurrently thread <-> (level, class): the five ratio vectors; thread <-> (level, group): consistency;
//   barrier;
//   the (level, sample) threads read their level's valid count from the slots, scale the Dice coefficients and write the
//     coefficients ONCE (no read-modify-write pass); thread L < n_levels forms level L's outputs (fixed summation order),
//     thread 0 the totals.
constexpr int SF_MAX_SLOTS = 256;  // (level, sample) pairs handled by the fast layout (else: strided passes below)

struct StepOffsets { size_t w, k, c, r; };
__device__ __forceinline__ StepOffsets step_offsets(const StepLevels& lv, int B, int L) {
  StepOffsets o{0, 0, 0, 2 + 4 * (size_t)lv.n_levels};
  for (int i = 0; i < L; ++i) {
    const int K = lv.K[i], nc = lv.child[i] ? K + 1 : K;
    o.w += (size_t)B * K * RHSEG_NSTAT + RHSEG_MAX_K + (size_t)nc * nc;
    o.k += K;
    o.c += (size_t)B * K * 3;
    o.r += 5 * (size_t)nc;
  }
  return o;
}

__global__ void __launch_bounds__(256)
step_finalize_kernel(const double* __restrict__ ws, const float* __restrict__ weights, StepLevels lv, int B,
                     double smooth, double inv_bn, unsigned level_mask, float* __restrict__ out, float* __restrict__ coef,
                     double* __restrict__ summary) {
  pdl_wait();
  __shared__ double slot[SF_MAX_SLOTS][4];  // per (level, sample): ce, dice (0 if dropped), dice_ok, ce_ok
  __shared__ double cons_part[RHSEG_MAX_LEVELS][RHSEG_MAX_K];  // per (level, group); entries g < G[L] are written below
  const int tid = threadIdx.x, nL = lv.n_levels;
  const int n_pairs = nL * B;
  // (1) per-sample losses: thread <-> (level, sample); more than SF_MAX_SLOTS pairs are handled in strided rounds
  for (int base = 0; base < n_pairs; base += SF_MAX_SLOTS) {
    const int e = base + tid;
    const bool live = e < n_pairs && tid < SF_MAX_SLOTS;
    float cf[RHSEG_KERNEL_MAX_K * 3];
    int L = 0, b = 0, K = 1;
    StepOffsets o{0, 0, 0, 0};
    SampleLoss r{0.0, 0.0, false, false};
    if (live) {
      L = e / B; b = e - L * B; K = lv.K[L];
      o = step_offsets(lv, B, L);
      r = sample_loss(ws + o.w + (size_t)b * K * RHSEG_NSTAT, weights + o.k, K, B, smooth, cf);
      slot[tid][0] = r.ce;
      slot[tid][1] = r.dice_ok ? r.dice : 0.0;
      slot[tid][2] = r.dice_ok ? 1.0 : 0.0;
      slot[tid][3] = r.ce_nan ? 0.0 : 1.0;
    }
    if (base == 0) {
      // (2) concurrently, from the top of the block: the five per-class ratios, thread <-> (level, class)
      int c = (int)blockDim.x - 1 - tid, Lr = 0;
      while (Lr < nL && c >= (lv.child[Lr] ? lv.K[Lr] + 1 : lv.K[Lr])) { c -= (lv.child[Lr] ? lv.K[Lr] + 1 : lv.K[Lr]); ++Lr; }
      if (Lr < nL) {
        const int Kr = lv.K[Lr], nc = lv.child[Lr] ? Kr + 1 : Kr;
        const StepOffsets orr = step_offsets(lv, B, Lr);
        const long long* conf = reinterpret_cast<const long long*>(ws + orr.w + (size_t)B * Kr * RHSEG_NSTAT + RHSEG_MAX_K);
        long long rowv[RHSEG_KERNEL_MAX_K + 1], colv[RHSEG_KERNEL_MAX_K + 1];
#pragma unroll
        for (int j = 0; j <= RHSEG_KERNEL_MAX_K; ++j) {
          rowv[j] = j < nc ? conf[c * nc + j] : 0;
          colv[j] = j < nc ? conf[j * nc + c] : 0;
        }
        long long tp = conf[c * nc + c], row = 0, col = 0;
#pragma unroll
        for (int j = 0; j <= RHSEG_KERNEL_MAX_K; ++j) { row += rowv[j]; col += colv[j]; }
        const long long fp = col - tp, fn = row - tp;
        auto safe = [](float num, float den) { return num / (den == 0.f ? 1.f : den); };
        const float tpf = (float)tp, fpf = (float)fp, fnf = (float)fn;
        float* orow = out + orr.r;
        orow[0 * nc + c] = safe(2.0f * tpf, (2.0f * tpf + 1.0f * fnf) + fpf);
        orow[1 * nc + c] = safe(tpf, (float)(col + row - tp));
        orow[2 * nc + c] = safe(tpf, (float)(tp + fn));
        orow[3 * nc + c] = safe(tpf, (float)(tp + fp));
        orow[4 * nc + c] = safe(tpf, (float)(tp + fn));
      }
      // (3) concurrently: consistency sums, thread <-> (level, group) in the middle of the block
      if (tid >= 64 && tid < 64 + nL * RHSEG_MAX_K) {
        const int Lc = (tid - 64) / RHSEG_MAX_K, g = (tid - 64) % RHSEG_MAX_K;
        if (g < lv.G[Lc]) {
          const StepOffsets oc = step_offsets(lv, B, Lc);
          cons_part[Lc][g] = (ws + oc.w + (size_t)B * lv.K[Lc] * RHSEG_NSTAT)[g] * inv_bn;
        }
      }
    }
    __syncthreads();
    // the level's valid-sample count is complete only when all its samples sit in this round; with more pairs than
    // slots the Dice coefficients are scaled by the pass at the end instead
    const bool one_round = n_pairs <= SF_MAX_SLOTS;
    if (live) {
      float inv_nv = 1.f;
      if (one_round) {
        double nv = 0.0;
        for (int bb = 0; bb < B; ++bb) nv += slot[L * B + bb][2];
        inv_nv = nv > 0.0 ? (float)fast_div(1.0, nv) : 0.f;
      }
      float* dst = coef + o.c + (size_t)b * K * 3;
#pragma unroll
      for (int c = 0; c < RHSEG_KERNEL_MAX_K; ++c)
        if (c < K) {
          dst[c * 3 + 0] = cf[c * 3 + 0];
          dst[c * 3 + 1] = cf[c * 3 + 1] * inv_nv;
          dst[c * 3 + 2] = cf[c * 3 + 2] * inv_nv;
        }
    }
    if (one_round) break;
    // many pairs: accumulate this round's slots into per-level sums kept in the first slots' shadow (rare path)
    __syncthreads();
  }
  const bool one_round = n_pairs <= SF_MAX_SLOTS;
  __shared__ double lvl[RHSEG_MAX_LEVELS][4];
  if (one_round) {
    if (tid < nL) {  // fixed summation order over the samples: deterministic
      double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
      for (int bb = 0; bb < B; ++bb) {
        const double* sl = slot[tid * B + bb];
        a0 += sl[0]; a1 += sl[1]; a2 += sl[2]; a3 += sl[3];
      }
      lvl[tid][0] = a0; lvl[tid][1] = a1; lvl[tid][2] = a2; lvl[tid][3] = a3;
    }
  } else {
    // rare path (more than 256 (level, sample) pairs): recompute the level sums from the statistics, then scale the Dice
    // coefficients in a second pass
    if (tid < nL) {
      const int K = lv.K[tid];
      const StepOffsets o = step_offsets(lv, B, tid);
      double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
      float scratch[RHSEG_KERNEL_MAX_K * 3];
      for (int bb = 0; bb < B; ++bb) {
        const SampleLoss r = sample_loss(ws + o.w + (size_t)bb * K * RHSEG_NSTAT, weights + o.k, K, B, smooth, scratch);
        a0 += r.ce;
        if (r.dice_ok) { a1 += r.dice; a2 += 1.0; }
        if (!r.ce_nan) a3 += 1.0;
      }
      lvl[tid][0] = a0; lvl[tid][1] = a1; lvl[tid][2] = a2; lvl[tid][3] = a3;
    }
  }
  __syncthreads();
  if (!one_round) {
    for (int L = 0; L < nL; ++L) {
      const float inv_nv = lvl[L][2] > 0.0 ? (float)fast_div(1.0, lvl[L][2]) : 0.f;
      float* cfl = coef + step_offsets(lv, B, L).c;
      for (int i = tid; i < B * lv.K[L]; i += blockDim.x) {
        cfl[(size_t)i * 3 + 1] *= inv_nv;
        cfl[(size_t)i * 3 + 2] *= inv_nv;
      }
    }
  }
  if (tid < nL) {  // level tid's outputs
    const int L = tid;
    const float ce = (float)fast_div(lvl[L][0], (double)B);
    const float dice = lvl[L][2] > 0.0 ? (float)fast_div(lvl[L][1], lvl[L][2]) : 0.f;
    out[2 + 4 * L] = ce; out[3 + 4 * L] = dice; out[4 + 4 * L] = (float)lvl[L][2]; out[5 + 4 * L] = (float)lvl[L][3];
    if (summary) {  // additive per-rank quantities for the data-parallel all-reduce (dist.py layout)
      summary[2 + 4 * L] = lvl[L][0];
      summary[3 + 4 * L] = lvl[L][1];
      summary[4 + 4 * L] = lvl[L][2];
      summary[5 + 4 * L] = lvl[L][3];
    }
  }
  if (tid == 0) {
    double cons_total = 0.0;
    int cons_count = 0;
    float total = 0.f;
    for (int L = 0; L < nL; ++L) {
      for (int g = 0; g < lv.G[L]; ++g) cons_total += cons_part[L][g];  // sum over groups of mean |children - parent|
      cons_count += lv.G[L];
      const float ce = (float)fast_div(lvl[L][0], (double)B);
      const float dice = lvl[L][2] > 0.0 ? (float)fast_div(lvl[L][1], lvl[L][2]) : 0.f;
      if ((level_mask >> L) & 1u) total += ce + dice;  // CE_L + Dice_L (0 when no sample is valid); curriculum: train.py:125-134
    }
    const float consf = cons_count > 0 ? (float)fast_div(cons_total, (double)cons_count) : 0.f;
    out[0] = total + consf;
    out[1] = consf;
    if (summary) {
      summary[0] = (double)B;
      summary[1] = (double)consf * (double)B;
    }
  }
  if (summary) {  // confusion counts as fp64 (exact below 2^53), level after level
    size_t s_off = 2 + 4 * (size_t)nL;
    for (int L = 0; L < nL; ++L) {
      const int K = lv.K[L], nc = lv.child[L] ? K + 1 : K;
      const StepOffsets o = step_offsets(lv, B, L);
      const long long* conf = reinterpret_cast<const long long*>(ws + o.w + (size_t)B * K * RHSEG_NSTAT + RHSEG_MAX_K);
      for (int i = tid; i < nc * nc; i += blockDim.x) summary[s_off + i] = (double)conf[i];
      s_off += (size_t)nc * nc;
    }
  }
}

// ------------------------------------------------------------------------------------
// gradient pass: dz = g_ce * dCE/dz + g_dice * dDice/dz
//   a_c = A_c m_c t_c ; g_c = (B_c t_c + C_c) m_c
//   logits:  dz_k = (a_k - p_k sum_c a_c) + p_k (g_k - sum_c g_c p_c)
//   raw:     dz_k = a_k + g_k
// ------------------------------------------------------------------------------------
template <int K, int VEC, int THREADS, bool LOGITS, typename LT = float>
__global__ void __launch_bounds__(THREADS)
loss_bwd_kernel(const LT* __restrict__ outs, const float* __restrict__ targets, long t_bstride,
                long t_cstride, const float* __restrict__ coef, const float* __restrict__ g_ce,
                const float* __restrict__ g_dice, long N, LT* __restrict__ dz) {
  pdl_wait();
  const int b = blockIdx.y;
  const long px = ((long)blockIdx.x * THREADS + threadIdx.x) * VEC;
  if (px >= N) return;
  const float gce = g_ce ? __ldg(g_ce) : 0.f, gdi = g_dice ? __ldg(g_dice) : 0.f;
  float A[K], Bc[K], Cc[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const float* cf = coef + ((size_t)b * K + k) * 3;
    A[k] = gce * __ldg(cf);
    Bc[k] = gdi * __ldg(cf + 1);
    Cc[k] = gdi * __ldg(cf + 2);
  }
  const LT* ob = outs + (size_t)b * K * N + px;
  const float* tb = targets + (size_t)b * t_bstride + px;
  float z[K][VEC], t[K][VEC];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const Vec<VEC> zv = ld_stream<VEC>(ob + (size_t)k * N);
    const Vec<VEC> tv = ld_cached<VEC>(tb + (size_t)k * t_cstride);
#pragma unroll
    for (int v = 0; v < VEC; ++v) { z[k][v] = zv.v[v]; t[k][v] = tv.v[v]; }
  }
  float o[K][VEC];
#pragma unroll
  for (int v = 0; v < VEC; ++v) {
    float zz[K], tt[K], ov[K];
#pragma unroll
    for (int k = 0; k < K; ++k) { zz[k] = z[k][v]; tt[k] = t[k][v]; }
    loss_dz_pixel<K, LOGITS>(zz, tt, A, Bc, Cc, ov);
#pragma unroll
    for (int k = 0; k < K; ++k) o[k][v] = ov[k];
  }
  LT* db = dz + (size_t)b * K * N + px;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    Vec<VEC> r;
#pragma unroll
    for (int v = 0; v < VEC; ++v) r.v[v] = o[k][v];
    st_grad<VEC>(db + (size_t)k * N, r);  // consumed right away by the head backward
  }
}

// ------------------------------------------------------------------------------------
// consistency sums: per group g, sum_{b,n} | sum_{c in g} cur - prev[parent(g)] |
// ------------------------------------------------------------------------------------
template <int K, int VEC, int THREADS>
__global__ void __launch_bounds__(THREADS)
consistency_kernel(const float* __restrict__ cur, const float* __restrict__ prev, const int32_t* __restrict__ table,
                   int K_prev, long N, double* __restrict__ sums) {
  pdl_wait();
  constexpr int NWARP = THREADS / 32;
  __shared__ float red[NWARP][K];
  const int b = blockIdx.y, tid = threadIdx.x;
  const LevelInfo li = load_level_info<K>(table);
  float acc[K];
#pragma unroll
  for (int k = 0; k < K; ++k) acc[k] = 0.f;
  for (long px = ((long)blockIdx.x * THREADS + tid) * VEC; px < N; px += (long)gridDim.x * THREADS * VEC) {
    float c[K][VEC], gs[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const Vec<VEC> t = ld_cached<VEC>(cur + ((size_t)b * K + k) * N + px);
#pragma unroll
      for (int v = 0; v < VEC; ++v) c[k][v] = t.v[v];
    }
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      float x[K];
#pragma unroll
      for (int k = 0; k < K; ++k) x[k] = c[k][v];
      group_sum<K>(x, li.start_mask, gs);
#pragma unroll
      for (int k = 0; k < K; ++k) c[k][v] = gs[k];
    }
#pragma unroll
    for (int k = 0; k < K; ++k)
      if ((li.start_mask >> k) & 1) {
        const Vec<VEC> pv = ld_cached<VEC>(prev + ((size_t)b * K_prev + li.parent[k]) * N + px);
#pragma unroll
        for (int v = 0; v < VEC; ++v) acc[k] += fabsf(c[k][v] - pv.v[v]);
      }
  }
  const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const float v = warp_sum(acc[k]);
    if (lane == 0) red[warp][k] = v;
  }
  __syncthreads();
  if (tid < K && ((li.start_mask >> tid) & 1)) {
    double a = 0.0;
#pragma unroll
    for (int w = 0; w < NWARP; ++w) a += (double)red[w][tid];
    atomicAdd(&sums[table[RHSEG_TBL_GROUP_OF + tid]], a);
  }
}

static bool can_vec4(const void* a, const void* b, long s0, long s1, long N) {
  return (N % 4 == 0) && ((reinterpret_cast<uintptr_t>(a) & 15u) == 0) && ((reinterpret_cast<uintptr_t>(b) & 15u) == 0) &&
         (s0 % 4 == 0) && (s1 % 4 == 0);
}

}  // namespace rhseg

using namespace rhseg;

namespace rhseg {
template <typename LT>
static int loss_stats_launch(const LT* outs, const float* targets, long t_bstride, long t_cstride, int B, int K, long N,
                             bool logits, double* stats, cudaStream_t st) {
  constexpr int THREADS = 256, ITER = 4;
  RHSEG_DISPATCH_K(K, {
    if (can_vec4(outs, targets, t_bstride, t_cstride, N)) {
      dim3 grid((unsigned)((N + THREADS * 4 * ITER - 1) / (THREADS * 4 * ITER)), B);
      if (logits) launch_pdl(loss_stats_kernel<KK, 4, ITER, THREADS, true, LT>, dim3(grid), dim3(THREADS), 0, st, outs, targets, t_bstride, t_cstride, N, stats);
      else launch_pdl(loss_stats_kernel<KK, 4, ITER, THREADS, false, LT>, dim3(grid), dim3(THREADS), 0, st, outs, targets, t_bstride, t_cstride, N, stats);
    } else {
      dim3 grid((unsigned)((N + THREADS * ITER - 1) / (THREADS * ITER)), B);
      if (logits) launch_pdl(loss_stats_kernel<KK, 1, ITER, THREADS, true, LT>, dim3(grid), dim3(THREADS), 0, st, outs, targets, t_bstride, t_cstride, N, stats);
      else launch_pdl(loss_stats_kernel<KK, 1, ITER, THREADS, false, LT>, dim3(grid), dim3(THREADS), 0, st, outs, targets, t_bstride, t_cstride, N, stats);
    }
  });
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}

template <typename LT>
static int loss_bwd_launch(const LT* outs, const float* targets, long t_bstride, long t_cstride, const float* coef,
                           const float* g_ce, const float* g_dice, int B, int K, long N, bool logits, LT* dz,
                           cudaStream_t st) {
  constexpr int THREADS = 256;
  RHSEG_DISPATCH_K(K, {
    if (can_vec4(outs, targets, t_bstride, t_cstride, N) && ((reinterpret_cast<uintptr_t>(dz) & 15u) == 0)) {
      dim3 grid((unsigned)((N / 4 + THREADS - 1) / THREADS), B);
      if (logits) launch_pdl(loss_bwd_kernel<KK, 4, THREADS, true, LT>, dim3(grid), dim3(THREADS), 0, st, outs, targets, t_bstride, t_cstride, coef, g_ce, g_dice, N, dz);
      else launch_pdl(loss_bwd_kernel<KK, 4, THREADS, false, LT>, dim3(grid), dim3(THREADS), 0, st, outs, targets, t_bstride, t_cstride, coef, g_ce, g_dice, N, dz);
    } else {
      dim3 grid((unsigned)((N + THREADS - 1) / THREADS), B);
      if (logits) launch_pdl(loss_bwd_kernel<KK, 1, THREADS, true, LT>, dim3(grid), dim3(THREADS), 0, st, outs, targets, t_bstride, t_cstride, coef, g_ce, g_dice, N, dz);
      else launch_pdl(loss_bwd_kernel<KK, 1, THREADS, false, LT>, dim3(grid), dim3(THREADS), 0, st, outs, targets, t_bstride, t_cstride, coef, g_ce, g_dice, N, dz);
    }
  });
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}
}  // namespace rhseg

// logits_input: 0 / 1 (outs are probabilities / logits), optionally | RHSEG_LOGITS_BF16
extern "C" int rhseg_loss_stats(const void* outs, const float* targets, long t_bstride, long t_cstride, int B,
                                int K, int n_pix, int logits_input, double* stats, void* stream) {
  if (!outs || !targets || !stats || B <= 0 || n_pix <= 0) return RHSEG_ERR_ARG;
  if (K < 1 || K > RHSEG_KERNEL_MAX_K) return RHSEG_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  RHSEG_CUDA(cudaMemsetAsync(stats, 0, sizeof(double) * (size_t)B * K * RHSEG_NSTAT, st));
  const bool logits = (logits_input & ~RHSEG_LOGITS_BF16) != 0;
  if (logits_input & RHSEG_LOGITS_BF16)
    return loss_stats_launch(static_cast<const uint16_t*>(outs), targets, t_bstride, t_cstride, B, K, n_pix, logits, stats, st);
  return loss_stats_launch(static_cast<const float*>(outs), targets, t_bstride, t_cstride, B, K, n_pix, logits, stats, st);
}

extern "C" int rhseg_loss_finalize(const double* stats, const float* weights, int B, int K, double smooth,
                                   float* out4, float* coef, void* stream) {
  if (!stats || !weights || !out4 || !coef || B <= 0 || K <= 0) return RHSEG_ERR_ARG;
  launch_pdl(loss_finalize_kernel, dim3(1), dim3(256), 0, (cudaStream_t)stream, stats, weights, B, K, smooth, out4, coef);
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}

extern "C" int rhseg_loss_bwd(const void* outs, const float* targets, long t_bstride, long t_cstride,
                              const float* coef, const float* g_ce, const float* g_dice, int B, int K, int n_pix,
                              int logits_input, void* dz, void* stream) {
  if (!outs || !targets || !coef || !dz || B <= 0 || n_pix <= 0) return RHSEG_ERR_ARG;
  if (K < 1 || K > RHSEG_KERNEL_MAX_K) return RHSEG_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  const bool logits = (logits_input & ~RHSEG_LOGITS_BF16) != 0;
  if (logits_input & RHSEG_LOGITS_BF16)
    return loss_bwd_launch(static_cast<const uint16_t*>(outs), targets, t_bstride, t_cstride, coef, g_ce, g_dice, B, K, n_pix,
                           logits, static_cast<uint16_t*>(dz), st);
  return loss_bwd_launch(static_cast<const float*>(outs), targets, t_bstride, t_cstride, coef, g_ce, g_dice, B, K, n_pix,
                         logits, static_cast<float*>(dz), st);
}

extern "C" int rhseg_consistency_sums(const float* cur, const float* prev, const int32_t* table, int B, int K,
                                      int K_prev, int n_pix, double* sums, void* stream) {
  if (!cur || !prev || !table || !sums || B <= 0 || n_pix <= 0 || K_prev <= 0) return RHSEG_ERR_ARG;
  if (K < 1 || K > RHSEG_KERNEL_MAX_K) return RHSEG_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  RHSEG_CUDA(cudaMemsetAsync(sums, 0, sizeof(double) * RHSEG_MAX_K, st));
  const long N = n_pix;
  constexpr int THREADS = 256;
  RHSEG_DISPATCH_K(K, {
    if (can_vec4(cur, prev, 0, 0, N)) {
      const long vecs = N / 4;
      dim3 grid((unsigned)min((long)1024, (vecs + THREADS - 1) / THREADS), B);
      launch_pdl(consistency_kernel<KK, 4, THREADS>, dim3(grid), dim3(THREADS), 0, st, cur, prev, table, K_prev, N, sums);
    } else {
      dim3 grid((unsigned)min((long)1024, (N + THREADS - 1) / THREADS), B);
      launch_pdl(consistency_kernel<KK, 1, THREADS>, dim3(grid), dim3(THREADS), 0, st, cur, prev, table, K_prev, N, sums);
    }
  });
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}

extern "C" int rhseg_step_finalize(const void* eval_words, const float* weights_all, int B, int n_levels,
                                   const int32_t* K_per_level, const int32_t* groups_per_level, double smooth,
                                   long n_pix, unsigned level_mask, float* out, float* coef_all, double* summary, void* stream) {
  if (!eval_words || !weights_all || !K_per_level || !groups_per_level || !out || !coef_all) return RHSEG_ERR_ARG;
  if (B <= 0 || n_levels < 1 || n_levels > RHSEG_MAX_LEVELS || n_pix <= 0) return RHSEG_ERR_ARG;
  StepLevels lv{};
  lv.n_levels = n_levels;
  for (int L = 0; L < n_levels; ++L) {
    if (K_per_level[L] < 1 || K_per_level[L] > RHSEG_KERNEL_MAX_K) return RHSEG_ERR_UNSUPPORTED;
    lv.K[L] = K_per_level[L];
    lv.G[L] = L == 0 ? 0 : groups_per_level[L];
    lv.child[L] = L == 0 ? 0 : 1;
  }
  launch_pdl(step_finalize_kernel, dim3(1), dim3(256), 0, (cudaStream_t)stream, reinterpret_cast<const double*>(eval_words), weights_all, lv, B,
                                                            smooth, 1.0 / ((double)B * (double)n_pix), level_mask, out, coef_all, summary);
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}

namespace rhseg {
// Data-parallel gradient factors (SURVEY.md 8(e)): the single-process reference averages CE over ALL samples of the
// global batch and Dice over the GLOBAL count of non-NaN samples (Metrics/losses.py:64-66, :117-119); a rank that
// back-propagates its local means and lets DDP average over ranks gets exactly that when its CE gradient is scaled
// by world*B_local/B_global and its Dice gradient by world*n_valid_local/n_valid_global.
__global__ void dp_grad_scales_kernel(const double* __restrict__ local, const double* __restrict__ global, int n_levels,
                                      double world, const float* __restrict__ g, float* __restrict__ out) {
  pdl_wait();
  const int L = threadIdx.x;
  if (L >= n_levels) return;
  const double up = g ? (double)g[0] : 1.0;
  const double bl = local[0], bg = global[0];
  const double nl = local[4 + 4 * L], ng = global[4 + 4 * L];
  out[2 * L + 0] = (float)(bg > 0.0 ? up * world * bl / bg : 0.0);
  out[2 * L + 1] = (float)(ng > 0.0 ? up * world * nl / ng : 0.0);
}
}  // namespace rhseg

extern "C" int rhseg_dp_grad_scales(const double* local_summary, const double* global_summary, int n_levels, int world,
                                    const float* g, float* out, void* stream) {
  if (!local_summary || !global_summary || !out || world < 1) return RHSEG_ERR_ARG;
  if (n_levels < 1 || n_levels > RHSEG_MAX_LEVELS) return RHSEG_ERR_ARG;
  launch_pdl(rhseg::dp_grad_scales_kernel, dim3(1), dim3(32), 0, (cudaStream_t)stream, local_summary, global_summary, n_levels,
             (double)world, g, out);
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}
