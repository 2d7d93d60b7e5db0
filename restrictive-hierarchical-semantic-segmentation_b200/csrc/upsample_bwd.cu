// Adjoint of the bilinear (align_corners=True) upsample, shared-memory tiled and separable,
// optionally fused with the hi-res gradient producers (HRNet path).
//
// The reference reaches this through autograd over F.interpolate (Models/models.py:766, :776):
//   dz_lo[i][j] = sum_{y,x} wy(y,i) wx(x,j) dz_hi[y][x]
// One CTA owns a tile of TH x TW low-res pixels of one sample (all K channels).  It stages the
// hi-res gradient of the tile's support region in shared memory, reduces along x, then along y.
// SRC 0: dz_hi is read from memory (what autograd hands us).
// SRC 1: dz_hi is formed on the fly per hi-res pixel as  loss gradient (closed form from logits,
//        targets, coefficients) + activation backward (sigmoid / restrictive softmax with the
//        gradient arriving at the probabilities), so the hi-res gradient tensor never exists.
#include <algorithm>
#include <cstdlib>
#include "common.cuh"
#include "hires.cuh"
#include "logits_io.cuh"

namespace rhseg {

constexpr int ADJ_TH = 8, ADJ_TW = 16, ADJ_THREADS = 256;
constexpr int ADJ_MAXW = 24;  // max hi-res taps per low-res index held in the weight tables (upsampling factor <= ~10)

struct FusedDzArgs {
  const float* logits;      // [B,K,H,W]
  const float* targets;     // strided
  long t_bstride, t_cstride;
  const float* coef;        // [B,K,3]
  const float* g_ce;        // device scalars (may be null)
  const float* g_dice;
  const float* prev_probs;  // [B,K_prev,H,W] (grouped)
  const int32_t* table;
  const double* g_uniform;  // [B,K] or null
  float inv_npix;
  const float* dp_pix;      // [B,K,H,W] or null
  uint32_t pix_mask;
  float* dp_prev;           // [B,K_prev,H,W] (+=) or null
  int K_prev;
};

template <int K, int SRC, int MODE>
__global__ void __launch_bounds__(ADJ_THREADS)
upsample_adjoint_tiled_kernel(const float* __restrict__ dz_hi, FusedDzArgs fa, int Hf, int Wf, int H, int W, float sy,
                              float sx, int ry_max, int rx_max, float* __restrict__ dz_lo) {
  pdl_wait();
  extern __shared__ __align__(16) float sm[];
  float* reg = sm;                                  // [K][ry_max][rx_max]   hi-res gradient of the support region
  float* tmp = sm + (size_t)K * ry_max * rx_max;    // [K][ry_max][ADJ_TW]   after the x reduction
  const int b = blockIdx.z, tid = threadIdx.x;
  const int i0 = blockIdx.y * ADJ_TH, j0 = blockIdx.x * ADJ_TW;
  const int th = min(ADJ_TH, Hf - i0), tw = min(ADJ_TW, Wf - j0);
  int y0, y1, x0, x1, dummy;
  lerp_support(i0, sy, H, y0, dummy);
  lerp_support(i0 + th - 1, sy, H, dummy, y1);
  lerp_support(j0, sx, W, x0, dummy);
  lerp_support(j0 + tw - 1, sx, W, dummy, x1);
  const int ry = y1 - y0 + 1, rx = x1 - x0 + 1;  // <= ry_max, rx_max by construction of the launcher
  const long N = (long)H * W;

  // interpolation weight tables of this tile: for output column j0+tj the contiguous run of hi-res
  // columns [wx_start, wx_start+wx_cnt) that read it, with their weights (same for rows)
  __shared__ float wx_tab[ADJ_TW * ADJ_MAXW], wy_tab[ADJ_TH * ADJ_MAXW];
  __shared__ int wx_start[ADJ_TW], wx_cnt[ADJ_TW], wy_start[ADJ_TH], wy_cnt[ADJ_TH];
  if (tid < ADJ_TW + ADJ_TH) {
    const bool is_x = tid < ADJ_TW;
    const int t = is_x ? tid : tid - ADJ_TW;
    const int lim = is_x ? tw : th;
    if (t < lim) {
      const int want = (is_x ? j0 : i0) + t;
      const float sc = is_x ? sx : sy;
      const int in_size = is_x ? Wf : Hf, out_size = is_x ? W : H;
      int lo, hi;
      lerp_support(want, sc, out_size, lo, hi);
      int first = -1, cnt = 0;
      float* tab = (is_x ? wx_tab : wy_tab) + t * ADJ_MAXW;
      for (int o = lo; o <= hi; ++o) {
        const float w = lerp_weight(o, sc, in_size, want);
        if (w != 0.f || first >= 0) {
          if (first < 0) first = o;
          if (cnt < ADJ_MAXW) tab[cnt] = w;
          ++cnt;
        }
      }
      // trailing zeros are harmless; the run is contiguous because the weights form a hat function
      (is_x ? wx_start : wy_start)[t] = first < 0 ? lo : first;
      (is_x ? wx_cnt : wy_cnt)[t] = cnt < ADJ_MAXW ? cnt : ADJ_MAXW;
    }
  }

  // ---- phase 1: hi-res gradient of the region -> shared memory ----
  if constexpr (SRC == 0) {
    const int lane = tid & 31, warp = tid >> 5;
    for (int yy = warp; yy < ry; yy += ADJ_THREADS / 32)
      for (int xx = lane; xx < rx; xx += 32) {
        const float* src = dz_hi + (size_t)b * K * N + (size_t)(y0 + yy) * W + x0 + xx;
#pragma unroll
        for (int k = 0; k < K; ++k) reg[((size_t)k * ry_max + yy) * rx_max + xx] = __ldg(src + (size_t)k * N);
      }
  } else {
    const LevelInfo li = load_level_info<K>(MODE == RHSEG_ACT_GROUPED ? fa.table : nullptr);
    const float gce = fa.g_ce ? __ldg(fa.g_ce) : 0.f, gdi = fa.g_dice ? __ldg(fa.g_dice) : 0.f;
    float A[K], Bc[K], Cc[K], gu[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const float* cf = fa.coef + ((size_t)b * K + k) * 3;
      A[k] = gce * __ldg(cf);
      Bc[k] = gdi * __ldg(cf + 1);
      Cc[k] = gdi * __ldg(cf + 2);
      gu[k] = fa.g_uniform ? (float)fa.g_uniform[b * K + k] * fa.inv_npix : 0.f;
    }
    const bool has_act = MODE != RHSEG_ACT_ZEROS && (fa.g_uniform != nullptr || (fa.dp_pix != nullptr && fa.pix_mask != 0));
    const int lane = tid & 31, warp = tid >> 5;
    for (int yy = warp; yy < ry; yy += ADJ_THREADS / 32)
     for (int xx = lane; xx < rx; xx += 32) {
      const int y = y0 + yy, x = x0 + xx;
      const size_t px = (size_t)y * W + x;
      float z[K], t[K], dz[K];
#pragma unroll
      for (int k = 0; k < K; ++k) {
        z[k] = __ldg(fa.logits + ((size_t)b * K + k) * N + px);
        t[k] = __ldg(fa.targets + (size_t)b * fa.t_bstride + (size_t)k * fa.t_cstride + px);
      }
      loss_dz_pixel<K, true>(z, t, A, Bc, Cc, dz);
      if (has_act) {
        float dP[K], pp[K], dpar[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
          dP[k] = gu[k];
          if (fa.dp_pix && ((fa.pix_mask >> k) & 1u)) dP[k] += __ldg(fa.dp_pix + ((size_t)b * K + k) * N + px);
          pp[k] = 0.f;
        }
        if constexpr (MODE == RHSEG_ACT_GROUPED) {
#pragma unroll
          for (int k = 0; k < K; ++k)
            pp[k] = ((li.start_mask >> k) & 1) ? __ldg(fa.prev_probs + ((size_t)b * fa.K_prev + li.parent[k]) * N + px)
                                               : pp[k > 0 ? k - 1 : 0];
        }
        act_dz_pixel<K, MODE>(z, dP, pp, li.start_mask, dz, dpar);
        if constexpr (MODE == RHSEG_ACT_GROUPED) {
          // every hi-res pixel is owned by exactly one tile: the one holding floor(src index)
          if (fa.dp_prev) {
            const int oi = (int)(sy * (float)y), oj = (int)(sx * (float)x);
            if (oi >= i0 && oi < i0 + th && oj >= j0 && oj < j0 + tw) {
#pragma unroll
              for (int k = 0; k < K; ++k)
                if ((li.start_mask >> k) & 1) fa.dp_prev[((size_t)b * fa.K_prev + li.parent[k]) * N + px] += dpar[k];
            }
          }
        }
      }
#pragma unroll
      for (int k = 0; k < K; ++k) reg[((size_t)k * ry_max + yy) * rx_max + xx] = dz[k];
    }
  }
  __syncthreads();

  // ---- phase 2: reduce along x: tmp[k][yy][tj] = sum_x wx(x, j0+tj) reg[k][yy][x] ----
  // (the few non-zero interpolation weights per output column / row were tabulated once per CTA)
  {
    const int tj = tid & (ADJ_TW - 1), rslot = tid / ADJ_TW;
    if (tj < tw) {
      const int xs = wx_start[tj] - x0, xn = wx_cnt[tj];
      const float* wt = wx_tab + tj * ADJ_MAXW;
#pragma unroll
      for (int k = 0; k < K; ++k)
        for (int yy = rslot; yy < ry; yy += ADJ_THREADS / ADJ_TW) {
          const float* row = reg + ((size_t)k * ry_max + yy) * rx_max + xs;
          float acc = 0.f;
          for (int q = 0; q < xn; ++q) acc = fmaf(wt[q], row[q], acc);
          tmp[((size_t)k * ry_max + yy) * ADJ_TW + tj] = acc;
        }
    }
  }
  __syncthreads();

  // ---- phase 3: reduce along y and store ----
  {
    const int tj = tid & (ADJ_TW - 1), ti = (tid / ADJ_TW) & (ADJ_TH - 1), kslot = tid / (ADJ_TW * ADJ_TH);
    if (tj < tw && ti < th) {
      const int ys = wy_start[ti] - y0, yn = wy_cnt[ti];
      const float* wt = wy_tab + ti * ADJ_MAXW;
      for (int k = kslot; k < K; k += ADJ_THREADS / (ADJ_TW * ADJ_TH)) {
        const float* col = tmp + ((size_t)k * ry_max + ys) * ADJ_TW + tj;
        float acc = 0.f;
        for (int q = 0; q < yn; ++q) acc = fmaf(wt[q], col[q * ADJ_TW], acc);
        dz_lo[((size_t)b * K + k) * Hf * Wf + (size_t)(i0 + ti) * Wf + j0 + tj] = acc;
      }
    }
  }
}

// ------------------------------------------------------------------------------------
// Band adjoint (the HRNet case: upsampling, W % 4 == 0, pre-zeroed dz_lo).  A CTA owns a band of consecutive hi-res
// rows of one sample; consumer thread t owns the VEC pixels x0 = t*VEC .. of every row of the band.
//   * a producer warp (one lane) streams one stage per hi-res row -- K logit rows, K target rows (+ parent
//     probabilities / per-pixel probability gradients when the level receives them) -- by bulk async copy;
//   * per row a consumer forms the gradient of its pixels exactly once (closed-form loss gradient + activation
//     backward) and applies the adjoint of the y interpolation IN REGISTERS: row y feeds the low-res rows i0(y),
//     i0(y)+1 with the forward's own lerp weights, so two running accumulators per pixel suffice;
//   * whenever i0 advances (every ~scale rows) the finished accumulator row goes through shared memory once: the
//     adjoint of the x interpolation (tabulated taps per low-res column) and one fp32 add into the pre-zeroed dz_lo.
//     Only the first / last low-res row of a band is shared with the neighbouring band, so every dz_lo element
//     receives at most two terms: the fp32 result does not depend on the order (deterministic).
// dz_hi, the former tmpx [B,K,H,Wf] and a second kernel never exist; the x reduction runs once per low-res row
// instead of once per hi-res row.
// SRC 0: dz_hi is read from memory (drop-in route, what autograd hands us);  SRC 1: formed on the fly.
// ACTK (SRC 1): 1 = no gradient reaches the level's probabilities (last level), 2 = sigmoid level that only
// receives the uniform FiLM-pool gradient (level 0 of a two-level tree), 0 = decided at run time (deeper trees).
// ------------------------------------------------------------------------------------
constexpr int XR_MAXW = 12;  // max hi-res taps per low-res column held in the weight table (upsampling factor <= ~5)

template <int K, int GSZ>
__device__ __forceinline__ void group_sum_g(const float (&x)[K], const Groups<K, GSZ>& gr, float (&out)[K]) {
  if constexpr (GSZ == 0) {
    group_sum<K>(x, gr.start_mask, out);
  } else {
#pragma unroll
    for (int g = 0; g < K / GSZ; ++g) {
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < GSZ; ++j) s += x[g * GSZ + j];
#pragma unroll
      for (int j = 0; j < GSZ; ++j) out[g * GSZ + j] = s;
    }
  }
}

template <int K, int VEC, int SRC, int MODE, int ACTK, int GSZ>
__global__ void __launch_bounds__(VEC == 4 ? 192 + 32 : 384 + 32)
dz_band_kernel(const float* __restrict__ dz_hi, FusedDzArgs fa, int Hf, int Wf, int H, int W, float sy, float sx, int band,
               int ns, int n_dp, float* __restrict__ dz_lo) {
  constexpr bool GROUPED = MODE == RHSEG_ACT_GROUPED;
  constexpr bool NOACT = SRC == 0 || ACTK == 1 || MODE == RHSEG_ACT_ZEROS, UNIF = SRC == 1 && ACTK == 2;
  static_assert(!UNIF || MODE == RHSEG_ACT_SIGMOID, "uniform-only kind: sigmoid levels");
  constexpr int NG = Groups<K, GSZ>::NG;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ncons = (int)blockDim.x - 32, ncw = ncons >> 5;
  const int b = blockIdx.y;
  const int y_begin = blockIdx.x * band, y_end = min(H, y_begin + band);
  const long N = (long)H * W;
  const int TP = W + XR_MAXW;  // pitch of a flush row (the tap window may run past the row end: zero pad)

  StageRing ring;
  ring.init(reinterpret_cast<uint64_t*>(smem_raw), ns, ncw);
  float* Tbuf = reinterpret_cast<float*>(smem_raw + 128);  // [2][K][TP]
  unsigned char* stage0 = smem_raw + 128 + (((size_t)2 * K * TP * 4 + 127) & ~(size_t)127);

  Groups<K, GSZ> gr;
  gr.load((SRC == 1 && GROUPED) ? fa.table : nullptr);  // the level table is constant device data
  const bool has_act = UNIF || (!NOACT && (fa.g_uniform != nullptr || (fa.dp_pix != nullptr && fa.pix_mask != 0)));
  const int n_pp = (GROUPED && !NOACT && has_act) ? gr.n : 0;
  const int n_dpr = (!NOACT && !UNIF && has_act && fa.dp_pix != nullptr) ? n_dp : 0;  // rows of dp_pix (channels in pix_mask)
  const uint32_t rowb = (uint32_t)W * 4u;
  // stage layout: SRC 0: [K dz rows];  SRC 1: [K logit rows][K target rows][n_pp parent-probability rows][n_dpr dP rows]
  const uint32_t stage_bytes = (uint32_t)(SRC == 0 ? K : 2 * K + n_pp + n_dpr) * rowb;
  __syncthreads();  // barriers initialised

  if (warp == ncw) {
    // ------------------------------ producer: starts fetching while the consumers set up ------------------------------
    if (lane == 0) {
      pdl_wait();
      int slot = 0;
      uint32_t phase = 1;
      for (int y = y_begin; y < y_end; ++y) {
        mbar_wait(ring.empty(slot), phase);
        uint32_t dst = smem_u32(stage0 + (size_t)slot * stage_bytes);
        const uint32_t bar = ring.full(slot);
        const long px = (long)y * W;
        if constexpr (SRC == 0) {
#pragma unroll
          for (int k = 0; k < K; ++k) { bulk_g2s_plain(dst, dz_hi + ((size_t)b * K + k) * N + px, rowb, bar); dst += rowb; }
        } else {
#pragma unroll
          for (int k = 0; k < K; ++k) { bulk_g2s_plain(dst, fa.logits + ((size_t)b * K + k) * N + px, rowb, bar); dst += rowb; }
#pragma unroll
          for (int k = 0; k < K; ++k) {
            bulk_g2s_plain(dst, fa.targets + (size_t)b * fa.t_bstride + (size_t)k * fa.t_cstride + px, rowb, bar);
            dst += rowb;
          }
          if constexpr (GROUPED && !NOACT) {
#pragma unroll
            for (int g = 0; g < NG; ++g)
              if (g < n_pp) { bulk_g2s_plain(dst, fa.prev_probs + ((size_t)b * fa.K_prev + gr.parent[g]) * N + px, rowb, bar); dst += rowb; }
          }
          if constexpr (!NOACT && !UNIF) {
            if (n_dpr) {
#pragma unroll
              for (int k = 0; k < K; ++k)
                if ((fa.pix_mask >> k) & 1u) { bulk_g2s_plain(dst, fa.dp_pix + ((size_t)b * K + k) * N + px, rowb, bar); dst += rowb; }
            }
          }
        }
        mbar_arrive_expect_tx(bar, stage_bytes);
        if (++slot == ns) { slot = 0; phase ^= 1u; }
      }
    }
    return;
  }

  // -------------------------------- consumers --------------------------------
  auto csync = [ncons] { consumer_sync(ncons); };
  const int x0 = tid * VEC;
  const bool ok = x0 < W;  // W % VEC == 0 (launcher)
  const int xr = ok ? x0 : 0;  // lanes past the row end process (and never publish) the row start
  // taps of the x adjoint of this thread's low-res column j = tid: the hi-res columns that read it form a contiguous
  // run of <= XR_MAXW - 3 pixels; the weights sit in registers over a 16-byte aligned window of XR_MAXW pixels
  float wtap[XR_MAXW];
  int wbase = 0;
  {
    const int j = tid;
    int lo = 0, hi = 0;
    if (j < Wf) {
      lerp_support(j, sx, W, lo, hi);
      while (lo < hi && lerp_weight(lo, sx, Wf, j) == 0.f) ++lo;
    }
    wbase = lo & ~3;
#pragma unroll
    for (int q = 0; q < XR_MAXW; ++q) wtap[q] = (j < Wf && wbase + q < W) ? lerp_weight(wbase + q, sx, Wf, j) : 0.f;
    // the launcher sized the window for every tap; a weight beyond it would silently be lost: fail loudly instead
    if (j < Wf && wbase + XR_MAXW < W && lerp_weight(wbase + XR_MAXW, sx, Wf, j) != 0.f) __trap();
  }
  for (int e = tid; e < 2 * K * XR_MAXW; e += ncons) Tbuf[(size_t)(e / XR_MAXW) * TP + W + e % XR_MAXW] = 0.f;  // pad columns
  float A[K], Bc[K], Cc[K], gu[K];
  pdl_wait();  // coef / g_uniform are produced by the previous kernels; dz_lo was zeroed by one
  if constexpr (SRC == 1) {
    const float gce = fa.g_ce ? __ldg(fa.g_ce) : 0.f, gdi = fa.g_dice ? __ldg(fa.g_dice) : 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const float* cf = fa.coef + ((size_t)b * K + k) * 3;
      A[k] = gce * __ldg(cf);
      Bc[k] = gdi * __ldg(cf + 1);
      Cc[k] = gdi * __ldg(cf + 2);
      gu[k] = (!NOACT && fa.g_uniform) ? (float)fa.g_uniform[b * K + k] * fa.inv_npix : 0.f;
    }
  }
  float accA[K][VEC], accB[K][VEC];
#pragma unroll
  for (int k = 0; k < K; ++k)
#pragma unroll
    for (int v = 0; v < VEC; ++v) { accA[k][v] = 0.f; accB[k][v] = 0.f; }
  int cur = make_lerp(y_begin, sy, Hf).i0;  // low-res row accA belongs to (accB: cur + 1)
  const int last_lo = y_begin < y_end ? make_lerp(y_end - 1, sy, Hf).i1 : cur - 1;
  int tb = 0;
  int slot = 0;
  uint32_t phase = 0;
  for (int y = y_begin;; ++y) {
    // adjoint of the y interpolation lives in registers: row y feeds the low-res rows i0(y) (accA) and i0(y)+1 (accB).
    // Rows below i0(y) are complete: each goes through shared memory once -- adjoint of the x interpolation -- and is
    // added into dz_lo.  After the last row everything up to last_lo is flushed.
    Lerp ly;
    ly.i0 = last_lo + 1; ly.i1 = ly.i0; ly.l0 = 0.f; ly.l1 = 0.f;
    if (y < y_end) ly = make_lerp(y, sy, Hf);
    while (cur < ly.i0) {  // uniform over the CTA
      float* T = Tbuf + (size_t)tb * K * TP;
      if (ok) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
          Vec<VEC> o;
#pragma unroll
          for (int v = 0; v < VEC; ++v) o.v[v] = accA[k][v];
          *reinterpret_cast<Vec<VEC>*>(T + (size_t)k * TP + x0) = o;
        }
      }
      csync();
      if (tid < Wf) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
          const float4* row = reinterpret_cast<const float4*>(T + (size_t)k * TP + wbase);
          float a = 0.f;
#pragma unroll
          for (int q4 = 0; q4 < XR_MAXW / 4; ++q4) {
            const float4 tv = row[q4];
            a = fmaf(wtap[4 * q4 + 0], tv.x, a);
            a = fmaf(wtap[4 * q4 + 1], tv.y, a);
            a = fmaf(wtap[4 * q4 + 2], tv.z, a);
            a = fmaf(wtap[4 * q4 + 3], tv.w, a);
          }
          atomicAdd(dz_lo + (((size_t)b * K + k) * Hf + cur) * Wf + tid, a);
        }
      }
      tb ^= 1;  // the next flush writes the other buffer: its barrier orders it after this one's readers
#pragma unroll
      for (int k = 0; k < K; ++k)
#pragma unroll
        for (int v = 0; v < VEC; ++v) { accA[k][v] = accB[k][v]; accB[k][v] = 0.f; }
      ++cur;
    }
    if (y >= y_end) break;

    mbar_wait(ring.full(slot), phase);
    const float* sf = reinterpret_cast<const float*>(stage0 + (size_t)slot * stage_bytes) + xr;
    float dz[K][VEC];
    if constexpr (SRC == 0) {
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const Vec<VEC> dv = *reinterpret_cast<const Vec<VEC>*>(sf + (size_t)k * W);
#pragma unroll
        for (int v = 0; v < VEC; ++v) dz[k][v] = dv.v[v];
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(ring.empty(slot));
    } else {
      float z[K][VEC], t[K][VEC], ppg[NG][VEC], ex[K][VEC];
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const Vec<VEC> zv = *reinterpret_cast<const Vec<VEC>*>(sf + (size_t)k * W);
        const Vec<VEC> tv = *reinterpret_cast<const Vec<VEC>*>(sf + (size_t)(K + k) * W);
#pragma unroll
        for (int v = 0; v < VEC; ++v) { z[k][v] = zv.v[v]; t[k][v] = tv.v[v]; ex[k][v] = 0.f; }
      }
      int row = 2 * K;
      if constexpr (GROUPED && !NOACT) {
#pragma unroll
        for (int g = 0; g < NG; ++g) {
#pragma unroll
          for (int v = 0; v < VEC; ++v) ppg[g][v] = 0.f;
          if (g < n_pp) {
            const Vec<VEC> pv = *reinterpret_cast<const Vec<VEC>*>(sf + (size_t)(row++) * W);
#pragma unroll
            for (int v = 0; v < VEC; ++v) ppg[g][v] = pv.v[v];
          }
        }
      }
      if constexpr (!NOACT && !UNIF) {
        if (n_dpr) {
#pragma unroll
          for (int k = 0; k < K; ++k)
            if ((fa.pix_mask >> k) & 1u) {
              const Vec<VEC> ev = *reinterpret_cast<const Vec<VEC>*>(sf + (size_t)(row++) * W);
#pragma unroll
              for (int v = 0; v < VEC; ++v) ex[k][v] = ev.v[v];
            }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(ring.empty(slot));  // the row is in registers
      float dpar[NG][VEC];
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        float zz[K], tt[K], o[K];
#pragma unroll
        for (int k = 0; k < K; ++k) { zz[k] = z[k][v]; tt[k] = t[k][v]; }
        loss_dz_pixel<K, true>(zz, tt, A, Bc, Cc, o);
        if constexpr (UNIF) {
#pragma unroll
          for (int k = 0; k < K; ++k) {
            const float p = sigmoidf_ref(zz[k]);
            o[k] = fmaf(gu[k], p * (1.0f - p), o[k]);
          }
        } else if constexpr (!NOACT) {
          if (has_act) {
            if constexpr (MODE == RHSEG_ACT_SIGMOID) {
#pragma unroll
              for (int k = 0; k < K; ++k) {
                const float p = sigmoidf_ref(zz[k]);
                o[k] = fmaf(gu[k] + ex[k][v], p * (1.0f - p), o[k]);
              }
            } else {
              // P_c = P_p Q_c: dQ_c = dP_c P_p; dz += Q (dQ - sum_group dQ Q); dP_p = sum_group dP_c Q_c
              float q[K], dpq[K], dq_q[K], inner[K], dpp[K], pg[NG];
#pragma unroll
              for (int g = 0; g < NG; ++g) pg[g] = ppg[g][v];
              softmax_groups<K, GSZ>(zz, gr, q);
#pragma unroll
              for (int k = 0; k < K; ++k) {
                dpq[k] = (gu[k] + ex[k][v]) * q[k];
                dq_q[k] = dpq[k] * group_value<K, GSZ>(pg, gr, k);
              }
              group_sum_g<K, GSZ>(dq_q, gr, inner);
              group_sum_g<K, GSZ>(dpq, gr, dpp);
#pragma unroll
              for (int k = 0; k < K; ++k) o[k] += dq_q[k] - q[k] * inner[k];
              // the group's sum sits at every member: pick the value at the group's first channel
#pragma unroll
              for (int g = 0; g < NG; ++g) {
                float val = 0.f;
                if constexpr (GSZ > 0) val = dpp[g * GSZ];
                else {
                  int seen = 0;
#pragma unroll
                  for (int k = 0; k < K; ++k)
                    if ((gr.start_mask >> k) & 1) { if (seen == g) val = dpp[k]; ++seen; }
                }
                dpar[g][v] = val;
              }
            }
          }
        }
#pragma unroll
        for (int k = 0; k < K; ++k) dz[k][v] = o[k];
      }
      if constexpr (GROUPED && !NOACT) {
        if (has_act && fa.dp_prev && ok) {  // every hi-res pixel is visited exactly once: plain stores
#pragma unroll
          for (int g = 0; g < NG; ++g)
            if (g < n_pp) {
              Vec<VEC> o;
#pragma unroll
              for (int v = 0; v < VEC; ++v) o.v[v] = dpar[g][v];
              *reinterpret_cast<Vec<VEC>*>(fa.dp_prev + ((size_t)b * fa.K_prev + gr.parent[g]) * N + (size_t)y * W + x0) = o;
            }
        }
      }
    }
    if (++slot == ns) { slot = 0; phase ^= 1u; }
    const bool two = ly.i1 > ly.i0;
#pragma unroll
    for (int k = 0; k < K; ++k)
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        accA[k][v] = fmaf(ly.l0, dz[k][v], accA[k][v]);
        if (two) accB[k][v] = fmaf(ly.l1, dz[k][v], accB[k][v]);
        else accA[k][v] = fmaf(ly.l1, dz[k][v], accA[k][v]);
      }
  }
}

template <int K, int VEC, int SRC, int MODE, int ACTK, int GSZ>
static int launch_dz_band(const float* dz_hi, const FusedDzArgs& fa, int B, int Hf, int Wf, int H, int W, float sy, float sx,
                          float* dz_lo, cudaStream_t st, bool* launched) {
  *launched = false;
  auto kern = dz_band_kernel<K, VEC, SRC, MODE, ACTK, GSZ>;
  const int ncons = ((W / VEC + 31) / 32) * 32;
  if (ncons > (VEC == 4 ? 192 : 384)) return RHSEG_OK;
  int n_dp = 0;
  for (int k = 0; k < K; ++k) n_dp += (fa.pix_mask >> k) & 1u;
  // worst-case stage (the kernel derives the actual row count from the table / flags)
  const int rows = SRC == 0 ? K : 2 * K + ((MODE == RHSEG_ACT_GROUPED && ACTK == 0) ? Groups<K, GSZ>::NG : 0) + (ACTK == 0 ? n_dp : 0);
  const size_t stage = (size_t)rows * W * 4;
  static int tune_ns = -1;
  if (tune_ns < 0) { const char* e = getenv("RHSEG_TUNE_DZ_NS"); tune_ns = e ? atoi(e) : 0; }
  const int ns = tune_ns > 0 ? std::min(tune_ns, 7) : 3;
  const size_t fixed = 128 + (((size_t)2 * K * (W + XR_MAXW) * 4 + 127) & ~(size_t)127);
  if (Wf > ncons) return RHSEG_OK;  // one low-res column per consumer thread in the x adjoint
  const size_t smem = fixed + (size_t)ns * stage;
  if (smem > 200 * 1024) return RHSEG_OK;
  int per_sm = 0;
  RHSEG_CUDA(cached_launch_prep(reinterpret_cast<const void*>(kern), ncons + 32, smem, smem, &per_sm));
  if (per_sm < 1) return RHSEG_OK;
  static int tune_ctas = -1;
  if (tune_ctas < 0) { const char* e = getenv("RHSEG_TUNE_DZ_CTAS"); tune_ctas = e ? atoi(e) : 0; }
  if (tune_ctas > 0) per_sm = std::min(per_sm, tune_ctas);
  const long slots = std::max<long>(1, (long)per_sm * device_sm_count() / B);
  // >= taps per low-res row, so that at most two CTAs feed one low-res row
  const int min_band = std::max(4, (int)ceilf(2.0f / sy));
  const int band = std::max(min_band, (int)((H + slots - 1) / slots));
  dim3 grid((unsigned)((H + band - 1) / band), B);
  launch_pdl(kern, dim3(grid), dim3(ncons + 32), smem, st, dz_hi, fa, Hf, Wf, H, W, sy, sx, band, ns, n_dp, dz_lo);
  RHSEG_LAUNCH_CHECK();
  *launched = true;
  return RHSEG_OK;
}

// Full-resolution donors (UNet): the same fused per-pixel gradient, written out once as dz.  LT: logit and dz element
// type (float, or uint16_t = bf16 bits: fa.logits then points at bf16 values; RHSEG_ACT_ZEROS only).
template <int K, int VEC, int MODE, int THREADS, typename LT = float>
__global__ void __launch_bounds__(THREADS)
dz_fullres_fused_kernel(FusedDzArgs fa, long N, LT* __restrict__ dz_out) {
  pdl_wait();
  const int b = blockIdx.y;
  const long px = ((long)blockIdx.x * THREADS + threadIdx.x) * VEC;
  if (px >= N) return;
  const LevelInfo li = load_level_info<K>(MODE == RHSEG_ACT_GROUPED ? fa.table : nullptr);
  const float gce = fa.g_ce ? __ldg(fa.g_ce) : 0.f, gdi = fa.g_dice ? __ldg(fa.g_dice) : 0.f;
  float A[K], Bc[K], Cc[K], gu[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const float* cf = fa.coef + ((size_t)b * K + k) * 3;
    A[k] = gce * __ldg(cf);
    Bc[k] = gdi * __ldg(cf + 1);
    Cc[k] = gdi * __ldg(cf + 2);
    gu[k] = fa.g_uniform ? (float)fa.g_uniform[b * K + k] * fa.inv_npix : 0.f;
  }
  const bool has_act = MODE != RHSEG_ACT_ZEROS && (fa.g_uniform != nullptr || (fa.dp_pix != nullptr && fa.pix_mask != 0));
  float z[K][VEC], t[K][VEC], e[K][VEC], pp[K][VEC], o[K][VEC], dpar[K][VEC];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const Vec<VEC> zv = ld_stream<VEC>(reinterpret_cast<const LT*>(fa.logits) + ((size_t)b * K + k) * N + px);
    const Vec<VEC> tv = ld_cached<VEC>(fa.targets + (size_t)b * fa.t_bstride + (size_t)k * fa.t_cstride + px);
    Vec<VEC> ev;
#pragma unroll
    for (int v = 0; v < VEC; ++v) ev.v[v] = 0.f;
    if (has_act && fa.dp_pix && ((fa.pix_mask >> k) & 1u)) ev = ld_stream<VEC>(fa.dp_pix + ((size_t)b * K + k) * N + px);
#pragma unroll
    for (int v = 0; v < VEC; ++v) { z[k][v] = zv.v[v]; t[k][v] = tv.v[v]; e[k][v] = ev.v[v]; pp[k][v] = 0.f; }
  }
  if constexpr (MODE == RHSEG_ACT_GROUPED) {
    if (has_act) {
#pragma unroll
      for (int k = 0; k < K; ++k) {
        if ((li.start_mask >> k) & 1) {
          const Vec<VEC> pv = ld_stream<VEC>(fa.prev_probs + ((size_t)b * fa.K_prev + li.parent[k]) * N + px);
#pragma unroll
          for (int v = 0; v < VEC; ++v) pp[k][v] = pv.v[v];
        } else {
#pragma unroll
          for (int v = 0; v < VEC; ++v) pp[k][v] = pp[k > 0 ? k - 1 : 0][v];
        }
      }
    }
  }
#pragma unroll
  for (int v = 0; v < VEC; ++v) {
    float zz[K], tt[K], dz[K], dP[K], ppv[K], dpv[K];
#pragma unroll
    for (int k = 0; k < K; ++k) { zz[k] = z[k][v]; tt[k] = t[k][v]; dP[k] = gu[k] + e[k][v]; ppv[k] = pp[k][v]; dpv[k] = 0.f; }
    loss_dz_pixel<K, true>(zz, tt, A, Bc, Cc, dz);
    if (has_act) act_dz_pixel<K, MODE>(zz, dP, ppv, li.start_mask, dz, dpv);
#pragma unroll
    for (int k = 0; k < K; ++k) { o[k][v] = dz[k]; dpar[k][v] = dpv[k]; }
  }
#pragma unroll
  for (int k = 0; k < K; ++k) {
    Vec<VEC> r;
#pragma unroll
    for (int v = 0; v < VEC; ++v) r.v[v] = o[k][v];
    st_grad<VEC>(dz_out + ((size_t)b * K + k) * N + px, r);  // re-read by the conv backward: keep cached
  }
  if constexpr (MODE == RHSEG_ACT_GROUPED) {
    if (has_act && fa.dp_prev) {
#pragma unroll
      for (int k = 0; k < K; ++k)
        if ((li.start_mask >> k) & 1) {
          float* dst = fa.dp_prev + ((size_t)b * fa.K_prev + li.parent[k]) * N + px;
          Vec<VEC> cur = *reinterpret_cast<const Vec<VEC>*>(dst);
#pragma unroll
          for (int v = 0; v < VEC; ++v) cur.v[v] += dpar[k][v];
          *reinterpret_cast<Vec<VEC>*>(dst) = cur;
        }
    }
  }
}

// host: worst-case support extent of a tile of `t` inputs (mirrors lerp_support)
static int region_extent(int t, float scale, int out_size) {
  if (scale <= 0.f) return out_size;
  const int e = (int)ceilf((float)(t + 1) / scale) + 5;
  return e < out_size ? e : out_size;
}

template <int K, int SRC, int MODE>
static int launch_adjoint(const float* dz_hi, const FusedDzArgs& fa, int hint, int B, int Hf, int Wf, int H, int W, float* dz_lo,
                          bool prezeroed, cudaStream_t st) {
  const float sy = H > 1 ? (float)(Hf - 1) / (float)(H - 1) : 0.f;
  const float sx = W > 1 ? (float)(Wf - 1) / (float)(W - 1) : 0.f;
  if constexpr (MODE != RHSEG_ACT_ZEROS || SRC == 0) {
    auto al = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
    // taps per low-res column (<= 2/sx + 1) plus the alignment slack of the 16-byte window must fit XR_MAXW
    // the hi-res columns with a non-zero weight for low-res column j lie in the open interval ((j-1)/sx, (j+1)/sx):
    // at most ceil(2/sx) of them, plus up to 3 columns of alignment slack in front
    bool band_ok = prezeroed && W % 4 == 0 && sx > 0.f && sy > 0.f && sy <= 1.0f && ceilf(2.0f / sx) + 3.0f <= (float)XR_MAXW &&
                   !getenv("RHSEG_NO_BAND_ADJOINT");
    if (SRC == 0) band_ok = band_ok && al(dz_hi);
    else band_ok = band_ok && al(fa.logits) && al(fa.targets) && fa.t_bstride % 4 == 0 && fa.t_cstride % 4 == 0 &&
                   al(fa.prev_probs) && al(fa.dp_pix) && al(fa.dp_prev);
    if (band_ok) {
      static int tune_vec = -1;
      if (tune_vec < 0) { const char* e = getenv("RHSEG_TUNE_DZ_VEC"); tune_vec = e ? atoi(e) : 0; }
      const bool no_pix = fa.dp_pix == nullptr || fa.pix_mask == 0;
      const bool no_act = SRC == 1 && fa.g_uniform == nullptr && no_pix;
      const bool unif = SRC == 1 && MODE == RHSEG_ACT_SIGMOID && fa.g_uniform != nullptr && no_pix;
      bool done = false;
      int rc = RHSEG_OK;
#define RHSEG_DZB(VEC, ACTK, GS) rc = launch_dz_band<K, VEC, SRC, MODE, ACTK, GS>(dz_hi, fa, B, Hf, Wf, H, W, sy, sx, dz_lo, st, &done)
#define RHSEG_DZB_V(ACTK, GS)                                   \
      do {                                                      \
        if (tune_vec != 2 || K > 4) RHSEG_DZB(4, ACTK, GS);     \
        if constexpr (K <= 4) { /* 2 px / thread: up to 416 threads, too few registers for K > 4 (spills) */ \
          if (!done && rc == RHSEG_OK) RHSEG_DZB(2, ACTK, GS);  \
        }                                                       \
      } while (0)
      if constexpr (SRC == 0) {
        RHSEG_DZB_V(1, K);
      } else if constexpr (MODE == RHSEG_ACT_SIGMOID) {
        if (no_act) RHSEG_DZB_V(1, K); else if (unif) RHSEG_DZB_V(2, K); else RHSEG_DZB_V(0, K);
      } else {
        bool uniform2 = false;
        if constexpr (K == 4) uniform2 = hint == 2;  // two parents with two children each (class_tree_tl_extended.json, level 2)
        if (no_act) RHSEG_DZB_V(1, K); else if (hint == K) RHSEG_DZB_V(0, K);
        else if (uniform2) { if constexpr (K == 4) RHSEG_DZB_V(0, 2); }
        else if constexpr (K <= 5) RHSEG_DZB_V(0, 0);  // table-driven group layout with K > 5 would spill: tiled kernel below
      }
#undef RHSEG_DZB_V
#undef RHSEG_DZB
      if (rc != RHSEG_OK) return rc;
      if (done) return RHSEG_OK;
    }
  }
  // generic: shared-memory tiled kernel (any alignment, halo recomputation); writes dz_lo
  const int ry_max = region_extent(ADJ_TH, sy, H), rx_max = region_extent(ADJ_TW, sx, W) | 1;  // odd pitch: fewer bank conflicts
  const size_t smem = ((size_t)K * ry_max * rx_max + (size_t)K * ry_max * ADJ_TW) * sizeof(float);
  if (smem > 200 * 1024) return RHSEG_ERR_UNSUPPORTED;  // upsampling factor too large for the tiled kernel
  if (sy > 0.f && 2.0f / sy + 4.0f > (float)ADJ_MAXW) return RHSEG_ERR_UNSUPPORTED;
  if (sx > 0.f && 2.0f / sx + 4.0f > (float)ADJ_MAXW) return RHSEG_ERR_UNSUPPORTED;
  if ((sy <= 0.f && H > ADJ_MAXW) || (sx <= 0.f && W > ADJ_MAXW)) return RHSEG_ERR_UNSUPPORTED;
  auto kern = upsample_adjoint_tiled_kernel<K, SRC, MODE>;
  if (smem > 48 * 1024) RHSEG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid((Wf + ADJ_TW - 1) / ADJ_TW, (Hf + ADJ_TH - 1) / ADJ_TH, B);
  launch_pdl(kern, dim3(grid), dim3(ADJ_THREADS), smem, st, dz_hi, fa, Hf, Wf, H, W, sy, sx, ry_max, rx_max, dz_lo);
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}

}  // namespace rhseg

using namespace rhseg;

extern "C" int rhseg_upsample_adjoint(const float* dz_hi, int B, int K, int Hf, int Wf, int H, int W, float* dz_lo,
                                      float* tmp, int flags, void* stream) {
  if (!dz_hi || !dz_lo || B <= 0 || Hf <= 0 || Wf <= 0 || H <= 0 || W <= 0) return RHSEG_ERR_ARG;
  if (K < 1 || K > RHSEG_KERNEL_MAX_K) return RHSEG_ERR_UNSUPPORTED;
  FusedDzArgs fa{};
  (void)tmp;  // workspace of an earlier two-kernel form; unused
  RHSEG_DISPATCH_K(K, return (launch_adjoint<KK, 0, 0>(dz_hi, fa, 0, B, Hf, Wf, H, W, dz_lo, (flags & RHSEG_DZ_PREZEROED) != 0, (cudaStream_t)stream)));
  return RHSEG_OK;
}

extern "C" int rhseg_head_dz_lowres_fused(const float* logits, const float* targets, long t_bstride, long t_cstride,
                                          const float* coef, const float* g_ce, const float* g_dice,
                                          const float* prev_probs, const int32_t* table, const double* g_uniform,
                                          double inv_npix, const float* dp_pix, uint32_t pix_mask, int B, int K,
                                          int K_prev, int Hf, int Wf, int H, int W, int act_mode, float* dz_lo,
                                          float* dp_prev, float* tmp, int flags, void* stream) {
  if (!logits || !targets || !coef || !dz_lo || B <= 0 || Hf <= 0 || Wf <= 0 || H <= 0 || W <= 0) return RHSEG_ERR_ARG;
  if (K < 1 || K > RHSEG_KERNEL_MAX_K) return RHSEG_ERR_UNSUPPORTED;
  const int hint = RHSEG_GROUP_HINT_OF(act_mode);
  act_mode &= 0xff;
  (void)tmp;  // workspace of an earlier two-kernel form; unused
  if (act_mode == RHSEG_ACT_GROUPED && (!prev_probs || !table)) return RHSEG_ERR_ARG;
  FusedDzArgs fa{logits, targets, t_bstride, t_cstride, coef, g_ce, g_dice, prev_probs, table, g_uniform,
                 (float)inv_npix, dp_pix, pix_mask, dp_prev, K_prev};
  cudaStream_t st = (cudaStream_t)stream;
  const bool pz = (flags & RHSEG_DZ_PREZEROED) != 0;
  RHSEG_DISPATCH_K(K, {
    if (act_mode == RHSEG_ACT_SIGMOID) return launch_adjoint<KK, 1, RHSEG_ACT_SIGMOID>(nullptr, fa, hint, B, Hf, Wf, H, W, dz_lo, pz, st);
    if (act_mode == RHSEG_ACT_GROUPED) return launch_adjoint<KK, 1, RHSEG_ACT_GROUPED>(nullptr, fa, hint, B, Hf, Wf, H, W, dz_lo, pz, st);
    return launch_adjoint<KK, 1, RHSEG_ACT_ZEROS>(nullptr, fa, hint, B, Hf, Wf, H, W, dz_lo, pz, st);
  });
  return RHSEG_OK;
}

extern "C" int rhseg_head_dz_fullres_fused(const void* logits, const float* targets, long t_bstride, long t_cstride,
                                           const float* coef, const float* g_ce, const float* g_dice,
                                           const float* prev_probs, const int32_t* table, const double* g_uniform,
                                           double inv_npix, const float* dp_pix, uint32_t pix_mask, int B, int K,
                                           int K_prev, int n_pix, int act_mode, void* dz_out, float* dp_prev,
                                           void* stream) {
  if (!logits || !targets || !coef || !dz_out || B <= 0 || n_pix <= 0) return RHSEG_ERR_ARG;
  if (K < 1 || K > RHSEG_KERNEL_MAX_K) return RHSEG_ERR_UNSUPPORTED;
  const bool bf16 = (act_mode & RHSEG_LOGITS_BF16) != 0;
  act_mode &= 0xff & ~RHSEG_LOGITS_BF16;
  if (bf16 && act_mode != RHSEG_ACT_ZEROS) return RHSEG_ERR_UNSUPPORTED;  // only the flat model's logits are bf16
  if (act_mode == RHSEG_ACT_GROUPED && (!prev_probs || !table)) return RHSEG_ERR_ARG;
  // bf16: fa.logits carries the bf16 pointer; the kernel instance reads it as such
  FusedDzArgs fa{static_cast<const float*>(logits), targets, t_bstride, t_cstride, coef, g_ce, g_dice, prev_probs, table,
                 g_uniform, (float)inv_npix, dp_pix, pix_mask, dp_prev, K_prev};
  cudaStream_t st = (cudaStream_t)stream;
  const long N = n_pix;
  constexpr int THREADS = 256;
  auto al = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
  const bool v4 = (N % 4 == 0) && al(logits) && al(targets) && t_bstride % 4 == 0 && t_cstride % 4 == 0 && al(dz_out) &&
                  al(prev_probs) && al(dp_pix) && al(dp_prev);
  const dim3 grid((unsigned)(v4 ? (N / 4 + THREADS - 1) / THREADS : (N + THREADS - 1) / THREADS), B);
  if (bf16) {
    auto* dz = static_cast<uint16_t*>(dz_out);
    RHSEG_DISPATCH_K(K, {
      if (v4) launch_pdl(dz_fullres_fused_kernel<KK, 4, RHSEG_ACT_ZEROS, THREADS, uint16_t>, grid, dim3(THREADS), 0, st, fa, N, dz);
      else launch_pdl(dz_fullres_fused_kernel<KK, 1, RHSEG_ACT_ZEROS, THREADS, uint16_t>, grid, dim3(THREADS), 0, st, fa, N, dz);
    });
    RHSEG_LAUNCH_CHECK();
    return RHSEG_OK;
  }
  float* dz = static_cast<float*>(dz_out);
  RHSEG_DISPATCH_K(K, {
    if (v4) {
      if (act_mode == RHSEG_ACT_SIGMOID) launch_pdl(dz_fullres_fused_kernel<KK, 4, RHSEG_ACT_SIGMOID, THREADS>, grid, dim3(THREADS), 0, st, fa, N, dz);
      else if (act_mode == RHSEG_ACT_GROUPED) launch_pdl(dz_fullres_fused_kernel<KK, 4, RHSEG_ACT_GROUPED, THREADS>, grid, dim3(THREADS), 0, st, fa, N, dz);
      else launch_pdl(dz_fullres_fused_kernel<KK, 4, RHSEG_ACT_ZEROS, THREADS>, grid, dim3(THREADS), 0, st, fa, N, dz);
    } else {
      if (act_mode == RHSEG_ACT_SIGMOID) launch_pdl(dz_fullres_fused_kernel<KK, 1, RHSEG_ACT_SIGMOID, THREADS>, grid, dim3(THREADS), 0, st, fa, N, dz);
      else if (act_mode == RHSEG_ACT_GROUPED) launch_pdl(dz_fullres_fused_kernel<KK, 1, RHSEG_ACT_GROUPED, THREADS>, grid, dim3(THREADS), 0, st, fa, N, dz);
      else launch_pdl(dz_fullres_fused_kernel<KK, 1, RHSEG_ACT_ZEROS, THREADS>, grid, dim3(THREADS), 0, st, fa, N, dz);
    }
  });
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}
