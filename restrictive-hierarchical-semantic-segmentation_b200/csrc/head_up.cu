// HRNet hi-res pass: bilinear (align_corners=True) upsample of the low-res logits fused with the activation,
// the composition, the FiLM pool sums and (optionally) the level's training evaluation.
// Reference semantics: Models/models.py:766/:776 (upsample), :767/:779-796 (activation, composition).
#include <algorithm>
#include <cstdlib>
#include <type_traits>
#include "common.cuh"
#include "hires.cuh"
#include "head_common.cuh"

namespace rhseg {

// ------------------------------------------------------------------------------------
// HRNet hi-res pass: bilinear (align_corners=True) upsample of the low-res logits fused with
// the activation.  Index/lambda arithmetic follows ATen's upsample_bilinear2d (fp32 scale =
// (in-1)/(out-1), src = scale*dst, i0 = (int)src, lambda1 = src - i0).
// ------------------------------------------------------------------------------------
template <int K, int VEC, int MODE, int THREADS>
__global__ void __launch_bounds__(THREADS)
upsample_act_kernel(const float* __restrict__ z_lo, const float* __restrict__ prev_probs,
                    const int32_t* __restrict__ table, int Hf, int Wf, int H, int W, int K_prev,
                    float sy, float sx, long total_vec, float* __restrict__ logits,
                    float* __restrict__ probs, double* __restrict__ psum, int vec_per_sample) {
  pdl_wait();
  __shared__ float red[(THREADS / 32) * K];
  const int b = blockIdx.y;
  const long vi = (long)blockIdx.x * THREADS + threadIdx.x;  // vector index inside the sample
  const bool ok = vi < vec_per_sample;
  const int wv = W / VEC;
  const int y = ok ? (int)(vi / wv) : 0;
  const int x0 = ok ? (int)(vi - (long)y * wv) * VEC : 0;
  const long N = (long)H * W, Nf = (long)Hf * Wf;
  const long px = (long)y * W + x0;

  float z[K][VEC], pp[K][VEC], prob[K][VEC];
  const LevelInfo li = load_level_info<K>(MODE == RHSEG_ACT_GROUPED ? table : nullptr);
  if (ok) {
    const Lerp ly = make_lerp(y, sy, Hf);
    Lerp lx[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) lx[v] = make_lerp(x0 + v, sx, Wf);
    const float* zb = z_lo + (size_t)b * K * Nf;
    // neighbour offsets are shared by all K channels
    int o00[VEC], o01[VEC], o10[VEC], o11[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      o00[v] = ly.i0 * Wf + lx[v].i0; o01[v] = ly.i0 * Wf + lx[v].i1;
      o10[v] = ly.i1 * Wf + lx[v].i0; o11[v] = ly.i1 * Wf + lx[v].i1;
    }
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const float* zk = zb + (size_t)k * Nf;
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        const float a = __ldg(zk + o00[v]), bq = __ldg(zk + o01[v]);
        const float c = __ldg(zk + o10[v]), d = __ldg(zk + o11[v]);
        z[k][v] = ly.l0 * (lx[v].l0 * a + lx[v].l1 * bq) + ly.l1 * (lx[v].l0 * c + lx[v].l1 * d);
      }
    }
    if constexpr (MODE == RHSEG_ACT_GROUPED) {
      const float* pb = prev_probs + (size_t)b * K_prev * N;
#pragma unroll
      for (int k = 0; k < K; ++k) {
        if ((li.start_mask >> k) & 1) {
          const Vec<VEC> t = ld_cached<VEC>(pb + (size_t)li.parent[k] * N + px);
#pragma unroll
          for (int v = 0; v < VEC; ++v) pp[k][v] = t.v[v];
        } else {
#pragma unroll
          for (int v = 0; v < VEC; ++v) pp[k][v] = pp[k > 0 ? k - 1 : 0][v];
        }
      }
    }
  } else {
#pragma unroll
    for (int k = 0; k < K; ++k)
#pragma unroll
      for (int v = 0; v < VEC; ++v) { z[k][v] = 0.f; pp[k][v] = 0.f; }
  }
  activate<K, VEC, MODE>(z, pp, li.start_mask, prob);
  float ps[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    ps[k] = 0.f;
    if (ok) {
      Vec<VEC> zo, po;
#pragma unroll
      for (int v = 0; v < VEC; ++v) { zo.v[v] = z[k][v]; po.v[v] = prob[k][v]; ps[k] += po.v[v]; }
      *reinterpret_cast<Vec<VEC>*>(logits + ((size_t)b * K + k) * N + px) = zo;
      *reinterpret_cast<Vec<VEC>*>(probs + ((size_t)b * K + k) * N + px) = po;
    }
  }
  block_psum<K, THREADS / 32>(ps, psum + (size_t)b * K, red, [] { __syncthreads(); });
}

// ------------------------------------------------------------------------------------
// Band kernel (the HRNet case: upsampling, W % 4 == 0).  A CTA owns a band of consecutive hi-res rows of one sample;
// consumer thread t owns the VEC pixels x0 = t*VEC .. of every row of the band.
//   * prologue (before griddepcontrol.wait: overlaps the previous kernel's tail): the thread's x interpolation is
//     folded into weights over the <= 3 low-res columns its pixels read; barriers;
//   * the producer warp (one lane) loads the band's low-res logit rows ONCE (K bulk copies of the enclosing
//     16-byte-aligned spans: HRNet planes are only 4-byte aligned) and then streams one stage per hi-res row:
//     parent probabilities (grouped levels) and, with the fused evaluation, targets / parent targets / previous
//     index map -- every per-pixel input arrives by bulk async copy, consumers never wait on global memory;
//   * per row a consumer lerps its 3 columns along y (2 x 3 shared-memory loads per channel), applies the x
//     weights, runs the activation (+ the evaluation, hires.cuh) and stores logits / probabilities.
// Interpolation arithmetic: ATen's index / lambda formulas (make_lerp); y is applied before x, which reorders the
// four-term sum (differences of a few 1e-8 relative; the tests compare at 1e-5).
// ------------------------------------------------------------------------------------
template <int K, int VEC, int MODE, int EVALK, int GSZ>
__global__ void __launch_bounds__(VEC == 4 ? 192 + 32 : 384 + 32)
upsample_band_kernel(const float* __restrict__ z_lo, const float* __restrict__ prev_probs,
                     const int32_t* __restrict__ table, int Hf, int Wf, int H, int W, int K_prev, float sy, float sx,
                     int band, int lok, int ns, int a0, float* __restrict__ logits, float* __restrict__ probs,
                     double* __restrict__ psum, EvalArgs ea) {
  constexpr bool EVAL = EVALK != 0, GROUPED = MODE == RHSEG_ACT_GROUPED;
  // EVALK 3: the validation evaluation (ValAcc) on the composed probabilities; its consistency term reads the parent
  // probabilities the activation already streams, so it needs no input beyond the targets
  constexpr bool COMPOSED = EVALK == 3;
  constexpr int CT = !GROUPED ? 0 : (EVALK == 2 || COMPOSED ? 2 : 1);
  constexpr bool CONS = EVAL && CT == 2 && !COMPOSED;
  using Acc = std::conditional_t<COMPOSED, ValAcc<K, CT, GSZ>, EvalAcc<K, CT, GSZ>>;
  constexpr int NG = Groups<K, GSZ>::NG;
  constexpr int MAXCW = VEC == 4 ? 6 : 12;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ float red[MAXCW * (EVAL ? Acc::NACC : K)];
  __shared__ int hist[EVAL ? Acc::NCELL : 1];
  __shared__ int cred[NG];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ncons = (int)blockDim.x - 32, ncw = ncons >> 5;
  const int b = blockIdx.y;
  const int y_begin = blockIdx.x * band, y_end = min(H, y_begin + band);
  const long N = (long)H * W, Nf = (long)Hf * Wf;

  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);
  StageRing ring;
  ring.init(bars, ns, ncw);
  uint64_t* lo_bar = bars + 2 * ns;
  if (tid == 0) { mbar_init(smem_u32(lo_bar), 1); mbar_fence_init(); }
  float* lo_s = reinterpret_cast<float*>(smem_raw + 128);             // [K][lok]
  unsigned char* stage0 = reinterpret_cast<unsigned char*>(lo_s + (size_t)K * lok);
  if constexpr (EVAL) {
    for (int i = tid; i < Acc::NCELL; i += blockDim.x) hist[i] = 0;
    if (tid < NG) cred[tid] = 0;
  }
  Groups<K, GSZ> gr;
  gr.load(GROUPED ? table : nullptr);
  const int n_pp = GROUPED ? gr.n : 0;
  // the index-map row starts 4-byte aligned only (W % 16 != 0): it is fetched as the enclosing 16-byte-aligned span
  const uint32_t rowb = (uint32_t)W * 4u, idxb = ((uint32_t)W + 30u) & ~15u;
  const int ia0 = CONS ? (int)(reinterpret_cast<uintptr_t>(ea.prev_idx) & 15u) : 0;
  // stage layout: [n_pp parent-probability rows][K target rows][n_pp parent-target rows][index row]
  const uint32_t stage_bytes = (uint32_t)(n_pp + (EVAL ? K : 0) + (CONS ? n_pp : 0)) * rowb + (CONS ? idxb : 0u);
  const bool streams = stage_bytes != 0u;
  const int r0 = make_lerp(y_begin, sy, Hf).i0;
  const int r1 = make_lerp(y_end - 1, sy, Hf).i1;
  __syncthreads();

  if (warp == ncw) {
    // ------------------------------ producer ------------------------------
    if (lane == 0) {
      pdl_wait();
      {
        const uint32_t bar = smem_u32(lo_bar);
        uint32_t total = 0;
        const int n_el = (r1 - r0 + 1) * Wf;
#pragma unroll
        for (int k = 0; k < K; ++k) {
          const long e0 = ((long)b * K + k) * Nf + (long)r0 * Wf;
          const int sh = row_shift(e0, a0);
          const uint32_t bytes = (uint32_t)(((sh + n_el + 3) >> 2) << 4);
          bulk_g2s_plain(smem_u32(lo_s + (size_t)k * lok), z_lo + (e0 - sh), bytes, bar);
          total += bytes;
        }
        mbar_arrive_expect_tx(bar, total);
      }
      if (streams) {
        int slot = 0;
        uint32_t phase = 1;
        for (int y = y_begin; y < y_end; ++y) {
          mbar_wait(ring.empty(slot), phase);
          uint32_t dst = smem_u32(stage0 + (size_t)slot * stage_bytes);
          const uint32_t bar = ring.full(slot);
          const long px = (long)y * W;
          uint32_t tx_bytes = stage_bytes;
          if constexpr (GROUPED) {
#pragma unroll
            for (int g = 0; g < NG; ++g)
              if (g < gr.n) { bulk_g2s_plain(dst, prev_probs + ((size_t)b * K_prev + gr.parent[g]) * N + px, rowb, bar); dst += rowb; }
          }
          if constexpr (EVAL) {
#pragma unroll
            for (int k = 0; k < K; ++k) {
              bulk_g2s_plain(dst, ea.targets + (size_t)b * ea.t_bstride + (size_t)k * ea.t_cstride + px, rowb, bar);
              dst += rowb;
            }
          }
          if constexpr (CONS) {
#pragma unroll
            for (int g = 0; g < NG; ++g)
              if (g < gr.n) {
                bulk_g2s_plain(dst, ea.parent_targets + (size_t)b * ea.pt_bstride + (size_t)gr.parent[g] * ea.pt_cstride + px, rowb, bar);
                dst += rowb;
              }
            const long e = (long)b * N + px;
            const uint32_t sh = (uint32_t)((e + ia0) & 15), bytes = (sh + (uint32_t)W + 15u) & ~15u;
            bulk_g2s_plain(dst, ea.prev_idx + (e - sh), bytes, bar);
            tx_bytes = tx_bytes - idxb + bytes;
          }
          mbar_arrive_expect_tx(bar, tx_bytes);
          if (++slot == ns) { slot = 0; phase ^= 1u; }
        }
      }
    }
    return;
  }

  // -------------------------------- consumers --------------------------------
  auto csync = [ncons] { consumer_sync(ncons); };
  const int x0 = tid * VEC;
  const bool ok = x0 < W;  // W % VEC == 0 (launcher)
  // x interpolation of the thread's VEC pixels as weights over the low-res columns c0, c0+1, c0+2
  float wx[VEC][3];
  int cofs[3];
  {
    const int xs = ok ? x0 : 0;
    const int c0 = make_lerp(xs, sx, Wf).i0;
#pragma unroll
    for (int c = 0; c < 3; ++c) cofs[c] = min(c0 + c, Wf - 1);
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      const Lerp lx = make_lerp(min(xs + v, W - 1), sx, Wf);
#pragma unroll
      for (int c = 0; c < 3; ++c) wx[v][c] = (lx.i0 - c0 == c ? lx.l0 : 0.f) + (lx.i1 - c0 == c ? lx.l1 : 0.f);
    }
  }
  int kbase[K];  // float offset of channel k's first row inside lo_s (shift of the aligned span included)
#pragma unroll
  for (int k = 0; k < K; ++k) kbase[k] = k * lok + row_shift(((long)b * K + k) * Nf + (long)r0 * Wf, a0);
  Acc ev;
  if constexpr (EVAL) ev.init();
  float ps[K];
#pragma unroll
  for (int k = 0; k < K; ++k) ps[k] = 0.f;
  pdl_wait();
  mbar_wait(smem_u32(lo_bar), 0);

  int slot = 0;
  uint32_t phase = 0;
  for (int y = y_begin; y < y_end; ++y) {
    const Lerp ly = make_lerp(y, sy, Hf);
    const int ro0 = (ly.i0 - r0) * Wf, ro1 = (ly.i1 - r0) * Wf;
    float z[K][VEC];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      float col[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float top = lo_s[kbase[k] + ro0 + cofs[c]], bot = lo_s[kbase[k] + ro1 + cofs[c]];
        col[c] = ly.l0 * top + ly.l1 * bot;
      }
#pragma unroll
      for (int v = 0; v < VEC; ++v) z[k][v] = wx[v][0] * col[0] + wx[v][1] * col[1] + wx[v][2] * col[2];
    }
    const long px = (long)y * W + x0;
    const unsigned char* sb = stage0 + (size_t)slot * stage_bytes;
    float ppg[NG][VEC], t[K][VEC], ptg[NG][VEC];
    unsigned pidxv = 0u;
    if (streams) {
      mbar_wait(ring.full(slot), phase);
      const int xr = ok ? x0 : 0;  // lanes past the row end read (and ignore) the row start
      const float* sf = reinterpret_cast<const float*>(sb) + xr;
      int row = 0;
      if constexpr (GROUPED) {
#pragma unroll
        for (int g = 0; g < NG; ++g) {
          if (g < gr.n) {
            const Vec<VEC> pv = *reinterpret_cast<const Vec<VEC>*>(sf + (size_t)(row++) * W);
#pragma unroll
            for (int v = 0; v < VEC; ++v) ppg[g][v] = pv.v[v];
          } else {
#pragma unroll
            for (int v = 0; v < VEC; ++v) ppg[g][v] = 0.f;
          }
        }
      }
      if constexpr (EVAL) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
          const Vec<VEC> tv = *reinterpret_cast<const Vec<VEC>*>(sf + (size_t)(row++) * W);
#pragma unroll
          for (int v = 0; v < VEC; ++v) t[k][v] = tv.v[v];
        }
      }
      if constexpr (CONS) {
#pragma unroll
        for (int g = 0; g < NG; ++g) {
          if (g < gr.n) {
            const Vec<VEC> pv = *reinterpret_cast<const Vec<VEC>*>(sf + (size_t)(row++) * W);
#pragma unroll
            for (int v = 0; v < VEC; ++v) ptg[g][v] = pv.v[v];
          } else {
#pragma unroll
            for (int v = 0; v < VEC; ++v) ptg[g][v] = -1.f;
          }
        }
        const unsigned char* ib = sb + (size_t)row * rowb + (((long)b * N + (long)y * W + ia0) & 15) + xr;
        if constexpr (VEC == 4) pidxv = *reinterpret_cast<const unsigned*>(ib);
        else if constexpr (VEC == 2) pidxv = *reinterpret_cast<const unsigned short*>(ib);
        else pidxv = *ib;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(ring.empty(slot));  // the row is in registers
      if (++slot == ns) { slot = 0; phase ^= 1u; }
    }
    unsigned my_idx = 0u;
    float prob[K][VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      float zz[K], p[K], mx = 0.f, sum = 1.f;
#pragma unroll
      for (int k = 0; k < K; ++k) zz[k] = z[k][v];
      constexpr bool SHARE = GROUPED && GSZ == K;  // one group spanning the level: the restrictive softmax is THE softmax
      if constexpr (EVAL || SHARE) softmax_all<K>(zz, p, mx, sum);
      if constexpr (MODE == RHSEG_ACT_SIGMOID) {
#pragma unroll
        for (int k = 0; k < K; ++k) prob[k][v] = sigmoidf_ref(zz[k]);
      } else {
        float q[K];
        if constexpr (SHARE) {
#pragma unroll
          for (int k = 0; k < K; ++k) q[k] = p[k];
        } else {
          softmax_groups<K, GSZ>(zz, gr, q);
        }
        // softmax(z_g + log(P_p + eps)) == softmax(z_g): the gate is constant inside a group (SURVEY F3)
        float pg[NG];
#pragma unroll
        for (int g = 0; g < NG; ++g) pg[g] = ppg[g][v];
#pragma unroll
        for (int k = 0; k < K; ++k) prob[k][v] = group_value<K, GSZ>(pg, gr, k) * q[k];
      }
      if constexpr (COMPOSED) {
        float tt[K], P[K], pp[NG];
#pragma unroll
        for (int k = 0; k < K; ++k) { tt[k] = t[k][v]; P[k] = prob[k][v]; }
#pragma unroll
        for (int g = 0; g < NG; ++g) pp[g] = GROUPED ? ppg[g][v] : 0.f;
        ev.pixel(zz, p, mx + log_fast(sum), tt, P, pp, ok, gr);  // lanes past the row end hold the row start: finite
      } else if constexpr (EVAL) {
        float tt[K], pt[NG];
#pragma unroll
        for (int k = 0; k < K; ++k) tt[k] = t[k][v];
#pragma unroll
        for (int g = 0; g < NG; ++g) pt[g] = ptg[g][v];
        const int idx = ev.pixel(zz, p, mx + log_fast(sum), tt, pt, (int)((pidxv >> (8 * v)) & 0xffu), ok, gr);
        my_idx |= (unsigned)idx << (8 * v);
      }
    }
    if (ok) {
#pragma unroll
      for (int k = 0; k < K; ++k) {
        Vec<VEC> zo, po;
#pragma unroll
        for (int v = 0; v < VEC; ++v) { zo.v[v] = z[k][v]; po.v[v] = prob[k][v]; ps[k] += prob[k][v]; }
        *reinterpret_cast<Vec<VEC>*>(logits + ((size_t)b * K + k) * N + px) = zo;
        *reinterpret_cast<Vec<VEC>*>(probs + ((size_t)b * K + k) * N + px) = po;
      }
      if constexpr (EVAL && !COMPOSED) {
        if (ea.idx_out) {
          unsigned char* dst = ea.idx_out + (size_t)b * N + px;
          if constexpr (VEC == 4) *reinterpret_cast<unsigned*>(dst) = my_idx;
          else if constexpr (VEC == 2) *reinterpret_cast<unsigned short*>(dst) = (unsigned short)my_idx;
          else *dst = (unsigned char)my_idx;
        }
      }
    }
  }
  // FiLM pool sums: one fp64 atomic per (CTA, channel)
  {
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const float v = warp_sum(ps[k]);
      if (lane == 0) red[warp * K + k] = v;
    }
    csync();
    if (tid < K) {
      double acc = 0.0;
      for (int w = 0; w < ncw; ++w) acc += (double)red[w * K + tid];
      atomicAdd(&psum[(size_t)b * K + tid], acc);
    }
    csync();
  }
  if constexpr (EVAL) {
    // block reduction of the evaluation (runtime warp count: sum the per-warp partials here)
    const int NACC = Acc::NACC;
#pragma unroll
    for (int k = 0; k < K; ++k)
#pragma unroll
      for (int j = 0; j < RHSEG_NSTAT; ++j) {
        const float v = warp_sum(ev.a[k][j]);
        if (lane == 0) red[warp * NACC + k * RHSEG_NSTAT + j] = v;
      }
    if constexpr (CONS) {
#pragma unroll
      for (int g = 0; g < NG; ++g) {
        const int v = __reduce_add_sync(0xffffffffu, ev.cm[g]);
        if (lane == 0 && v) atomicAdd(&cred[g], v);
      }
    }
    if constexpr (COMPOSED) {
#pragma unroll
      for (int g = 0; g < Acc::NCS; ++g) {
        const float v = warp_sum(ev.cs[g]);
        if (lane == 0) red[warp * NACC + K * RHSEG_NSTAT + g] = v;
      }
    }
    ev.cc.flush(hist);
    csync();
    for (int i = tid; i < NACC; i += ncons) {  // narrow images run a single consumer warp
      double acc = 0.0;
      for (int w = 0; w < ncw; ++w) acc += (double)red[w * NACC + i];
      if constexpr (COMPOSED) {
        if (i < K * RHSEG_NSTAT) atomicAdd(&ea.stats[(size_t)b * K * RHSEG_NSTAT + i], acc);
        else if (acc != 0.0) atomicAdd(&ea.cons[i - K * RHSEG_NSTAT], acc);
      } else {
        atomicAdd(&ea.stats[(size_t)b * K * RHSEG_NSTAT + i], acc);
      }
    }
    if constexpr (CONS) {
      if (tid < NG && cred[tid]) atomicAdd(&ea.cons[tid], (double)cred[tid]);
    }
    for (int i = tid; i < Acc::NCELL; i += ncons)
      if (hist[i]) atomicAdd(&ea.conf[i], (unsigned long long)hist[i]);
  }
}

// host: launch the band kernel when the shape allows it; returns false when the generic kernel must be used
template <int K, int VEC, int MODE, int EVALK, int GSZ>
static int launch_band(const float* z_lo, const float* prev_probs, const int32_t* table, int B, int Hf, int Wf, int H, int W,
                       int K_prev, float sy, float sx, float* logits, float* probs, double* psum, cudaStream_t st,
                       const EvalArgs& ea, bool* launched) {
  *launched = false;
  auto kern = upsample_band_kernel<K, VEC, MODE, EVALK, GSZ>;
  constexpr bool EVAL = EVALK != 0, GROUPED = MODE == RHSEG_ACT_GROUPED;
  const int ncons = ((W / VEC + 31) / 32) * 32;
  if (ncons > (VEC == 4 ? 192 : 384)) return RHSEG_OK;
  // worst-case stage: the kernel reads the actual number of groups from the level table
  const int n_pp = GROUPED ? Groups<K, GSZ>::NG : 0;
  const size_t stage = (size_t)(n_pp + (EVAL ? K : 0) + (EVALK == 2 ? n_pp : 0)) * W * 4 + (EVALK == 2 ? ((W + 30) & ~15) : 0);
  static int tune_ns = -1;
  if (tune_ns < 0) { const char* e = getenv("RHSEG_TUNE_UP_NS"); tune_ns = e ? atoi(e) : 0; }
  const int ns = stage == 0 ? 1 : (tune_ns > 0 ? std::min(tune_ns, 7) : 3);
  auto smem_for = [&](int band) {
    const int nlo = (int)floorf(sy * (float)(band - 1)) + 3;
    const int lok = ((nlo * Wf + 8) + 3) & ~3;
    return 128 + (size_t)K * lok * 4 + (size_t)ns * stage;
  };
  // one resident wave: the occupancy at a nominal band decides the number of CTA slots, the slots the band
  int per_sm = 0;
  const size_t smem0 = smem_for(8);
  if (smem0 > 200 * 1024) return RHSEG_OK;
  RHSEG_CUDA(cached_launch_prep(reinterpret_cast<const void*>(kern), ncons + 32, smem0, std::min<size_t>(smem_for(H), 200 * 1024), &per_sm));
  if (per_sm < 1) return RHSEG_OK;
  static int tune_ctas = -1;
  if (tune_ctas < 0) { const char* e = getenv("RHSEG_TUNE_UP_CTAS"); tune_ctas = e ? atoi(e) : 0; }
  if (tune_ctas > 0) per_sm = std::min(per_sm, tune_ctas);
  const long slots = std::max<long>(1, (long)per_sm * device_sm_count() / B);
  int band = std::max(4, (int)((H + slots - 1) / slots));
  while (band > 4 && smem_for(band) > 200 * 1024) --band;
  if (smem_for(band) > 200 * 1024) return RHSEG_OK;
  const int nlo = (int)floorf(sy * (float)(band - 1)) + 3;
  const int lok = ((nlo * Wf + 8) + 3) & ~3;
  const int a0 = (int)((reinterpret_cast<uintptr_t>(z_lo) >> 2) & 3);
  dim3 grid((unsigned)((H + band - 1) / band), B);
  launch_pdl(kern, dim3(grid), dim3(ncons + 32), smem_for(band), st, z_lo, prev_probs, table, Hf, Wf, H, W, K_prev, sy, sx, band, lok,
             ns, a0, logits, probs, psum, ea);
  RHSEG_LAUNCH_CHECK();
  *launched = true;
  return RHSEG_OK;
}

template <int K, int MODE>
static int fwd_upsampled(const float* z_lo, const float* prev_probs, const int32_t* table, int B, int Hf, int Wf,
                         int H, int W, int K_prev, int hint, float* logits, float* probs, double* psum,
                         cudaStream_t st, const EvalArgs* ea, bool* need_eval) {
  const float sy = H > 1 ? (float)(Hf - 1) / (float)(H - 1) : 0.f;
  const float sx = W > 1 ? (float)(Wf - 1) / (float)(W - 1) : 0.f;
  constexpr int THREADS = 256;
  *need_eval = false;
  auto al4 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 3u) == 0; };
  auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
  static int tune_vec = -1;
  if (tune_vec < 0) { const char* e = getenv("RHSEG_TUNE_UP_VEC"); tune_vec = e ? atoi(e) : 0; }
  bool band_ok = MODE != RHSEG_ACT_ZEROS && W % 4 == 0 && sy > 0.f && sy <= 1.0f && sx > 0.f && al16(logits) && al16(probs) &&
                 (MODE != RHSEG_ACT_GROUPED || al16(prev_probs)) && !getenv("RHSEG_NO_BAND_FWD");
  if (ea) band_ok = band_ok && al16(ea->targets) && ea->t_bstride % 4 == 0 && ea->t_cstride % 4 == 0 && al4(ea->idx_out) &&
                    (!ea->parent_targets || (al16(ea->parent_targets) && ea->pt_bstride % 4 == 0 && ea->pt_cstride % 4 == 0)) &&
                    (!ea->prev_idx || al4(ea->prev_idx));
  if constexpr (MODE != RHSEG_ACT_ZEROS) {
    if (band_ok) {
      const EvalArgs none{};
      const EvalArgs& e = ea ? *ea : none;
      const int evalk = !ea ? 0 : ea->composed ? 3 : ((MODE == RHSEG_ACT_GROUPED && ea->prev_idx && ea->parent_targets) ? 2 : 1);
      // pixels per thread: 4 when three low-res columns cover them (sx <= 1/3), else 2
      const bool v4 = 3.0f * sx <= 0.999f && tune_vec != 2;
      const bool v2 = 1.0f * sx <= 0.999f;
      bool done = false;
      int rc = RHSEG_OK;
#define RHSEG_BAND(VEC, EK, GS) rc = launch_band<K, VEC, MODE, EK, GS>(z_lo, prev_probs, table, B, Hf, Wf, H, W, K_prev, sy, sx, logits, probs, psum, st, e, &done)
#define RHSEG_BAND_V(EK, GS)                                  \
      do {                                                    \
        if (v4) RHSEG_BAND(4, EK, GS);                        \
        if constexpr (K <= 4) { /* 2 px / thread needs > 256 threads for wide rows: too few registers for K > 4 (spills) */ \
          if (!done && rc == RHSEG_OK && v2) RHSEG_BAND(2, EK, GS); \
        }                                                     \
      } while (0)
      if constexpr (MODE == RHSEG_ACT_SIGMOID) {
        if (evalk == 0) RHSEG_BAND_V(0, K); else if (evalk == 3) RHSEG_BAND_V(3, K); else RHSEG_BAND_V(1, K);
      } else {
        const bool single = hint == K;
        bool uniform2 = false;
        if constexpr (K == 4) uniform2 = hint == 2;  // two parents with two children each (extended tree, level 2)
        if (single) {
          if (evalk == 0) RHSEG_BAND_V(0, K); else if (evalk == 1) RHSEG_BAND_V(1, K); else if (evalk == 3) RHSEG_BAND_V(3, K); else RHSEG_BAND_V(2, K);
        } else if (uniform2) {
          if constexpr (K == 4) { if (evalk == 0) RHSEG_BAND_V(0, 2); else if (evalk == 1) RHSEG_BAND_V(1, 2); else if (evalk == 3) RHSEG_BAND_V(3, 2); else RHSEG_BAND_V(2, 2); }
        } else {
          if (evalk == 0) RHSEG_BAND_V(0, 0);
          else if constexpr (K <= 6) { if (evalk == 1) RHSEG_BAND_V(1, 0); else if (evalk == 3) RHSEG_BAND_V(3, 0); else RHSEG_BAND_V(2, 0); }
          // K > 6 with a table-driven group layout and the fused evaluation would spill: generic kernel + rhseg_level_eval
        }
      }
#undef RHSEG_BAND_V
#undef RHSEG_BAND
      if (rc != RHSEG_OK) return rc;
      if (done) return RHSEG_OK;
    }
  }
  // generic kernel: any shape / alignment; the evaluation (if requested) runs as its own kernel afterwards
  *need_eval = ea != nullptr;
  if (W % 4 == 0 && al16(logits) && al16(probs) && (!prev_probs || al16(prev_probs))) {
    const int vps = H * (W / 4);
    dim3 grid((vps + THREADS - 1) / THREADS, B);
    launch_pdl(upsample_act_kernel<K, 4, MODE, THREADS>, dim3(grid), dim3(THREADS), 0, st, z_lo, prev_probs, table, Hf, Wf, H, W, K_prev,
                                                                       sy, sx, 0, logits, probs, psum, vps);
  } else {
    const int vps = H * W;
    dim3 grid((vps + THREADS - 1) / THREADS, B);
    launch_pdl(upsample_act_kernel<K, 1, MODE, THREADS>, dim3(grid), dim3(THREADS), 0, st, z_lo, prev_probs, table, Hf, Wf, H, W, K_prev,
                                                                       sy, sx, 0, logits, probs, psum, vps);
  }
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}


int fwd_upsampled_dispatch(int K, int act_arg, const float* z_lo, const float* prev_probs, const int32_t* table,
                           int B, int Hf, int Wf, int H, int W, int K_prev, float* logits, float* probs, double* psum,
                           cudaStream_t st, const EvalArgs* ea, bool* need_eval) {
  const int act_mode = act_arg & 0xff, hint = RHSEG_GROUP_HINT_OF(act_arg);
  RHSEG_DISPATCH_K(K, {
    if (act_mode == RHSEG_ACT_SIGMOID)
      return fwd_upsampled<KK, RHSEG_ACT_SIGMOID>(z_lo, prev_probs, table, B, Hf, Wf, H, W, K_prev, hint, logits, probs, psum, st, ea, need_eval);
    if (act_mode == RHSEG_ACT_GROUPED)
      return fwd_upsampled<KK, RHSEG_ACT_GROUPED>(z_lo, prev_probs, table, B, Hf, Wf, H, W, K_prev, hint, logits, probs, psum, st, ea, need_eval);
    return fwd_upsampled<KK, RHSEG_ACT_ZEROS>(z_lo, prev_probs, table, B, Hf, Wf, H, W, K_prev, hint, logits, probs, psum, st, ea, need_eval);
  });
  return RHSEG_OK;
}

}  // namespace rhseg
