// Metrics: integer confusion matrix (ProcessClasses + torchmetrics multiclass semantics,
// Metrics/performance_metrics.py:27-141) and the train-loop prediction glue
// (train.py:206-231, predictEval.py:409-422).
#include <algorithm>
#include <cstdlib>
#include <type_traits>
#include "common.cuh"
#include "eval_accum.cuh"
#include "hires.cuh"
#include "logits_io.cuh"

namespace rhseg {

// argmax(softmax(z)) with ATen's op order (train.py:219-221)
template <int K>
__device__ __forceinline__ int argmax_softmax(const float (&z)[K]) {
  return argmax_softmax_aten<K>(z);
}

// warp-aggregated histogram update: lanes holding the same cell elect one leader
__device__ __forceinline__ void hist_add(int* hist, int cell) {
  const unsigned peers = __match_any_sync(0xffffffffu, cell);
  if (cell >= 0 && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&hist[cell], __popc(peers));
}

// MODE 0: inputs are (probs, targets) exactly as the metric wrappers receive them.
// MODE 1: inputs are (logits, ternary targets); the train-loop glue is applied on the fly.
template <int K, int VEC, int ITER, int THREADS, int MODE>
__global__ void __launch_bounds__(THREADS)
confusion_kernel(const float* __restrict__ probs, long p_bstride, long p_cstride, const float* __restrict__ targets,
                 long t_bstride, long t_cstride, long N, int child, unsigned long long* __restrict__ conf) {
  pdl_wait();
  constexpr int NCMAX = K + 1;
  __shared__ int hist[NCMAX * NCMAX];
  const int nc = child ? K + 1 : K;
  const int b = blockIdx.y, tid = threadIdx.x;
  for (int i = tid; i < nc * nc; i += THREADS) hist[i] = 0;
  __syncthreads();
  const float* pb = probs + (size_t)b * p_bstride;
  const float* tb = targets + (size_t)b * t_bstride;
  WarpConfusion<K + 1> wc;
  wc.init(nc);
  const long chunk0 = (long)blockIdx.x * (THREADS * VEC * ITER);
#pragma unroll
  for (int it = 0; it < ITER; ++it) {
    const long px = chunk0 + (long)it * THREADS * VEC + (long)tid * VEC;
    const bool ok = px < N;
    float p[K][VEC], t[K][VEC];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      Vec<VEC> pv, tv;
#pragma unroll
      for (int v = 0; v < VEC; ++v) { pv.v[v] = 0.f; tv.v[v] = 0.f; }
      if (ok) {
        pv = ld_stream<VEC>(pb + (size_t)k * p_cstride + px);
        tv = ld_stream<VEC>(tb + (size_t)k * t_cstride + px);
      }
#pragma unroll
      for (int v = 0; v < VEC; ++v) { p[k][v] = pv.v[v]; t[k][v] = tv.v[v]; }
    }
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      float pr[K], tg[K];
#pragma unroll
      for (int k = 0; k < K; ++k) { pr[k] = p[k][v]; tg[k] = t[k][v]; }
      if constexpr (MODE == 1) {
        const int idx = argmax_softmax<K>(pr);
#pragma unroll
        for (int k = 0; k < K; ++k) {
          const bool ign = tg[k] == -1.0f;
          pr[k] = (k == idx && !ign) ? 1.0f : 0.0f;  // one-hot, zeroed where the target is -1
          tg[k] = ign ? 0.0f : tg[k];                // eval target
        }
      }
      const int pc = process_class<K>(pr, child != 0);
      int tc = process_class<K>(tg, child != 0);
      if (!ok || (child && tc == 0)) tc = -1;  // torchmetrics ignore_index=0 on child levels
      wc.add(tc, pc);
    }
  }
  wc.flush(hist, nc);
  __syncthreads();
  for (int i = tid; i < nc * nc; i += THREADS)
    if (hist[i]) atomicAdd(&conf[i], (unsigned long long)hist[i]);
}

template <int K, int VEC, int THREADS>
__global__ void __launch_bounds__(THREADS)
predict_kernel(const float* __restrict__ logits, const float* __restrict__ targets, long t_bstride, long t_cstride,
               long N, float* __restrict__ onehot, float* __restrict__ eval_t, int32_t* __restrict__ pred_idx) {
  pdl_wait();
  const int b = blockIdx.y;
  const long px = ((long)blockIdx.x * THREADS + threadIdx.x) * VEC;
  if (px >= N) return;
  float z[K][VEC], t[K][VEC];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const Vec<VEC> zv = ld_stream<VEC>(logits + ((size_t)b * K + k) * N + px);
    const Vec<VEC> tv = ld_stream<VEC>(targets + (size_t)b * t_bstride + (size_t)k * t_cstride + px);
#pragma unroll
    for (int v = 0; v < VEC; ++v) { z[k][v] = zv.v[v]; t[k][v] = tv.v[v]; }
  }
  int idx[VEC];
#pragma unroll
  for (int v = 0; v < VEC; ++v) {
    float zz[K];
#pragma unroll
    for (int k = 0; k < K; ++k) zz[k] = z[k][v];
    idx[v] = argmax_softmax<K>(zz);
    if (pred_idx) pred_idx[(size_t)b * N + px + v] = idx[v];
  }
#pragma unroll
  for (int k = 0; k < K; ++k) {
    Vec<VEC> oh, et;
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      const bool ign = t[k][v] == -1.0f;
      oh.v[v] = (idx[v] == k && !ign) ? 1.0f : 0.0f;
      et.v[v] = ign ? 0.0f : t[k][v];
    }
    if (onehot) *reinterpret_cast<Vec<VEC>*>(onehot + ((size_t)b * K + k) * N + px) = oh;
    if (eval_t) *reinterpret_cast<Vec<VEC>*>(eval_t + ((size_t)b * K + k) * N + px) = et;
  }
}

// The five per-class ratios from the confusion matrix, with torchmetrics' arithmetic order
// (int64 -> fp32, then the ratio; zero denominator -> 0):
//   row 0 F1 = 2tp / (2tp + fn + fp)     row 1 Jaccard = tp / (colsum + rowsum - tp)
//   row 2 Accuracy(average=None) = tp / (tp + fn)   row 3 Precision = tp / (tp + fp)   row 4 Recall
__global__ void metric_ratios_kernel(const long long* __restrict__ conf, int nc, float* __restrict__ out) {
  pdl_wait();
  const int c = threadIdx.x;
  if (c >= nc) return;
  long long tp = conf[c * nc + c], row = 0, col = 0;
  for (int j = 0; j < nc; ++j) { row += conf[c * nc + j]; col += conf[j * nc + c]; }
  const long long fp = col - tp, fn = row - tp;
  auto safe = [](float num, float den) { return num / (den == 0.f ? 1.f : den); };
  const float tpf = (float)tp, fpf = (float)fp, fnf = (float)fn;
  out[0 * nc + c] = safe(2.0f * tpf, (2.0f * tpf + 1.0f * fnf) + fpf);
  out[1 * nc + c] = safe(tpf, (float)(col + row - tp));
  out[2 * nc + c] = safe(tpf, (float)(tp + fn));
  out[3 * nc + c] = safe(tpf, (float)(tp + fp));
  out[4 * nc + c] = safe(tpf, (float)(tp + fn));
}

// ------------------------------------------------------------------------------------
// Fused per-level training evaluation: ONE pass over (logits, ternary targets) of a level yields
//   * the CE/Dice statistics of rhseg_loss_stats                       (Metrics/losses.py:16-134)
//   * the train-path prediction argmax(softmax(z)) (train.py:219-221), kept only as a uint8 index map
//   * the confusion matrix of the masked one-hot prediction vs the eval target
//     (train.py:226-232 + performance_metrics.py:27-141)
//   * the consistency sums of the masked one-hot predictions against the previous level's
//     (losses.py:150-177 as train_epoch calls it, train.py:237-239)
// so neither the one-hot tensors nor the eval targets are ever materialised.
// out layout (8-byte words): [B*K*5 fp64 stats][RHSEG_MAX_K fp64 consistency sums][nc*nc int64 confusion]
// LT: logit element type (float, or uint16_t = bf16 bits of a flat head under autocast, widened at the load)
// ------------------------------------------------------------------------------------
template <int K, int VEC, int MINB, int THREADS, int CT = -1, typename LT = float>
__global__ void __launch_bounds__(THREADS, MINB)
level_eval_kernel(const LT* __restrict__ logits, const float* __restrict__ targets, long t_bstride, long t_cstride,
                  const float* __restrict__ parent_targets, long pt_bstride, long pt_cstride,
                  const unsigned char* __restrict__ prev_idx, const int32_t* __restrict__ table, long N, int child,
                  double* __restrict__ stats, double* __restrict__ cons, unsigned long long* __restrict__ conf,
                  unsigned char* __restrict__ idx_out) {
  pdl_wait();
  __shared__ float red[THREADS / 32][EvalAccum<K>::NACC];
  __shared__ int hist[(K + 1) * (K + 1)];
  const int b = blockIdx.y, tid = threadIdx.x;
  EvalAccum<K, CT> ev;
  ev.init(child, child && prev_idx != nullptr && parent_targets != nullptr, table, hist, THREADS);
  const LT* zb = logits + (size_t)b * K * N;
  // persistent over the sample's pixel vectors: one resident wave, statistics reduced once per CTA
  for (long px0 = (long)blockIdx.x * (THREADS * VEC); px0 < N; px0 += (long)gridDim.x * (THREADS * VEC)) {
    const long px = px0 + (long)tid * VEC;
    const bool ok = px < N;
    float z[K][VEC], t[K][VEC], ptv[K][VEC];
    unsigned char pidx[VEC], my_idx[VEC];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      Vec<VEC> zv;
#pragma unroll
      for (int v = 0; v < VEC; ++v) zv.v[v] = 0.f;
      if (ok) zv = ld_cached<VEC>(zb + (size_t)k * N + px);
#pragma unroll
      for (int v = 0; v < VEC; ++v) z[k][v] = zv.v[v];
    }
    ev.template load_targets<VEC>(targets, t_bstride, t_cstride, parent_targets, pt_bstride, pt_cstride, prev_idx, b, N, px,
                                  ok, t, ptv, pidx);
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      float zz[K], tt[K], pt[K];
#pragma unroll
      for (int k = 0; k < K; ++k) { zz[k] = z[k][v]; tt[k] = t[k][v]; pt[k] = ptv[k][v]; }
      my_idx[v] = (unsigned char)ev.pixel(zz, tt, pt, pidx[v], ok);
    }
    ev.template store_idx<VEC>(idx_out, b, N, px, ok, my_idx);
  }
  ev.template finish<THREADS / 32>(&red[0][0], hist, stats, cons, conf, table, b);
}

// ------------------------------------------------------------------------------------
// The same evaluation as a bulk-copy pipeline (the fast path: 16-byte aligned planes, N % 16 == 0).
// The flattened (sample, pixel) range is split EVENLY over one resident wave of CTAs in units of 16 pixels.  A
// producer warp streams stages of up to EVP_PX consecutive pixels of one sample -- K logit planes, K target
// planes and, for the consistency term, the parent's target plane per group and the previous level's index map --
// into a shared-memory ring with 1-D bulk async copies; eight consumer warps read only shared memory, so no
// global-load latency is exposed and the per-pixel code (hires.cuh: EvalAcc) is all that is left.
// ------------------------------------------------------------------------------------
constexpr int EVP_CW = 8, EVP_CONSUMERS = EVP_CW * 32, EVP_THREADS = EVP_CONSUMERS + 32, EVP_PX = EVP_CONSUMERS * 4;

// stage layout: K logit planes (EVP_PX elements of LT each), then K target planes, the NG parent target planes and the
// index map (fp32 / uint8)
template <int K, int CT, int GSZ, typename LT = float>
__host__ __device__ constexpr int evp_stage_bytes() {
  return K * EVP_PX * (int)sizeof(LT) + (K + (CT == 2 ? Groups<K, GSZ>::NG : 0)) * EVP_PX * 4 + (CT == 2 ? EVP_PX : 0);
}

template <int K, int CT, int GSZ, typename LT = float>
__global__ void __launch_bounds__(EVP_THREADS)
level_eval_pipe_kernel(const LT* __restrict__ logits, const float* __restrict__ targets, long t_bstride, long t_cstride,
                       const float* __restrict__ parent_targets, long pt_bstride, long pt_cstride,
                       const unsigned char* __restrict__ prev_idx, const int32_t* __restrict__ table, long N,
                       long units_total, int ns, double* __restrict__ stats, double* __restrict__ cons,
                       unsigned long long* __restrict__ conf, unsigned char* __restrict__ idx_out) {
  using Acc = EvalAcc<K, CT, GSZ>;
  constexpr bool CONS = CT == 2;
  constexpr int NG = Groups<K, GSZ>::NG;
  constexpr int STAGE = evp_stage_bytes<K, CT, GSZ, LT>();
  constexpr int ZF = K * EVP_PX * (int)sizeof(LT) / 4;  // 4-byte words of a stage's logit planes
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ float red[EVP_CW * Acc::NACC];
  __shared__ int hist[Acc::NCELL];
  __shared__ int cred[NG];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  StageRing ring;
  ring.init(reinterpret_cast<uint64_t*>(smem_raw), ns, EVP_CW);
  unsigned char* stage0 = smem_raw + 128;
  for (int i = tid; i < Acc::NCELL; i += EVP_THREADS) hist[i] = 0;
  if (tid < NG) cred[tid] = 0;
  Groups<K, GSZ> gr;
  gr.load(CT >= 1 ? table : nullptr);  // the level table is uploaded once per device: not produced by the previous kernel
  const long g0 = (units_total * blockIdx.x / gridDim.x) * 16, g1 = (units_total * (blockIdx.x + 1) / gridDim.x) * 16;
  int b = (int)(g0 / N);
  long off = g0 - (long)b * N;
  __syncthreads();
  pdl_wait();

  if (warp == EVP_CW) {
    // ------------------------------ producer ------------------------------
    if (lane == 0) {
      int slot = 0;
      uint32_t phase = 1;
      for (long cur = g0; cur < g1;) {
        const int len = (int)min((long)EVP_PX, min(N - off, g1 - cur));
        mbar_wait(ring.empty(slot), phase);
        const uint32_t dst = smem_u32(stage0 + (size_t)slot * STAGE), bar = ring.full(slot);
        const uint32_t bytes = (uint32_t)len * 4u, zbytes = (uint32_t)len * (uint32_t)sizeof(LT);
        uint32_t total = 0;
#pragma unroll
        for (int k = 0; k < K; ++k) {
          bulk_g2s_plain(dst + k * EVP_PX * (int)sizeof(LT), logits + ((size_t)b * K + k) * N + off, zbytes, bar);
          bulk_g2s_plain(dst + (ZF + k * EVP_PX) * 4, targets + (size_t)b * t_bstride + (size_t)k * t_cstride + off, bytes, bar);
          total += zbytes + bytes;
        }
        if constexpr (CONS) {
#pragma unroll
          for (int g = 0; g < NG; ++g)
            if (g < gr.n) {
              bulk_g2s_plain(dst + (ZF + (K + g) * EVP_PX) * 4,
                             parent_targets + (size_t)b * pt_bstride + (size_t)gr.parent[g] * pt_cstride + off, bytes, bar);
              total += bytes;
            }
          bulk_g2s_plain(dst + (ZF + (K + NG) * EVP_PX) * 4, prev_idx + (size_t)b * N + off, (uint32_t)len, bar);
          total += (uint32_t)len;
        }
        mbar_arrive_expect_tx(bar, total);
        if (++slot == ns) { slot = 0; phase ^= 1u; }
        cur += len;
        off += len;
        if (off == N) { off = 0; ++b; }
      }
    }
    return;
  }

  // -------------------------------- consumers --------------------------------
  auto csync = [] { consumer_sync(EVP_CONSUMERS); };
  Acc ev;
  ev.init();
  int cur_b = b, slot = 0;
  uint32_t phase = 0;
  for (long cur = g0; cur < g1;) {
    const int len = (int)min((long)EVP_PX, min(N - off, g1 - cur));
    if (b != cur_b) {  // the range crosses into the next sample: hand over the finished sample's sums
      ev.template finish<EVP_CW>(red, cred, hist, stats + (size_t)cur_b * K * RHSEG_NSTAT, cons, conf, tid, EVP_CONSUMERS, csync);
      cur_b = b;
    }
    mbar_wait(ring.full(slot), phase);
    const float* sf = reinterpret_cast<const float*>(stage0 + (size_t)slot * STAGE);
    // full stages (all but the last of a sample or of the CTA's range) run code without any range predicate
    auto body = [&](auto full_tag) {
      constexpr bool FULL = decltype(full_tag)::value;
      const bool ok = FULL ? true : tid * 4 < len;
      float z[K][4], t[K][4], ptg[NG][4];
      unsigned pidx4 = 0u;
#pragma unroll
      for (int k = 0; k < K; ++k) {
        if constexpr (std::is_same_v<LT, float>) {
          const float4 zv = *reinterpret_cast<const float4*>(sf + k * EVP_PX + tid * 4);
          z[k][0] = zv.x; z[k][1] = zv.y; z[k][2] = zv.z; z[k][3] = zv.w;
        } else {  // bf16: four logits in 8 bytes, widened exactly
          const uint2 zv = *reinterpret_cast<const uint2*>(reinterpret_cast<const uint16_t*>(sf) + k * EVP_PX + tid * 4);
          z[k][0] = bf16_lo(zv.x); z[k][1] = bf16_hi(zv.x); z[k][2] = bf16_lo(zv.y); z[k][3] = bf16_hi(zv.y);
        }
        const float4 tv = *reinterpret_cast<const float4*>(sf + ZF + k * EVP_PX + tid * 4);
        t[k][0] = tv.x; t[k][1] = tv.y; t[k][2] = tv.z; t[k][3] = tv.w;
      }
#pragma unroll
      for (int g = 0; g < NG; ++g) {
        if (CONS && g < gr.n) {
          const float4 pv = *reinterpret_cast<const float4*>(sf + ZF + (K + g) * EVP_PX + tid * 4);
          ptg[g][0] = pv.x; ptg[g][1] = pv.y; ptg[g][2] = pv.z; ptg[g][3] = pv.w;
        } else {
          ptg[g][0] = ptg[g][1] = ptg[g][2] = ptg[g][3] = -1.0f;
        }
      }
      if constexpr (CONS) pidx4 = *reinterpret_cast<const unsigned*>(reinterpret_cast<const unsigned char*>(sf + ZF + (K + NG) * EVP_PX) + tid * 4);
      __syncwarp();
      if (lane == 0) mbar_arrive(ring.empty(slot));  // the stage is in registers: the producer may refill the slot
      unsigned my_idx = 0u;
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        float zz[K], tt[K], pg[NG], p[K], mx, sum;
#pragma unroll
        for (int k = 0; k < K; ++k) { zz[k] = ok ? z[k][v] : 0.f; tt[k] = t[k][v]; }  // stale shared memory may hold NaNs
#pragma unroll
        for (int g = 0; g < NG; ++g) pg[g] = ptg[g][v];
        softmax_all<K>(zz, p, mx, sum);
        const int idx = ev.pixel(zz, p, mx + log_fast(sum), tt, pg, (int)((pidx4 >> (8 * v)) & 0xffu), ok, gr);
        my_idx |= (unsigned)idx << (8 * v);
      }
      if (ok && idx_out) *reinterpret_cast<unsigned*>(idx_out + (size_t)b * N + off + tid * 4) = my_idx;
    };
    if (len == EVP_PX) body(std::true_type{});
    else body(std::false_type{});
    if (++slot == ns) { slot = 0; phase ^= 1u; }
    cur += len;
    off += len;
    if (off == N) { off = 0; ++b; }
  }
  if (g0 < g1) ev.template finish<EVP_CW>(red, cred, hist, stats + (size_t)cur_b * K * RHSEG_NSTAT, cons, conf, tid, EVP_CONSUMERS, csync);
}

template <int K, int CT, int GSZ, typename LT = float>
static int launch_eval_pipe(const LT* logits, const float* targets, long t_bs, long t_cs, const float* parent_targets,
                            long pt_bs, long pt_cs, const unsigned char* prev_idx, const int32_t* table, int B, long N,
                            double* stats, double* cons, unsigned long long* conf, unsigned char* idx_out, cudaStream_t st) {
  auto kern = level_eval_pipe_kernel<K, CT, GSZ, LT>;
  constexpr int STAGE = evp_stage_bytes<K, CT, GSZ, LT>();
  static int tune = -1;
  if (tune < 0) { const char* e = getenv("RHSEG_TUNE_EVAL"); tune = e ? atoi(e) : 0; }
  const int ns = tune == 1 ? 3 : (tune == 2 ? 4 : 2);
  const size_t smem = 128 + (size_t)ns * STAGE;
  int per_sm = 0;
  RHSEG_CUDA(cached_launch_prep(reinterpret_cast<const void*>(kern), EVP_THREADS, smem, smem, &per_sm));
  if (per_sm < 1) return RHSEG_ERR_UNSUPPORTED;
  const long units = (long)B * N / 16;
  // every CTA gets at least two full stages of work; one resident wave at most
  const long grid = std::max<long>(1, std::min<long>((long)device_sm_count() * per_sm, units / (2 * EVP_PX / 16)));
  launch_pdl(kern, dim3((unsigned)grid), dim3(EVP_THREADS), smem, st, logits, targets, t_bs, t_cs, parent_targets, pt_bs, pt_cs,
             prev_idx, table, N, units, ns, stats, cons, conf, idx_out);
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}

// ------------------------------------------------------------------------------------
// Per-level VALIDATION evaluation (the reference's test(), train.py:324-339; hires.cuh: ValAcc), ONE pass over the
// logits, the composed probabilities, the ternary targets and, for the consistency term, the previous level's
// probability plane of each group's parent.  Nothing is written but the fp64 / int64 sums.
//   level_val_pipe_kernel  bulk-copy pipeline (16-byte aligned planes and target strides, N % 4 == 0): the same
//                          even split and producer warp as level_eval_pipe_kernel; a consumer thread takes the stage's
//                          pixels tid, tid + 256, ... straight from shared memory (conflict-free 4-byte reads), so
//                          only one pixel's values are in registers at a time.
//   level_val_kernel       any alignment and size: one pixel per thread, the group layout read from the table.
// ------------------------------------------------------------------------------------
template <int K, int CT, int GSZ>
__host__ __device__ constexpr int vp_planes() { return 3 * K + (CT == 2 ? Groups<K, GSZ>::NG : 0); }
// pixels per stage: a stage stays within 64 KB, so that three of them fit one CTA's shared memory
template <int K, int CT, int GSZ>
__host__ __device__ constexpr int vp_px() { return vp_planes<K, CT, GSZ>() <= 16 ? 1024 : 512; }
constexpr int VP_STAGES = 3;

template <int K, int CT, int GSZ>
__global__ void __launch_bounds__(EVP_THREADS)
level_val_pipe_kernel(const float* __restrict__ logits, const float* __restrict__ probs, const float* __restrict__ prev_probs,
                      int K_prev, const float* __restrict__ targets, long t_bstride, long t_cstride,
                      const int32_t* __restrict__ table, long N, long units_total, double* __restrict__ stats,
                      double* __restrict__ cons, unsigned long long* __restrict__ conf) {
  using Acc = ValAcc<K, CT, GSZ>;
  constexpr bool CONS = CT == 2;
  constexpr int NG = Groups<K, GSZ>::NG;
  constexpr int PX = vp_px<K, CT, GSZ>(), PPT = PX / EVP_CONSUMERS;
  constexpr int STAGE = vp_planes<K, CT, GSZ>() * PX * 4;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ float red[EVP_CW * Acc::NACC];
  __shared__ int hist[Acc::NCELL];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  StageRing ring;
  ring.init(reinterpret_cast<uint64_t*>(smem_raw), VP_STAGES, EVP_CW);
  unsigned char* stage0 = smem_raw + 128;
  for (int i = tid; i < Acc::NCELL; i += EVP_THREADS) hist[i] = 0;
  Groups<K, GSZ> gr;
  gr.load(CT >= 1 ? table : nullptr);  // uploaded once per device: not produced by the previous kernel
  const long g0 = (units_total * blockIdx.x / gridDim.x) * 4, g1 = (units_total * (blockIdx.x + 1) / gridDim.x) * 4;
  int b = (int)(g0 / N);
  long off = g0 - (long)b * N;
  __syncthreads();
  pdl_wait();

  if (warp == EVP_CW) {
    // ------------------------------ producer ------------------------------
    if (lane == 0) {
      int slot = 0;
      uint32_t phase = 1;
      for (long cur = g0; cur < g1;) {
        const int len = (int)min((long)PX, min(N - off, g1 - cur));
        mbar_wait(ring.empty(slot), phase);
        const uint32_t dst = smem_u32(stage0 + (size_t)slot * STAGE), bar = ring.full(slot);
        const uint32_t bytes = (uint32_t)len * 4u;
        uint32_t total = 0;
#pragma unroll
        for (int k = 0; k < K; ++k) {
          bulk_g2s_plain(dst + k * PX * 4, logits + ((size_t)b * K + k) * N + off, bytes, bar);
          bulk_g2s_plain(dst + (K + k) * PX * 4, probs + ((size_t)b * K + k) * N + off, bytes, bar);
          bulk_g2s_plain(dst + (2 * K + k) * PX * 4, targets + (size_t)b * t_bstride + (size_t)k * t_cstride + off, bytes, bar);
          total += 3 * bytes;
        }
        if constexpr (CONS) {
#pragma unroll
          for (int g = 0; g < NG; ++g)
            if (g < gr.n) {
              bulk_g2s_plain(dst + (3 * K + g) * PX * 4, prev_probs + ((size_t)b * K_prev + gr.parent[g]) * N + off, bytes, bar);
              total += bytes;
            }
        }
        mbar_arrive_expect_tx(bar, total);
        if (++slot == VP_STAGES) { slot = 0; phase ^= 1u; }
        cur += len;
        off += len;
        if (off == N) { off = 0; ++b; }
      }
    }
    return;
  }

  // -------------------------------- consumers --------------------------------
  auto csync = [] { consumer_sync(EVP_CONSUMERS); };
  Acc ev;
  ev.init();
  int cur_b = b, slot = 0;
  uint32_t phase = 0;
  for (long cur = g0; cur < g1;) {
    const int len = (int)min((long)PX, min(N - off, g1 - cur));
    if (b != cur_b) {  // the range crosses into the next sample: hand over the finished sample's sums
      ev.template finish<EVP_CW>(red, hist, stats + (size_t)cur_b * K * RHSEG_NSTAT, cons, conf, tid, EVP_CONSUMERS, csync);
      cur_b = b;
    }
    mbar_wait(ring.full(slot), phase);
    const float* sf = reinterpret_cast<const float*>(stage0 + (size_t)slot * STAGE);
#pragma unroll 1
    for (int v = 0; v < PPT; ++v) {
      const int i = tid + v * EVP_CONSUMERS;
      const bool ok = i < len;
      float z[K], P[K], t[K], pp[NG], p[K], mx, sum;
#pragma unroll
      for (int k = 0; k < K; ++k) {  // stale shared memory past `len` may hold NaNs
        z[k] = ok ? sf[k * PX + i] : 0.f;
        P[k] = ok ? sf[(K + k) * PX + i] : 0.f;
        t[k] = ok ? sf[(2 * K + k) * PX + i] : -1.f;
      }
#pragma unroll
      for (int g = 0; g < NG; ++g) pp[g] = (CONS && ok && g < gr.n) ? sf[(3 * K + g) * PX + i] : 0.f;
      softmax_all<K>(z, p, mx, sum);
      ev.pixel(z, p, mx + log_fast(sum), t, P, pp, ok, gr);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(ring.empty(slot));  // the warp is done with the stage: the producer may refill it
    if (++slot == VP_STAGES) { slot = 0; phase ^= 1u; }
    cur += len;
    off += len;
    if (off == N) { off = 0; ++b; }
  }
  if (g0 < g1) ev.template finish<EVP_CW>(red, hist, stats + (size_t)cur_b * K * RHSEG_NSTAT, cons, conf, tid, EVP_CONSUMERS, csync);
}

template <int K, int CT, int GSZ>
static int launch_val_pipe(const float* logits, const float* probs, const float* prev_probs, int K_prev, const float* targets,
                           long t_bs, long t_cs, const int32_t* table, int B, long N, double* stats, double* cons,
                           unsigned long long* conf, cudaStream_t st) {
  auto kern = level_val_pipe_kernel<K, CT, GSZ>;
  const size_t smem = 128 + (size_t)VP_STAGES * vp_planes<K, CT, GSZ>() * vp_px<K, CT, GSZ>() * 4;
  int per_sm = 0;
  RHSEG_CUDA(cached_launch_prep(reinterpret_cast<const void*>(kern), EVP_THREADS, smem, smem, &per_sm));
  if (per_sm < 1) return RHSEG_ERR_UNSUPPORTED;
  const long units = (long)B * N / 4;
  // every CTA gets at least two full stages of work; one resident wave at most
  const long grid = std::max<long>(1, std::min<long>((long)device_sm_count() * per_sm, units / (2 * vp_px<K, CT, GSZ>() / 4)));
  launch_pdl(kern, dim3((unsigned)grid), dim3(EVP_THREADS), smem, st, logits, probs, prev_probs, K_prev, targets, t_bs, t_cs,
             table, N, units, stats, cons, conf);
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}

template <int K, int CT>
__global__ void __launch_bounds__(256)
level_val_kernel(const float* __restrict__ logits, const float* __restrict__ probs, const float* __restrict__ prev_probs,
                 int K_prev, const float* __restrict__ targets, long t_bstride, long t_cstride,
                 const int32_t* __restrict__ table, long N, double* __restrict__ stats, double* __restrict__ cons,
                 unsigned long long* __restrict__ conf) {
  using Acc = ValAcc<K, CT, 0>;
  constexpr int NG = Groups<K, 0>::NG;
  __shared__ float red[8 * Acc::NACC];
  __shared__ int hist[Acc::NCELL];
  const int tid = threadIdx.x, b = blockIdx.y;
  for (int i = tid; i < Acc::NCELL; i += 256) hist[i] = 0;
  Groups<K, 0> gr;
  gr.load(CT >= 1 ? table : nullptr);
  __syncthreads();
  pdl_wait();
  Acc ev;
  ev.init();
  const float* zb = logits + (size_t)b * K * N;
  const float* Pb = probs + (size_t)b * K * N;
  for (long px0 = (long)blockIdx.x * 256; px0 < N; px0 += (long)gridDim.x * 256) {  // uniform trip count: ballots
    const long px = px0 + tid;
    const bool ok = px < N;
    float z[K], P[K], t[K], pp[NG], p[K], mx, sum;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      z[k] = ok ? zb[(size_t)k * N + px] : 0.f;
      P[k] = ok ? Pb[(size_t)k * N + px] : 0.f;
      t[k] = ok ? targets[(size_t)b * t_bstride + (size_t)k * t_cstride + px] : -1.f;
    }
#pragma unroll
    for (int g = 0; g < NG; ++g)
      pp[g] = (CT == 2 && ok && g < gr.n) ? prev_probs[((size_t)b * K_prev + gr.parent[g]) * N + px] : 0.f;
    softmax_all<K>(z, p, mx, sum);
    ev.pixel(z, p, mx + log_fast(sum), t, P, pp, ok, gr);
  }
  ev.template finish<8>(red, hist, stats + (size_t)b * K * RHSEG_NSTAT, cons, conf, tid, 256, [] { __syncthreads(); });
}

// ------------------------------------------------------------------------------------
// Flat -> hierarchy stitching (predictEval.py:85-185, :381-388): the flat model predicts the
// leaves only; every node of the tree becomes one output channel: a leaf copies its flat channel,
// a parent is the union (any > 0) of its descendant leaves.  Table driven: one uint32 leaf mask
// per output channel, bit 31 set = "copy" (leaf), clear = "union" (parent).
// ------------------------------------------------------------------------------------
struct StitchTable {
  int n_out;
  uint32_t mask[RHSEG_STITCH_MAX_OUT];
};

template <int VEC, int THREADS>
__global__ void __launch_bounds__(THREADS)
stitch_kernel(const float* __restrict__ leaves, int n_leaves, long N, StitchTable tab, float* __restrict__ out) {
  pdl_wait();
  const int b = blockIdx.y;
  const long px = ((long)blockIdx.x * THREADS + threadIdx.x) * VEC;
  if (px >= N) return;
  float x[RHSEG_STITCH_MAX_LEAVES][VEC];
#pragma unroll
  for (int l = 0; l < RHSEG_STITCH_MAX_LEAVES; ++l) {
    if (l < n_leaves) {
      const Vec<VEC> v = ld_stream<VEC>(leaves + ((size_t)b * n_leaves + l) * N + px);
#pragma unroll
      for (int q = 0; q < VEC; ++q) x[l][q] = v.v[q];
    } else {
#pragma unroll
      for (int q = 0; q < VEC; ++q) x[l][q] = 0.f;
    }
  }
  for (int o = 0; o < tab.n_out; ++o) {
    const uint32_t m = tab.mask[o];
    const bool copy = (m >> 31) != 0u;
    Vec<VEC> r;
#pragma unroll
    for (int q = 0; q < VEC; ++q) {
      float cp = 0.f;
      bool any = false;
#pragma unroll
      for (int l = 0; l < RHSEG_STITCH_MAX_LEAVES; ++l)
        if ((m >> l) & 1u) { cp = x[l][q]; any |= x[l][q] > 0.f; }
      r.v[q] = copy ? cp : (any ? 1.0f : 0.0f);
    }
    st_stream<VEC>(out + ((size_t)b * tab.n_out + o) * N + px, r);
  }
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

template <int MODE>
static int confusion_launch(const float* probs, long p_bs, long p_cs, const float* targets, long t_bs, long t_cs,
                            int B, int K, long N, int child, int64_t* conf, cudaStream_t st) {
  const int nc = child ? K + 1 : K;
  RHSEG_CUDA(cudaMemsetAsync(conf, 0, sizeof(int64_t) * nc * nc, st));
  constexpr int THREADS = 256, ITER = 4;
  const bool v4 = (N % 4 == 0) && aligned16(probs) && aligned16(targets) && p_bs % 4 == 0 && p_cs % 4 == 0 &&
                  t_bs % 4 == 0 && t_cs % 4 == 0;
  auto* c = reinterpret_cast<unsigned long long*>(conf);
  RHSEG_DISPATCH_K(K, {
    if (v4) {
      dim3 grid((unsigned)((N + THREADS * 4 * ITER - 1) / (THREADS * 4 * ITER)), B);
      launch_pdl(confusion_kernel<KK, 4, ITER, THREADS, MODE>, dim3(grid), dim3(THREADS), 0, st, probs, p_bs, p_cs, targets, t_bs, t_cs, N, child, c);
    } else {
      dim3 grid((unsigned)((N + THREADS * ITER - 1) / (THREADS * ITER)), B);
      launch_pdl(confusion_kernel<KK, 1, ITER, THREADS, MODE>, dim3(grid), dim3(THREADS), 0, st, probs, p_bs, p_cs, targets, t_bs, t_cs, N, child, c);
    }
  });
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}

// generic path of rhseg_level_eval: any alignment, any size (level kind decided at run time)
template <typename LT>
static int launch_eval_generic(const LT* logits, const float* targets, long t_bstride, long t_cstride,
                               const float* parent_targets, long pt_bstride, long pt_cstride, const unsigned char* prev_idx,
                               const int32_t* table, int B, int K, long N, int child, bool v4, double* stats, double* cons,
                               unsigned long long* conf, unsigned char* idx_out, cudaStream_t st) {
  constexpr int THREADS = 256;
  const int slots = std::max(1, device_sm_count() * 2 / B);  // CTAs per sample for one resident wave
  RHSEG_DISPATCH_K(K, {
    if (v4 && KK <= 4) {  // 4 pixels per thread spill beyond K = 4 at two CTAs per SM: wider levels take one pixel per thread
      dim3 grid((unsigned)balanced_grid((N + THREADS * 4 - 1) / (THREADS * 4), slots), B);
      launch_pdl(level_eval_kernel<(KK <= 4 ? KK : 1), 4, 2, THREADS, -1, LT>, dim3(grid), dim3(THREADS), 0, st, logits, targets, t_bstride, t_cstride,
          parent_targets, pt_bstride, pt_cstride, prev_idx, table, N, child, stats, cons, conf, idx_out);
    } else {
      dim3 grid((unsigned)balanced_grid((N + THREADS - 1) / THREADS, slots), B);
      launch_pdl(level_eval_kernel<KK, 1, (KK > 6 ? 1 : 2), THREADS, -1, LT>, dim3(grid), dim3(THREADS), 0, st, logits, targets, t_bstride, t_cstride,
          parent_targets, pt_bstride, pt_cstride, prev_idx, table, N, child, stats, cons, conf, idx_out);
    }
  });
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}

}  // namespace rhseg

using namespace rhseg;

extern "C" int rhseg_confusion_matrix(const float* probs, long p_bstride, long p_cstride, const float* targets,
                                      long t_bstride, long t_cstride, int B, int K, int n_pix, int child,
                                      int64_t* conf, void* stream) {
  if (!probs || !targets || !conf || B <= 0 || n_pix <= 0) return RHSEG_ERR_ARG;
  if (K < 1 || K > RHSEG_KERNEL_MAX_K) return RHSEG_ERR_UNSUPPORTED;
  return confusion_launch<0>(probs, p_bstride, p_cstride, targets, t_bstride, t_cstride, B, K, n_pix, child, conf,
                             (cudaStream_t)stream);
}

extern "C" int rhseg_confusion_from_logits(const float* logits, const float* targets, long t_bstride,
                                           long t_cstride, int B, int K, int n_pix, int child, int64_t* conf,
                                           void* stream) {
  if (!logits || !targets || !conf || B <= 0 || n_pix <= 0) return RHSEG_ERR_ARG;
  if (K < 1 || K > RHSEG_KERNEL_MAX_K) return RHSEG_ERR_UNSUPPORTED;
  return confusion_launch<1>(logits, (long)K * n_pix, (long)n_pix, targets, t_bstride, t_cstride, B, K, n_pix, child,
                             conf, (cudaStream_t)stream);
}

extern "C" int rhseg_predict_onehot(const float* logits, const float* targets, long t_bstride, long t_cstride,
                                    int B, int K, int n_pix, float* onehot, float* eval_t, int32_t* pred_idx,
                                    void* stream) {
  if (!logits || !targets || B <= 0 || n_pix <= 0) return RHSEG_ERR_ARG;
  if (K < 1 || K > RHSEG_KERNEL_MAX_K) return RHSEG_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  const long N = n_pix;
  constexpr int THREADS = 256;
  const bool v4 = (N % 4 == 0) && aligned16(logits) && aligned16(targets) && t_bstride % 4 == 0 && t_cstride % 4 == 0 &&
                  aligned16(onehot) && aligned16(eval_t);
  RHSEG_DISPATCH_K(K, {
    if (v4) {
      dim3 grid((unsigned)((N / 4 + THREADS - 1) / THREADS), B);
      launch_pdl(predict_kernel<KK, 4, THREADS>, dim3(grid), dim3(THREADS), 0, st, logits, targets, t_bstride, t_cstride, N, onehot, eval_t, pred_idx);
    } else {
      dim3 grid((unsigned)((N + THREADS - 1) / THREADS), B);
      launch_pdl(predict_kernel<KK, 1, THREADS>, dim3(grid), dim3(THREADS), 0, st, logits, targets, t_bstride, t_cstride, N, onehot, eval_t, pred_idx);
    }
  });
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}

extern "C" int rhseg_metric_ratios(const int64_t* conf, int nc, float* out5, void* stream) {
  if (!conf || !out5 || nc < 1 || nc > RHSEG_MAX_K + 1) return RHSEG_ERR_ARG;
  launch_pdl(metric_ratios_kernel, dim3(1), dim3(32), 0, (cudaStream_t)stream, reinterpret_cast<const long long*>(conf), nc, out5);
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}

extern "C" int rhseg_level_eval(const void* logits_in, const float* targets, long t_bstride, long t_cstride,
                                const float* parent_targets, long pt_bstride, long pt_cstride,
                                const unsigned char* prev_idx, const int32_t* table, int B, int K, int n_pix,
                                int child_arg, void* out_words, unsigned char* idx_out, int flags, void* stream) {
  if (!logits_in || !targets || !out_words || B <= 0 || n_pix <= 0) return RHSEG_ERR_ARG;
  if (K < 1 || K > RHSEG_KERNEL_MAX_K) return RHSEG_ERR_UNSUPPORTED;
  const int child = child_arg & 1, hint = RHSEG_GROUP_HINT_OF(child_arg);
  // bf16 logits come from the flat model: its one (root) level only, no consistency inputs or index map
  const bool bf16 = (flags & RHSEG_LOGITS_BF16) != 0;
  if (bf16 && (child || parent_targets || prev_idx || idx_out)) return RHSEG_ERR_UNSUPPORTED;
  if (child && !table) return RHSEG_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const int nc = child ? K + 1 : K;
  const size_t words = (size_t)B * K * RHSEG_NSTAT + RHSEG_MAX_K + (size_t)nc * nc;
  if (!(flags & RHSEG_EVAL_PREZEROED)) RHSEG_CUDA(cudaMemsetAsync(out_words, 0, words * 8, st));
  double* stats = reinterpret_cast<double*>(out_words);
  double* cons = stats + (size_t)B * K * RHSEG_NSTAT;
  unsigned long long* conf = reinterpret_cast<unsigned long long*>(cons + RHSEG_MAX_K);
  const long N = n_pix;
  bool v4 = (N % 4 == 0) && aligned16(logits_in) && aligned16(targets) && t_bstride % 4 == 0 && t_cstride % 4 == 0 &&
            (reinterpret_cast<uintptr_t>(prev_idx) % 4 == 0) && (reinterpret_cast<uintptr_t>(idx_out) % 4 == 0);
  if (parent_targets) v4 = v4 && aligned16(parent_targets) && pt_bstride % 4 == 0 && pt_cstride % 4 == 0;
  const bool cons_in = child && prev_idx != nullptr && parent_targets != nullptr;
  const bool pipe = v4 && N % 16 == 0 && aligned16(prev_idx) && (long)B * N >= 4 * EVP_PX && !getenv("RHSEG_NO_EVAL_PIPE");
  if (bf16) {
    const uint16_t* z16 = static_cast<const uint16_t*>(logits_in);
    if (pipe) RHSEG_DISPATCH_K(K, return (launch_eval_pipe<KK, 0, KK, uint16_t>(z16, targets, t_bstride, t_cstride, nullptr, 0, 0, nullptr, nullptr, B, N, stats, cons, conf, nullptr, st)));
    return launch_eval_generic(z16, targets, t_bstride, t_cstride, nullptr, 0, 0, nullptr, table, B, K, N, 0, v4, stats, cons, conf, nullptr, st);
  }
  const float* logits = static_cast<const float*>(logits_in);
  if (pipe) {
    // level kind and group structure fixed at compile time: no flag tests per pixel
    RHSEG_DISPATCH_K(K, {
      if (!child)
        return launch_eval_pipe<KK, 0, KK>(logits, targets, t_bstride, t_cstride, nullptr, 0, 0, nullptr, nullptr, B, N, stats, cons, conf, idx_out, st);
      if (hint == KK) {
        if (cons_in) return launch_eval_pipe<KK, 2, KK>(logits, targets, t_bstride, t_cstride, parent_targets, pt_bstride, pt_cstride, prev_idx, table, B, N, stats, cons, conf, idx_out, st);
        return launch_eval_pipe<KK, 1, KK>(logits, targets, t_bstride, t_cstride, nullptr, 0, 0, nullptr, table, B, N, stats, cons, conf, idx_out, st);
      }
      if constexpr (KK == 4) {
        if (hint == 2) {  // two parents with two children each (extended tree, level 2): layout fixed at compile time
          if (cons_in) return launch_eval_pipe<KK, 2, 2>(logits, targets, t_bstride, t_cstride, parent_targets, pt_bstride, pt_cstride, prev_idx, table, B, N, stats, cons, conf, idx_out, st);
          return launch_eval_pipe<KK, 1, 2>(logits, targets, t_bstride, t_cstride, nullptr, 0, 0, nullptr, table, B, N, stats, cons, conf, idx_out, st);
        }
      }
      if (cons_in) {
        // table-driven group layout + consistency with K > 6 would spill in the pipelined kernel: generic kernel below
        if constexpr (KK <= 6) return launch_eval_pipe<KK, 2, 0>(logits, targets, t_bstride, t_cstride, parent_targets, pt_bstride, pt_cstride, prev_idx, table, B, N, stats, cons, conf, idx_out, st);
      } else
      return launch_eval_pipe<KK, 1, 0>(logits, targets, t_bstride, t_cstride, nullptr, 0, 0, nullptr, table, B, N, stats, cons, conf, idx_out, st);
    });
  }
  return launch_eval_generic(logits, targets, t_bstride, t_cstride, parent_targets, pt_bstride, pt_cstride, prev_idx, table, B, K, N,
                             child, v4, stats, cons, conf, idx_out, st);
}

extern "C" int rhseg_level_eval_composed(const float* logits, const float* probs, const float* prev_probs,
                                         const float* targets, long t_bstride, long t_cstride, const int32_t* table,
                                         int B, int K, int K_prev, int n_pix, int child_arg, void* out_words, int flags,
                                         void* stream) {
  if (!logits || !probs || !targets || !out_words || B <= 0 || n_pix <= 0) return RHSEG_ERR_ARG;
  if (K < 1 || K > RHSEG_KERNEL_MAX_K) return RHSEG_ERR_UNSUPPORTED;
  const int child = child_arg & 1, hint = RHSEG_GROUP_HINT_OF(child_arg);
  if (child && !table) return RHSEG_ERR_ARG;
  const bool cons_in = child && prev_probs != nullptr;
  if (cons_in && (K_prev < 1 || K_prev > RHSEG_KERNEL_MAX_K)) return RHSEG_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const int nc = child ? K + 1 : K;
  const size_t words = (size_t)B * K * RHSEG_NSTAT + RHSEG_MAX_K + (size_t)nc * nc;
  if (!(flags & RHSEG_EVAL_PREZEROED)) RHSEG_CUDA(cudaMemsetAsync(out_words, 0, words * 8, st));
  double* stats = reinterpret_cast<double*>(out_words);
  double* cons = stats + (size_t)B * K * RHSEG_NSTAT;
  unsigned long long* conf = reinterpret_cast<unsigned long long*>(cons + RHSEG_MAX_K);
  const long N = n_pix;
  // bulk copies need 16-byte sizes and addresses: every plane and target slice starts on a 16-byte boundary and
  // every stage boundary (a multiple of 4 pixels) stays on one
  const bool pipe = N % 4 == 0 && aligned16(logits) && aligned16(probs) && aligned16(targets) && t_bstride % 4 == 0 &&
                    t_cstride % 4 == 0 && (!cons_in || aligned16(prev_probs)) && !getenv("RHSEG_NO_EVAL_PIPE");
  if (pipe) {
    RHSEG_DISPATCH_K(K, {
      if (!child)
        return launch_val_pipe<KK, 0, KK>(logits, probs, nullptr, 0, targets, t_bstride, t_cstride, nullptr, B, N, stats, cons, conf, st);
      if (hint == KK) {
        if (cons_in) return launch_val_pipe<KK, 2, KK>(logits, probs, prev_probs, K_prev, targets, t_bstride, t_cstride, table, B, N, stats, cons, conf, st);
        return launch_val_pipe<KK, 1, KK>(logits, probs, nullptr, 0, targets, t_bstride, t_cstride, table, B, N, stats, cons, conf, st);
      }
      if constexpr (KK == 4) {
        if (hint == 2) {  // two parents with two children each (extended tree, level 2)
          if (cons_in) return launch_val_pipe<KK, 2, 2>(logits, probs, prev_probs, K_prev, targets, t_bstride, t_cstride, table, B, N, stats, cons, conf, st);
          return launch_val_pipe<KK, 1, 2>(logits, probs, nullptr, 0, targets, t_bstride, t_cstride, table, B, N, stats, cons, conf, st);
        }
      }
      if (cons_in) return launch_val_pipe<KK, 2, 0>(logits, probs, prev_probs, K_prev, targets, t_bstride, t_cstride, table, B, N, stats, cons, conf, st);
      return launch_val_pipe<KK, 1, 0>(logits, probs, nullptr, 0, targets, t_bstride, t_cstride, table, B, N, stats, cons, conf, st);
    });
  }
  constexpr int THREADS = 256;
  const int slots = std::max(1, device_sm_count() * 4 / B);  // CTAs per sample for about one resident wave
  const dim3 grid((unsigned)balanced_grid((N + THREADS - 1) / THREADS, slots), B);
  RHSEG_DISPATCH_K(K, {
    if (!child) launch_pdl(level_val_kernel<KK, 0>, grid, dim3(THREADS), 0, st, logits, probs, prev_probs, K_prev, targets, t_bstride, t_cstride, table, N, stats, cons, conf);
    else if (cons_in) launch_pdl(level_val_kernel<KK, 2>, grid, dim3(THREADS), 0, st, logits, probs, prev_probs, K_prev, targets, t_bstride, t_cstride, table, N, stats, cons, conf);
    else launch_pdl(level_val_kernel<KK, 1>, grid, dim3(THREADS), 0, st, logits, probs, prev_probs, K_prev, targets, t_bstride, t_cstride, table, N, stats, cons, conf);
  });
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}

extern "C" int rhseg_stitch_levels(const float* leaves, int B, int n_leaves, int n_pix, const uint32_t* masks,
                                   int n_out, float* out, void* stream) {
  if (!leaves || !masks || !out || B <= 0 || n_pix <= 0) return RHSEG_ERR_ARG;
  if (n_leaves < 1 || n_leaves > RHSEG_STITCH_MAX_LEAVES || n_out < 1 || n_out > RHSEG_STITCH_MAX_OUT) return RHSEG_ERR_UNSUPPORTED;
  StitchTable tab{};
  tab.n_out = n_out;
  for (int o = 0; o < n_out; ++o) {
    if ((masks[o] & 0x7fffffffu) >> n_leaves) return RHSEG_ERR_TREE;  // references a leaf that does not exist
    tab.mask[o] = masks[o];
  }
  const long N = n_pix;
  constexpr int THREADS = 256;
  cudaStream_t st = (cudaStream_t)stream;
  if (N % 4 == 0 && aligned16(leaves) && aligned16(out)) {
    dim3 grid((unsigned)((N / 4 + THREADS - 1) / THREADS), B);
    launch_pdl(stitch_kernel<4, THREADS>, dim3(grid), dim3(THREADS), 0, st, leaves, n_leaves, N, tab, out);
  } else {
    dim3 grid((unsigned)((N + THREADS - 1) / THREADS), B);
    launch_pdl(stitch_kernel<1, THREADS>, dim3(grid), dim3(THREADS), 0, st, leaves, n_leaves, N, tab, out);
  }
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}

// ------------------------------------------------------------------------------------
// Image (+) logits concat (north_star item 2, SURVEY row a4'): out = cat([image, logits], dim=1).
// The reference never performs this concat (its recurrent passes re-run the donor on the unchanged
// image, Models/models.py:277, :773), so it is a stand-alone utility and is not wired into forward.
// ------------------------------------------------------------------------------------
template <int VEC>
__global__ void __launch_bounds__(256)
concat_planes_kernel(const float* __restrict__ a, int ca, const float* __restrict__ b, int cb, long N,
                     float* __restrict__ out) {
  pdl_wait();
  const int plane = blockIdx.y;              // (sample, output channel)
  const int c_out = ca + cb;
  const int s = plane / c_out, c = plane - s * c_out;
  const float* src = c < ca ? a + ((size_t)s * ca + c) * N : b + ((size_t)s * cb + (c - ca)) * N;
  float* dst = out + (size_t)plane * N;
  for (long px = ((long)blockIdx.x * 256 + threadIdx.x) * VEC; px < N; px += (long)gridDim.x * 256 * VEC)
    st_stream<VEC>(dst + px, ld_stream<VEC>(src + px));
}

// ------------------------------------------------------------------------------------
// Ternary targets shipped as int8 ({1, 0, -1}: what Data/dataset.py:227-265 produces, a quarter of the fp32 bytes over
// PCIe) -> the fp32 tensor every kernel of the path reads.  16 values per thread: one 16-byte load, four 16-byte stores.
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) widen_i8_kernel(const signed char* __restrict__ in, long n, float* __restrict__ out) {
  pdl_wait();
  const long n16 = n / 16;
  for (long i = (long)blockIdx.x * 256 + threadIdx.x; i < n16; i += (long)gridDim.x * 256) {
    const int4 v = __ldg(reinterpret_cast<const int4*>(in) + i);
    const int w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float4 o;
      o.x = (float)(signed char)(w[q] & 0xff);
      o.y = (float)(signed char)((w[q] >> 8) & 0xff);
      o.z = (float)(signed char)((w[q] >> 16) & 0xff);
      o.w = (float)(signed char)((w[q] >> 24) & 0xff);
      reinterpret_cast<float4*>(out)[i * 4 + q] = o;
    }
  }
  for (long i = n16 * 16 + (long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long)gridDim.x * 256) out[i] = (float)in[i];
}

extern "C" int rhseg_targets_i8_to_f32(const signed char* in, long n, float* out, void* stream) {
  if (!in || !out || n <= 0) return RHSEG_ERR_ARG;
  if (!aligned16(in) || !aligned16(out)) return RHSEG_ERR_ARG;
  const unsigned grid = (unsigned)std::min<long>((n / 16 + 255) / 256 + 1, 8L * device_sm_count());
  launch_pdl(widen_i8_kernel, dim3(grid), dim3(256), 0, (cudaStream_t)stream, in, n, out);
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}

extern "C" int rhseg_concat_image_logits(const float* image, int c_image, const float* logits, int K, int B, int n_pix,
                                         float* out, void* stream) {
  if (!image || !logits || !out || B <= 0 || c_image < 1 || K < 1 || n_pix <= 0) return RHSEG_ERR_ARG;
  const long N = n_pix;
  cudaStream_t st = (cudaStream_t)stream;
  const bool v4 = N % 4 == 0 && aligned16(image) && aligned16(logits) && aligned16(out);
  const long per = v4 ? 1024 : 256;
  dim3 grid((unsigned)std::min<long>(64, (N + per - 1) / per), (unsigned)(B * (c_image + K)));
  if (v4) launch_pdl(concat_planes_kernel<4>, dim3(grid), dim3(256), 0, st, image, c_image, logits, K, N, out);
  else launch_pdl(concat_planes_kernel<1>, dim3(grid), dim3(256), 0, st, image, c_image, logits, K, N, out);
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}
