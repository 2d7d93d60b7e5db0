// Output-resolution building blocks shared by the hi-res forward (head_up.cu), the per-level evaluation
// (metrics.cu) and the hi-res gradient (upsample_bwd.cu):
//   * Groups<K, GSZ>      the level's parent groups with the group size fixed at compile time when it is uniform
//   * softmax helpers     one exp per channel, shared between activation, statistics and prediction
//   * CellCounter         warp-cooperative confusion counting on the cell index (ballots, no atomics)
//   * EvalAcc<K, CT, GSZ> CE/Dice statistics + train-path prediction + confusion + consistency of one pixel
//   * StageRing           mbarrier ring of shared-memory stages fed by 1-D bulk async copies (a producer warp
//                         streams every per-pixel input of the kernel; consumer warps only touch shared memory)
// Reference semantics: Metrics/losses.py:16-177, Metrics/performance_metrics.py:27-47, train.py:206-239.
#pragma once
#include "common.cuh"
#include "pipeline.cuh"

namespace rhseg {

// ------------------------------------------------------------------------------------------------
// Group structure.  GSZ > 0: every group has exactly GSZ channels (the launcher checked the hint against
// nothing: the caller's act_mode / child argument carries it, see RHSEG_GROUP_HINT in rhseg_b200.h);
// GSZ == 0: generic, read from the level table.
// ------------------------------------------------------------------------------------------------
template <int K, int GSZ>
struct Groups {
  static constexpr int NG = GSZ > 0 ? K / GSZ : K;
  static_assert(GSZ == 0 || K % GSZ == 0, "uniform group size divides K");
  int n;              // number of groups
  int parent[NG];     // channel of the group's parent in level L-1
  int start_mask;     // generic: bit k set = channel k starts a group
  unsigned gof;       // generic: 4-bit group index per channel (K <= 8)
  __device__ __forceinline__ void load(const int32_t* __restrict__ table) {
    n = GSZ > 0 ? NG : (table ? table[1] : K);
    start_mask = 0;
    gof = 0u;
#pragma unroll
    for (int g = 0; g < NG; ++g) parent[g] = (table && g < n) ? table[RHSEG_TBL_GPARENT + g] : -1;
    if constexpr (GSZ == 0) {
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const int g = table ? table[RHSEG_TBL_GROUP_OF + k] : k;
        const int gs = table ? table[RHSEG_TBL_GSTART + g] : k;
        if (gs == k) start_mask |= (1 << k);
        gof |= (unsigned)(g & 15) << (4 * k);
      }
    }
  }
  __device__ __forceinline__ int group_of(int k) const {
    if constexpr (GSZ == K) return 0;
    else if constexpr (GSZ > 0) return k / GSZ;
    else return (int)((gof >> (4 * k)) & 15u);
  }
};

// softmax over all K channels: p, max, sum of exp(z - max)  (SFU math; integer decisions never use it)
template <int K>
__device__ __forceinline__ void softmax_all(const float (&z)[K], float (&p)[K], float& mx, float& sum) {
  fast_softmax<K>(z, p, mx, sum);
}

// restrictive (per parent group) softmax.  GSZ == K is the plain softmax.
template <int K, int GSZ>
__device__ __forceinline__ void softmax_groups(const float (&z)[K], const Groups<K, GSZ>& gr, float (&q)[K]) {
  if constexpr (GSZ == 0) {
    grouped_softmax<K>(z, gr.start_mask, q);
  } else {
#pragma unroll
    for (int g = 0; g < K / GSZ; ++g) {
      float mx = z[g * GSZ];
#pragma unroll
      for (int j = 1; j < GSZ; ++j) mx = fmaxf(mx, z[g * GSZ + j]);
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < GSZ; ++j) { q[g * GSZ + j] = exp_fast(z[g * GSZ + j] - mx); s += q[g * GSZ + j]; }
      const float inv = rcp_approx(s);
#pragma unroll
      for (int j = 0; j < GSZ; ++j) q[g * GSZ + j] *= inv;
    }
  }
}

// per-channel copy of a per-group value (parent probability, parent target)
template <int K, int GSZ>
__device__ __forceinline__ float group_value(const float (&per_group)[Groups<K, GSZ>::NG], const Groups<K, GSZ>& gr, int k) {
  if constexpr (GSZ > 0) {
    return per_group[k / GSZ];
  } else {
    float v = per_group[0];
#pragma unroll
    for (int g = 1; g < K; ++g) v = (gr.group_of(k) == g) ? per_group[g] : v;
    return v;
  }
}

// ------------------------------------------------------------------------------------------------
// Confusion counting.  cell = target_class * nc + predicted_class (< 0: pixel ignored).  The warp ballots the
// bits of the cell index; lane l (slot s) owns cell l + 32 s and ANDs the votes (or their complements) that
// spell its own index.  BITS + 1 ballots and about as many logic ops per pixel, no atomics, no match.
// ------------------------------------------------------------------------------------------------
template <int NCELL>
struct CellCounter {
  static constexpr int SLOTS = (NCELL + 31) / 32;
  static constexpr int BITS = NCELL <= 2 ? 1 : NCELL <= 4 ? 2 : NCELL <= 8 ? 3 : NCELL <= 16 ? 4 : NCELL <= 32 ? 5 : NCELL <= 64 ? 6 : 7;
  static constexpr int LB = BITS < 5 ? BITS : 5;
  int cnt[SLOTS];
  unsigned xl[LB];  // ~0 where the lane's bit i is clear (vote ^ xl selects the lanes that agree with this lane)
  __device__ __forceinline__ void init() {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) cnt[s] = 0;
#pragma unroll
    for (int i = 0; i < LB; ++i) xl[i] = ((lane >> i) & 1) ? 0u : 0xffffffffu;
  }
  __device__ __forceinline__ void add(int cell) {
    unsigned m = __ballot_sync(0xffffffffu, cell >= 0);
#pragma unroll
    for (int i = 0; i < LB; ++i) m &= __ballot_sync(0xffffffffu, (cell & (1 << i)) != 0) ^ xl[i];
    if constexpr (SLOTS == 1) {
      cnt[0] += __popc(m);
    } else {
      unsigned vh[BITS - 5];
#pragma unroll
      for (int i = 5; i < BITS; ++i) vh[i - 5] = __ballot_sync(0xffffffffu, (cell & (1 << i)) != 0);
#pragma unroll
      for (int s = 0; s < SLOTS; ++s) {
        unsigned ms = m;
#pragma unroll
        for (int i = 5; i < BITS; ++i) ms &= ((s >> (i - 5)) & 1) ? vh[i - 5] : ~vh[i - 5];
        cnt[s] += __popc(ms);
      }
    }
  }
  // hist: shared int[NCELL] (zeroed by the caller)
  __device__ __forceinline__ void flush(int* hist) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
      const int cell = lane + 32 * s;
      if (cell < NCELL && cnt[s]) atomicAdd(&hist[cell], cnt[s]);
      cnt[s] = 0;
    }
  }
};

// class index of one pixel following ProcessClasses (performance_metrics.py:31-47): argmax (first maximum, NaN
// wins) over the channels, with the prepended "nothing positive" channel on child levels.  `sum` = x[0] + ... in
// channel order; a NaN sum (a NaN or inf - inf among the values) takes the NaN-aware path.
template <int K, bool CHILD>
__device__ __noinline__ int process_class_nan(const float* xp) {
  float x[K];
#pragma unroll
  for (int k = 0; k < K; ++k) x[k] = xp[k];
  if constexpr (CHILD) {
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) sum += x[k];
    float best = (sum == 0.f) ? 1.0f : 0.0f;
    int idx = 0;
#pragma unroll
    for (int k = 0; k < K; ++k)
      if (beats(x[k], best)) { best = x[k]; idx = k + 1; }
    return idx;
  } else {
    float best = x[0];
    int idx = 0;
#pragma unroll
    for (int k = 1; k < K; ++k)
      if (beats(x[k], best)) { best = x[k]; idx = k; }
    return idx;
  }
}
template <int K, bool CHILD>
__device__ __forceinline__ int process_class2(const float (&x)[K]) {
  float sum = 0.f;
#pragma unroll
  for (int k = 0; k < K; ++k) sum += x[k];
  int idx = 0;
  if (sum != sum) {
    float xl[K];
#pragma unroll
    for (int k = 0; k < K; ++k) xl[k] = x[k];
    idx = process_class_nan<K, CHILD>(xl);
  } else if constexpr (CHILD) {
    float best = (sum == 0.f) ? 1.0f : 0.0f;  // prepended "nothing positive" channel
#pragma unroll
    for (int k = 0; k < K; ++k)
      if (x[k] > best) { best = x[k]; idx = k + 1; }
  } else {
    float best = x[0];
#pragma unroll
    for (int k = 1; k < K; ++k)
      if (x[k] > best) { best = x[k]; idx = k; }
  }
  return idx;
}

// ------------------------------------------------------------------------------------------------
// Per-pixel training evaluation (train.py:206-239 for one level): CE/Dice statistics, the bit-exact train-path
// prediction, the confusion cell of the masked one-hot prediction against the eval target, and the consistency
// mismatch of the masked one-hot predictions of this level and the previous one.
//   CT 0: root level (no background class, no consistency)   1: child level   2: child level + consistency
// ------------------------------------------------------------------------------------------------
template <int K, int CT, int GSZ>
struct EvalAcc {
  static constexpr int NS = RHSEG_NSTAT;
  static constexpr bool CHILD = CT >= 1, CONS = CT == 2;
  static constexpr int NC = CHILD ? K + 1 : K;
  static constexpr int NCELL = NC * NC;
  static constexpr int NG = Groups<K, GSZ>::NG;
  static constexpr int NACC = K * NS;
  float a[K][NS];
  int cm[CONS ? NG : 1];  // consistency: number of pixels where (children one-hot sum) != (parent one-hot)
  CellCounter<NCELL> cc;

  __device__ __forceinline__ void init() {
    cc.init();
#pragma unroll
    for (int g = 0; g < (CONS ? NG : 1); ++g) cm[g] = 0;
#pragma unroll
    for (int k = 0; k < K; ++k)
#pragma unroll
      for (int j = 0; j < NS; ++j) a[k][j] = 0.f;
  }

  // z: logits, p: softmax(z) over all K channels, mlse = max + log(sum exp(z - max)), t: ternary targets of the
  // level (out-of-range pixels arrive with ok == false and any t), ptg: the parent's target per group, pidx: the
  // previous level's predicted channel.  All lanes of the warp call it (ballots).  Returns the predicted channel.
  __device__ __forceinline__ int pixel(const float (&z)[K], const float (&p)[K], float mlse, const float (&t)[K],
                                       const float (&ptg)[NG], int pidx, bool ok, const Groups<K, GSZ>& gr) {
    float et[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const bool m = ok && t[k] != -1.0f;
      const float mf = m ? 1.0f : 0.0f;
      et[k] = m ? t[k] : 0.0f;  // eval target (train.py:226-229); also t * mask for the statistics
      const float lp = z[k] - mlse;
      a[k][0] = fmaf(et[k], lp, a[k][0]);
      a[k][1] += mf;
      a[k][2] = fmaf(p[k], et[k], a[k][2]);
      a[k][3] = fmaf(p[k], mf, a[k][3]);
      a[k][4] += et[k];
    }
    const int idx = argmax_softmax_aten<K>(z);  // train.py:219-221, bit-exact
    float t_idx = t[0];
#pragma unroll
    for (int k = 1; k < K; ++k) t_idx = (idx == k) ? t[k] : t_idx;
    const bool m_idx = t_idx != -1.0f;  // the one-hot survives the ignore mask (train.py:230-231)
    // ProcessClasses of the masked one-hot prediction: its channel, or "nothing positive"
    const int pc = m_idx ? (CHILD ? idx + 1 : idx) : 0;
    int tc = process_class2<K, CHILD>(et);
    const bool counted = ok && !(CHILD && tc == 0);  // torchmetrics ignore_index=0 on child levels
    cc.add(counted ? tc * NC + pc : -1);
    if constexpr (CONS) {
      const int gi = gr.group_of(idx);
#pragma unroll
      for (int g = 0; g < NG; ++g) {
        const bool child_hot = m_idx && gi == g;
        const bool parent_hot = pidx == gr.parent[g] && ptg[g] != -1.0f;
        cm[g] += (ok && g < gr.n && child_hot != parent_hot) ? 1 : 0;
      }
    }
    return idx;
  }

  // Block reduction + one fp64 / int64 atomic per CTA and quantity, then the accumulators are cleared.
  //   red: shared float[NWARP][NACC]; cred: shared int[NG]; hist: shared int[NCELL] (both zeroed by the caller
  //   before the first pixel and left zeroed here).  SYNC(): barrier of the participating threads; tid / nthreads /
  //   warp: position among them.
  template <int NWARP, typename SyncFn>
  __device__ __forceinline__ void finish(float* red, int* cred, int* hist, double* __restrict__ stats_b,
                                         double* __restrict__ cons, unsigned long long* __restrict__ conf, int tid,
                                         int nthreads, SyncFn sync) {
    const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int k = 0; k < K; ++k)
#pragma unroll
      for (int j = 0; j < NS; ++j) {
        const float v = warp_sum(a[k][j]);
        if (lane == 0) red[warp * NACC + k * NS + j] = v;
        a[k][j] = 0.f;
      }
    if constexpr (CONS) {
#pragma unroll
      for (int g = 0; g < NG; ++g) {
        const int v = __reduce_add_sync(0xffffffffu, cm[g]);
        if (lane == 0 && v) atomicAdd(&cred[g], v);
        cm[g] = 0;
      }
    }
    cc.flush(hist);
    sync();
    if (tid < NACC) {
      double acc = 0.0;
#pragma unroll
      for (int w = 0; w < NWARP; ++w) acc += (double)red[w * NACC + tid];
      atomicAdd(&stats_b[tid], acc);
    }
    if constexpr (CONS) {
      if (tid < NG && cred[tid]) { atomicAdd(&cons[tid], (double)cred[tid]); cred[tid] = 0; }
    }
    for (int i = tid; i < NCELL; i += nthreads)
      if (hist[i]) { atomicAdd(&conf[i], (unsigned long long)hist[i]); hist[i] = 0; }
    sync();
  }
};

// ------------------------------------------------------------------------------------------------
// Per-pixel VALIDATION evaluation (the reference's test(), train.py:324-339, for one level): the CE/Dice statistics
// of EvalAcc, the confusion cell of ProcessClasses over the composed probabilities P against the RAW ternary targets
// (no one-hot, no -1 -> 0), and per group g the consistency |sum_{c in g} P_c - P_prev[parent(g)]| of the real
// probabilities, without an ignore mask.  Level kinds (CT) as in EvalAcc.  Kept apart from EvalAcc so that the
// training instances keep their code.
// ------------------------------------------------------------------------------------------------
template <int K, int CT, int GSZ>
struct ValAcc {
  static constexpr int NS = RHSEG_NSTAT;
  static constexpr bool CHILD = CT >= 1, CONS = CT == 2;
  static constexpr int NC = CHILD ? K + 1 : K;
  static constexpr int NCELL = NC * NC;
  static constexpr int NG = Groups<K, GSZ>::NG;
  static constexpr int NCS = CONS ? NG : 0;
  static constexpr int NACC = K * NS + NCS;  // statistics, then one consistency partial per group
  float a[K][NS];
  float cs[CONS ? NG : 1];
  CellCounter<NCELL> cc;

  __device__ __forceinline__ void init() {
    cc.init();
#pragma unroll
    for (int g = 0; g < (CONS ? NG : 1); ++g) cs[g] = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k)
#pragma unroll
      for (int j = 0; j < NS; ++j) a[k][j] = 0.f;
  }

  // z, p, mlse, t, ok as in EvalAcc::pixel (t: the raw ternary targets); P: the level's composed probabilities,
  // pp: the previous level's probability of each group's parent (CT 2).  Out-of-range pixels (ok == false) must
  // arrive with finite P.  All lanes of the warp call it (ballots).
  __device__ __forceinline__ void pixel(const float (&z)[K], const float (&p)[K], float mlse, const float (&t)[K],
                                        const float (&P)[K], const float (&pp)[NG], bool ok, const Groups<K, GSZ>& gr) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const bool m = ok && t[k] != -1.0f;
      const float mf = m ? 1.0f : 0.0f;
      const float et = m ? t[k] : 0.0f;
      const float lp = z[k] - mlse;
      a[k][0] = fmaf(et, lp, a[k][0]);
      a[k][1] += mf;
      a[k][2] = fmaf(p[k], et, a[k][2]);
      a[k][3] = fmaf(p[k], mf, a[k][3]);
      a[k][4] += et;
    }
    const int pc = process_class2<K, CHILD>(P);
    const int tc = process_class2<K, CHILD>(t);
    const bool counted = ok && !(CHILD && tc == 0);  // torchmetrics ignore_index=0 on child levels
    cc.add(counted ? tc * NC + pc : -1);
    if constexpr (CONS) {
#pragma unroll
      for (int g = 0; g < NG; ++g) {
        float s = 0.f;
        if constexpr (GSZ > 0) {
#pragma unroll
          for (int j = 0; j < GSZ; ++j) s += P[g * GSZ + j];
        } else {
#pragma unroll
          for (int k = 0; k < K; ++k) s += (gr.group_of(k) == g) ? P[k] : 0.0f;
        }
        cs[g] += (ok && g < gr.n) ? fabsf(s - pp[g]) : 0.0f;
      }
    }
  }

  // Block reduction + one fp64 / int64 atomic per CTA and quantity, then the accumulators are cleared.
  //   red: shared float[NWARP][NACC]; hist: shared int[NCELL] (zeroed by the caller before the first pixel and left
  //   zeroed here); cons: the level's consistency slots, indexed by group.  sync / tid / nthreads as in EvalAcc.
  template <int NWARP, typename SyncFn>
  __device__ __forceinline__ void finish(float* red, int* hist, double* __restrict__ stats_b, double* __restrict__ cons,
                                         unsigned long long* __restrict__ conf, int tid, int nthreads, SyncFn sync) {
    const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int k = 0; k < K; ++k)
#pragma unroll
      for (int j = 0; j < NS; ++j) {
        const float v = warp_sum(a[k][j]);
        if (lane == 0) red[warp * NACC + k * NS + j] = v;
        a[k][j] = 0.f;
      }
#pragma unroll
    for (int g = 0; g < NCS; ++g) {
      const float v = warp_sum(cs[g]);
      if (lane == 0) red[warp * NACC + K * NS + g] = v;
      cs[g] = 0.f;
    }
    cc.flush(hist);
    sync();
    if (tid < NACC) {
      double acc = 0.0;
#pragma unroll
      for (int w = 0; w < NWARP; ++w) acc += (double)red[w * NACC + tid];
      if (tid < K * NS) atomicAdd(&stats_b[tid], acc);
      else if (acc != 0.0) atomicAdd(&cons[tid - K * NS], acc);
    }
    for (int i = tid; i < NCELL; i += nthreads)
      if (hist[i]) { atomicAdd(&conf[i], (unsigned long long)hist[i]); hist[i] = 0; }
    sync();
  }
};

// ------------------------------------------------------------------------------------------------
// Shared-memory stage ring.  bars[0..NS) = "full" (expect_tx bytes of the stage's copies, one producer arrival),
// bars[NS..2NS) = "empty" (one arrival per consumer warp).  The producer is one elected lane.
// ------------------------------------------------------------------------------------------------
struct StageRing {
  uint64_t* bars;
  int ns;
  __device__ __forceinline__ void init(uint64_t* b, int n_stages, int consumer_warps) {
    bars = b;
    ns = n_stages;
    if (threadIdx.x == 0) {
      for (int i = 0; i < n_stages; ++i) {
        mbar_init(smem_u32(&bars[i]), 1);
        mbar_init(smem_u32(&bars[n_stages + i]), consumer_warps);
      }
      mbar_fence_init();
    }
  }
  __device__ __forceinline__ uint32_t full(int slot) const { return smem_u32(&bars[slot]); }
  __device__ __forceinline__ uint32_t empty(int slot) const { return smem_u32(&bars[ns + slot]); }
};

// plain (no cache hint) 1-D bulk copy global -> shared: data other kernels re-read stays in L2 normally
__device__ __forceinline__ void bulk_g2s_plain(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

// magic-number division of a non-negative int by a runtime constant d >= 1 (d fixed per launch)
struct FastDiv {
  unsigned mul, shift, d;
  __host__ __device__ FastDiv() : mul(0), shift(0), d(1) {}
  __host__ explicit FastDiv(unsigned dd) : d(dd) {
    if (dd <= 1) { mul = 0; shift = 0; return; }
    unsigned s = 0;
    while ((1ull << s) < dd) ++s;
    shift = s;
    mul = (unsigned)(((1ull << 32) * ((1ull << s) - dd)) / dd + 1);
  }
  __device__ __forceinline__ unsigned div(unsigned n) const {
    if (d == 1) return n;
    const unsigned t = __umulhi(n, mul);
    return (t + ((n - t) >> 1)) >> (shift - 1);
  }
};

}  // namespace rhseg
