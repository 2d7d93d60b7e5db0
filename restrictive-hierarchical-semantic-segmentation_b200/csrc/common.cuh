// Shared device helpers for the rhseg_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <mutex>
#include <vector>
#include <stdint.h>
#include <cstdlib>
#pragma GCC visibility push(default)
#include "rhseg_b200.h"
#pragma GCC visibility pop

#define RHSEG_TBL_PARENT (4)
#define RHSEG_TBL_GROUP_OF (4 + RHSEG_MAX_K)
#define RHSEG_TBL_GSTART (4 + 2 * RHSEG_MAX_K)
#define RHSEG_TBL_GLEN (4 + 3 * RHSEG_MAX_K)
#define RHSEG_TBL_GPARENT (4 + 4 * RHSEG_MAX_K)

#define RHSEG_LAUNCH_CHECK()                      \
  do {                                            \
    cudaError_t e__ = cudaGetLastError();         \
    if (e__ != cudaSuccess) return (int)e__;      \
  } while (0)

#define RHSEG_CUDA(call)                          \
  do {                                            \
    cudaError_t e__ = (call);                     \
    if (e__ != cudaSuccess) return (int)e__;      \
  } while (0)

// K -> template dispatch (K in [1, RHSEG_KERNEL_MAX_K])
#define RHSEG_DISPATCH_K(K, ...)                                 \
  switch (K) {                                                   \
    case 1: { constexpr int KK = 1; __VA_ARGS__; } break;        \
    case 2: { constexpr int KK = 2; __VA_ARGS__; } break;        \
    case 3: { constexpr int KK = 3; __VA_ARGS__; } break;        \
    case 4: { constexpr int KK = 4; __VA_ARGS__; } break;        \
    case 5: { constexpr int KK = 5; __VA_ARGS__; } break;        \
    case 6: { constexpr int KK = 6; __VA_ARGS__; } break;        \
    case 7: { constexpr int KK = 7; __VA_ARGS__; } break;        \
    case 8: { constexpr int KK = 8; __VA_ARGS__; } break;        \
    default: return RHSEG_ERR_UNSUPPORTED;                       \
  }

namespace rhseg {

// ---- programmatic dependent launch (PDL) ----
// Every kernel of the library begins with pdl_wait() and can be launched with the programmatic-stream-serialization
// attribute: its CTAs may then become resident (and pay launch latency / run setup code) while the previous kernel of the
// stream drains, and block at the wait until that kernel has completed and its writes are visible.
// When: the attribute saves GPU time between kernels (~1.5 % of a captured step) but costs ~2.8 us of HOST time per launch
// (measured: 27 launches of the eager drop-in route, 1.029 -> 0.953 ms of host time per step without it).  A captured
// graph pays the host cost once, an eager caller on every call and is usually host-bound there.  Default: the attribute
// is set while the stream is being captured (CUDA graphs) and left out for eager launches.
//   RHSEG_PDL=always | capture (default) | off;  RHSEG_NO_PDL=1 is the same as off.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

inline int pdl_mode() {  // 0 off, 1 while capturing, 2 always
  static int cached = -1;
  if (cached < 0) {
    const char* off = getenv("RHSEG_NO_PDL");
    const char* e = getenv("RHSEG_PDL");
    int m = 1;
    if (e && e[0] == 'a') m = 2;
    if (e && e[0] == 'o') m = 0;
    if (off && off[0] == '1') m = 0;
    cached = m;
  }
  return cached;
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  const int mode = pdl_mode();
  bool use = mode == 2;
  if (mode == 1) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    use = cudaStreamIsCapturing(st, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusActive;
  }
  cfg.numAttrs = use ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

// SM count of the current device (cached per process; grids are sized from it)
inline int device_sm_count() {  // of the CURRENT device (a process may drive several)
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    cached[dev] = n > 0 ? n : 148;
  }
  return cached[dev];
}

// Launch preparation of the persistent kernels, cached: raising the dynamic shared-memory limit and asking for the
// resident CTAs per SM are driver calls of several microseconds each -- noticeable on the eager drop-in route, which is
// bound by host time per launch.  Keyed by (device, kernel, threads, shared memory); the limit only ever grows.
inline cudaError_t cached_launch_prep(const void* kern, int threads, size_t smem, size_t smem_limit, int* per_sm) {
  struct Entry { int dev; const void* f; int threads; size_t smem; int per_sm; };
  struct Limit { int dev; const void* f; size_t limit; };
  static std::mutex mu;
  static std::vector<Entry> occ;
  static std::vector<Limit> lim;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  std::lock_guard<std::mutex> lock(mu);
  Limit* l = nullptr;
  for (auto& x : lim)
    if (x.dev == dev && x.f == kern) { l = &x; break; }
  if (l == nullptr || l->limit < smem_limit) {
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_limit);
    if (e != cudaSuccess) return e;
    if (l) l->limit = smem_limit; else lim.push_back(Limit{dev, kern, smem_limit});
  }
  for (const auto& x : occ)
    if (x.dev == dev && x.f == kern && x.threads == threads && x.smem == smem) { *per_sm = x.per_sm; return cudaSuccess; }
  int n = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, threads, smem);
  if (e != cudaSuccess) return e;
  occ.push_back(Entry{dev, kern, threads, smem, n});
  *per_sm = n;
  return cudaSuccess;
}

// Persistent grid for `units` equal work items and `slots` resident CTAs: the smallest grid that keeps the
// per-CTA iteration count at its minimum, so that every CTA runs the same number of iterations (+-1 unit)
// instead of a few CTAs running one extra.
inline int balanced_grid(long units, long slots) {
  if (units <= 0) return 1;
  if (slots < 1) slots = 1;
  const long iters = (units + slots - 1) / slots;
  return (int)((units + iters - 1) / iters);
}

__host__ __device__ constexpr int pad_k(int K) { return K <= 1 ? 1 : (K <= 2 ? 2 : (K <= 4 ? 4 : 8)); }
__host__ __device__ constexpr int log2_pow2(int v) { return v <= 1 ? 0 : 1 + log2_pow2(v / 2); }

// ---- streaming global memory access (read-once data: do not allocate in L1) ----
template <int VEC> struct Vec;
template <> struct Vec<1> { float v[1]; };
template <> struct __align__(8) Vec<2> { float v[2]; };
template <> struct __align__(16) Vec<4> { float v[4]; };

template <int VEC>
__device__ __forceinline__ Vec<VEC> ld_stream(const float* p) {
  Vec<VEC> r;
  if constexpr (VEC == 4) {
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]) : "l"(p));
  } else if constexpr (VEC == 2) {
    asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(r.v[0]), "=f"(r.v[1]) : "l"(p));
  } else {
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r.v[0]) : "l"(p));
  }
  return r;
}

// cached variant (data that is re-read by neighbouring threads / CTAs: keep it in L1/L2)
template <int VEC>
__device__ __forceinline__ Vec<VEC> ld_cached(const float* p) {
  Vec<VEC> r;
  if constexpr (VEC == 4) {
    float4 t = __ldg(reinterpret_cast<const float4*>(p));
    r.v[0] = t.x; r.v[1] = t.y; r.v[2] = t.z; r.v[3] = t.w;
  } else if constexpr (VEC == 2) {
    float2 t = __ldg(reinterpret_cast<const float2*>(p));
    r.v[0] = t.x; r.v[1] = t.y;
  } else {
    r.v[0] = __ldg(p);
  }
  return r;
}

// the KP weights of one channel in a [C][KP] shared-memory table of the conv kernels (p = its row): vector loads that
// every thread of a warp reads at the same address (broadcast)
template <int KP>
__device__ __forceinline__ void ld_wvec(const float* p, float (&w)[KP]) {
  if constexpr (KP == 4) {
    const float4 t = *reinterpret_cast<const float4*>(p);
    w[0] = t.x; w[1] = t.y; w[2] = t.z; w[3] = t.w;
  } else if constexpr (KP == 8) {
    const float4 t0 = *reinterpret_cast<const float4*>(p);
    const float4 t1 = *reinterpret_cast<const float4*>(p + 4);
    w[0] = t0.x; w[1] = t0.y; w[2] = t0.z; w[3] = t0.w; w[4] = t1.x; w[5] = t1.y; w[6] = t1.z; w[7] = t1.w;
  } else if constexpr (KP == 2) {
    const float2 t = *reinterpret_cast<const float2*>(p);
    w[0] = t.x; w[1] = t.y;
  } else {
    w[0] = p[0];
  }
}

template <int VEC>
__device__ __forceinline__ void st_stream(float* p, const Vec<VEC>& r) {
  if constexpr (VEC == 4) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "f"(r.v[0]), "f"(r.v[1]), "f"(r.v[2]), "f"(r.v[3]) : "memory");
  } else if constexpr (VEC == 2) {
    asm volatile("st.global.L1::no_allocate.v2.f32 [%0], {%1,%2};" :: "l"(p), "f"(r.v[0]), "f"(r.v[1]) : "memory");
  } else {
    asm volatile("st.global.L1::no_allocate.f32 [%0], %1;" :: "l"(p), "f"(r.v[0]) : "memory");
  }
}

// ---- warp / block reductions ----
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Reduce NV (power of two, <= 32) per-lane values across the warp with NV-1 + (5-log2 NV)
// shuffles (recursive halving, then butterfly).  On return every lane holds in v[0] the warp
// total of value index `transposed_index<NV>(lane)`.
template <int NV>
__device__ __forceinline__ void warp_reduce_transposed(float (&v)[NV], int lane) {
  int off = 16;
#pragma unroll
  for (int n = NV; n > 1; n >>= 1) {
    const bool hi = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < n / 2; ++i) {
      const float keep = hi ? v[i + n / 2] : v[i];
      const float send = hi ? v[i] : v[i + n / 2];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
    off >>= 1;
  }
#pragma unroll
  for (; off > 0; off >>= 1) v[0] += __shfl_xor_sync(0xffffffffu, v[0], off);
}
template <int NV>
__device__ __forceinline__ int transposed_index(int lane) {
  // bits of the lane id consumed by the halving steps, most significant first
  constexpr int L = log2_pow2(NV);
  return (lane >> (5 - L)) & (NV - 1);
}
// lanes for which (lane & low_mask) == 0 are the designated writers (one per value index)
template <int NV>
__device__ __forceinline__ bool transposed_writer(int lane) {
  constexpr int L = log2_pow2(NV);
  return (lane & ((1 << (5 - L)) - 1)) == 0;
}

// ---- per-pixel activation math (uniform table fields live in registers) ----
struct LevelInfo {
  int start_mask;  // bit k set: channel k is the first channel of its group
  int parent[RHSEG_KERNEL_MAX_K];
};

// Probability math uses the SFU approximations (ex2.approx / rcp with ~1-2 ulp error): the outputs
// are compared with the reference at 1e-5 relative, three orders of magnitude above that error,
// and the kernels that evaluate them are instruction-bound otherwise.  Anything that decides an
// INTEGER result (argmax of softmax) goes through argmax_softmax_aten() below instead.
__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
// exp / log on the SFU without the denormal fix-up code __expf / __logf carry (4-5 instructions each): the
// probability math only sees exp(x <= 0) -- results below 2^-126 flush to zero -- and log(sum >= 1).
__device__ __forceinline__ float exp_fast(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x * 1.4426950408889634f));
  return r;
}
__device__ __forceinline__ float log_fast(float x) {
  float r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r * 0.6931471805599453f;
}
// 1 / (1 + exp(-z)); exp(-z) overflows to +inf for z < -88.7 and the reciprocal is then 0, as in the exact formula
__device__ __forceinline__ float sigmoidf_ref(float z) { return rcp_approx(1.0f + exp_fast(-z)); }

// x / y for the tiny latency-bound kernels (finalize, parameter gradients): fp32 reciprocal seed + two Newton steps
// in fp64 (~1 ulp) instead of the ~40-instruction IEEE division routine on the critical thread.  y == 0 gives NaN
// (callers treat 0/0 as "invalid", as IEEE does; x/0 with x != 0 does not occur there).
__device__ __forceinline__ double fast_div(double x, double y) {
  double r = (double)__frcp_rn((float)y);
  r = r * (2.0 - y * r);
  r = r * (2.0 - y * r);
  return x * r;
}

// Segmented (per contiguous group) softmax over K channels; groups start where start_mask has a bit.
template <int K>
__device__ __forceinline__ void grouped_softmax(const float (&z)[K], int start_mask, float (&q)[K]) {
  float m[K];
  m[0] = z[0];
#pragma unroll
  for (int k = 1; k < K; ++k) m[k] = ((start_mask >> k) & 1) ? z[k] : fmaxf(m[k - 1], z[k]);
#pragma unroll
  for (int k = K - 2; k >= 0; --k) m[k] = ((start_mask >> (k + 1)) & 1) ? m[k] : m[k + 1];
  float e[K], s[K];
#pragma unroll
  for (int k = 0; k < K; ++k) e[k] = exp_fast(z[k] - m[k]);
  s[0] = e[0];
#pragma unroll
  for (int k = 1; k < K; ++k) s[k] = ((start_mask >> k) & 1) ? e[k] : s[k - 1] + e[k];
#pragma unroll
  for (int k = K - 2; k >= 0; --k) s[k] = ((start_mask >> (k + 1)) & 1) ? s[k] : s[k + 1];
  // one reciprocal per group (computed at the group's first channel, copied forward)
  float r[K];
  r[0] = rcp_approx(s[0]);
#pragma unroll
  for (int k = 1; k < K; ++k) r[k] = ((start_mask >> k) & 1) ? rcp_approx(s[k]) : r[k - 1];
#pragma unroll
  for (int k = 0; k < K; ++k) q[k] = e[k] * r[k];
}

// Per-group sum broadcast back to every member: out[k] = sum_{j in group(k)} x[j].
template <int K>
__device__ __forceinline__ void group_sum(const float (&x)[K], int start_mask, float (&out)[K]) {
  out[0] = x[0];
#pragma unroll
  for (int k = 1; k < K; ++k) out[k] = ((start_mask >> k) & 1) ? x[k] : out[k - 1] + x[k];
#pragma unroll
  for (int k = K - 2; k >= 0; --k) out[k] = ((start_mask >> (k + 1)) & 1) ? out[k] : out[k + 1];
}

// softmax over all K channels, ATen op order (max, sequential sum of expf(z-max), expf/sum)
template <int K>
__device__ __forceinline__ void full_softmax(const float (&z)[K], float (&p)[K], float& mx, float& sum) {
  mx = z[0];
#pragma unroll
  for (int k = 1; k < K; ++k) mx = fmaxf(mx, z[k]);
  sum = 0.f;
#pragma unroll
  for (int k = 0; k < K; ++k) { p[k] = expf(z[k] - mx); sum += p[k]; }
#pragma unroll
  for (int k = 0; k < K; ++k) p[k] = p[k] / sum;
}

// softmax over all K channels with SFU math (statistics / gradients; see the note above)
template <int K>
__device__ __forceinline__ void fast_softmax(const float (&z)[K], float (&p)[K], float& mx, float& sum) {
  mx = z[0];
#pragma unroll
  for (int k = 1; k < K; ++k) mx = fmaxf(mx, z[k]);
  sum = 0.f;
#pragma unroll
  for (int k = 0; k < K; ++k) { p[k] = exp_fast(z[k] - mx); sum += p[k]; }
  const float inv = rcp_approx(sum);
#pragma unroll
  for (int k = 0; k < K; ++k) p[k] *= inv;
}

// torch.argmax semantics: first maximum, NaN counts as the maximum.
__device__ __forceinline__ bool beats(float v, float best) { return (v > best) || (v != v && best == best); }

// torch.argmax(torch.softmax(z, 1), 1) of one pixel, bit-exact with ATen's float kernels.
// softmax is monotone, so the answer is the first maximum of z unless rounding inside softmax
// creates a tie with an EARLIER channel; that needs a logit within ~2.4e-7 of the maximum
// (exp(-d) must round to 1 or 1-ulp).  Only such near-ties (and non-finite inputs) take the slow
// path that replays ATen's arithmetic: max, sequential sum of expf(z-max), IEEE division.
template <int K>
__device__ __noinline__ int argmax_softmax_slow(const float* zp) {
  float z[K], p[K], mx, sum;
#pragma unroll
  for (int k = 0; k < K; ++k) z[k] = zp[k];
  full_softmax<K>(z, p, mx, sum);
  float best = p[0];
  int idx = 0;
#pragma unroll
  for (int k = 1; k < K; ++k)
    if (beats(p[k], best)) { best = p[k]; idx = k; }
  return idx;
}

template <int K>
__device__ __forceinline__ int argmax_softmax_aten(const float (&z)[K]) {
  float best = z[0];
  int idx = 0;
#pragma unroll
  for (int k = 1; k < K; ++k)
    if (z[k] > best) { best = z[k]; idx = k; }
  // second-largest logit (ties with the maximum included): a near-tie is the only way softmax rounding
  // can move the argmax to an earlier channel
  float second = -3.4e38f;
#pragma unroll
  for (int k = 0; k < K; ++k) second = (k != idx) ? fmaxf(second, z[k]) : second;
  const bool slow = !(best - second > 2.0e-6f) || !(fabsf(best) <= 3.0e38f);  // near-tie, inf or NaN
  if (K > 1 && slow) {
    float zl[K];
#pragma unroll
    for (int k = 0; k < K; ++k) zl[k] = z[k];
    idx = argmax_softmax_slow<K>(zl);
  }
  return idx;
}

// ---- per-pixel gradient math shared by the stand-alone and the fused backward kernels ----

// d(g_ce*CE + g_dice*Dice)/dz at one pixel from the closed-form coefficients
//   a_c = A_c m_c t_c ; g_c = (B_c t_c + C_c) m_c ,  m_c = (t_c != -1)
//   logits:  dz_k = (a_k - p_k sum_c a_c) + p_k (g_k - sum_c g_c p_c)      raw:  dz_k = a_k + g_k
template <int K, bool LOGITS>
__device__ __forceinline__ void loss_dz_pixel(const float (&z)[K], const float (&t)[K], const float (&A)[K],
                                              const float (&Bc)[K], const float (&Cc)[K], float (&o)[K]) {
  float a[K], g[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const bool m = t[k] != -1.0f;
    a[k] = m ? A[k] * t[k] : 0.f;
    g[k] = m ? fmaf(Bc[k], t[k], Cc[k]) : 0.f;
  }
  if constexpr (LOGITS) {
    float p[K], mx, sum, sa = 0.f, sgp = 0.f;
    fast_softmax<K>(z, p, mx, sum);
#pragma unroll
    for (int k = 0; k < K; ++k) { sa += a[k]; sgp = fmaf(g[k], p[k], sgp); }
#pragma unroll
    for (int k = 0; k < K; ++k) o[k] = (a[k] - p[k] * sa) + p[k] * (g[k] - sgp);
  } else {
#pragma unroll
    for (int k = 0; k < K; ++k) o[k] = a[k] + g[k];
  }
}

// Activation backward at one pixel: adds the gradient that arrives at the probabilities (dP)
// to dz, and returns dL/dP_parent per channel (same value for all members of a group).
//   sigmoid : dz += dP * P (1 - P)
//   grouped : P_c = P_p * Q_c ; dQ_c = dP_c P_p ; dz += Q (dQ - sum_group dQ Q) ; dP_p = sum_group dP_c Q_c
// (the log(P_p + eps) gate of the reference contributes exactly zero: softmax is shift invariant)
template <int K, int MODE>
__device__ __forceinline__ void act_dz_pixel(const float (&z)[K], const float (&dP)[K], const float (&pp)[K],
                                             int start_mask, float (&dz)[K], float (&dparent)[K]) {
  if constexpr (MODE == RHSEG_ACT_SIGMOID) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const float p = sigmoidf_ref(z[k]);
      dz[k] = fmaf(dP[k], p * (1.0f - p), dz[k]);
      dparent[k] = 0.f;
    }
  } else if constexpr (MODE == RHSEG_ACT_GROUPED) {
    float q[K], dq_q[K], inner[K], dpq[K];
    grouped_softmax<K>(z, start_mask, q);
#pragma unroll
    for (int k = 0; k < K; ++k) {
      dpq[k] = dP[k] * q[k];
      dq_q[k] = dpq[k] * pp[k];
    }
    group_sum<K>(dq_q, start_mask, inner);
    group_sum<K>(dpq, start_mask, dparent);
#pragma unroll
    for (int k = 0; k < K; ++k) dz[k] += dq_q[k] - q[k] * inner[k];
  } else {
#pragma unroll
    for (int k = 0; k < K; ++k) dparent[k] = 0.f;
  }
}

// ATen upsample_bilinear2d (align_corners=True) source index / lambdas for one output index
struct Lerp {
  int i0, i1;
  float l0, l1;
};
__device__ __forceinline__ Lerp make_lerp(int dst, float scale, int in_size) {
  Lerp r;
  const float src = scale * (float)dst;
  r.i0 = (int)src;
  r.i1 = r.i0 + ((r.i0 < in_size - 1) ? 1 : 0);
  r.l1 = src - (float)r.i0;
  r.l0 = 1.0f - r.l1;
  return r;
}
// weight with which output index `dst` reads input index `want`
__device__ __forceinline__ float lerp_weight(int dst, float scale, int in_size, int want) {
  const Lerp l = make_lerp(dst, scale, in_size);
  return (l.i0 == want ? l.l0 : 0.f) + (l.i1 == want ? l.l1 : 0.f);
}
// conservative range [lo, hi] of output indices that read input index i
__device__ __forceinline__ void lerp_support(int i, float scale, int out_size, int& lo, int& hi) {
  if (scale <= 0.f) { lo = 0; hi = out_size - 1; return; }
  lo = max(0, (int)floorf((float)(i - 1) / scale) - 1);
  hi = min(out_size - 1, (int)ceilf((float)(i + 1) / scale) + 1);
}

template <int K>
__device__ __forceinline__ LevelInfo load_level_info(const int32_t* __restrict__ table) {
  LevelInfo li;
  li.start_mask = 0;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    li.parent[k] = table ? table[RHSEG_TBL_PARENT + k] : -1;
    const int g = table ? table[RHSEG_TBL_GROUP_OF + k] : k;
    const int gs = table ? table[RHSEG_TBL_GSTART + g] : k;
    if (gs == k) li.start_mask |= (1 << k);
  }
  return li;
}

}  // namespace rhseg
