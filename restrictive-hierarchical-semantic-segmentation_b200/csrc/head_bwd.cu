// Head backward: activation backward (composition / restrictive softmax / sigmoid), adjoint
// of the align_corners bilinear upsample, 1x1-conv backward (dfeats + fp64 weight-gradient
// sums) and the tiny parameter-gradient kernel (head conv, FiLM linear, uniform gradient to
// the previous level's pooled probabilities).  The reference obtains all of this from
// autograd over Models/models.py:58-77 and :263-306 / :757-802; closed forms in DESIGN.md.
#include <algorithm>
#include <cstdlib>
#include "conv_bwd_kernel.cuh"

namespace rhseg {

// the fp32 instances of the NCHW conv backward compile here, the bf16 ones in head_bwd_bf16.cu
template int conv_bwd_nchw<float>(int, const float*, const float*, const float*, int, int, int, float*, double*, double*, int,
                                  cudaStream_t, int, const ParamTail&);
extern template int conv_bwd_nchw<uint16_t>(int, const uint16_t*, const float*, const float*, int, int, int, uint16_t*, double*,
                                            double*, int, cudaStream_t, int, const ParamTail&);

// ------------------------------------------------------------------------------------
// activation backward, output resolution, elementwise
// ------------------------------------------------------------------------------------
template <int K, int VEC, int MODE, int THREADS>
__global__ void __launch_bounds__(THREADS)
act_bwd_kernel(const float* __restrict__ logits, const float* __restrict__ prev_probs,
               const int32_t* __restrict__ table, const float* __restrict__ dz_in,
               const double* __restrict__ g_uniform, float inv_npix, const float* __restrict__ dp_pix,
               uint32_t pix_mask, int K_prev, long N, float* __restrict__ dz_out, float* __restrict__ dp_prev) {
  pdl_wait();
  const int b = blockIdx.y;
  const long px = ((long)blockIdx.x * THREADS + threadIdx.x) * VEC;
  if (px >= N) return;
  const LevelInfo li = load_level_info<K>(MODE == RHSEG_ACT_GROUPED ? table : nullptr);
  const size_t base = (size_t)b * K * N + px;

  float z[K][VEC], dP[K][VEC], dz[K][VEC];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const Vec<VEC> t = ld_stream<VEC>(logits + base + (size_t)k * N);
    const float gu = g_uniform ? (float)(g_uniform[b * K + k]) * inv_npix : 0.f;
    Vec<VEC> d, e;
#pragma unroll
    for (int v = 0; v < VEC; ++v) { d.v[v] = 0.f; e.v[v] = 0.f; }
    if (dz_in) d = ld_stream<VEC>(dz_in + base + (size_t)k * N);
    if (dp_pix && ((pix_mask >> k) & 1u)) e = ld_stream<VEC>(dp_pix + base + (size_t)k * N);
#pragma unroll
    for (int v = 0; v < VEC; ++v) { z[k][v] = t.v[v]; dz[k][v] = d.v[v]; dP[k][v] = gu + e.v[v]; }
  }

  float pp[K][VEC], dpar[K][VEC];
  if constexpr (MODE == RHSEG_ACT_GROUPED) {
    const float* pb = prev_probs + (size_t)b * K_prev * N + px;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      if ((li.start_mask >> k) & 1) {
        const Vec<VEC> t = ld_stream<VEC>(pb + (size_t)li.parent[k] * N);
#pragma unroll
        for (int v = 0; v < VEC; ++v) pp[k][v] = t.v[v];
      } else {
#pragma unroll
        for (int v = 0; v < VEC; ++v) pp[k][v] = pp[k > 0 ? k - 1 : 0][v];
      }
    }
  }
#pragma unroll
  for (int v = 0; v < VEC; ++v) {
    float zz[K], dPv[K], ppv[K], dzv[K], dparv[K];
#pragma unroll
    for (int k = 0; k < K; ++k) { zz[k] = z[k][v]; dPv[k] = dP[k][v]; ppv[k] = pp[k][v]; dzv[k] = dz[k][v]; }
    act_dz_pixel<K, MODE>(zz, dPv, ppv, li.start_mask, dzv, dparv);
#pragma unroll
    for (int k = 0; k < K; ++k) { dz[k][v] = dzv[k]; dpar[k][v] = dparv[k]; }
  }
  if constexpr (MODE == RHSEG_ACT_GROUPED) {
    if (dp_prev) {
      float* dpb = dp_prev + (size_t)b * K_prev * N + px;
#pragma unroll
      for (int k = 0; k < K; ++k)
        if ((li.start_mask >> k) & 1) {
          float* dst = dpb + (size_t)li.parent[k] * N;
          Vec<VEC> cur = *reinterpret_cast<const Vec<VEC>*>(dst);
#pragma unroll
          for (int v = 0; v < VEC; ++v) cur.v[v] += dpar[k][v];
          *reinterpret_cast<Vec<VEC>*>(dst) = cur;
        }
    }
  }
#pragma unroll
  for (int k = 0; k < K; ++k) {
    Vec<VEC> o;
#pragma unroll
    for (int v = 0; v < VEC; ++v) o.v[v] = dz[k][v];
    *reinterpret_cast<Vec<VEC>*>(dz_out + base + (size_t)k * N) = o;
  }
}

// ------------------------------------------------------------------------------------
// parameter gradients (tiny): one thread per feature channel
// ------------------------------------------------------------------------------------
// Thread (cl, bl): channel blockIdx.x*PG_CH + cl, samples b = bl, bl+PG_BL, ...  All global loads of a
// thread are independent (one sample per thread when B <= PG_BL), the sums over samples and over
// channels go through shared memory.
constexpr int PG_CH = 64, PG_BL = 4, PG_THREADS = PG_CH * PG_BL;

__global__ void __launch_bounds__(PG_THREADS)
param_grads_kernel(const double* __restrict__ S, const double* __restrict__ s, const float* __restrict__ head_w,
                   const float* __restrict__ film_w, const float* __restrict__ gamma_beta,
                   const double* __restrict__ prev_psum, double n_pix, int B, int C, int K, int K_prev,
                   float* __restrict__ d_head_w, float* __restrict__ d_head_b, float* __restrict__ d_film_w,
                   float* __restrict__ d_film_b, double* __restrict__ g_prev) {
  pdl_wait();
  constexpr int NV = RHSEG_KERNEL_MAX_K + 2 + 2 * RHSEG_MAX_K;  // dw[k], dfb_g, dfb_b, dfw_g[j], dfw_b[j]
  __shared__ float red[PG_BL][PG_CH][NV + 1];
  __shared__ float gsm[PG_THREADS / 32][RHSEG_MAX_K];
  const int cl = threadIdx.x % PG_CH, bl = threadIdx.x / PG_CH;
  const int c = blockIdx.x * PG_CH + cl;
  const bool ok = c < C;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (blockIdx.x == 0 && threadIdx.x < K) {
    double acc = 0.0;
    for (int b = 0; b < B; ++b) acc += s[b * K + threadIdx.x];
    d_head_b[threadIdx.x] = (float)acc;
  }
  float w[RHSEG_KERNEL_MAX_K], fwg[RHSEG_MAX_K], fwb[RHSEG_MAX_K];
#pragma unroll
  for (int k = 0; k < RHSEG_KERNEL_MAX_K; ++k) w[k] = (ok && k < K) ? head_w[(size_t)k * C + c] : 0.f;
#pragma unroll
  for (int j = 0; j < RHSEG_MAX_K; ++j) {
    fwg[j] = (ok && film_w && j < K_prev) ? film_w[(size_t)c * K_prev + j] : 0.f;
    fwb[j] = (ok && film_w && j < K_prev) ? film_w[(size_t)(C + c) * K_prev + j] : 0.f;
  }
  float acc[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) acc[i] = 0.f;
  for (int b = bl; b < ((B + PG_BL - 1) / PG_BL) * PG_BL; b += PG_BL) {  // uniform trip count for the block reductions
    const bool live = ok && b < B;
    double dgam = 0.0, dbet = 0.0;
    if (live) {
      const double gam = film_w ? (double)gamma_beta[(size_t)b * 2 * C + c] : 1.0;
      const double bet = film_w ? (double)gamma_beta[(size_t)b * 2 * C + C + c] : 0.0;
#pragma unroll
      for (int k = 0; k < RHSEG_KERNEL_MAX_K; ++k)
        if (k < K) {
          const double Sv = S[((size_t)b * K + k) * C + c], sv = s[b * K + k];
          acc[k] += (float)(Sv * gam + sv * bet);
          dgam += Sv * (double)w[k];
          dbet += (double)w[k] * sv;
        }
    }
    if (film_w) {
      acc[RHSEG_KERNEL_MAX_K] += (float)dgam;
      acc[RHSEG_KERNEL_MAX_K + 1] += (float)dbet;
      for (int j = 0; j < K_prev; ++j) {
        const double cond = b < B ? (double)(float)fast_div(prev_psum[b * K_prev + j], n_pix) : 0.0;
        acc[RHSEG_KERNEL_MAX_K + 2 + j] += (float)(dgam * cond);
        acc[RHSEG_KERNEL_MAX_K + 2 + RHSEG_MAX_K + j] += (float)(dbet * cond);
        // g_prev[b][j] = sum over channels of film_w^T [dgamma|dbeta]: warp sums now, one block step below
        const float contrib = warp_sum((float)((double)fwg[j] * dgam + (double)fwb[j] * dbet));
        if (lane == 0) gsm[warp][j] = contrib;
      }
      __syncthreads();
      if (cl < K_prev && b < B) {  // thread (cl = j, bl): the PG_CH/32 warps that share this sample slot
        double tsum = 0.0;
        for (int q = 0; q < PG_CH / 32; ++q) tsum += (double)gsm[bl * (PG_CH / 32) + q][cl];
        atomicAdd(&g_prev[b * K_prev + cl], tsum);
      }
      __syncthreads();
    }
  }
#pragma unroll
  for (int i = 0; i < NV; ++i) red[bl][cl][i] = acc[i];
  __syncthreads();
  if (bl != 0 || !ok) return;
  float tot[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    tot[i] = 0.f;
#pragma unroll
    for (int q = 0; q < PG_BL; ++q) tot[i] += red[q][cl][i];
  }
#pragma unroll
  for (int k = 0; k < RHSEG_KERNEL_MAX_K; ++k)
    if (k < K) d_head_w[(size_t)k * C + c] = tot[k];
  if (film_w) {
    d_film_b[c] = tot[RHSEG_KERNEL_MAX_K];
    d_film_b[C + c] = tot[RHSEG_KERNEL_MAX_K + 1];
#pragma unroll
    for (int j = 0; j < RHSEG_MAX_K; ++j)
      if (j < K_prev) {
        d_film_w[(size_t)c * K_prev + j] = tot[RHSEG_KERNEL_MAX_K + 2 + j];
        d_film_w[(size_t)(C + c) * K_prev + j] = tot[RHSEG_KERNEL_MAX_K + 2 + RHSEG_MAX_K + j];
      }
  }
}

}  // namespace rhseg

using namespace rhseg;

extern "C" int rhseg_head_act_bwd(const float* logits, const float* prev_probs, const int32_t* table,
                                  const float* dz_in, const double* g_uniform, double inv_npix,
                                  const float* dp_pix, uint32_t pix_mask, int B, int K, int K_prev, int H, int W,
                                  int act_mode, float* dz_out, float* dp_prev, void* stream) {
  if (!logits || !dz_out || B <= 0 || H <= 0 || W <= 0) return RHSEG_ERR_ARG;
  if (K < 1 || K > RHSEG_KERNEL_MAX_K) return RHSEG_ERR_UNSUPPORTED;
  if (act_mode == RHSEG_ACT_GROUPED && (!prev_probs || !table)) return RHSEG_ERR_ARG;
  if (dz_out == dz_in) return RHSEG_ERR_ARG;
  const long N = (long)H * W;
  cudaStream_t st = (cudaStream_t)stream;
  constexpr int THREADS = 256;
  const float inv = (float)inv_npix;
  RHSEG_DISPATCH_K(K, {
    if (N % 4 == 0) {
      dim3 grid((unsigned)((N / 4 + THREADS - 1) / THREADS), B);
      if (act_mode == RHSEG_ACT_SIGMOID)
        launch_pdl(act_bwd_kernel<KK, 4, RHSEG_ACT_SIGMOID, THREADS>, dim3(grid), dim3(THREADS), 0, st, logits, prev_probs, table, dz_in, g_uniform, inv, dp_pix, pix_mask, K_prev, N, dz_out, dp_prev);
      else if (act_mode == RHSEG_ACT_GROUPED)
        launch_pdl(act_bwd_kernel<KK, 4, RHSEG_ACT_GROUPED, THREADS>, dim3(grid), dim3(THREADS), 0, st, logits, prev_probs, table, dz_in, g_uniform, inv, dp_pix, pix_mask, K_prev, N, dz_out, dp_prev);
      else
        launch_pdl(act_bwd_kernel<KK, 4, RHSEG_ACT_ZEROS, THREADS>, dim3(grid), dim3(THREADS), 0, st, logits, prev_probs, table, dz_in, g_uniform, inv, dp_pix, pix_mask, K_prev, N, dz_out, dp_prev);
    } else {
      dim3 grid((unsigned)((N + THREADS - 1) / THREADS), B);
      if (act_mode == RHSEG_ACT_SIGMOID)
        launch_pdl(act_bwd_kernel<KK, 1, RHSEG_ACT_SIGMOID, THREADS>, dim3(grid), dim3(THREADS), 0, st, logits, prev_probs, table, dz_in, g_uniform, inv, dp_pix, pix_mask, K_prev, N, dz_out, dp_prev);
      else if (act_mode == RHSEG_ACT_GROUPED)
        launch_pdl(act_bwd_kernel<KK, 1, RHSEG_ACT_GROUPED, THREADS>, dim3(grid), dim3(THREADS), 0, st, logits, prev_probs, table, dz_in, g_uniform, inv, dp_pix, pix_mask, K_prev, N, dz_out, dp_prev);
      else
        launch_pdl(act_bwd_kernel<KK, 1, RHSEG_ACT_ZEROS, THREADS>, dim3(grid), dim3(THREADS), 0, st, logits, prev_probs, table, dz_in, g_uniform, inv, dp_pix, pix_mask, K_prev, N, dz_out, dp_prev);
    }
  });
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}

static int conv_bwd_impl(const void* feats_v, const float* dz, const float* eff_w, int B, int C, int K, int n_pix,
                         void* dfeats_v, double* S, double* s, int zero_sums, void* stream, const ParamTail& pt) {
  if (!feats_v || !dz || !eff_w || !S || !s || B <= 0 || C <= 0 || n_pix <= 0) return RHSEG_ERR_ARG;
  if (K < 1 || K > RHSEG_KERNEL_MAX_K) return RHSEG_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  const int w_shared = (zero_sums & 2) ? 1 : 0;
  if (zero_sums & 1) {
    RHSEG_CUDA(cudaMemsetAsync(S, 0, sizeof(double) * (size_t)B * K * C, st));
    RHSEG_CUDA(cudaMemsetAsync(s, 0, sizeof(double) * (size_t)B * K, st));
  }
  const bool nhwc = (zero_sums & RHSEG_FEATS_NHWC) != 0, bf16 = (zero_sums & RHSEG_FEATS_BF16) != 0;
  const uintptr_t addr = reinterpret_cast<uintptr_t>(feats_v) | reinterpret_cast<uintptr_t>(dfeats_v);
  if (nhwc) {
    if (((size_t)C * (bf16 ? 2 : 4)) % 16 != 0 || (addr & 15u) != 0) return RHSEG_ERR_UNSUPPORTED;
  } else if (bf16 && (addr & 1u)) {
    return RHSEG_ERR_ARG;
  }
  const int sms = device_sm_count();
  auto conv = [&](auto feats, auto dfeats) {
    return nhwc ? conv_bwd_nhwc(K, feats, dz, eff_w, B, C, n_pix, dfeats, S, s, sms, st, w_shared, pt)
                : conv_bwd_nchw(K, feats, dz, eff_w, B, C, n_pix, dfeats, S, s, sms, st, w_shared, pt);
  };
  return bf16 ? conv(static_cast<const uint16_t*>(feats_v), static_cast<uint16_t*>(dfeats_v))
              : conv(static_cast<const float*>(feats_v), static_cast<float*>(dfeats_v));
}

extern "C" int rhseg_head_conv_bwd(const void* feats, const float* dz, const float* eff_w, int B, int C, int K,
                                   int n_pix, void* dfeats, double* S, double* s, int zero_sums, void* stream) {
  return conv_bwd_impl(feats, dz, eff_w, B, C, K, n_pix, dfeats, S, s, zero_sums, stream, ParamTail{});
}

extern "C" int rhseg_head_conv_bwd_params(const void* feats, const float* dz, const float* eff_w, int B, int C, int K,
                                          int n_pix, void* dfeats, double* S, double* s, int flags, const float* head_w,
                                          const float* film_w, const float* gamma_beta, const double* prev_psum,
                                          double n_pix_out, int K_prev, float* d_head_w, float* d_head_b, float* d_film_w,
                                          float* d_film_b, double* g_prev, unsigned* ticket, void* stream) {
  if (!head_w || !d_head_w || !d_head_b || !ticket) return RHSEG_ERR_ARG;
  if (film_w) {
    if (!gamma_beta || !prev_psum || !d_film_w || !d_film_b || !g_prev || n_pix_out <= 0) return RHSEG_ERR_ARG;
    if (K_prev < 1 || K_prev > RHSEG_MAX_K) return RHSEG_ERR_UNSUPPORTED;
  }
  // level 0 of a narrow donor: the batch sums are formed by the conv kernel's last CTA.  Measured: UNet (K*C*B = 1024 sums)
  // 0.5507 vs 0.5538 ms per step with the separate kernel; HRNet-W48 (11520 sums through one CTA) 0.4207 vs 0.4166 -> kept
  // for small heads only.
  if (!film_w && (long)K * C * B <= 4096 && !getenv("RHSEG_NO_L0_TAIL"))
    return conv_bwd_impl(feats, dz, eff_w, B, C, K, n_pix, dfeats, S, s, flags, stream, ParamTail{ticket, B, d_head_w, d_head_b});
  const int rc = conv_bwd_impl(feats, dz, eff_w, B, C, K, n_pix, dfeats, S, s, flags, stream, ParamTail{});
  if (rc != RHSEG_OK) return rc;
  // g_prev: the caller's buffer is zero on entry when bit 2 (value 4) of flags is set (part of a larger zero fill)
  return rhseg_head_param_grads(S, s, head_w, film_w, gamma_beta, prev_psum, n_pix_out, B, C, K, K_prev, d_head_w, d_head_b,
                                d_film_w, d_film_b, g_prev, (flags & 4) ? 1 : 0, stream);
}

extern "C" int rhseg_head_param_grads(const double* S, const double* s, const float* head_w, const float* film_w,
                                      const float* gamma_beta, const double* prev_psum, double n_pix, int B, int C,
                                      int K, int K_prev, float* d_head_w, float* d_head_b, float* d_film_w,
                                      float* d_film_b, double* g_prev, int g_prev_zeroed, void* stream) {
  if (!S || !s || !head_w || !d_head_w || !d_head_b || B <= 0 || C <= 0) return RHSEG_ERR_ARG;
  if (K < 1 || K > RHSEG_KERNEL_MAX_K) return RHSEG_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  if (film_w) {
    if (!gamma_beta || !prev_psum || !d_film_w || !d_film_b || !g_prev || n_pix <= 0) return RHSEG_ERR_ARG;
    if (K_prev < 1 || K_prev > RHSEG_MAX_K) return RHSEG_ERR_UNSUPPORTED;
    if (!g_prev_zeroed) RHSEG_CUDA(cudaMemsetAsync(g_prev, 0, sizeof(double) * (size_t)B * K_prev, st));
  }
  launch_pdl(param_grads_kernel, dim3((C + PG_CH - 1) / PG_CH), dim3(PG_THREADS), 0, st, S, s, head_w, film_w, gamma_beta, prev_psum, n_pix, B, C, K, K_prev,
                                                      d_head_w, d_head_b, d_film_w, d_film_b, g_prev);
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}
