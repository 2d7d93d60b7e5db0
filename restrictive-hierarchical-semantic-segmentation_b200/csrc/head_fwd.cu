// Head forward: FiLM fold, fused 1x1 conv + activation (full-resolution donors, UNet), and the
// low-resolution conv of upsampled heads (HRNet; the hi-res pass lives in head_up.cu).
// Reference semantics: Models/models.py:58-77 (FiLM), :177-184/:268/:280 (1x1 heads),
// :269/:288-302 (sigmoid, restrictive softmax, composition, concat), :766/:776 (upsample).
#include "head_fwd_kernel.cuh"

namespace rhseg {

// ------------------------------------------------------------------------------------
// FiLM fold (tiny): one CTA per sample.
// ------------------------------------------------------------------------------------
__global__ void film_fold_kernel(const float* __restrict__ head_w, const float* __restrict__ head_b,
                                 const float* __restrict__ film_w, const float* __restrict__ film_b,
                                 const double* __restrict__ prev_psum, double n_pix, int C, int K, int K_prev,
                                 float* __restrict__ gamma_beta, float* __restrict__ eff_w,
                                 float* __restrict__ eff_b) {
  pdl_wait();
  extern __shared__ float sm[];  // cond[K_prev] | beta-dot partials[K * nwarps]
  const int b = blockIdx.x, tid = threadIdx.x, nthr = blockDim.x;
  float* cond = sm;
  float* part = sm + RHSEG_MAX_K;
  if (film_w == nullptr) {
    for (int i = tid; i < K * C; i += nthr) eff_w[(size_t)b * K * C + i] = head_w[i];
    for (int k = tid; k < K; k += nthr) eff_b[b * K + k] = head_b[k];
    return;
  }
  if (tid < K_prev) cond[tid] = (float)fast_div(prev_psum[b * K_prev + tid], n_pix);  // AdaptiveAvgPool2d(1)
  __syncthreads();
  float bdot[RHSEG_KERNEL_MAX_K];
#pragma unroll
  for (int k = 0; k < RHSEG_KERNEL_MAX_K; ++k) bdot[k] = 0.f;
  for (int c = tid; c < C; c += nthr) {
    float g = film_b[c], be = film_b[C + c];
    for (int j = 0; j < K_prev; ++j) {  // Linear(K_prev, 2C): same accumulation order as a dot product
      g = fmaf(film_w[(size_t)c * K_prev + j], cond[j], g);
      be = fmaf(film_w[(size_t)(C + c) * K_prev + j], cond[j], be);
    }
    gamma_beta[(size_t)b * 2 * C + c] = g;
    gamma_beta[(size_t)b * 2 * C + C + c] = be;
#pragma unroll
    for (int k = 0; k < RHSEG_KERNEL_MAX_K; ++k)
      if (k < K) {
        const float w = head_w[(size_t)k * C + c];
        eff_w[((size_t)b * K + k) * C + c] = w * g;
        bdot[k] = fmaf(w, be, bdot[k]);
      }
  }
  const int lane = tid & 31, warp = tid >> 5, nwarp = nthr >> 5;
#pragma unroll
  for (int k = 0; k < RHSEG_KERNEL_MAX_K; ++k) {
    const float v = warp_sum(bdot[k]);
    if (lane == 0 && k < K) part[k * nwarp + warp] = v;
  }
  __syncthreads();
  if (tid < K) {
    float acc = head_b[tid];
    for (int w = 0; w < nwarp; ++w) acc += part[tid * nwarp + w];
    eff_b[b * K + tid] = acc;
  }
}

// the fp32 instances of the NCHW feature conv compile here, the bf16 ones in head_fwd_bf16.cu
template int level_conv_nchw<float>(const float*, const float*, const float*, const float*, const int32_t*, int, int, int,
                                    int, int, int, float*, bool, float*, float*, double*, int, cudaStream_t);
extern template int level_conv_nchw<uint16_t>(const uint16_t*, const float*, const float*, const float*, const int32_t*,
                                              int, int, int, int, int, int, float*, bool, float*, float*, double*, int,
                                              cudaStream_t);

}  // namespace rhseg

using namespace rhseg;

extern "C" int rhseg_film_fold(const float* head_w, const float* head_b, const float* film_w, const float* film_b,
                               const double* prev_psum, double n_pix, int B, int C, int K, int K_prev,
                               float* gamma_beta, float* eff_w, float* eff_b, void* stream) {
  if (!head_w || !head_b || !eff_w || !eff_b || B <= 0 || C <= 0) return RHSEG_ERR_ARG;
  if (K < 1 || K > RHSEG_KERNEL_MAX_K) return RHSEG_ERR_UNSUPPORTED;
  if (film_w) {
    if (!film_b || !prev_psum || !gamma_beta || n_pix <= 0) return RHSEG_ERR_ARG;
    if (K_prev < 1 || K_prev > RHSEG_MAX_K) return RHSEG_ERR_UNSUPPORTED;
  }
  const int threads = C >= 512 ? 768 : 256;
  const size_t smem = (RHSEG_MAX_K + RHSEG_KERNEL_MAX_K * (threads / 32)) * sizeof(float);
  launch_pdl(film_fold_kernel, dim3(B), dim3(threads), smem, (cudaStream_t)stream, head_w, head_b, film_w, film_b, prev_psum, n_pix, C, K,
                                                             K_prev, gamma_beta, eff_w, eff_b);
  RHSEG_LAUNCH_CHECK();
  return RHSEG_OK;
}

static int level_fwd_impl(const void* feats_v, const float* eff_w, const float* eff_b,
                          const float* prev_probs, const int32_t* table, int B, int C, int Hf, int Wf,
                          int H, int W, int K, int K_prev, int act_arg, float* z_lo, float* logits,
                          float* probs, double* psum, int zero_psum, void* stream, const EvalArgs* ea, bool* need_eval) {
  const int act_mode = act_arg & 0xff;
  if (need_eval) *need_eval = false;
  if (!feats_v || !eff_w || !eff_b || !logits || !probs || !psum) return RHSEG_ERR_ARG;
  if (B <= 0 || C <= 0 || Hf <= 0 || Wf <= 0 || H <= 0 || W <= 0) return RHSEG_ERR_ARG;
  if (K < 1 || K > RHSEG_KERNEL_MAX_K) return RHSEG_ERR_UNSUPPORTED;
  if (act_mode == RHSEG_ACT_GROUPED && (!prev_probs || !table || K_prev < 1)) return RHSEG_ERR_ARG;
  if (act_mode < 0 || act_mode > RHSEG_ACT_ZEROS) return RHSEG_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  if (zero_psum & 1) RHSEG_CUDA(cudaMemsetAsync(psum, 0, sizeof(double) * B * K, st));
  const bool zlo_zeroed = (zero_psum & 2) != 0;
  const int w_shared = (zero_psum & 4) ? 1 : 0;
  const bool up = (H != Hf) || (W != Wf);
  if (ea && !up) return RHSEG_ERR_UNSUPPORTED;
  if (act_mode == RHSEG_ACT_GROUPED && table == nullptr) return RHSEG_ERR_ARG;
  const int Nf = Hf * Wf;
  const bool nhwc = (zero_psum & RHSEG_FEATS_NHWC) != 0, bf16 = (zero_psum & RHSEG_FEATS_BF16) != 0;
  if (nhwc) {
    if (((size_t)C * (bf16 ? 2 : 4)) % 16 != 0 || (reinterpret_cast<uintptr_t>(feats_v) & 15u) != 0) return RHSEG_ERR_UNSUPPORTED;
  } else if (bf16 && (reinterpret_cast<uintptr_t>(feats_v) & 1u)) {
    return RHSEG_ERR_ARG;
  }
  if (up && !z_lo) return RHSEG_ERR_ARG;
  float* conv_out = up ? z_lo : nullptr;  // the feature conv of an upsampled head writes z_lo
  auto conv = [&](auto feats) {
    return nhwc ? level_conv_nhwc(feats, eff_w, eff_b, prev_probs, table, B, C, Nf, K, K_prev, act_mode, conv_out, zlo_zeroed,
                                  logits, probs, psum, w_shared, st)
                : level_conv_nchw(feats, eff_w, eff_b, prev_probs, table, B, C, Nf, K, K_prev, act_mode, conv_out, zlo_zeroed,
                                  logits, probs, psum, w_shared, st);
  };
  int rc = bf16 ? conv(static_cast<const uint16_t*>(feats_v)) : conv(static_cast<const float*>(feats_v));
  if (rc != RHSEG_OK || !up) return rc;
  bool ne = false;
  rc = fwd_upsampled_dispatch(K, act_arg, z_lo, prev_probs, table, B, Hf, Wf, H, W, K_prev, logits, probs, psum, st, ea, &ne);
  if (need_eval) *need_eval = ne;
  return rc;
}

extern "C" int rhseg_head_level_fwd(const void* feats, const float* eff_w, const float* eff_b,
                                    const float* prev_probs, const int32_t* table, int B, int C, int Hf, int Wf,
                                    int H, int W, int K, int K_prev, int act_mode, float* z_lo, float* logits,
                                    float* probs, double* psum, int zero_psum, void* stream) {
  return level_fwd_impl(feats, eff_w, eff_b, prev_probs, table, B, C, Hf, Wf, H, W, K, K_prev, act_mode, z_lo, logits, probs,
                        psum, zero_psum, stream, nullptr, nullptr);
}

extern "C" int rhseg_head_level_fwd_eval(const void* feats, const float* eff_w, const float* eff_b,
                                         const float* prev_probs, const int32_t* table, int B, int C, int Hf, int Wf,
                                         int H, int W, int K, int K_prev, int act_mode, float* z_lo, float* logits,
                                         float* probs, double* psum, const float* targets, long t_bstride,
                                         long t_cstride, const float* parent_targets, long pt_bstride, long pt_cstride,
                                         const unsigned char* prev_idx, void* out_words, unsigned char* idx_out,
                                         int flags, void* stream) {
  if (!targets || !out_words) return RHSEG_ERR_ARG;
  if (K < 1 || K > RHSEG_KERNEL_MAX_K) return RHSEG_ERR_UNSUPPORTED;
  const int child = (act_mode & 0xff) == RHSEG_ACT_SIGMOID ? 0 : 1;
  const int nc = child ? K + 1 : K;
  const size_t words = (size_t)B * K * RHSEG_NSTAT + RHSEG_MAX_K + (size_t)nc * nc;
  if (!(flags & RHSEG_EVAL_PREZEROED)) RHSEG_CUDA(cudaMemsetAsync(out_words, 0, words * 8, (cudaStream_t)stream));
  double* stats = reinterpret_cast<double*>(out_words);
  double* cons = stats + (size_t)B * K * RHSEG_NSTAT;
  const bool composed = (flags & RHSEG_EVAL_COMPOSED) != 0;
  if (composed) parent_targets = nullptr, prev_idx = nullptr, idx_out = nullptr;
  EvalArgs ea{targets, t_bstride, t_cstride, parent_targets, pt_bstride, pt_cstride, prev_idx, child, stats, cons,
              reinterpret_cast<unsigned long long*>(cons + RHSEG_MAX_K), idx_out, composed ? 1 : 0};
  bool need_eval = false;
  const int rc = level_fwd_impl(feats, eff_w, eff_b, prev_probs, table, B, C, Hf, Wf, H, W, K, K_prev, act_mode, z_lo, logits,
                                probs, psum, (flags & (2 | 4 | RHSEG_FEATS_BF16 | RHSEG_FEATS_NHWC)), stream, &ea, &need_eval);
  if (rc != RHSEG_OK || !need_eval) return rc;
  // shapes the band kernel does not take: the evaluation runs as its own kernel on the finished logits
  if (composed)
    return rhseg_level_eval_composed(logits, probs, child ? prev_probs : nullptr, targets, t_bstride, t_cstride, table, B, K,
                                     K_prev, H * W, child | RHSEG_GROUP_HINT(RHSEG_GROUP_HINT_OF(act_mode)), out_words,
                                     RHSEG_EVAL_PREZEROED, stream);
  return rhseg_level_eval(logits, targets, t_bstride, t_cstride, parent_targets, pt_bstride, pt_cstride, prev_idx, table, B, K,
                          H * W, child | RHSEG_GROUP_HINT(RHSEG_GROUP_HINT_OF(act_mode)), out_words, idx_out,
                          RHSEG_EVAL_PREZEROED, stream);
}
