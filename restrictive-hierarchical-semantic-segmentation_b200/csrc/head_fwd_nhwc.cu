// Head forward conv for channels-last fp32 features (RHSEG_FEATS_NHWC): the fp32 instances of head_fwd_nhwc.cuh, in a
// translation unit of their own so that they compile in parallel with the others.
#include "head_fwd_nhwc.cuh"

namespace rhseg {

int level_conv_nhwc(const float* feats, const float* eff_w, const float* eff_b, const float* prev_probs,
                    const int32_t* table, int B, int C, int Nf, int K, int K_prev, int act_mode, float* z_lo,
                    bool zlo_zeroed, float* logits, float* probs, double* psum, int w_shared, cudaStream_t st) {
  return level_conv_nhwc_impl<float>(feats, eff_w, eff_b, prev_probs, table, B, C, Nf, K, K_prev, act_mode, z_lo,
                                     zlo_zeroed, logits, probs, psum, w_shared, st);
}

}  // namespace rhseg
