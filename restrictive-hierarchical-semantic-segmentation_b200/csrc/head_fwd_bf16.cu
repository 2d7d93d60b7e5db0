// Head forward conv for bf16 donor features (autocast-trained backbones): the instances of head_fwd_kernel.cuh with
// 16-bit elements, in a translation unit of their own so that they compile in parallel with the fp32 ones.  Every
// feature value is converted to fp32 exactly in registers; weights, sums, logits and probabilities are fp32 as in
// the fp32 path, so the results equal that path's on the upcast features (DESIGN.md 3.7).
#include "head_fwd_kernel.cuh"

namespace rhseg {

// Ring shapes for 2-byte elements (DESIGN.md 3.7): the fp32 shapes would halve every row copy; these keep the
// scalar-row copies at 1 KB (T = 512 px) and the vector-row copies at 2 KB.
using FwdCfgV4Bf16 = FwdCfgV4;   // T = 1024 px, 2 KB row copies, 8 channels per stage
using FwdCfgS1Bf16 = FwdCfgS1;   // with J = 4: T = 512 px, 1 KB row copies
constexpr int FWD_S1_J_BF16 = 4;

template <int K, int MODE>
static int fwd_fullres_bf16(const uint16_t* feats, const float* eff_w, const float* eff_b, const float* prev_probs,
                            const int32_t* table, int B, int C, int N, int K_prev, float* logits, float* probs,
                            double* psum, cudaStream_t st, int w_shared) {
  const bool v4 = rows_vec4(feats, N) && rows_vec4(logits, N) && rows_vec4(probs, N) && (!prev_probs || rows_vec4(prev_probs, N));
  if (v4)
    return launch_fwd<uint16_t, K, 4, 1, MODE, FwdCfgV4Bf16>(feats, eff_w, eff_b, prev_probs, table, B, C, N, K_prev, logits, probs, psum, st, false, w_shared);
  return launch_fwd<uint16_t, K, 1, FWD_S1_J_BF16, MODE, FwdCfgS1Bf16>(feats, eff_w, eff_b, prev_probs, table, B, C, N, K_prev, logits, probs, psum, st, false, w_shared);
}

int level_conv_bf16(const uint16_t* feats, const float* eff_w, const float* eff_b, const float* prev_probs,
                    const int32_t* table, int B, int C, int Nf, int K, int K_prev, int act_mode, float* z_lo,
                    bool zlo_zeroed, float* logits, float* probs, double* psum, int w_shared, cudaStream_t st) {
  if (z_lo == nullptr) {
    RHSEG_DISPATCH_K(K, {
      if (act_mode == RHSEG_ACT_SIGMOID)
        return fwd_fullres_bf16<KK, RHSEG_ACT_SIGMOID>(feats, eff_w, eff_b, prev_probs, table, B, C, Nf, K_prev, logits, probs, psum, st, w_shared);
      if (act_mode == RHSEG_ACT_GROUPED)
        return fwd_fullres_bf16<KK, RHSEG_ACT_GROUPED>(feats, eff_w, eff_b, prev_probs, table, B, C, Nf, K_prev, logits, probs, psum, st, w_shared);
      return fwd_fullres_bf16<KK, RHSEG_ACT_ZEROS>(feats, eff_w, eff_b, prev_probs, table, B, C, Nf, K_prev, logits, probs, psum, st, w_shared);
    });
  }
  RHSEG_DISPATCH_K(K, {
    if (rows_vec4(feats, Nf) && rows_vec4(z_lo, Nf))
      return launch_fwd<uint16_t, KK, 4, 1, MODE_CONV_ONLY, FwdCfgV4Bf16>(feats, eff_w, eff_b, nullptr, nullptr, B, C, Nf, K_prev, z_lo, nullptr, nullptr, st, zlo_zeroed, w_shared);
    return launch_fwd<uint16_t, KK, 1, FWD_S1_J_BF16, MODE_CONV_ONLY, FwdCfgS1Bf16>(feats, eff_w, eff_b, nullptr, nullptr, B, C, Nf, K_prev, z_lo, nullptr, nullptr, st, zlo_zeroed, w_shared);
  });
  return RHSEG_OK;
}

}  // namespace rhseg
