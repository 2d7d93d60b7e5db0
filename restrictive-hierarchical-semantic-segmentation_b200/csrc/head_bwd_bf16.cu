// Conv backward for bf16 donor features (autocast-trained backbones): the instances of conv_bwd_kernel.cuh with 16-bit
// elements, in a translation unit of their own so that they compile in parallel with the fp32 ones.  Features are
// converted to fp32 exactly, S / s accumulate as in the fp32 path, and dfeats is formed in fp32 and rounded to bf16
// (nearest even) once, when it is stored (DESIGN.md 3.7).
#include "conv_bwd_kernel.cuh"

namespace rhseg {

// Ring shapes for 2-byte elements (DESIGN.md 3.7).  Vector rows: T = 1024 px, 2 KB row copies.  Scalar rows (odd
// planes): T = 1024 px (J = 4 for K <= 4), 2 KB row copies, 16 channels per stage.
using BwdCfgV4Bf16 = BwdCfgV4;
using BwdCfgS1Bf16 = BwdCfgS1;

int conv_bwd_bf16(int K, const uint16_t* feats, const float* dz, const float* eff_w, int B, int C, int N, uint16_t* dfeats,
                  double* S, double* s, int sm_count, cudaStream_t st, int w_shared, const ParamTail& pt) {
  RHSEG_DISPATCH_K(K, {
    const bool v4 = (N % 8 == 0) && ((reinterpret_cast<uintptr_t>(feats) & 15u) == 0) &&
                    ((reinterpret_cast<uintptr_t>(dz) & 15u) == 0) && ((reinterpret_cast<uintptr_t>(dfeats) & 15u) == 0);
    if (v4) return launch_conv_bwd<uint16_t, KK, 4, 1, BwdCfgV4Bf16>(feats, dz, eff_w, B, C, N, dfeats, S, s, sm_count, st, w_shared, pt);
    return launch_conv_bwd<uint16_t, KK, 1, (KK <= 4 ? 4 : 2), BwdCfgS1Bf16>(feats, dz, eff_w, B, C, N, dfeats, S, s, sm_count, st, w_shared, pt);
  });
  return RHSEG_OK;
}

}  // namespace rhseg
