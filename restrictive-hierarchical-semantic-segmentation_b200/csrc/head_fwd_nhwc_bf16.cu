// Head forward conv for channels-last bf16 features (RHSEG_FEATS_NHWC | RHSEG_FEATS_BF16): the 16-bit instances of
// head_fwd_nhwc.cuh, in a translation unit of their own so that they compile in parallel with the others.
#include "head_fwd_nhwc.cuh"

namespace rhseg {

template int level_conv_nhwc<uint16_t>(const uint16_t*, const float*, const float*, const float*, const int32_t*, int, int,
                                       int, int, int, int, float*, bool, float*, float*, double*, int, cudaStream_t);

}  // namespace rhseg
