// Head forward conv for bf16 donor features (autocast-trained backbones): the instances of head_fwd_kernel.cuh with
// 16-bit elements, in a translation unit of their own so that they compile in parallel with the fp32 ones.  Every
// feature value is converted to fp32 exactly in registers; weights, sums, logits and probabilities are fp32 as in
// the fp32 path, so the results equal that path's on the upcast features (DESIGN.md 3.7).
#include "head_fwd_kernel.cuh"

namespace rhseg {

template int level_conv_nchw<uint16_t>(const uint16_t*, const float*, const float*, const float*, const int32_t*, int, int,
                                       int, int, int, int, float*, bool, float*, float*, double*, int, cudaStream_t);

}  // namespace rhseg
