// Head forward conv for channels-last fp32 features (RHSEG_FEATS_NHWC): the fp32 instances of head_fwd_nhwc.cuh, in a
// translation unit of their own so that they compile in parallel with the others.
#include "head_fwd_nhwc.cuh"

namespace rhseg {

template int level_conv_nhwc<float>(const float*, const float*, const float*, const float*, const int32_t*, int, int, int,
                                    int, int, int, float*, bool, float*, float*, double*, int, cudaStream_t);

}  // namespace rhseg
