// Conv backward for bf16 donor features (autocast-trained backbones): the instances of conv_bwd_kernel.cuh with 16-bit
// elements, in a translation unit of their own so that they compile in parallel with the fp32 ones.  Features are
// converted to fp32 exactly, S / s accumulate as in the fp32 path, and dfeats is formed in fp32 and rounded to bf16
// (nearest even) once, when it is stored (DESIGN.md 3.7).  The ring shapes are the fp32 ones: T = 1024 px with 2 KB
// row copies on vector rows, and on scalar rows (odd planes) for K <= 4.
#include "conv_bwd_kernel.cuh"

namespace rhseg {

template int conv_bwd_nchw<uint16_t>(int, const uint16_t*, const float*, const float*, int, int, int, uint16_t*, double*,
                                     double*, int, cudaStream_t, int, const ParamTail&);

}  // namespace rhseg
