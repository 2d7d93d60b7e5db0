// Pieces shared by the feature-streaming forward conv (head_fwd*.cu) and head_up.cu (output-resolution upsample +
// activation + fused evaluation): the activation epilogue, the FiLM-pool block sum, the evaluation arguments and
// the dispatchers of both passes.  Separate translation units so that they compile in parallel.
#pragma once
#include "common.cuh"

namespace rhseg {

// Arguments of the fused per-level training evaluation (eval_accum.cuh): statistics, prediction index map,
// confusion matrix, consistency sums, computed on the pixels while their logits are in registers.
struct EvalArgs {
  const float* targets;
  long t_bstride, t_cstride;
  const float* parent_targets;
  long pt_bstride, pt_cstride;
  const unsigned char* prev_idx;
  int child;
  double* stats;
  double* cons;
  unsigned long long* conf;
  unsigned char* idx_out;
};

// hi-res pass of an upsampled head (head_up.cu): K / activation mode dispatch included.  act_arg = activation mode |
// RHSEG_GROUP_HINT.  *need_eval is set when `ea` was given but the shape took the generic kernel, which does not
// evaluate: the caller then runs rhseg_level_eval on the logits.
int fwd_upsampled_dispatch(int K, int act_arg, const float* z_lo, const float* prev_probs, const int32_t* table, int B,
                           int Hf, int Wf, int H, int W, int K_prev, float* logits, float* probs, double* psum,
                           cudaStream_t st, const EvalArgs* ea, bool* need_eval);

// Feature conv of the level forward, FT = float or uint16_t (bf16 bit patterns).  z_lo == nullptr: a head at feature
// resolution, conv + activation into logits / probs / psum; otherwise the low-res conv of an upsampled head into
// z_lo [B,K,Nf] (zeroed by the caller when zlo_zeroed).  K dispatch and tile shapes included.
// NCHW features [B,C,Nf], element-aligned (head_fwd_kernel.cuh; instances in head_fwd.cu, head_fwd_bf16.cu):
template <typename FT>
int level_conv_nchw(const FT* feats, const float* eff_w, const float* eff_b, const float* prev_probs, const int32_t* table,
                    int B, int C, int Nf, int K, int K_prev, int act_mode, float* z_lo, bool zlo_zeroed, float* logits,
                    float* probs, double* psum, int w_shared, cudaStream_t st);
// channels-last features [B,Nf,C], C * element size and the base address multiples of 16 bytes (head_fwd_nhwc.cuh;
// instances in head_fwd_nhwc.cu, head_fwd_nhwc_bf16.cu):
template <typename FT>
int level_conv_nhwc(const FT* feats, const float* eff_w, const float* eff_b, const float* prev_probs, const int32_t* table,
                    int B, int C, int Nf, int K, int K_prev, int act_mode, float* z_lo, bool zlo_zeroed, float* logits,
                    float* probs, double* psum, int w_shared, cudaStream_t st);

// ------------------------------------------------------------------------------------
// Activation epilogue shared by the fused and the upsampled path.  P pixels per thread.
// ------------------------------------------------------------------------------------
template <int K, int P, int MODE>
__device__ __forceinline__ void activate(const float (&z)[K][P], const float (&pp)[K][P], int start_mask,
                                         float (&prob)[K][P]) {
#pragma unroll
  for (int p = 0; p < P; ++p) {
    if constexpr (MODE == RHSEG_ACT_SIGMOID) {
#pragma unroll
      for (int k = 0; k < K; ++k) prob[k][p] = sigmoidf_ref(z[k][p]);
    } else if constexpr (MODE == RHSEG_ACT_GROUPED) {
      float zz[K], q[K];
#pragma unroll
      for (int k = 0; k < K; ++k) zz[k] = z[k][p];
      // softmax(z_g + log(P_p + eps)) == softmax(z_g): the gate is constant inside a group
      grouped_softmax<K>(zz, start_mask, q);
#pragma unroll
      for (int k = 0; k < K; ++k) prob[k][p] = pp[k][p] * q[k];
    } else {
#pragma unroll
      for (int k = 0; k < K; ++k) prob[k][p] = 0.f;
    }
  }
}

// per-thread partial sums of the probabilities -> one fp64 atomic per (CTA, channel).
// SYNC() is the barrier of the participating threads (whole CTA or the consumer warps only).
template <int K, int NWARP, typename SyncFn>
__device__ __forceinline__ void block_psum(const float (&ps)[K], double* __restrict__ psum_b, float* red, SyncFn sync) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const float v = warp_sum(ps[k]);
    if (lane == 0) red[warp * K + k] = v;
  }
  sync();
  if (threadIdx.x < K) {
    double acc = 0.0;
#pragma unroll
    for (int w = 0; w < NWARP; ++w) acc += (double)red[w * K + threadIdx.x];
    atomicAdd(&psum_b[threadIdx.x], acc);
  }
  sync();
}


}  // namespace rhseg
