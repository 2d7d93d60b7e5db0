// Channels-last (NHWC) donor features: [B, Hf*Wf, C] in memory, fp32 or bf16 bits (RHSEG_FEATS_NHWC).  Pieces shared by
// the NHWC forward (head_fwd_nhwc.cuh) and the NHWC conv backward (head_bwd_nhwc.cu): the 3-D tensor map the forward
// streams the features through, the TMA tile copy and the 16-byte channel-group loads.  DESIGN.md 3.8.
#pragma once
#include <cuda.h>
#include <cudaTypedefs.h>
#include <mutex>
#include "common.cuh"
#include "pipeline.cuh"

namespace rhseg {

// cuTensorMapEncodeTiled through the runtime's driver entry point (the library links cudart statically, not libcuda)
inline PFN_cuTensorMapEncodeTiled tensor_map_encoder() {
  static std::once_flag once;
  static PFN_cuTensorMapEncodeTiled fn = nullptr;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled>(p);
  });
  return fn;
}

// Tensor map [C, N, B] (innermost first) of NHWC features; box = [box_c channels, box_p pixels, 1 sample].  Boxes that
// reach past a sample's last pixel or past the last channel are zero-filled, so a tile never reads the next sample.
// box_c * element size = 32 bytes uses the 32-byte swizzle (16-byte chunk index ^= bit 7 of the shared address: pixel
// rows 4 apart alternate their two chunks), which makes the per-pixel 128-bit reads of a warp conflict-free.
template <typename FT>
inline int encode_feats_map(CUtensorMap* map, const FT* feats, int B, int C, long N, int box_c, int box_p) {
  const PFN_cuTensorMapEncodeTiled enc = tensor_map_encoder();
  if (!enc) return RHSEG_ERR_UNSUPPORTED;
  const cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)N, (cuuint64_t)B};
  const cuuint64_t strides[2] = {(cuuint64_t)C * sizeof(FT), (cuuint64_t)C * sizeof(FT) * (cuuint64_t)N};
  const cuuint32_t box[3] = {(cuuint32_t)box_c, (cuuint32_t)box_p, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  const int ib = box_c * (int)sizeof(FT);
  const CUresult r = enc(map, sizeof(FT) == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_UINT16, 3,
                         const_cast<FT*>(feats), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         ib == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? RHSEG_OK : RHSEG_ERR_UNSUPPORTED;
}

// 3-D tile copy global -> shared (box of `map` at coordinates (c, p, b)), completion (bytes) signalled on `bar`
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, int c, int p, int b, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(c), "r"(p), "r"(b), "r"(bar)
      : "memory");
}

// 16-byte loads from shared memory / of one pixel's channel group
__device__ __forceinline__ uint4 lds128(const void* p) { return *reinterpret_cast<const uint4*>(p); }

// the 8 channels of a 16-byte chunk as fp32 (4 fp32 per chunk: two chunks; 8 bf16: one)
__device__ __forceinline__ void chunk_f32(const uint4& t, float* f, float) {
  f[0] = __uint_as_float(t.x); f[1] = __uint_as_float(t.y); f[2] = __uint_as_float(t.z); f[3] = __uint_as_float(t.w);
}
__device__ __forceinline__ void chunk_f32(const uint4& t, float* f, uint16_t) {
  f[0] = bf16_lo(t.x); f[1] = bf16_hi(t.x); f[2] = bf16_lo(t.y); f[3] = bf16_hi(t.y);
  f[4] = bf16_lo(t.z); f[5] = bf16_hi(t.z); f[6] = bf16_lo(t.w); f[7] = bf16_hi(t.w);
}

}  // namespace rhseg
