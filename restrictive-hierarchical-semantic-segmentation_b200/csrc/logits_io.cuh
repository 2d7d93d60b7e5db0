// Logit element types of the flat-model loss / evaluation / gradient kernels: float, or uint16_t = the bit pattern of a
// bf16 value (a flat head run under bf16 autocast).  A bf16 logit is widened to fp32 exactly when it is loaded, so the
// per-pixel code after the load is the fp32 code; a bf16 gradient is formed in fp32 and rounded to nearest even once,
// when it is stored.  The float overloads are the plain fp32 loads and stores.
#pragma once
#include "common.cuh"
#include "pipeline.cuh"

namespace rhseg {

// streaming load of VEC consecutive bf16 logits (VEC * 2 bytes, aligned to that size)
template <int VEC>
__device__ __forceinline__ Vec<VEC> ld_stream(const uint16_t* p) {
  static_assert(VEC == 1 || VEC == 4, "bf16 logit loads: 1 or 4 elements");
  Vec<VEC> r;
  if constexpr (VEC == 4) {
    uint32_t a, b;
    asm volatile("ld.global.nc.L1::no_allocate.v2.b32 {%0,%1}, [%2];" : "=r"(a), "=r"(b) : "l"(p));
    r.v[0] = bf16_lo(a); r.v[1] = bf16_hi(a); r.v[2] = bf16_lo(b); r.v[3] = bf16_hi(b);
  } else {
    unsigned short h;
    asm volatile("ld.global.nc.L1::no_allocate.b16 %0, [%1];" : "=h"(h) : "l"(p));
    r.v[0] = feat_f32((uint16_t)h);
  }
  return r;
}

template <int VEC>
__device__ __forceinline__ Vec<VEC> ld_cached(const uint16_t* p) {
  static_assert(VEC == 1 || VEC == 4, "bf16 logit loads: 1 or 4 elements");
  Vec<VEC> r;
  if constexpr (VEC == 4) {
    const uint2 t = __ldg(reinterpret_cast<const uint2*>(p));
    r.v[0] = bf16_lo(t.x); r.v[1] = bf16_hi(t.x); r.v[2] = bf16_lo(t.y); r.v[3] = bf16_hi(t.y);
  } else {
    r.v[0] = feat_f32((uint16_t)__ldg(reinterpret_cast<const unsigned short*>(p)));
  }
  return r;
}

// gradient store (cached: the donor's backward reads it next)
template <int VEC>
__device__ __forceinline__ void st_grad(float* p, const Vec<VEC>& r) { *reinterpret_cast<Vec<VEC>*>(p) = r; }
template <int VEC>
__device__ __forceinline__ void st_grad(uint16_t* p, const Vec<VEC>& r) {
  static_assert(VEC == 1 || VEC == 4, "bf16 gradient stores: 1 or 4 elements");
  if constexpr (VEC == 4) *reinterpret_cast<uint2*>(p) = make_uint2(pack_bf16x2(r.v[0], r.v[1]), pack_bf16x2(r.v[2], r.v[3]));
  else *p = to_bf16_bits(r.v[0]);
}

}  // namespace rhseg
