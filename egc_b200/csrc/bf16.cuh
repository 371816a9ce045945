// bf16 storage of the gathered tensors (basis rows, target-side streams): conversions only.  Values are rounded to
// nearest-even when stored and widened exactly (a 16-bit shift) when loaded; every sum, product and comparison of the
// kernels that read them stays fp32.
#pragma once

#include <cuda_bf16.h>

#include <type_traits>

#include "common.cuh"

namespace egc {

using bf16 = __nv_bfloat16;
template <class ST>
constexpr bool kBf16 = std::is_same<ST, bf16>::value;

__device__ __forceinline__ float bf16_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }
__device__ __forceinline__ float4 widen_bf16x4(uint2 w) { return make_float4(bf16_lo(w.x), bf16_hi(w.x), bf16_lo(w.y), bf16_hi(w.y)); }
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  return static_cast<uint32_t>(__bfloat16_as_ushort(__float2bfloat16_rn(a))) |
         (static_cast<uint32_t>(__bfloat16_as_ushort(__float2bfloat16_rn(b))) << 16);
}

// four consecutive stored values -> fp32 (read-only cache path)
template <class ST>
__device__ __forceinline__ float4 ldg4(const ST* p) {
  if constexpr (kBf16<ST>) return widen_bf16x4(__ldg(reinterpret_cast<const uint2*>(p)));
  else return __ldg(reinterpret_cast<const float4*>(p));
}
template <class ST>
__device__ __forceinline__ void ldg4(float (&v)[4], const ST* p) {
  const float4 t = ldg4<ST>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
// fp32 -> four consecutive stored values (round to nearest even for bf16)
template <class ST>
__device__ __forceinline__ void st4(ST* p, const float (&v)[4]) {
  if constexpr (kBf16<ST>) *reinterpret_cast<uint2*>(p) = make_uint2(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]));
  else *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
}
template <class ST>
__device__ __forceinline__ void st1(ST* p, float v) {
  if constexpr (kBf16<ST>) *p = __float2bfloat16_rn(v);
  else *p = v;
}

}  // namespace egc
