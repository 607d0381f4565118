// msda_scalar.cuh -- one element of any value dtype in and out of the compute type of the generic kernels
// (float for float / bf16 / f16 values, double for double): msda_generic.cuh and the generic DCNv2 kernels.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

namespace msda {

template <typename VT> struct Compute { using type = float; };
template <> struct Compute<double> { using type = double; };
template <> struct Compute<__half> { using type = float; };

template <typename CT, typename VT> __device__ __forceinline__ CT load_as(const VT* p) { return (CT)(*p); }
template <> __device__ __forceinline__ float load_as<float, __nv_bfloat16>(const __nv_bfloat16* p) {
  return __bfloat162float(*p);
}
template <> __device__ __forceinline__ float load_as<float, __half>(const __half* p) { return __half2float(*p); }
template <typename VT, typename CT> __device__ __forceinline__ void store_as(VT* p, CT v) { *p = (VT)v; }
template <> __device__ __forceinline__ void store_as<__nv_bfloat16, float>(__nv_bfloat16* p, float v) {
  *p = __float2bfloat16_rn(v);
}
template <> __device__ __forceinline__ void store_as<__half, float>(__half* p, float v) { *p = __float2half_rn(v); }

}  // namespace msda
