// Shared device/host helpers for the chgnet_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/chgnet_b200.h"

namespace chg {

// ---- host side ---------------------------------------------------------
void set_error(const char* fmt, ...);
void count_launch();
int sm_count();

#define CHG_CHECK_ARG(cond, msg)                \
  do {                                          \
    if (!(cond)) {                              \
      chg::set_error("%s: %s", __func__, msg);  \
      return CHG_ERR_ARG;                       \
    }                                           \
  } while (0)

#define CHG_CUDA(expr)                                                              \
  do {                                                                              \
    cudaError_t _e = (expr);                                                        \
    if (_e != cudaSuccess) {                                                        \
      chg::set_error("%s: %s failed: %s", __func__, #expr, cudaGetErrorString(_e)); \
      return CHG_ERR_CUDA;                                                          \
    }                                                                               \
  } while (0)

#define CHG_LAUNCH_END()                                                            \
  do {                                                                              \
    cudaError_t _e = cudaGetLastError();                                            \
    if (_e != cudaSuccess) {                                                        \
      chg::set_error("%s: launch failed: %s", __func__, cudaGetErrorString(_e));    \
      return CHG_ERR_CUDA;                                                          \
    }                                                                               \
    chg::count_launch();                                                            \
    return CHG_OK;                                                                  \
  } while (0)

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// ---- device side -------------------------------------------------------
#ifdef __CUDACC__

constexpr int F = CHG_FEA;  // 64

// sigmoid / silu in fp32.  MUFU.EX2 + MUFU.RCP (about 2 ulp each); define
// CHG_ACCURATE_MATH to fall back to expf + IEEE division.
__device__ __forceinline__ float sigmoid_f(float x) {
#ifdef CHG_ACCURATE_MATH
  return 1.f / (1.f + expf(-x));
#else
  return __fdividef(1.f, 1.f + __expf(-x));
#endif
}
__device__ __forceinline__ float silu_f(float x) { return x * sigmoid_f(x); }
// d silu / dx = s (1 + x (1 - s))
__device__ __forceinline__ float dsilu_f(float x) {
  const float s = sigmoid_f(x);
  return s * fmaf(x, 1.f - s, 1.f);
}

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void stg4(float* p, const float4& v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ float4 lds4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void sts4(float* p, const float4& v) { *reinterpret_cast<float4*>(p) = v; }

__device__ __forceinline__ float4 operator+(const float4& a, const float4& b) {
  return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}
__device__ __forceinline__ float4 operator*(const float4& a, const float4& b) {
  return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w);
}
__device__ __forceinline__ float4 operator*(const float4& a, float s) {
  return make_float4(a.x * s, a.y * s, a.z * s, a.w * s);
}
__device__ __forceinline__ float& f4at(float4& v, int i) { return reinterpret_cast<float*>(&v)[i]; }
__device__ __forceinline__ float f4at(const float4& v, int i) { return reinterpret_cast<const float*>(&v)[i]; }

// sum over the 16 lanes that share (lane >> 4)
__device__ __forceinline__ float sum16(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  v += __shfl_xor_sync(0xffffffffu, v, 4);
  v += __shfl_xor_sync(0xffffffffu, v, 8);
  return v;
}
__device__ __forceinline__ float sum32(float v) {
  v = sum16(v);
  v += __shfl_xor_sync(0xffffffffu, v, 16);
  return v;
}
__device__ __forceinline__ double sum32d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

#endif  // __CUDACC__
}  // namespace chg
