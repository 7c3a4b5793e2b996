// Shared helpers for libemr2a.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/emr2a.h"

#define EMR2A_EPS 1e-8f

namespace emr2a {

// ---- thread-local error text -------------------------------------------------
int fail(int code, const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* where);

#define EMR2A_CUDA_TRY(expr)                                        \
  do {                                                              \
    cudaError_t _e = (expr);                                        \
    if (_e != cudaSuccess) return ::emr2a::cuda_fail(_e, #expr);    \
  } while (0)

#define EMR2A_LAUNCH_CHECK(name)                                    \
  do {                                                              \
    cudaError_t _e = cudaGetLastError();                            \
    if (_e != cudaSuccess) return ::emr2a::cuda_fail(_e, name);     \
  } while (0)

int sm_count();

// ---- packed Top-K keys -------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t order_f32(float s) {
#ifdef __CUDA_ARCH__
  uint32_t b = __float_as_uint(s);
#else
  union { float f; uint32_t u; } c; c.f = s; uint32_t b = c.u;
#endif
  return (b & 0x80000000u) ? ~b : (b ^ 0x80000000u);
}
__host__ __device__ __forceinline__ float unorder_f32(uint32_t o) {
  uint32_t b = (o & 0x80000000u) ? (o ^ 0x80000000u) : ~o;
#ifdef __CUDA_ARCH__
  return __uint_as_float(b);
#else
  union { float f; uint32_t u; } c; c.u = b; return c.f;
#endif
}
__host__ __device__ __forceinline__ uint64_t pack_key(float score, uint32_t idx) {
  return (static_cast<uint64_t>(order_f32(score)) << 32) | static_cast<uint64_t>(0xFFFFFFFFu - idx);
}
__host__ __device__ __forceinline__ float key_score(uint64_t k) { return unorder_f32(static_cast<uint32_t>(k >> 32)); }
__host__ __device__ __forceinline__ uint32_t key_index(uint64_t k) { return 0xFFFFFFFFu - static_cast<uint32_t>(k & 0xFFFFFFFFu); }

// ---- warp helpers --------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ uint64_t warp_max_u64(uint64_t v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    uint64_t t = __shfl_xor_sync(0xffffffffu, v, o);
    v = t > v ? t : v;
  }
  return v;
}

// 128-bit streaming loads / stores (read-once data: do not pollute L1)
__device__ __forceinline__ float4 ldg_stream_f4(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ uint4 ldg_stream_u4(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ uint2 ldg_stream_u2(const uint2* p) {
  uint2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
  return r;
}

// Bound E on |s~ - s| of the rescore arm (derivation: rescore.cu), from the query's norms nq, rq and the database's
// K1 stats ds.  Shared by the re-scoring kernels and the range epilogue of the tensor-core filter (tc_common.cuh).
__device__ __forceinline__ float error_bound(float nq, float rq, const float* ds, int D) {
  // the four norms are fp32 sums of D squares (relative error of a norm <= D * 2^-25): widen them accordingly
  const float up = 1.f + static_cast<float>(D) * 5.9604645e-8f;
  const float nd = ds[0] * up, rd = ds[1] * up;
  nq *= up; rq *= up;
  const float arith = (1.02f * static_cast<float>(D) + 8.f) * 1.1920929e-7f * (nq + rq) * (nd + rd);
  return (rq * nd + (nq + rq) * rd + arith) * 1.000001f + 1e-30f;      // rounded up: the bound must stay a bound
}

// split an fp32 value into bf16 hi + bf16 lo (2-way split, x ~= hi + lo, rel. residual ~2^-17)
__device__ __forceinline__ void split_bf16(float x, uint16_t& hi, uint16_t& lo) {
  __nv_bfloat16 h = __float2bfloat16_rn(x);
  float r = x - __bfloat162float(h);
  __nv_bfloat16 l = __float2bfloat16_rn(r);
  hi = __bfloat16_as_ushort(h);
  lo = __bfloat16_as_ushort(l);
}

}  // namespace emr2a
