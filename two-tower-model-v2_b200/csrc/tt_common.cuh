// Shared host/device helpers for the tt_b200 library (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string>

#include "../../include/tt_b200.h"

namespace tt {

// ---- host-side error plumbing -------------------------------------------------------------
void set_error(const std::string& msg);   // defined in api.cu (thread-local)

#define TT_CHECK_ARG(cond, msg)                                                     \
  do {                                                                              \
    if (!(cond)) {                                                                  \
      ::tt::set_error(std::string(__func__) + ": " + (msg));                        \
      return TT_ERR_INVALID;                                                        \
    }                                                                               \
  } while (0)

#define TT_CHECK_CUDA(expr)                                                         \
  do {                                                                              \
    cudaError_t _e = (expr);                                                        \
    if (_e != cudaSuccess) {                                                        \
      ::tt::set_error(std::string(__func__) + ": " #expr " failed: " +              \
                      cudaGetErrorString(_e));                                      \
      return TT_ERR_CUDA;                                                           \
    }                                                                               \
  } while (0)

void count_launch();                      // api.cu: kernels launched by this library (process-wide)
#define TT_CHECK_LAUNCH()                 \
  do {                                    \
    ::tt::count_launch();                 \
    TT_CHECK_CUDA(cudaGetLastError());    \
  } while (0)

inline int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
  }
  return n;
}

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---- programmatic dependent launch (PDL) ------------------------------------------------------
// The kernels of one search call form a chain on one stream.  Each is launched with the programmatic-stream-
// serialization attribute, calls pdl_trigger() first thing (its successor may be scheduled as soon as every CTA of
// this grid has started) and pdl_wait() before it touches global memory (returns once the predecessor grid has
// completed and its writes are visible).  The successor's launch latency and prologue (barrier init, TMEM
// allocation, descriptor prefetch) then hide under the predecessor's tail.  The device-side instructions are no-ops
// in a kernel launched without the attribute.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---- device helpers ------------------------------------------------------------------------
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Streaming 128-bit load that does not allocate in L1 (data is touched once).
__device__ __forceinline__ float4 ldg_stream(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}

// Monotone map float -> uint32 (larger float <=> larger key); NaN sorts above +inf.
__device__ __host__ __forceinline__ uint32_t float_to_ordered(float f) {
  uint32_t b;
#ifdef __CUDA_ARCH__
  b = __float_as_uint(f);
#else
  union { float f; uint32_t u; } c; c.f = f; b = c.u;
#endif
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __host__ __forceinline__ float ordered_to_float(uint32_t k) {
  uint32_t b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
#ifdef __CUDA_ARCH__
  return __uint_as_float(b);
#else
  union { float f; uint32_t u; } c; c.u = b; return c.f;
#endif
}
// 64-bit sort key: descending order of the key == (score descending, row index ascending).
__device__ __host__ __forceinline__ uint64_t make_key(float score, uint32_t row) {
  return ((uint64_t)float_to_ordered(score) << 32) | (uint64_t)(~row);
}
__device__ __host__ __forceinline__ float key_score(uint64_t k) { return ordered_to_float((uint32_t)(k >> 32)); }
__device__ __host__ __forceinline__ uint32_t key_row(uint64_t k) { return ~(uint32_t)(k & 0xffffffffu); }

}  // namespace tt
