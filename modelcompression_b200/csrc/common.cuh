// common.cuh — shared helpers for libmcb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <stdlib.h>
#include "../../include/mcb200.h"

#define MC_ERR_ARG (-1)
#define MC_ERR_SHAPE (-2)
#define MC_ERR_WS (-3)

int mc_set_error(int code, const char* fmt, ...);

#define MC_CHECK_ARG(cond, ...)                      \
  do {                                               \
    if (!(cond)) return mc_set_error(MC_ERR_ARG, __VA_ARGS__); \
  } while (0)

#define MC_CUDA(call)                                                                       \
  do {                                                                                      \
    cudaError_t e_ = (call);                                                                \
    if (e_ != cudaSuccess)                                                                  \
      return mc_set_error(-(1000 + (int)e_), "%s failed: %s (%s:%d)", #call,                \
                          cudaGetErrorString(e_), __FILE__, __LINE__);                      \
  } while (0)

#define MC_LAUNCH_CHECK(name)                                                               \
  do {                                                                                      \
    cudaError_t e_ = cudaGetLastError();                                                    \
    if (e_ != cudaSuccess)                                                                  \
      return mc_set_error(-(1000 + (int)e_), "launch of %s failed: %s", name,               \
                          cudaGetErrorString(e_));                                          \
  } while (0)

static inline int mc_num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
  }
  return n;
}

// Multi-tensor segment table passed by value as a kernel parameter (<= 4 KB).
struct SegTable {
  const float* ptr[MC_MAX_SEGMENTS];
  float* out[MC_MAX_SEGMENTS];
  long long start[MC_MAX_SEGMENTS + 1];  // prefix sums of element counts
  int nseg;
};

// Streaming 128-bit accesses (bypass L1 allocation; data is touched once).
__device__ __forceinline__ float4 ld_stream_f4(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream_f4(float4* p, const float4& v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y),
               "f"(v.z), "f"(v.w)
               : "memory");
}
