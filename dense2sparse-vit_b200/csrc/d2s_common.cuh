// Shared helpers for libd2s_b200.so (sm_100a only).
#pragma once
#include <stdlib.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/d2s.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libd2s_b200 is written for sm_100a only"
#endif

namespace d2s {

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs; grids are sized in multiples of this

void set_error(const char* fmt, ...);
int  check_launch(const char* what);
void count_launch(int n = 1);

#define D2S_REQUIRE(cond, code, ...)            \
  do {                                          \
    if (!(cond)) {                              \
      d2s::set_error(__VA_ARGS__);              \
      return (code);                            \
    }                                           \
  } while (0)

// The opt-in to more than 48 KB of dynamic shared memory is a per-DEVICE function attribute: remembered per call site and per
// device ordinal, so that a process driving several GPUs (model on cuda:1 while cuda:0 is current elsewhere) sets it on each.
struct SmemOptIn { unsigned long long done = 0; };
template <typename K>
static inline cudaError_t opt_in_smem(SmemOptIn& st, K kern, int bytes) {
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && ((st.done >> dev) & 1ull)) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess && dev >= 0 && dev < 64) st.done |= 1ull << dev;
  return e;
}

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
static inline int  ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline size_t elem_size(int dtype) { return dtype == D2S_BF16 ? 2 : 4; }

// ---- device helpers --------------------------------------------------------------------------
__device__ __forceinline__ float ld_as_float(const float* p, size_t i) { return p[i]; }
__device__ __forceinline__ float ld_as_float(const __nv_bfloat16* p, size_t i) { return __bfloat162float(p[i]); }
__device__ __forceinline__ void  st_from_float(float* p, size_t i, float v) { p[i] = v; }
__device__ __forceinline__ void  st_from_float(__nv_bfloat16* p, size_t i, float v) { p[i] = __float2bfloat16_rn(v); }

// streaming 16-byte accesses: gathered rows are touched once, keep them out of L1
__device__ __forceinline__ int4 ld_stream16(const void* p) {
  int4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream16(void* p, const int4& v) {
  asm volatile("st.global.L1::no_allocate.v4.s32 [%0], {%1,%2,%3,%4};"
               :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

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

// Order-preserving map float -> uint32 with torch.sort semantics: NaN largest, -0.0 == +0.0.
__device__ __forceinline__ uint32_t float_to_ordered(float f) {
  if (f != f) return 0xffffffffu;
  uint32_t u = __float_as_uint(f + 0.0f);  // -0.0 + 0.0 = +0.0
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

}  // namespace d2s
