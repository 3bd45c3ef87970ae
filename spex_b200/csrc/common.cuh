// common.cuh — shared device helpers for libspex_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/spex_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libspex_b200 is written for sm_100a only; there is no fallback path."
#endif

namespace spex {

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

// launch counter (bench.py reports it as gpu_launches)
extern int64_t g_launches;
inline void count_launch(int n = 1) { g_launches += n; }

inline int check_last() {
  cudaError_t e = cudaGetLastError();
  return (int)e;
}

#define SPEX_RETURN_IF(cond, code) \
  do {                             \
    if (cond) return (code);       \
  } while (0)

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ---- cache-hinted memory ops -----------------------------------------------------------------
// Streaming (read-once) data: col / val / rowptr tiles and output rows.  Keep them out of L1 and
// mark them evict-first (ld.global.cs) so the 126 MB L2 is left to the gathered embedding rows.
__device__ __forceinline__ int ld_stream_s32(const int32_t* p) { return __ldcs(p); }
__device__ __forceinline__ float ld_stream_f32(const float* p) { return __ldcs(p); }
__device__ __forceinline__ float4 ld_stream_f4(const float* p) {
  return __ldcs(reinterpret_cast<const float4*>(p));
}
// Gathered embedding rows: read-only path, no L1 allocation (each 256 B row is consumed once by
// one warp), default L2 policy so hot rows stay resident.
__device__ __forceinline__ float4 ld_gather_f4(const float* p) {
  float4 v;
  asm("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p));
  return v;
}
// Software-managed L2 residency: hot embedding rows (columns flagged by the graph plan) are loaded
// with an evict_last policy, everything else with evict_first, so the 126 MB L2 keeps the rows that
// are gathered thousands of times instead of whatever was touched most recently.
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ float4 ld_gather_f4_hint(const float* p, uint64_t policy) {
  float4 v;
  asm("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
      : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
      : "l"(p), "l"(policy));
  return v;
}
// 128-bit store to an NVSwitch multicast address (cuMulticast mapping of the same buffer on every
// GPU of the group): the switch delivers it to all of them.
__device__ __forceinline__ void st_multimem_f4(float* p, float4 v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x),
               "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}
// plain (coherent) 128-bit load: for buffers that the same kernel also writes (in-place Z).
__device__ __forceinline__ float4 ld_f4(const float* p) {
  return *reinterpret_cast<const float4*>(p);
}
__device__ __forceinline__ void st_stream_f4(float* p, float4 v) {
  __stcs(reinterpret_cast<float4*>(p), v);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}

// SplitMix64 finaliser (Steele, Lea, Flood 2014): the counter-based hash of the device samplers
// (sampler.cu) and of the edge-dropout mask (spmm.cu).
__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

__device__ __forceinline__ float4 f4_zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ void f4_fma(float4& a, float s, const float4& x) {
  a.x = fmaf(s, x.x, a.x);
  a.y = fmaf(s, x.y, a.y);
  a.z = fmaf(s, x.z, a.z);
  a.w = fmaf(s, x.w, a.w);
}
__device__ __forceinline__ float4 f4_shfl_xor(const float4& a, int m) {
  float4 r;
  r.x = __shfl_xor_sync(kFull, a.x, m);
  r.y = __shfl_xor_sync(kFull, a.y, m);
  r.z = __shfl_xor_sync(kFull, a.z, m);
  r.w = __shfl_xor_sync(kFull, a.w, m);
  return r;
}
__device__ __forceinline__ void f4_add(float4& a, const float4& b) {
  a.x += b.x;
  a.y += b.y;
  a.z += b.z;
  a.w += b.w;
}

}  // namespace spex
