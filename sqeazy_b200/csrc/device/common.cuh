// Shared device-side helpers for the sqeazy_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace sqyb {

#define SQYB_CUDA_OK(expr)                                   \
  do {                                                       \
    cudaError_t _e = (expr);                                 \
    if (_e != cudaSuccess) return (int)_e;                   \
  } while (0)

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs; grids are sized in multiples of this

// blocks of `threads` for `work_items` grid-stride items, at most 32 waves of the 148 SMs
inline int grid_for(uint64_t work_items, int threads) {
  uint64_t blocks = (work_items + threads - 1) / threads;
  const uint64_t cap = (uint64_t)kNumSMs * 32;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

// 128-bit streaming load/store: data crosses the SM exactly once, keep it out of L1.
__device__ __forceinline__ uint4 ld_stream(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ uint32_t ld_stream(const uint32_t* p) {
  uint32_t r;
  asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream(uint4* p, const uint4& v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}
__device__ __forceinline__ void st_stream(uint2* p, const uint2& v) {
  asm volatile("st.global.L1::no_allocate.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(v.x), "r"(v.y) : "memory");
}
__device__ __forceinline__ void st_stream(uint32_t* p, uint32_t v) {
  asm volatile("st.global.L1::no_allocate.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// Saturating subtraction of a threshold (remove_background, encoders/remove_background_scheme_impl.hpp:82-89) from
// packed unsigned fields, written with plain integer operations on purpose. ptxas 12.9 miscompiles the emulation of
// __vsubus2 when the loop around it is unrolled: the unrolled copies rebuild the packed constant -thr and one of them
// gets the two's-complement +1 in only one halfword (SASS: `VIADD.16x2 R0, ~thr2, 0x0` next to `VIADD.16x2 R2, ~thr2,
// 0x10001`, merged by PRMT), so every other voxel lost thr+1 in all grid-stride sweeps of the unrolled body — invisible
// below ~39 M voxels, found by tests/test_gpu_fullsize.py.
__device__ __forceinline__ uint32_t sat_sub_u16x2(uint32_t v, uint32_t thr) {
  const int lo = (int)(v & 0xffffu) - (int)thr, hi = (int)(v >> 16) - (int)thr;
  return (uint32_t)max(lo, 0) | ((uint32_t)max(hi, 0) << 16);
}
__device__ __forceinline__ uint32_t sat_sub_u8x4(uint32_t v, uint32_t thr) {
  uint32_t r = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) r |= (uint32_t)max((int)((v >> (8 * k)) & 0xffu) - (int)thr, 0) << (8 * k);
  return r;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

}  // namespace sqyb
