// bitswapN: bit-plane (w-bit field) transpose of a uint16 buffer, one read + one write of the
// volume (the reference makes 16 passes: encoders/sse_utils.hpp:1366-1433, and decodes on one
// scalar thread: encoders/bitplane_reorder_scalar.hpp:81-116).
//
// Semantics (encoders/bitplane_reorder_scalar.hpp:27-74, bitswap_scheme_impl.hpp:97-157):
//   P = 16/w planes, N' = N - N % P, S = N'/P.  For i < N', field p (p = 0 lowest w bits) of in[i]
//   lands in out[(P-1-p)*S + i/P] at bit offset (16-w) - (i%P)*w.  in[i >= N'] is copied verbatim.
//
// Fast path (N % 128 == 0, 32-byte aligned pointers): a thread owns 32 consecutive voxels
// (two 256-bit loads), packs two neighbouring groups per 32-bit register, runs log2(P) masked
// delta-swap stages (a PxP transpose of w-bit atoms in registers), and stores W consecutive
// 32-bit words per plane, so a warp writes 128*W contiguous bytes per plane. The optional
// threshold filter (remove_background, encoders/remove_background_scheme_impl.hpp:82-89) is
// fused into the load (sat_sub_u16x2, common.cuh). The thread program lives in bitswap_thread.h.
#include "bitswap_thread.h"
#include "common.cuh"
#include "kernels.h"

namespace sqyb {

namespace {

using bitswap_thread::Geo;

// ---- encode: n32 = number of 32-voxel chunks, S = words per segment --------------------------
template <int W, bool SUB>
__global__ void __launch_bounds__(256) bitswap_encode_fast(const uint16_t* __restrict__ in, uint16_t* __restrict__ out,
                                                            uint64_t n32, uint64_t S, uint32_t thr /* threshold, < 65536 */) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n32; t += stride)
    bitswap_thread::encode_chunk<W, SUB>(in, out, t, S, thr);
}

template <int W>
__global__ void __launch_bounds__(256) bitswap_decode_fast(const uint16_t* __restrict__ in, uint16_t* __restrict__ out,
                                                            uint64_t n32, uint64_t S) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n32; t += stride)
    bitswap_thread::decode_chunk<W, false>(in, out, t, S);
}

// ---- generic path: any N, any alignment; one thread per group of P voxels --------------------
template <int W, bool SUB>
__global__ void bitswap_encode_generic(const uint16_t* __restrict__ in, uint16_t* __restrict__ out, uint64_t n,
                                       uint32_t thr) {
  constexpr int P = Geo<W>::P;
  const uint64_t S = n / P;
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; g < S; g += stride) {
    uint32_t v[P];
#pragma unroll
    for (int j = 0; j < P; ++j) {
      uint32_t x = in[g * P + j];
      if (SUB) x = x > thr ? x - thr : 0;
      v[j] = x;
    }
#pragma unroll
    for (int p = 0; p < P; ++p) {
      uint32_t word = 0;
#pragma unroll
      for (int j = 0; j < P; ++j) word |= ((v[j] >> (p * W)) & ((1u << W) - 1u)) << ((16 - W) - j * W);
      out[(uint64_t)(P - 1 - p) * S + g] = (uint16_t)word;
    }
  }
  // verbatim tail (bitswap_scheme_impl.hpp:99-103)
  if (blockIdx.x == 0) {
    for (uint64_t i = S * P + threadIdx.x; i < n; i += blockDim.x) {
      uint32_t x = in[i];
      if (SUB) x = x > thr ? x - thr : 0;
      out[i] = (uint16_t)x;
    }
  }
}

template <int W>
__global__ void bitswap_decode_generic(const uint16_t* __restrict__ in, uint16_t* __restrict__ out, uint64_t n) {
  constexpr int P = Geo<W>::P;
  const uint64_t S = n / P;
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; g < S; g += stride) {
    uint32_t w[P];
#pragma unroll
    for (int p = 0; p < P; ++p) w[p] = in[(uint64_t)(P - 1 - p) * S + g];
#pragma unroll
    for (int j = 0; j < P; ++j) {
      uint32_t x = 0;
#pragma unroll
      for (int p = 0; p < P; ++p) x |= ((w[p] >> ((16 - W) - j * W)) & ((1u << W) - 1u)) << (p * W);
      out[g * P + j] = (uint16_t)x;
    }
  }
  if (blockIdx.x == 0)
    for (uint64_t i = S * P + threadIdx.x; i < n; i += blockDim.x) out[i] = in[i];
}

inline int grid_for(uint64_t work_items, int threads) {
  uint64_t blocks = (work_items + threads - 1) / threads;
  const uint64_t cap = (uint64_t)kNumSMs * 32;  // persistent-ish grid-stride: 32 waves of 148
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

inline bool fast_ok(const void* a, const void* b, uint64_t n) {
  return n >= 128 && (n % 128 == 0) && (((uintptr_t)a | (uintptr_t)b) & 31) == 0;
}

template <int W>
int launch_encode(const uint16_t* in, uint16_t* out, uint64_t n, int threshold, cudaStream_t st) {
  constexpr int P = Geo<W>::P;
  const bool sub = threshold > 0;
  const uint32_t thr = (uint32_t)threshold & 0xffffu;
  if (n == 0) return 0;
  if (fast_ok(in, out, n)) {
    const uint64_t n32 = n / 32, S = n / P;
    const int g = grid_for(n32, 256);
    if (sub) bitswap_encode_fast<W, true><<<g, 256, 0, st>>>(in, out, n32, S, thr);
    else bitswap_encode_fast<W, false><<<g, 256, 0, st>>>(in, out, n32, S, 0);
  } else {
    const int g = grid_for(n / P + 1, 256);
    if (sub) bitswap_encode_generic<W, true><<<g, 256, 0, st>>>(in, out, n, thr);
    else bitswap_encode_generic<W, false><<<g, 256, 0, st>>>(in, out, n, 0);
  }
  SQYB_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

template <int W>
int launch_decode(const uint16_t* in, uint16_t* out, uint64_t n, cudaStream_t st) {
  constexpr int P = Geo<W>::P;
  if (n == 0) return 0;
  if (fast_ok(in, out, n)) {
    const uint64_t n32 = n / 32, S = n / P;
    bitswap_decode_fast<W><<<grid_for(n32, 256), 256, 0, st>>>(in, out, n32, S);
  } else {
    bitswap_decode_generic<W><<<grid_for(n / P + 1, 256), 256, 0, st>>>(in, out, n);
  }
  SQYB_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

// ---- plain threshold filter (no bitswap following) -------------------------------------------
__global__ void __launch_bounds__(256) remove_background_kernel(const uint16_t* __restrict__ in, uint16_t* __restrict__ out,
                                                                uint64_t n, uint32_t thr) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool aligned = ((((uintptr_t)in) | ((uintptr_t)out)) & 15) == 0;
  const uint64_t nv = aligned ? n / 8 : 0;
  for (uint64_t i = tid; i < nv; i += stride) {
    uint4 v = ld_stream(reinterpret_cast<const uint4*>(in) + i);
    v.x = sat_sub_u16x2(v.x, thr); v.y = sat_sub_u16x2(v.y, thr); v.z = sat_sub_u16x2(v.z, thr); v.w = sat_sub_u16x2(v.w, thr);
    st_stream(reinterpret_cast<uint4*>(out) + i, v);
  }
  for (uint64_t i = nv * 8 + tid; i < n; i += stride) {
    uint32_t x = in[i];
    out[i] = (uint16_t)(x > thr ? x - thr : 0);
  }
}

// voxel range [first, first+count) of a volume of n voxels: same kernels, same plane-major destination (segment stride n/P),
// pointers moved to the range. Ranges are cut at multiples of 128 voxels of 32-byte aligned buffers (fast kernels only).
template <int W>
int launch_encode_range(const uint16_t* in, uint16_t* out, uint64_t n, uint64_t first, uint64_t count, int threshold, cudaStream_t st) {
  constexpr int P = Geo<W>::P;
  if (count == 0) return 0;
  if (!fast_ok(in, out, n) || first % 128 || count % 128 || first + count > n) return -3;
  const uint64_t n32 = count / 32, S = n / P;
  const int g = grid_for(n32, 256);
  if (threshold > 0) bitswap_encode_fast<W, true><<<g, 256, 0, st>>>(in + first, out + first / P, n32, S, (uint32_t)threshold & 0xffffu);
  else bitswap_encode_fast<W, false><<<g, 256, 0, st>>>(in + first, out + first / P, n32, S, 0);
  SQYB_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

template <int W>
int launch_decode_range(const uint16_t* in, uint16_t* out, uint64_t n, uint64_t first, uint64_t count, cudaStream_t st) {
  constexpr int P = Geo<W>::P;
  if (count == 0) return 0;
  if (!fast_ok(in, out, n) || first % 128 || count % 128 || first + count > n) return -3;
  bitswap_decode_fast<W><<<grid_for(count / 32, 256), 256, 0, st>>>(in + first / P, out + first, count / 32, n / P);
  SQYB_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

}  // namespace

int k_bitswap_encode_range(int w, const uint16_t* in, uint16_t* out, uint64_t n, uint64_t first, uint64_t count, int threshold,
                           cudaStream_t st) {
  switch (w) {
    case 1: return launch_encode_range<1>(in, out, n, first, count, threshold, st);
    case 2: return launch_encode_range<2>(in, out, n, first, count, threshold, st);
    case 4: return launch_encode_range<4>(in, out, n, first, count, threshold, st);
    case 8: return launch_encode_range<8>(in, out, n, first, count, threshold, st);
  }
  return -1;
}

int k_bitswap_decode_range(int w, const uint16_t* in, uint16_t* out, uint64_t n, uint64_t first, uint64_t count, cudaStream_t st) {
  switch (w) {
    case 1: return launch_decode_range<1>(in, out, n, first, count, st);
    case 2: return launch_decode_range<2>(in, out, n, first, count, st);
    case 4: return launch_decode_range<4>(in, out, n, first, count, st);
    case 8: return launch_decode_range<8>(in, out, n, first, count, st);
  }
  return -1;
}

int k_bitswap_encode(int w, const uint16_t* in, uint16_t* out, uint64_t n, int threshold, cudaStream_t st) {
  switch (w) {
    case 1: return launch_encode<1>(in, out, n, threshold, st);
    case 2: return launch_encode<2>(in, out, n, threshold, st);
    case 4: return launch_encode<4>(in, out, n, threshold, st);
    case 8: return launch_encode<8>(in, out, n, threshold, st);
  }
  return -1;
}

int k_bitswap_decode(int w, const uint16_t* in, uint16_t* out, uint64_t n, cudaStream_t st) {
  switch (w) {
    case 1: return launch_decode<1>(in, out, n, st);
    case 2: return launch_decode<2>(in, out, n, st);
    case 4: return launch_decode<4>(in, out, n, st);
    case 8: return launch_decode<8>(in, out, n, st);
  }
  return -1;
}

int k_remove_background(const uint16_t* in, uint16_t* out, uint64_t n, int threshold, cudaStream_t st) {
  if (n == 0) return 0;
  const uint32_t thr = (uint32_t)threshold & 0xffffu;
  remove_background_kernel<<<grid_for(n / 8 + 1, 256), 256, 0, st>>>(in, out, n, thr);
  SQYB_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

}  // namespace sqyb
