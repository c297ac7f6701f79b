// bitswapN: bit-plane (w-bit field) transpose of a uint16 or uint8 buffer, one read + one write of the
// volume (the reference makes 16 passes: encoders/sse_utils.hpp:1366-1433, and decodes on one
// scalar thread: encoders/bitplane_reorder_scalar.hpp:81-116).
//
// Semantics (encoders/bitplane_reorder_scalar.hpp:27-74, bitswap_scheme_impl.hpp:97-157), B = bits per voxel:
//   P = B/w planes, N' = N - N % P, S = N'/P.  For i < N', field p (p = 0 lowest w bits) of in[i]
//   lands in out[(P-1-p)*S + i/P] at bit offset (B-w) - (i%P)*w.  in[i >= N'] is copied verbatim.
// uint8 volumes are the *_UI8 entry points (src/sqeazy.cpp:72-106,309-335 over dypeline<uint8_t>,
// sqeazy_pipelines.hpp:31-77); the reference excludes its SSE path for sizeof(raw_type) == 1, so the scalar
// code defines the result (bitswap_scheme_impl.hpp:97-197).
//
// Fast path, uint16 (N % 128 == 0, 32-byte aligned pointers): a thread owns 32 consecutive voxels
// (two 256-bit loads), packs two neighbouring groups per 32-bit register, runs log2(P) masked
// delta-swap stages (a PxP transpose of w-bit atoms in registers), and stores W consecutive
// 32-bit words per plane, so a warp writes 128*W contiguous bytes per plane. The optional
// threshold filter (remove_background, encoders/remove_background_scheme_impl.hpp:82-89) is
// fused into the load (sat_sub_u16x2, common.cuh). The thread program lives in bitswap_thread.h.
//
// Fast path, uint8 (N % 128 == 0, 16-byte aligned pointers): a thread owns 32 consecutive bytes (two 128-bit loads = four
// 64-bit chunks). Inside a chunk every group of P bytes is byte-reversed (the first element of a group goes to the
// most significant field) and the PxP matrix of w-bit atoms is transposed with log2(P) masked delta swaps; byte p of a
// transposed group is then exactly the group's output byte for plane p. A thread stores 32/P consecutive bytes per
// plane, so a warp writes 128*w contiguous bytes per plane. Decoding runs the same two involutions in reverse order.
//
// The kernels of both element sizes share their names and parameters (overloads on the pointer type), so one launch
// helper per direction serves both.
#include "bitswap_thread.h"
#include "common.cuh"
#include "kernels.h"

namespace sqyb {

namespace {

using bitswap_thread::Geo;

// ---- uint16, encode: n32 = number of 32-voxel chunks, S = words per segment -----------------
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

// ---- uint16, generic path: any N, any alignment; one thread per group of P voxels -----------
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

// ---- uint8, fast path ------------------------------------------------------------------------
template <int W>
__device__ __forceinline__ unsigned long long reverse_groups(unsigned long long x) {
  uint32_t lo = (uint32_t)x, hi = (uint32_t)(x >> 32);
  if (W == 1) {  // groups of 8 bytes
    const uint32_t l2 = __byte_perm(hi, 0, 0x0123), h2 = __byte_perm(lo, 0, 0x0123);
    lo = l2; hi = h2;
  } else if (W == 2) {  // groups of 4 bytes
    lo = __byte_perm(lo, 0, 0x0123);
    hi = __byte_perm(hi, 0, 0x0123);
  } else {  // groups of 2 bytes
    lo = __byte_perm(lo, 0, 0x2301);
    hi = __byte_perm(hi, 0, 0x2301);
  }
  return ((unsigned long long)hi << 32) | lo;
}

template <int W>
__device__ __forceinline__ unsigned long long transpose_atoms(unsigned long long x) {
  unsigned long long t;
  if (W == 1) {
    t = (x ^ (x >> 7)) & 0x00AA00AA00AA00AAull;  x ^= t ^ (t << 7);
    t = (x ^ (x >> 14)) & 0x0000CCCC0000CCCCull; x ^= t ^ (t << 14);
    t = (x ^ (x >> 28)) & 0x00000000F0F0F0F0ull; x ^= t ^ (t << 28);
  } else if (W == 2) {
    t = (x ^ (x >> 6)) & 0x00CC00CC00CC00CCull;  x ^= t ^ (t << 6);
    t = (x ^ (x >> 12)) & 0x0000F0F00000F0F0ull; x ^= t ^ (t << 12);
  } else {
    t = (x ^ (x >> 4)) & 0x00F000F000F000F0ull;  x ^= t ^ (t << 4);
  }
  return x;
}

// n32 = number of 32-byte chunks, S = bytes per segment
template <int W, bool SUB>
__global__ void __launch_bounds__(256) bitswap_encode_fast(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, uint64_t n32,
                                                            uint64_t S, uint32_t thr /* threshold, < 256 */) {
  constexpr int P = 8 / W;          // planes = bytes per group
  constexpr int G = 32 / P;         // groups per thread = output bytes per plane per thread
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n32; t += stride) {
    uint4 a = ld_stream(reinterpret_cast<const uint4*>(in + t * 32));
    uint4 b = ld_stream(reinterpret_cast<const uint4*>(in + t * 32) + 1);
    if (SUB) {
      a.x = sat_sub_u8x4(a.x, thr); a.y = sat_sub_u8x4(a.y, thr); a.z = sat_sub_u8x4(a.z, thr); a.w = sat_sub_u8x4(a.w, thr);
      b.x = sat_sub_u8x4(b.x, thr); b.y = sat_sub_u8x4(b.y, thr); b.z = sat_sub_u8x4(b.z, thr); b.w = sat_sub_u8x4(b.w, thr);
    }
    unsigned long long c[4] = {((unsigned long long)a.y << 32) | a.x, ((unsigned long long)a.w << 32) | a.z,
                               ((unsigned long long)b.y << 32) | b.x, ((unsigned long long)b.w << 32) | b.z};
#pragma unroll
    for (int k = 0; k < 4; ++k) c[k] = transpose_atoms<W>(reverse_groups<W>(c[k]));
    // byte (o + p) of chunk k, o = start of group q inside the chunk, is plane p's byte for group q
#pragma unroll
    for (int p = 0; p < P; ++p) {
      uint32_t w[G / 4 > 0 ? G / 4 : 1];
#pragma unroll
      for (int k = 0; k < G / 4; ++k) w[k] = 0;
#pragma unroll
      for (int q = 0; q < G; ++q) {
        const int byte_index = q * P + p;          // in the thread's 32 transformed bytes
        const uint32_t v = (uint32_t)(c[byte_index >> 3] >> (8 * (byte_index & 7))) & 0xffu;
        w[q >> 2] |= v << (8 * (q & 3));
      }
      uint8_t* dst = out + (uint64_t)(P - 1 - p) * S + t * G;
      if (G == 4) st_stream(reinterpret_cast<uint32_t*>(dst), w[0]);
      else if (G == 8) st_stream(reinterpret_cast<uint2*>(dst), make_uint2(w[0], w[1]));
      else st_stream(reinterpret_cast<uint4*>(dst), make_uint4(w[0], w[1], w[2], w[3]));
    }
  }
}

template <int W>
__global__ void __launch_bounds__(256) bitswap_decode_fast(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, uint64_t n32,
                                                            uint64_t S) {
  constexpr int P = 8 / W;
  constexpr int G = 32 / P;
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n32; t += stride) {
    unsigned long long c[4] = {0, 0, 0, 0};
#pragma unroll
    for (int p = 0; p < P; ++p) {
      const uint8_t* src = in + (uint64_t)(P - 1 - p) * S + t * G;
      uint32_t w[4] = {0, 0, 0, 0};
      if (G == 4) w[0] = __ldg(reinterpret_cast<const uint32_t*>(src));
      else if (G == 8) { const uint2 v = __ldg(reinterpret_cast<const uint2*>(src)); w[0] = v.x; w[1] = v.y; }
      else { const uint4 v = ld_stream(reinterpret_cast<const uint4*>(src)); w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w; }
#pragma unroll
      for (int q = 0; q < G; ++q) {
        const int byte_index = q * P + p;
        const unsigned long long v = (w[q >> 2] >> (8 * (q & 3))) & 0xffu;
        c[byte_index >> 3] |= v << (8 * (byte_index & 7));
      }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) c[k] = reverse_groups<W>(transpose_atoms<W>(c[k]));
    st_stream(reinterpret_cast<uint4*>(out + t * 32), make_uint4((uint32_t)c[0], (uint32_t)(c[0] >> 32), (uint32_t)c[1], (uint32_t)(c[1] >> 32)));
    st_stream(reinterpret_cast<uint4*>(out + t * 32) + 1, make_uint4((uint32_t)c[2], (uint32_t)(c[2] >> 32), (uint32_t)c[3], (uint32_t)(c[3] >> 32)));
  }
}

// ---- uint8, generic path: any N, any alignment; one thread per group of P bytes -------------
template <int W, bool SUB>
__global__ void bitswap_encode_generic(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, uint64_t n, uint32_t thr) {
  constexpr int P = 8 / W;
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
      for (int j = 0; j < P; ++j) word |= ((v[j] >> (p * W)) & ((1u << W) - 1u)) << ((8 - W) - j * W);
      out[(uint64_t)(P - 1 - p) * S + g] = (uint8_t)word;
    }
  }
  if (blockIdx.x == 0) {  // verbatim tail (bitswap_scheme_impl.hpp:99-103)
    for (uint64_t i = S * P + threadIdx.x; i < n; i += blockDim.x) {
      uint32_t x = in[i];
      if (SUB) x = x > thr ? x - thr : 0;
      out[i] = (uint8_t)x;
    }
  }
}

template <int W>
__global__ void bitswap_decode_generic(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, uint64_t n) {
  constexpr int P = 8 / W;
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
      for (int p = 0; p < P; ++p) x |= ((w[p] >> ((8 - W) - j * W)) & ((1u << W) - 1u)) << (p * W);
      out[g * P + j] = (uint8_t)x;
    }
  }
  if (blockIdx.x == 0)
    for (uint64_t i = S * P + threadIdx.x; i < n; i += blockDim.x) out[i] = in[i];
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

// remove_background on uint8 (remove_background_scheme_impl.hpp:73-95 with raw_type = uint8_t)
__global__ void __launch_bounds__(256) remove_background_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, uint64_t n,
                                                                uint32_t thr) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool aligned = ((((uintptr_t)in) | ((uintptr_t)out)) & 15) == 0;
  const uint64_t nv = aligned ? n / 16 : 0;
  for (uint64_t i = tid; i < nv; i += stride) {
    uint4 v = ld_stream(reinterpret_cast<const uint4*>(in) + i);
    v.x = sat_sub_u8x4(v.x, thr); v.y = sat_sub_u8x4(v.y, thr); v.z = sat_sub_u8x4(v.z, thr); v.w = sat_sub_u8x4(v.w, thr);
    st_stream(reinterpret_cast<uint4*>(out) + i, v);
  }
  for (uint64_t i = nv * 16 + tid; i < n; i += stride) {
    const uint32_t x = in[i];
    out[i] = (uint8_t)(x > thr ? x - thr : 0);
  }
}

// the fast kernels take whole 128-voxel groups of 16-byte (uint8) / 32-byte (uint16) aligned buffers
template <typename T>
bool fast_ok(const T* a, const T* b, uint64_t n) {
  return n >= 128 && (n % 128 == 0) && (((uintptr_t)a | (uintptr_t)b) & (16 * sizeof(T) - 1)) == 0;
}

// T = uint8_t (W = 1, 2, 4) or uint16_t (W = 1, 2, 4, 8); the threshold is taken as a T, as the reference stores it
template <typename T, int W>
int launch_encode(const void* in_v, void* out_v, uint64_t n, int threshold, cudaStream_t st) {
  constexpr int P = 8 * (int)sizeof(T) / W;
  const T* in = static_cast<const T*>(in_v);
  T* out = static_cast<T*>(out_v);
  const bool sub = threshold > 0;
  const uint32_t thr = (T)threshold;
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

template <typename T, int W>
int launch_decode(const void* in_v, void* out_v, uint64_t n, cudaStream_t st) {
  constexpr int P = 8 * (int)sizeof(T) / W;
  const T* in = static_cast<const T*>(in_v);
  T* out = static_cast<T*>(out_v);
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

template <typename T>
int launch_remove_background(const void* in, void* out, uint64_t n, int threshold, cudaStream_t st) {
  if (n == 0) return 0;
  remove_background_kernel<<<grid_for(n * sizeof(T) / 16 + 1, 256), 256, 0, st>>>(static_cast<const T*>(in), static_cast<T*>(out), n,
                                                                                 (uint32_t)(T)threshold);
  SQYB_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
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

int k_bitswap_encode(int elem, int w, const void* in, void* out, uint64_t n, int threshold, cudaStream_t st) {
  const bool u8 = elem == 1;
  switch (w) {
    case 1: return u8 ? launch_encode<uint8_t, 1>(in, out, n, threshold, st) : launch_encode<uint16_t, 1>(in, out, n, threshold, st);
    case 2: return u8 ? launch_encode<uint8_t, 2>(in, out, n, threshold, st) : launch_encode<uint16_t, 2>(in, out, n, threshold, st);
    case 4: return u8 ? launch_encode<uint8_t, 4>(in, out, n, threshold, st) : launch_encode<uint16_t, 4>(in, out, n, threshold, st);
    case 8: return u8 ? -1 : launch_encode<uint16_t, 8>(in, out, n, threshold, st);
  }
  return -1;
}

int k_bitswap_decode(int elem, int w, const void* in, void* out, uint64_t n, cudaStream_t st) {
  const bool u8 = elem == 1;
  switch (w) {
    case 1: return u8 ? launch_decode<uint8_t, 1>(in, out, n, st) : launch_decode<uint16_t, 1>(in, out, n, st);
    case 2: return u8 ? launch_decode<uint8_t, 2>(in, out, n, st) : launch_decode<uint16_t, 2>(in, out, n, st);
    case 4: return u8 ? launch_decode<uint8_t, 4>(in, out, n, st) : launch_decode<uint16_t, 4>(in, out, n, st);
    case 8: return u8 ? -1 : launch_decode<uint16_t, 8>(in, out, n, st);
  }
  return -1;
}

int k_remove_background(int elem, const void* in, void* out, uint64_t n, int threshold, cudaStream_t st) {
  return elem == 1 ? launch_remove_background<uint8_t>(in, out, n, threshold, st)
                   : launch_remove_background<uint16_t>(in, out, n, threshold, st);
}

}  // namespace sqyb
