// bitshuffle head filter for uint16 and uint8 stacks on sm_100a (SURVEY §8f-4).
//
// Replaces bitshuffle_scheme<uint16_t>::encode/decode (encoders/bitshuffle_scheme_impl.hpp:91-160), which hands the buffer
// to bshuf_bitshuffle / bshuf_bitunshuffle of the third-party bitshuffle library (github.com/kiyo-masui/bitshuffle,
// downloaded at cmake time by the reference, not in its tree). Layout of that library's output (bitshuffle_core.c:
// bshuf_blocked_wrap_fun + bshuf_trans_bit_elem), restated in oracle/sqy_oracle.c:
//   * the elements are cut into blocks of `block_size` elements (0 = default: 8192 bytes / element size = 4096, a multiple
//     of 8), then one block of the remaining elements rounded down to a multiple of 8, then < 8 left-over elements verbatim;
//   * a block of S elements becomes 16 bit rows of S/8 bytes: row r = bit r of every element (row 0 = least significant
//     bit), element e of the block in byte e/8 at bit e%8.
// One pass: a thread takes 32 consecutive elements with two 256-bit loads, transposes the two 16x16 bit matrices they form
// (both at once, one in each half of 16 registers: 4 masked delta-swap stages) and stores one 32-bit word per bit row; a
// warp's words are 128 contiguous bytes of every row. Blocks whose size is not a multiple of 32 (odd block_size, the last
// partial block) and unaligned buffers take a thread-per-8-elements kernel.
#include "bit_transpose16.h"
#include "common.cuh"
#include "kernels.h"

namespace sqyb {
namespace {

__device__ __forceinline__ void ld256(const void* p, uint32_t* r) {
  asm volatile("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "l"(p));
}
__device__ __forceinline__ void st256(void* p, const uint32_t* r) {
  asm volatile("st.global.L1::no_allocate.v8.u32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(r[0]), "r"(r[1]),
               "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}

// n32 chunks of 32 elements inside whole blocks of bs elements (bs % 32 == 0)
__global__ void __launch_bounds__(256) bitshuffle16_encode_fast(const uint16_t* __restrict__ in, uint8_t* __restrict__ out,
                                                                 uint64_t n32, uint32_t bs) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  const uint32_t row_bytes = bs / 8, per_block = bs / 32;
  for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n32; t += stride) {
    uint32_t L[16], w[16];
    ld256(in + t * 32, L);
    ld256(in + t * 32 + 16, L + 8);
    // w[i] = element i | element 16+i << 16
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      w[2 * k] = __byte_perm(L[k], L[8 + k], 0x5410);
      w[2 * k + 1] = __byte_perm(L[k], L[8 + k], 0x7632);
    }
    transpose16x16_pairs(w);   // w[r] = bit r of the 32 elements, element e at bit e
    const uint64_t blk = t / per_block;
    const uint32_t c = (uint32_t)(t - blk * per_block);
    uint8_t* o = out + blk * 2ull * bs + 4u * c;
#pragma unroll
    for (int r = 0; r < 16; ++r) st_stream(reinterpret_cast<uint32_t*>(o + (uint64_t)r * row_bytes), w[r]);
  }
}

__global__ void __launch_bounds__(256) bitshuffle16_decode_fast(const uint8_t* __restrict__ in, uint16_t* __restrict__ out,
                                                                 uint64_t n32, uint32_t bs) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  const uint32_t row_bytes = bs / 8, per_block = bs / 32;
  for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n32; t += stride) {
    const uint64_t blk = t / per_block;
    const uint32_t c = (uint32_t)(t - blk * per_block);
    const uint8_t* s = in + blk * 2ull * bs + 4u * c;
    uint32_t w[16], L[16];
#pragma unroll
    for (int r = 0; r < 16; ++r) w[r] = ld_stream(reinterpret_cast<const uint32_t*>(s + (uint64_t)r * row_bytes));
    transpose16x16_pairs(w);   // w[i] = element i | element 16+i << 16
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      L[k] = __byte_perm(w[2 * k], w[2 * k + 1], 0x5410);
      L[8 + k] = __byte_perm(w[2 * k], w[2 * k + 1], 0x7632);
    }
    st256(out + t * 32, L);
    st256(out + t * 32 + 16, L + 8);
  }
}

// any block geometry, any alignment: a thread per group of 8 elements (one byte of each of the 16 rows).
// groups are numbered over the whole buffer; `first` elements precede the region, its blocks have bs elements, the
// region holds `count` elements (multiple of 8) = whole blocks, or one partial block (bs = count).
__global__ void __launch_bounds__(256) bitshuffle16_encode_generic(const uint16_t* __restrict__ in, uint8_t* __restrict__ out,
                                                                    uint64_t first, uint64_t count, uint32_t bs) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x, groups = count / 8;
  const uint32_t row_bytes = bs / 8;
  for (uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += stride) {
    const uint64_t blk = g / row_bytes;
    const uint32_t c = (uint32_t)(g - blk * row_bytes);
    const uint16_t* s = in + first + g * 8;
    uint32_t x[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] = s[i];
    uint8_t* o = out + 2 * first + blk * 2ull * bs + c;
#pragma unroll
    for (int r = 0; r < 16; ++r) {
      uint32_t b = 0;
#pragma unroll
      for (int i = 0; i < 8; ++i) b |= ((x[i] >> r) & 1u) << i;
      o[(uint64_t)r * row_bytes] = (uint8_t)b;
    }
  }
}

__global__ void __launch_bounds__(256) bitshuffle16_decode_generic(const uint8_t* __restrict__ in, uint16_t* __restrict__ out,
                                                                    uint64_t first, uint64_t count, uint32_t bs) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x, groups = count / 8;
  const uint32_t row_bytes = bs / 8;
  for (uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += stride) {
    const uint64_t blk = g / row_bytes;
    const uint32_t c = (uint32_t)(g - blk * row_bytes);
    const uint8_t* s = in + 2 * first + blk * 2ull * bs + c;
    uint32_t x[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int r = 0; r < 16; ++r) {
      const uint32_t b = s[(uint64_t)r * row_bytes];
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i] |= ((b >> i) & 1u) << r;
    }
    uint16_t* o = out + first + g * 8;
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = (uint16_t)x[i];
  }
}

__global__ void copy_tail16(const uint16_t* __restrict__ in, uint16_t* __restrict__ out, uint64_t first, uint32_t count) {
  if (threadIdx.x < count) out[first + threadIdx.x] = in[first + threadIdx.x];
}

// ---- uint8 elements (the *_UI8 entry points): 8 bit rows per block, default blocks of 8192 elements ----
// A thread takes 32 bytes (one 256-bit load) = four groups of 8; the 8x8 bit transpose of a group (64-bit delta swaps) leaves
// in byte r the bits r of its 8 elements, i.e. the group's byte of row r; the four groups' bytes make the 32-bit word the
// thread stores into row r.
__global__ void __launch_bounds__(256) bitshuffle8_encode_fast(const uint8_t* __restrict__ in, uint8_t* __restrict__ out,
                                                                uint64_t n32, uint32_t bs) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  const uint32_t row_bytes = bs / 8, per_block = bs / 32;
  for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n32; t += stride) {
    uint32_t L[8];
    ld256(in + t * 32, L);
    uint32_t lo[4], hi[4];
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      const uint64_t x = transpose8x8((uint64_t)L[2 * g] | ((uint64_t)L[2 * g + 1] << 32));
      lo[g] = (uint32_t)x;          // rows 0..3 of group g
      hi[g] = (uint32_t)(x >> 32);  // rows 4..7
    }
    const uint64_t blk = t / per_block;
    const uint32_t c = (uint32_t)(t - blk * per_block);
    uint8_t* o = out + blk * (uint64_t)bs + 4u * c;
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const uint32_t* q = r < 4 ? lo : hi;
      const int b = r & 3;          // byte b of the four group words
      const uint32_t s01 = __byte_perm(q[0], q[1], 0x0040 + b * 0x0011);   // (q0.b, q1.b, -, -)
      const uint32_t s23 = __byte_perm(q[2], q[3], 0x0040 + b * 0x0011);
      st_stream(reinterpret_cast<uint32_t*>(o + (uint64_t)r * row_bytes), __byte_perm(s01, s23, 0x5410));
    }
  }
}

__global__ void __launch_bounds__(256) bitshuffle8_decode_fast(const uint8_t* __restrict__ in, uint8_t* __restrict__ out,
                                                                uint64_t n32, uint32_t bs) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  const uint32_t row_bytes = bs / 8, per_block = bs / 32;
  for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n32; t += stride) {
    const uint64_t blk = t / per_block;
    const uint32_t c = (uint32_t)(t - blk * per_block);
    const uint8_t* s = in + blk * (uint64_t)bs + 4u * c;
    uint32_t w[8], L[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) w[r] = ld_stream(reinterpret_cast<const uint32_t*>(s + (uint64_t)r * row_bytes));
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      // byte g of the eight row words = the transposed group g
      const uint32_t sel = 0x0040 + g * 0x0011;
      const uint32_t lo = __byte_perm(__byte_perm(w[0], w[1], sel), __byte_perm(w[2], w[3], sel), 0x5410);
      const uint32_t hi = __byte_perm(__byte_perm(w[4], w[5], sel), __byte_perm(w[6], w[7], sel), 0x5410);
      const uint64_t x = transpose8x8((uint64_t)lo | ((uint64_t)hi << 32));
      L[2 * g] = (uint32_t)x;
      L[2 * g + 1] = (uint32_t)(x >> 32);
    }
    st256(out + t * 32, L);
  }
}

// any geometry / alignment: a thread per group of 8 elements
__global__ void __launch_bounds__(256) bitshuffle8_generic(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, uint64_t first,
                                                            uint64_t count, uint32_t bs, int decode) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x, groups = count / 8;
  const uint32_t row_bytes = bs / 8;
  for (uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += stride) {
    const uint64_t blk = g / row_bytes;
    const uint32_t c = (uint32_t)(g - blk * row_bytes);
    const uint64_t rows = first + blk * (uint64_t)bs + c, elems = first + g * 8;
    uint64_t x = 0;
    if (decode) {
#pragma unroll
      for (int r = 0; r < 8; ++r) x |= (uint64_t)in[rows + (uint64_t)r * row_bytes] << (8 * r);
      x = transpose8x8(x);
#pragma unroll
      for (int i = 0; i < 8; ++i) out[elems + i] = (uint8_t)(x >> (8 * i));
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) x |= (uint64_t)in[elems + i] << (8 * i);
      x = transpose8x8(x);
#pragma unroll
      for (int r = 0; r < 8; ++r) out[rows + (uint64_t)r * row_bytes] = (uint8_t)(x >> (8 * r));
    }
  }
}

__global__ void copy_tail8(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, uint64_t first, uint32_t count) {
  if (threadIdx.x < count) out[first + threadIdx.x] = in[first + threadIdx.x];
}

}  // namespace

uint32_t bitshuffle_block_elems(uint32_t block_size, int elem_size) {
  // bshuf_default_block_size: 8192 target bytes / element size, rounded down to a multiple of 8, at least 128
  if (block_size) return block_size;
  uint32_t b = 8192u / (uint32_t)elem_size;
  b = (b / 8u) * 8u;
  return b < 128u ? 128u : b;
}

// encode == true: in = elements, out = shuffled bytes; false: the inverse. Returns -81 (the library's code) for a block
// size that is not a multiple of 8.
static int run_bitshuffle16(bool encode, const void* in, void* out, uint64_t n, uint32_t block_size, cudaStream_t st) {
  const uint32_t bs = bitshuffle_block_elems(block_size, 2);
  if (bs % 8u) return -81;
  if (n == 0) return 0;
  const uint64_t full = (n / bs) * bs;                 // elements in whole blocks
  const uint64_t last = ((n - full) / 8) * 8;          // one more block of the rest, rounded down to a multiple of 8
  const uint64_t left = n - full - last;               // < 8 elements, verbatim
  const bool aligned = ((((uintptr_t)in) | ((uintptr_t)out)) & 31) == 0;
  const uint16_t* e_in = static_cast<const uint16_t*>(in);
  uint16_t* e_out = static_cast<uint16_t*>(out);
  const uint8_t* b_in = static_cast<const uint8_t*>(in);
  uint8_t* b_out = static_cast<uint8_t*>(out);
  if (full) {
    if (aligned && bs % 32u == 0) {
      if (encode) bitshuffle16_encode_fast<<<grid_for(full / 32, 256), 256, 0, st>>>(e_in, b_out, full / 32, bs);
      else bitshuffle16_decode_fast<<<grid_for(full / 32, 256), 256, 0, st>>>(b_in, e_out, full / 32, bs);
    } else {
      if (encode) bitshuffle16_encode_generic<<<grid_for(full / 8, 256), 256, 0, st>>>(e_in, b_out, 0, full, bs);
      else bitshuffle16_decode_generic<<<grid_for(full / 8, 256), 256, 0, st>>>(b_in, e_out, 0, full, bs);
    }
    SQYB_COUNT_LAUNCH(1);
  }
  if (last) {
    if (encode) bitshuffle16_encode_generic<<<grid_for(last / 8, 256), 256, 0, st>>>(e_in, b_out, full, last, (uint32_t)last);
    else bitshuffle16_decode_generic<<<grid_for(last / 8, 256), 256, 0, st>>>(b_in, e_out, full, last, (uint32_t)last);
    SQYB_COUNT_LAUNCH(1);
  }
  if (left) {
    copy_tail16<<<1, 32, 0, st>>>(e_in, e_out, full + last, (uint32_t)left);
    SQYB_COUNT_LAUNCH(1);
  }
  return (int)cudaGetLastError();
}

static int run_bitshuffle8(bool encode, const uint8_t* in, uint8_t* out, uint64_t n, uint32_t block_size, cudaStream_t st) {
  const uint32_t bs = bitshuffle_block_elems(block_size, 1);
  if (bs % 8u) return -81;
  if (n == 0) return 0;
  const uint64_t full = (n / bs) * bs, last = ((n - full) / 8) * 8, left = n - full - last;
  const bool aligned = ((((uintptr_t)in) | ((uintptr_t)out)) & 31) == 0;
  if (full) {
    if (aligned && bs % 32u == 0) {
      if (encode) bitshuffle8_encode_fast<<<grid_for(full / 32, 256), 256, 0, st>>>(in, out, full / 32, bs);
      else bitshuffle8_decode_fast<<<grid_for(full / 32, 256), 256, 0, st>>>(in, out, full / 32, bs);
    } else {
      bitshuffle8_generic<<<grid_for(full / 8, 256), 256, 0, st>>>(in, out, 0, full, bs, encode ? 0 : 1);
    }
    SQYB_COUNT_LAUNCH(1);
  }
  if (last) {
    bitshuffle8_generic<<<grid_for(last / 8, 256), 256, 0, st>>>(in, out, full, last, (uint32_t)last, encode ? 0 : 1);
    SQYB_COUNT_LAUNCH(1);
  }
  if (left) {
    copy_tail8<<<1, 32, 0, st>>>(in, out, full + last, (uint32_t)left);
    SQYB_COUNT_LAUNCH(1);
  }
  return (int)cudaGetLastError();
}

int k_bitshuffle_encode(int elem, const void* in, void* out, uint64_t n, uint32_t block_size, cudaStream_t st) {
  return elem == 1 ? run_bitshuffle8(true, static_cast<const uint8_t*>(in), static_cast<uint8_t*>(out), n, block_size, st)
                   : run_bitshuffle16(true, in, out, n, block_size, st);
}
int k_bitshuffle_decode(int elem, const void* in, void* out, uint64_t n, uint32_t block_size, cudaStream_t st) {
  return elem == 1 ? run_bitshuffle8(false, static_cast<const uint8_t*>(in), static_cast<uint8_t*>(out), n, block_size, st)
                   : run_bitshuffle16(false, in, out, n, block_size, st);
}

}  // namespace sqyb
