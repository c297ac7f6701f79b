// Thread program of the fast bitswapN transpose (uint16, w = W bits per plane): one thread turns 32 consecutive voxels
// into W consecutive 32-bit words of each of the P = 16/W planes, or back. bitswap.cu runs it over a whole volume; the
// LZ4 block decoder (lz4_decode.cu) runs it over the voxels of one range of 16 KiB plane blocks as soon as the range is
// decoded. Layout and semantics: bitswap.cu.
#pragma once
#include "common.cuh"

namespace sqyb {
namespace bitswap_thread {

template <int W>
struct Geo {
  static constexpr int P = 16 / W;   // planes == voxels per group
  static constexpr int SETS = W;     // register sets per thread (32 voxels / 2P)
};

__host__ __device__ constexpr uint32_t atom_mask16(int W, int k) {
  // atoms c (c = 0 at bit 0) with (c & k) == 0
  uint32_t m = 0;
  for (int c = 0; c < 16 / W; ++c)
    if ((c & k) == 0) m |= ((1u << W) - 1u) << (c * W);
  return m;
}

// PxP transpose of W-bit atoms in registers: log2(P) masked delta-swap stages. The stage that moves whole bytes (shift 8,
// mask 0x00ff00ff for every W) is two byte permutes per register pair instead of shifts and masks.
template <int W>
__device__ __forceinline__ void transpose_sets(uint32_t (&reg)[16]) {
  constexpr int P = Geo<W>::P;
#pragma unroll
  for (int s = 0; s < Geo<W>::SETS; ++s) {
#pragma unroll
    for (int k = P / 2; k >= 1; k >>= 1) {
      const uint32_t m16 = atom_mask16(W, k);
      const uint32_t mask = m16 | (m16 << 16);
      const int sh = k * W;
#pragma unroll
      for (int r = 0; r < P; ++r) {
        if ((r & k) == 0) {
          uint32_t a = reg[s * P + r], b = reg[s * P + r + k];
          if (sh == 8) {
            const uint32_t a2 = __byte_perm(a, b, 0x6240);   // a0 b0 a2 b2
            b = __byte_perm(a, b, 0x7351);                   // a1 b1 a3 b3
            a = a2;
          } else {
            const uint32_t t = ((a >> sh) ^ b) & mask;
            b ^= t;
            a ^= t << sh;
          }
          reg[s * P + r] = a;
          reg[s * P + r + k] = b;
        }
      }
    }
  }
}

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

// Plane loads of the decode. A buffer written by an earlier launch goes through the read-only path; one written by other
// warps of the same launch (the fused decoder) must not: ld.global.cg reads it from L2, after the writers' fence + counter.
template <bool L2ONLY>
__device__ __forceinline__ uint32_t ld_plane(const uint32_t* p) {
  if (!L2ONLY) return __ldg(p);
  uint32_t r;
  asm volatile("ld.global.cg.u32 %0, [%1];" : "=r"(r) : "l"(p));
  return r;
}
template <bool L2ONLY>
__device__ __forceinline__ uint2 ld_plane(const uint2* p) {
  if (!L2ONLY) return __ldg(p);
  uint2 r;
  asm volatile("ld.global.cg.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
  return r;
}
template <bool L2ONLY>
__device__ __forceinline__ uint4 ld_plane(const uint4* p) {
  if (!L2ONLY) return ld_stream(p);
  uint4 r;
  asm volatile("ld.global.cg.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
template <bool L2ONLY>
__device__ __forceinline__ void ld_plane256(const void* p, uint32_t* r) {
  if (!L2ONLY) {
    ld256(p, r);
    return;
  }
  asm volatile("ld.global.cg.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "l"(p));
}

// voxels [32t, 32t+32) of `in` -> words of every plane; plane p lands in segment P-1-p of `out` (segment stride S words of
// 16 bits). SUB: the threshold `thr` is subtracted (saturating) on the way in.
template <int W, bool SUB>
__device__ __forceinline__ void encode_chunk(const uint16_t* __restrict__ in, uint16_t* __restrict__ out, uint64_t t, uint64_t S,
                                             uint32_t thr) {
  constexpr int P = Geo<W>::P;
  uint32_t L[16];
  ld256(in + t * 32, L);
  ld256(in + t * 32 + 16, L + 8);
  if (SUB) {
#pragma unroll
    for (int k = 0; k < 16; ++k) L[k] = sat_sub_u16x2(L[k], thr);
  }
  uint32_t reg[16];
#pragma unroll
  for (int s = 0; s < Geo<W>::SETS; ++s) {
#pragma unroll
    for (int r = 0; r < P; ++r) {
      const int j = P - 1 - r;
      const int a = (2 * s) * P + j, b = (2 * s + 1) * P + j;
      const uint32_t sel = (2 * (a & 1)) | ((2 * (a & 1) + 1) << 4) | ((4 + 2 * (b & 1)) << 8) | ((5 + 2 * (b & 1)) << 12);
      reg[s * P + r] = __byte_perm(L[a >> 1], L[b >> 1], sel);
    }
  }
  transpose_sets<W>(reg);
  // plane p -> segment (P-1-p); this chunk's first group index is t*32/P
#pragma unroll
  for (int p = 0; p < P; ++p) {
    uint32_t* dst = reinterpret_cast<uint32_t*>(out + (uint64_t)(P - 1 - p) * S + t * (32 / P));
    if (W == 1) {
      st_stream(dst, reg[p]);
    } else if (W == 2) {
      st_stream(reinterpret_cast<uint2*>(dst), make_uint2(reg[p], reg[P + p]));
    } else if (W == 4) {
      st_stream(reinterpret_cast<uint4*>(dst), make_uint4(reg[p], reg[P + p], reg[2 * P + p], reg[3 * P + p]));
    } else {
      uint32_t v[8];
#pragma unroll
      for (int s = 0; s < 8; ++s) v[s] = reg[s * P + p];
      st256(dst, v);
    }
  }
}

// the inverse in two steps, so that a caller can have the loads of several chunks in flight: the words of every plane that
// voxels [32t, 32t+32) were turned into ...
template <int W, bool L2ONLY>
__device__ __forceinline__ void load_planes(const uint16_t* __restrict__ in, uint64_t t, uint64_t S, uint32_t (&reg)[16]) {
  constexpr int P = Geo<W>::P;
#pragma unroll
  for (int p = 0; p < P; ++p) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(in + (uint64_t)(P - 1 - p) * S + t * (32 / P));
    if (W == 1) {
      reg[p] = ld_plane<L2ONLY>(src);
    } else if (W == 2) {
      const uint2 v = ld_plane<L2ONLY>(reinterpret_cast<const uint2*>(src));
      reg[p] = v.x; reg[P + p] = v.y;
    } else if (W == 4) {
      const uint4 v = ld_plane<L2ONLY>(reinterpret_cast<const uint4*>(src));
      reg[p] = v.x; reg[P + p] = v.y; reg[2 * P + p] = v.z; reg[3 * P + p] = v.w;
    } else {
      uint32_t v[8];
      ld_plane256<L2ONLY>(src, v);
#pragma unroll
      for (int s = 0; s < 8; ++s) reg[s * P + p] = v[s];
    }
  }
}

// ... and those words back into the 32 voxels, two to a word (voxel 2k in the low half of L[k]) ...
template <int W>
__device__ __forceinline__ void voxels_of(uint32_t (&reg)[16], uint32_t (&L)[16]) {
  constexpr int P = Geo<W>::P;
  transpose_sets<W>(reg);  // the atom transpose is an involution
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const int m0 = 2 * k;
    const int g = m0 / P, j0 = m0 % P, s = g / 2, h = g & 1;
    const uint32_t sel = (2 * h) | ((2 * h + 1) << 4) | ((4 + 2 * h) << 8) | ((5 + 2 * h) << 12);
    L[k] = __byte_perm(reg[s * P + (P - 1 - j0)], reg[s * P + (P - 2 - j0)], sel);
  }
}

// ... stored in place
template <int W>
__device__ __forceinline__ void store_voxels(uint32_t (&reg)[16], uint16_t* __restrict__ out, uint64_t t) {
  uint32_t L[16];
  voxels_of<W>(reg, L);
  st256(out + t * 32, L);
  st256(out + t * 32 + 16, L + 8);
}

template <int W, bool L2ONLY>
__device__ __forceinline__ void decode_chunk(const uint16_t* __restrict__ in, uint16_t* __restrict__ out, uint64_t t, uint64_t S) {
  uint32_t reg[16];
  load_planes<W, L2ONLY>(in, t, S, reg);
  store_voxels<W>(reg, out, t);
}

}  // namespace bitswap_thread
}  // namespace sqyb
