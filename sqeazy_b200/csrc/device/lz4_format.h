// LZ4 frame / block format constants shared by the GPU encoder, the GPU decoder and the host code.
// The reference's `lz4` stage emits LZ4 *Frame* streams through liblz4 (encoders/lz4.hpp:58-114,
// 214-242; encoders/lz4_utils.hpp:99-173); liblz4 itself is an un-vendored dependency, so the
// format below follows the published LZ4 Frame Format / Block Format descriptions (lz4 >= 1.8).
//
// Payload layout written by this library for `...->lz4`:
//   [skippable frame  : u32 magic 0x184D2A5B | u32 size | SqybIndex header | u32 block_word[nblocks]]
//   [LZ4 frame header : 04 22 4D 18 | FLG 0x60 (v1, independent blocks) | BD 0x40 (64 KiB max) | HC 0x82]
//   [block]*          : u32 size (bit31 = stored) | data        (blocks hold kLz4BlockBytes of input)
//   [EndMark          : u32 0]
// Everything in front of the first block is written by lz4_write_prefix and read back by lz4_read_prefix (below).
// The skippable frame is legal LZ4F (decoders skip it; verified against the reference's own decode
// loop, encoders/lz4.hpp:257-339 + liblz4 1.9.4) and lets the GPU decoder find every block without
// walking the stream sequentially.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define SQYB_HD __host__ __device__
#else
#define SQYB_HD
#endif

namespace sqyb {

constexpr uint32_t kLz4FrameMagic = 0x184D2204u;
constexpr uint32_t kLz4SkippableMagicBase = 0x184D2A50u;   // ..5F
constexpr uint32_t kSqybSkippableMagic = 0x184D2A5Bu;
constexpr uint32_t kSqybIndexMagic = 0x42595153u;           // "SQYB"
constexpr uint32_t kLz4StoredFlag = 0x80000000u;

constexpr int kLz4BlockBytes = 16384;   // input bytes per LZ4 block produced by the GPU encoder
constexpr int kLz4MinMatch = 4;
constexpr int kLz4LastLiterals = 5;     // the last 5 bytes of a block are always literals
constexpr int kLz4MFLimit = 12;         // the last match starts at least 12 bytes before the block end

struct SqybIndexHeader {                // 32 bytes, little endian
  uint32_t magic;                       // kSqybIndexMagic
  uint32_t version;                     // 1
  uint32_t block_bytes;                 // input bytes per block (last block may be shorter)
  uint32_t nblocks;
  uint64_t raw_bytes;                   // total decoded bytes of the frame that follows
  uint64_t frame_bytes;                 // bytes of the LZ4 frame that follows (header .. EndMark), filled by the encoder
};

constexpr uint64_t kSkippableHeaderBytes = 8;
constexpr uint64_t kLz4FrameHeaderBytes = 7;
constexpr uint64_t kLz4EndMarkBytes = 4;

SQYB_HD static inline uint64_t lz4_nblocks(uint64_t raw_bytes) { return (raw_bytes + kLz4BlockBytes - 1) / kLz4BlockBytes; }
// bytes in front of the first LZ4 block header
SQYB_HD static inline uint64_t lz4_prefix_bytes(uint64_t nblocks) {
  return kSkippableHeaderBytes + sizeof(SqybIndexHeader) + 4 * nblocks + kLz4FrameHeaderBytes;
}
// worst case payload: every block stored
SQYB_HD static inline uint64_t lz4_payload_bound(uint64_t raw_bytes) {
  const uint64_t nb = lz4_nblocks(raw_bytes);
  return lz4_prefix_bytes(nb) + raw_bytes + 4 * nb + kLz4EndMarkBytes;
}

SQYB_HD static inline void lz4_put32(uint8_t* p, uint32_t v) { for (int k = 0; k < 4; ++k) p[k] = (uint8_t)(v >> (8 * k)); }
SQYB_HD static inline void lz4_put64(uint8_t* p, uint64_t v) { for (int k = 0; k < 8; ++k) p[k] = (uint8_t)(v >> (8 * k)); }
SQYB_HD static inline uint32_t lz4_get32(const uint8_t* p) { uint32_t v = 0; for (int k = 0; k < 4; ++k) v |= (uint32_t)p[k] << (8 * k); return v; }
SQYB_HD static inline uint64_t lz4_get64(const uint8_t* p) { return lz4_get32(p) | (uint64_t)lz4_get32(p + 4) << 32; }

// the lz4_prefix_bytes(nblocks) bytes in front of the first block header: skippable header, index header and LZ4 frame header.
// The block words (dst + kSkippableHeaderBytes + sizeof(SqybIndexHeader)) are left to the caller. Returns lz4_prefix_bytes(nblocks).
SQYB_HD static inline uint64_t lz4_write_prefix(uint8_t* dst, uint32_t nblocks, uint64_t raw_bytes, uint64_t frame_bytes) {
  lz4_put32(dst, kSqybSkippableMagic);
  lz4_put32(dst + 4, (uint32_t)(sizeof(SqybIndexHeader) + 4ull * nblocks));
  lz4_put32(dst + 8, kSqybIndexMagic);
  lz4_put32(dst + 12, 1u);
  lz4_put32(dst + 16, (uint32_t)kLz4BlockBytes);
  lz4_put32(dst + 20, nblocks);
  lz4_put64(dst + 24, raw_bytes);
  lz4_put64(dst + 32, frame_bytes);
  const uint64_t f = kSkippableHeaderBytes + sizeof(SqybIndexHeader) + 4ull * nblocks;
  lz4_put32(dst + f, kLz4FrameMagic);
  dst[f + 4] = 0x60;  // FLG: version 01, block independent
  dst[f + 5] = 0x40;  // BD: 64 KiB max block
  dst[f + 6] = 0x82;  // HC = (xxh32(FLG BD) >> 8) & 0xff
  return f + kLz4FrameHeaderBytes;
}

// reads the prefix lz4_write_prefix writes from the front of an n-byte payload (host memory). False when the payload does not
// start with one whose frame runs to the end of the payload. The `nblocks` block words behind the index header are not checked.
static inline bool lz4_read_prefix(const uint8_t* p, uint64_t n, SqybIndexHeader* out) {
  constexpr uint64_t kIndexEnd = kSkippableHeaderBytes + sizeof(SqybIndexHeader);
  if (n < kIndexEnd || lz4_get32(p) != kSqybSkippableMagic || lz4_get32(p + 8) != kSqybIndexMagic || lz4_get32(p + 12) != 1u)
    return false;
  SqybIndexHeader h{kSqybIndexMagic, 1u, lz4_get32(p + 16), lz4_get32(p + 20), lz4_get64(p + 24), lz4_get64(p + 32)};
  const uint64_t prefix = lz4_prefix_bytes(h.nblocks), f = prefix - kLz4FrameHeaderBytes;
  if (lz4_get32(p + 4) != sizeof(SqybIndexHeader) + 4ull * h.nblocks || n < prefix + kLz4EndMarkBytes ||
      lz4_get32(p + f) != kLz4FrameMagic || f + h.frame_bytes != n)
    return false;
  *out = h;
  return true;
}

}  // namespace sqyb
