// LZ4 frame decoder for sm_100a: decodes any concatenation of LZ4 frames (what the reference's
// sequential loop accepts, encoders/lz4.hpp:257-339): frames written by this library (independent
// 16 KiB blocks + block index in a skippable frame), by the reference's parallel mode (one frame
// per chunk, encoders/lz4_utils.hpp:193-274) and by its serial mode / the sqy CLI default (one frame
// of block-LINKED 256 KiB blocks, encoders/lz4_utils.hpp:99-173, SURVEY F6).
//
// Stages (all on the GPU, no host round trip):
//   directory : one CTA parses the frame structure. A stream that is exactly one frame of this library (the common
//               case) is handed to lz4_tile_sums_kernel + lz4_expand_kernel, which build the block table from the
//               index frame with many CTAs; other index frames are scanned in place; foreign frames -> thread 0
//               walks the 4-byte block headers.
//   sizes     : only for foreign blocks whose decoded size is not implied (last block of a frame):
//               a warp per block walks the tokens without copying.
//   offsets   : one CTA prefix-sums decoded sizes into output offsets and validates the total (skipped on the fast path).
//   decode    : persistent grid, a warp per block of any size; stored blocks are copied and closed-form run blocks
//               filled with 16-byte stores in passing. Sequence headers are parsed 32 at a time (every lane
//               parses the bytes at ip+lane as if a token started there, the real chain is followed with one shuffle
//               per sequence), literals are copied by the lanes that own them, matches are replayed in order. The
//               last 2 KiB of output live in a shared-memory ring (match sources), the compressed stream in a 1 KiB
//               ring; complete 512-byte chunks are flushed with 16-byte stores. Far matches and bytes in front of a
//               linked block are read back from global memory; linked blocks wait on their predecessor's flag only
//               when a match reaches in front of the block.
#include "bitswap_thread.h"
#include "common.cuh"
#include "kernels.h"
#include "lz4_format.h"

#include <cstdlib>

namespace sqyb {
namespace {

constexpr uint32_t kNoLink = 0xFFFFFFFFu;
constexpr uint32_t kLinkHead = 0xFFFFFFFEu;   // first block of a block-linked frame: nothing in front of it, but successors link to it
constexpr uint32_t kDeferMin = 8;             // default: streams with at least this many linked blocks take the deferred-reference path

enum DecErr : uint32_t {
  kErrNone = 0,
  kErrBadMagic = 1,
  kErrTruncated = 2,
  kErrTooManyBlocks = 3,
  kErrBadBlock = 4,
  kErrSizeMismatch = 5,
  kErrBadHeader = 6,
};

struct DecCtl {          // lives at the start of the workspace
  uint32_t nblocks;
  uint32_t error;
  uint32_t ticket_size;
  uint32_t ticket_decode;
  uint32_t need_sizes;   // number of blocks whose decoded size must be measured
  uint32_t own;          // the stream is exactly one frame of this library; fast_nblk / fast_bb hold its geometry
  uint32_t reserved[2];
  // fast path: the stream is exactly one frame of this library -> the block table is built by many CTAs
  uint32_t fast, fast_nblk, fast_bb, fast_pad;
  unsigned long long fast_idx, fast_first, fast_raw;
  unsigned long long fast_end;   // first byte behind the frame's EndMark, as promised by the index header
  unsigned long long total_decoded;
  uint32_t nlinked;      // blocks that belong to block-linked frames
  uint32_t deferred;     // 1: those blocks are left to lz4_decode_deferred_kernel + the two resolve passes (k_lz4_decode_linked)
  uint32_t ticket_deferred, pad1;
  uint32_t set_ticket[32];   // work counters of the block-set launches (k_lz4_decode_run with count != 0)
};
static_assert(sizeof(DecCtl) <= 256, "DecCtl lives in the first 256 bytes of the workspace");

struct DecTables {
  unsigned long long* src_off;   // offset of block data in the stream
  unsigned long long* dst_off;   // offset in the output
  uint32_t* word;                // block header word (bit31 = stored)
  uint32_t* dsize;               // decoded size (0 = unknown until the size pass)
  uint32_t* link;                // previous block of the same linked frame or kNoLink
  uint32_t* done;                // completion flags for linked frames
  uint32_t* reach;               // linked blocks: bytes of their frame in front of them, at most 65535 (the directory stores
                                 // the frame's first block here, lz4_offsets_kernel turns it into the byte count)
  uint32_t* range;               // fused transpose: decoded blocks of each range of bit-plane blocks (lz4_decode_kernel)
};

__device__ __forceinline__ uint32_t rd32(const uint8_t* p) {
  return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}
__device__ __forceinline__ unsigned long long rd64(const uint8_t* p) {
  return (unsigned long long)rd32(p) | ((unsigned long long)rd32(p + 4) << 32);
}

// inclusive block scan of one value per thread (1024 threads); returns inclusive sum, total via smem
__device__ __forceinline__ unsigned long long block_scan_incl(unsigned long long v, unsigned long long* warp_sums,
                                                              unsigned long long& total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const unsigned long long t = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= d) v += t;
  }
  __syncthreads();
  if (lane == 31) warp_sums[warp] = v;
  __syncthreads();
  if (warp == 0) {
    unsigned long long w = warp_sums[lane];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const unsigned long long t = __shfl_up_sync(0xffffffffu, w, d);
      if (lane >= d) w += t;
    }
    warp_sums[lane] = w;
  }
  __syncthreads();
  total = warp_sums[31];
  return v + (warp > 0 ? warp_sums[warp - 1] : 0ull);
}

constexpr int kDirThreads = 1024;
constexpr int kPerThread = 16;
constexpr uint32_t kTile = 4096;        // blocks per CTA tile of the fast table build (256 threads x 16)

__global__ void __launch_bounds__(kDirThreads) lz4_directory_kernel(const uint8_t* __restrict__ src, uint64_t src_bytes,
                                                                    DecCtl* ctl, DecTables T, uint32_t capacity,
                                                                    int measure_all, int defer_min) {
  __shared__ unsigned long long warp_sums[32];
  __shared__ unsigned long long sh_pos;
  __shared__ uint32_t sh_nb, sh_err, sh_mode, sh_need, sh_linked;
  __shared__ unsigned long long sh_args[4];
  const int tid = threadIdx.x;
  if (tid == 0) { sh_pos = 0; sh_nb = 0; sh_err = 0; sh_need = 0; sh_linked = 0; }
  __syncthreads();
  while (true) {
    // ---- thread 0 classifies what starts at pos ----
    if (tid == 0) {
      sh_mode = 0;  // 0 stop, 1 our indexed frame (parallel), 2 handled serially / continue
      const unsigned long long pos = sh_pos;
      if (sh_err == 0 && pos + 4 <= src_bytes) {
        const uint32_t magic = rd32(src + pos);
        if ((magic & 0xFFFFFFF0u) == kLz4SkippableMagicBase) {
          if (pos + 8 > src_bytes) { sh_err = kErrTruncated; }
          else {
            const unsigned long long size = rd32(src + pos + 4);
            const unsigned long long body = pos + 8;
            bool ours = false;
            if (magic == kSqybSkippableMagic && size >= sizeof(SqybIndexHeader) && body + size <= src_bytes &&
                rd32(src + body) == kSqybIndexMagic && rd32(src + body + 4) == 1u) {
              const uint32_t bb = rd32(src + body + 8), nblk = rd32(src + body + 12);
              const unsigned long long raw = rd64(src + body + 16), fbytes = rd64(src + body + 24);
              const unsigned long long fstart = body + size;
              if (size == sizeof(SqybIndexHeader) + 4ull * nblk && bb > 0 && fstart + fbytes <= src_bytes &&
                  fbytes >= kLz4FrameHeaderBytes + kLz4EndMarkBytes && rd32(src + fstart) == kLz4FrameMagic &&
                  (src[fstart + 4] & 0x1D) == 0 /* no checksums, no content size, no dict */ &&
                  (unsigned long long)nblk * bb >= raw && (nblk == 0 || (unsigned long long)(nblk - 1) * bb < raw)) {
                ours = true;
                const bool whole = pos == 0 && sh_nb == 0 && fstart + fbytes == src_bytes;
                if (whole) {
                  ctl->own = 1u;
                  ctl->fast_nblk = nblk;
                  ctl->fast_bb = bb;
                }
                if ((unsigned long long)sh_nb + nblk > capacity) sh_err = kErrTooManyBlocks;
                else if (whole && nblk >= 2u * kTile && bb <= 65536u) {
                  // the whole stream is one frame of ours: lz4_tile_sums_kernel + lz4_expand_kernel build the table
                  ctl->fast = 1u;
                  ctl->fast_idx = body + sizeof(SqybIndexHeader);
                  ctl->fast_first = fstart + kLz4FrameHeaderBytes;
                  ctl->fast_raw = raw;
                  ctl->fast_end = fstart + fbytes;
                  sh_nb = nblk;
                  sh_pos = src_bytes;
                  sh_mode = 2;
                } else {
                  sh_args[0] = body + sizeof(SqybIndexHeader);   // index words
                  sh_args[1] = fstart + kLz4FrameHeaderBytes;    // first block header
                  sh_args[2] = ((unsigned long long)bb << 32) | nblk;
                  sh_args[3] = raw;
                  sh_pos = fstart + fbytes;
                  sh_mode = 1;
                }
              }
            }
            if (!ours && sh_err == 0) {
              if (body + size > src_bytes) sh_err = kErrTruncated;
              else { sh_pos = body + size; sh_mode = 2; }
            }
          }
        } else if (magic == kLz4FrameMagic) {
          // ---- foreign frames: serial walk of the block headers. Consecutive foreign frames (the reference's multi-threaded
          // mode writes one per 256 KiB chunk: 8192 for a 2 GiB stack) are walked without leaving this thread — a round of
          // CTA barriers per frame cost more than the walk itself.
          unsigned long long fpos = pos;
          uint32_t nb = sh_nb;
          uint32_t pending = kNoLink, pending_max = 0;   // single-block frame whose size is still to be settled
          while (sh_err == 0) {
            if (fpos + 7 > src_bytes) { sh_err = kErrTruncated; break; }
            // another frame follows the pending single-block frame: a chunked writer fills every chunk but the last, so
            // its block is taken as full instead of being measured by a token walk (a wrong guess shows up as a size
            // mismatch and the caller retries with measure_all)
            if (pending != kNoLink) {
              T.dsize[pending] = pending_max;
              sh_need--;
              pending = kNoLink;
            }
            const uint32_t flg = src[fpos + 4], bd = src[fpos + 5];
            const bool indep = (flg >> 5) & 1, bchk = (flg >> 4) & 1, csz = (flg >> 3) & 1, cchk = (flg >> 2) & 1, dict = flg & 1;
            const uint32_t bsid = (bd >> 4) & 7;
            if ((flg >> 6) != 1 || bsid < 4) { sh_err = kErrBadHeader; break; }
            const uint32_t maxblock = 1u << (8 + 2 * bsid);
            unsigned long long p = fpos + 7 + (csz ? 8 : 0) + (dict ? 4 : 0);
            const uint32_t first_of_frame = nb;
            while (true) {
              if (p + 4 > src_bytes) { sh_err = kErrTruncated; break; }
              const uint32_t word = rd32(src + p);
              if (word == 0) { p += 4; break; }
              const uint32_t sz = word & 0x7FFFFFFFu;
              if (sz > maxblock || p + 4 + sz > src_bytes) { sh_err = kErrBadBlock; break; }
              if (nb >= capacity) { sh_err = kErrTooManyBlocks; break; }
              T.src_off[nb] = p + 4;
              T.word[nb] = word;
              // non-final blocks of liblz4 frames are full; measure_all drops that assumption
              T.dsize[nb] = (word & kLz4StoredFlag) ? sz : (measure_all ? 0u : maxblock);
              if (measure_all && !(word & kLz4StoredFlag)) sh_need++;
              T.link[nb] = indep ? kNoLink : (nb > first_of_frame ? nb - 1 : kLinkHead);
              T.reach[nb] = first_of_frame;
              if (!indep && nb > first_of_frame) sh_linked++;
              nb++;
              p += 4ull + sz + (bchk ? 4 : 0);
            }
            if (sh_err) break;
            if (cchk) p += 4;
            // the last block of a frame may be short: its size has to be measured
            if (!measure_all && nb > first_of_frame && !(T.word[nb - 1] & kLz4StoredFlag)) {
              T.dsize[nb - 1] = 0;
              sh_need++;
              if (nb == first_of_frame + 1) { pending = nb - 1; pending_max = maxblock; }
            }
            // a "linked" frame of a single block (the reference's multi-threaded mode: one frame per chunk) links nothing
            if (!indep && nb == first_of_frame + 1) T.link[first_of_frame] = kNoLink;
            fpos = p;
            if (fpos + 4 > src_bytes || rd32(src + fpos) != kLz4FrameMagic) break;   // something else follows: back to the classifier
          }
          if (sh_err == 0) {
            sh_nb = nb;
            sh_pos = fpos;
            sh_mode = 2;
          }
        } else {
          sh_err = kErrBadMagic;
        }
      }
    }
    __syncthreads();
    const uint32_t mode = sh_mode;
    if (mode == 0) break;
    if (mode == 1) {
      // ---- our frame: block table by parallel prefix sum over the index words ----
      const uint8_t* idx = src + sh_args[0];
      const bool idx_aligned = (((uintptr_t)idx) & 3) == 0;
      const unsigned long long first_hdr = sh_args[1];
      const uint32_t nblk = (uint32_t)(sh_args[2] & 0xFFFFFFFFu), bb = (uint32_t)(sh_args[2] >> 32);
      const unsigned long long raw = sh_args[3];
      const uint32_t nb0 = sh_nb;
      unsigned long long running = 0;
      for (uint32_t base = 0; base < nblk; base += kDirThreads * kPerThread) {
        uint32_t w[kPerThread];
        unsigned long long local = 0;
#pragma unroll
        for (int k = 0; k < kPerThread; ++k) {
          const uint32_t i = base + tid * kPerThread + k;
          w[k] = i < nblk ? (idx_aligned ? __ldg(reinterpret_cast<const uint32_t*>(idx) + i) : rd32(idx + 4ull * i)) : 0u;
          local += i < nblk ? 4ull + (w[k] & 0x7FFFFFFFu) : 0ull;
        }
        unsigned long long total;
        const unsigned long long incl = block_scan_incl(local, warp_sums, total);
        unsigned long long off = running + incl - local;
#pragma unroll
        for (int k = 0; k < kPerThread; ++k) {
          const uint32_t i = base + tid * kPerThread + k;
          if (i < nblk) {
            T.src_off[nb0 + i] = first_hdr + off + 4;
            T.word[nb0 + i] = w[k];
            const unsigned long long rem = raw - (unsigned long long)i * bb;
            T.dsize[nb0 + i] = (uint32_t)(rem < bb ? rem : bb);
            T.link[nb0 + i] = kNoLink;
            off += 4ull + (w[k] & 0x7FFFFFFFu);
          }
        }
        running += total;
        __syncthreads();
      }
      // The index words are untrusted input: the block offsets derived from them are only used when they add up to exactly
      // the frame the index header promised (which was checked against src_bytes above). Every src_off + csize then lies
      // inside the stream.
      if (tid == 0) {
        sh_nb = nb0 + nblk;
        if (first_hdr + running + kLz4EndMarkBytes != sh_pos) sh_err = kErrBadBlock;
      }
    }
    __syncthreads();
  }
  if (tid == 0) {
    ctl->nblocks = sh_nb;
    ctl->error = sh_err;
    ctl->need_sizes = sh_need;
    ctl->nlinked = sh_linked;
    ctl->deferred = (defer_min > 0 && sh_linked >= (uint32_t)defer_min) ? 1u : 0u;
  }
}

// ------------------------------------------------------------------------------------------------
// warp-level block decode
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t read_ext(const uint8_t* __restrict__ src, uint32_t& ip, uint32_t csize, int lane) {
  uint32_t add = 0;
  while (true) {
    const uint32_t idx = ip + lane;
    const uint32_t bval = idx < csize ? (uint32_t)__ldg(src + idx) : 0u;
    const uint32_t nz = __ballot_sync(0xffffffffu, bval != 255u);
    if (nz) {
      const int f = __ffs(nz) - 1;
      add += 255u * f + __shfl_sync(0xffffffffu, bval, f);
      ip += f + 1;
      return add;
    }
    add += 255u * 32u;
    ip += 32;
  }
}

// copy n bytes src -> dst (src read-only stream, arbitrary alignment), warp-cooperative
__device__ __forceinline__ void warp_copy_from_stream(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, uint32_t n,
                                                      int lane) {
  if (n >= 256 && (((uintptr_t)dst) & 15) == 0) {
    // 16-byte stores; source words fetched 4-byte aligned and funnel-shifted
    const uint32_t sh = ((uintptr_t)src & 3) * 8;
    const uint32_t* sw = reinterpret_cast<const uint32_t*>((uintptr_t)src & ~(uintptr_t)3);
    const uint32_t nvec = (n - 8) >> 4;  // keep the 5-word read inside [src, src+n)
    for (uint32_t v = lane; v < nvec; v += 32) {
      const uint32_t* p = sw + v * 4;
      const uint32_t x0 = __ldg(p), x1 = __ldg(p + 1), x2 = __ldg(p + 2), x3 = __ldg(p + 3), x4 = __ldg(p + 4);
      uint4 o;
      o.x = __funnelshift_r(x0, x1, sh);
      o.y = __funnelshift_r(x1, x2, sh);
      o.z = __funnelshift_r(x2, x3, sh);
      o.w = __funnelshift_r(x3, x4, sh);
      reinterpret_cast<uint4*>(dst)[v] = o;
    }
    const uint32_t done = nvec << 4;
    for (uint32_t k = done + lane; k < n; k += 32) dst[k] = __ldg(src + k);
  } else {
    for (uint32_t k = lane; k < n; k += 32) dst[k] = __ldg(src + k);
  }
}

// token walk without copying: decoded size of one block (for foreign blocks whose size is not implied)
__device__ __forceinline__ uint32_t measure_block_warp(const uint8_t* __restrict__ src, uint32_t csize, uint32_t& err, int lane) {
  uint32_t ip = 0, op = 0;
  while (ip < csize) {
    const uint32_t token = __ldg(src + ip);
    ip++;
    uint32_t lit = token >> 4;
    if (lit == 15) lit += read_ext(src, ip, csize, lane);
    if (ip + lit > csize) { err = kErrBadBlock; return op; }
    ip += lit;
    op += lit;
    if (ip >= csize) break;
    if (ip + 2 > csize) { err = kErrBadBlock; return op; }
    ip += 2;
    uint32_t mlen = token & 15u;
    if (mlen == 15) mlen += read_ext(src, ip, csize, lane);
    op += mlen + 4;
  }
  return op;
}

constexpr int kDecThreads = 128;

// ------------------------------------------------------------------------------------------------
// windowed block decoder: a warp per block of ANY size, independent or linked.
// The last kWin output bytes live in a shared-memory ring (match sources with offset <= kWin-64 — the
// overwhelming majority — never leave the SM); the ring is flushed to global memory in 512-byte chunks of
// 16-byte stores as soon as a chunk is complete. Matches that reach further back (or, in a linked frame, in
// front of the block) read the already flushed bytes with L1-bypassing loads. 3 KiB of shared memory per warp
// keeps 48 blocks in flight per SM instead of the 13 a whole 16 KiB block per warp would allow.
// ------------------------------------------------------------------------------------------------
constexpr uint32_t kWin = 2048;   // output ring bytes per warp
constexpr uint32_t kRing = 1024;  // compressed-stream ring per warp (two 512-byte chunks)
constexpr int kWinWarps = 8;
constexpr size_t kWinWarpSmem = kWin + kRing;
constexpr uint64_t kSmallStreamBytes = uint64_t(128) << 20;   // streams up to this size take the 64-register decoder
constexpr uint32_t kLitOwn = 4;          // literals an owner lane copies itself
constexpr uint32_t kBatchOut = 512;       // output bytes a batch of sequences may produce before the next flush
constexpr uint32_t kNear = kWin - kBatchOut - 64;
constexpr int kFarW = 8;                  // lanes that copy one short far match of a batch (four matches at a time) ...
constexpr uint32_t kFarMax = 24;          // ... of up to this many bytes; longer ones take the whole warp
                                          // (measured, cfg2 / plain planes / cfg1 decode in ms: off 5.81 / 6.60 / 0.76; 8 lanes, any length
                                          //  5.81 / 5.55 / 0.60; 8 lanes, <= 16 / 24 / 32 bytes 5.39 / 5.37 / 5.40 (plain 5.49, cfg1 0.61);
                                          //  16 lanes, <= 32: 5.38 / 5.76 / 0.66; 4 lanes: 6.23; the three steps' loads issued before the stores: 5.38 / 5.62 / 0.60)

__device__ __forceinline__ uint4 load_stream_piece(const uint8_t* addr, const uint8_t* sbeg, const uint8_t* send) {
  if (addr >= sbeg && addr + 16 <= send) return __ldg(reinterpret_cast<const uint4*>(addr));
  uint32_t w[4] = {0, 0, 0, 0};
  for (int k = 0; k < 16; ++k) {
    const uint8_t* p = addr + k;
    if (p >= sbeg && p < send) w[k >> 2] |= (uint32_t)__ldg(p) << (8 * (k & 3));
  }
  return make_uint4(w[0], w[1], w[2], w[3]);
}

// byte load that may be served by L1 (ld.global.ca); only for lines that no longer change, see the far-source copy
__device__ __forceinline__ uint8_t ld_l1_u8(const uint8_t* p) {
  uint32_t v;
  asm volatile("ld.global.ca.u8 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return (uint8_t)v;
}

struct WinOut {
  uint8_t* win;        // shared ring
  uint8_t* d;          // block's output in global memory
  uint32_t flushed;    // bytes of this block already written to global (multiple of 512 until the end)
  uint32_t dcap;       // decoded size the block table promises: nothing is ever written to global beyond it
  bool aligned;        // d is 16-byte aligned
  bool line_aligned;   // d is 128-byte aligned: the flushed part of the block ends on a cache line boundary
  bool overflow;
  int lane;
  // writes every complete 512-byte chunk below `op` to global memory
  __device__ __forceinline__ void flush_to(uint32_t op) {
    while (op - flushed >= 512u) {
      if (flushed + 512u > dcap) { overflow = true; return; }
      __syncwarp();
      if (aligned) {
        const uint4 v = *reinterpret_cast<const uint4*>(win + ((flushed + 16u * lane) & (kWin - 1)));
        st_stream(reinterpret_cast<uint4*>(d + flushed) + lane, v);
      } else {
        for (uint32_t k = lane; k < 512u; k += 32) d[flushed + k] = win[(flushed + k) & (kWin - 1)];
      }
      flushed += 512u;
    }
  }
  __device__ __forceinline__ void finish(uint32_t op) {
    __syncwarp();
    if (op > dcap) { overflow = true; return; }
    for (uint32_t k = flushed + lane; k < op; k += 32) d[k] = win[k & (kWin - 1)];
    flushed = op;
  }
};

// returns decoded size; err set on malformed input. Shared-memory accesses are masked into their rings and
// global writes are fenced by WinOut::dcap, so a corrupt stream can produce garbage but never an out-of-bounds
// access; the per-sequence work therefore carries no bounds branches, only a sticky `bad` flag.
__device__ __forceinline__ uint32_t decode_block_window(const uint8_t* __restrict__ s, uint32_t csize, WinOut& O,
                                                        uint8_t* ring8, const uint8_t* sbeg, const uint8_t* send,
                                                        const uint32_t* reach, uint32_t link, const uint32_t* done,
                                                        bool& waited, uint32_t& err, int lane) {
  const uint8_t* A = reinterpret_cast<const uint8_t*>((uintptr_t)s & ~(uintptr_t)15);
  const uint32_t shift = (uint32_t)(s - A);
  uint4* ring4 = reinterpret_cast<uint4*>(ring8);
  uint32_t cur = 0;
  ring4[lane] = load_stream_piece(A + 16u * lane, sbeg, send);
  ring4[32 + lane] = load_stream_piece(A + 512u + 16u * lane, sbeg, send);
  uint4 pre = load_stream_piece(A + 1024u + 16u * lane, sbeg, send);
  __syncwarp();
  auto ensure = [&](uint32_t pos) {
    const uint32_t c = pos >> 9;
    if (c == cur) return;
    __syncwarp();
    if (c == cur + 1) {
      ring4[((cur + 2) & 1) * 32 + lane] = pre;
      cur = c;
    } else {  // jumped over a long literal run: re-prime
      cur = c;
      ring4[(c & 1) * 32 + lane] = load_stream_piece(A + 512ull * c + 16u * lane, sbeg, send);
      ring4[((c + 1) & 1) * 32 + lane] = load_stream_piece(A + 512ull * (c + 1) + 16u * lane, sbeg, send);
    }
    pre = load_stream_piece(A + 512ull * (cur + 2) + 16u * lane, sbeg, send);
    __syncwarp();
  };
#define SQYB_RB(pos) ((uint32_t)ring8[(pos) & (kRing - 1)])
#define SQYB_W(pos) O.win[(pos) & (kWin - 1)]
  uint32_t ip = shift, op = 0;
  const uint32_t end = shift + csize;
  bool bad = false;
  // copies one match to output position op (warp-cooperative); false on a malformed stream
  auto do_match = [&](uint32_t op, uint32_t offset, uint32_t mlen) -> bool {
    if (offset > op) {
        // reaches in front of this block: only legal inside a linked frame, after the predecessor is complete
        // (a linked block behind its frame's first one is block link + 1; its window is looked up only here, off the hot path)
        if (link == kNoLink || offset - op > reach[link + 1]) { err = kErrBadBlock; return false; }
        if (!waited) {
          if (lane == 0) {
            while (atomicAdd(const_cast<uint32_t*>(done) + link, 0u) == 0u) __nanosleep(100);
            __threadfence();
          }
          waited = true;
        }
      }
      __syncwarp();
      if (offset <= kNear && offset <= op) {
        // ---- source inside the ring ----
        if (mlen <= 32 && offset >= mlen) {
          if ((uint32_t)lane < mlen) SQYB_W(op + lane) = SQYB_W(op + lane - offset);
        } else if (offset >= 32) {
          for (uint32_t kb = 0; kb < mlen; kb += 32) {
            const uint32_t k = kb + lane;
            if (k < mlen) SQYB_W(op + k) = SQYB_W(op + k - offset);
            const uint32_t step = mlen - kb < 32u ? mlen - kb : 32u;
            O.flush_to(op + kb + step);
            __syncwarp();                 // orders overlapping steps
          }
        } else if (mlen >= 256 && (offset == 1 || offset == 2 || offset == 4)) {
          // run fill: for a period dividing 4 every 4-byte aligned output word holds the same value
          const uint32_t al = (op + 3u) & ~3u;          // first aligned output position
          const uint32_t om = offset - 1u;              // period is a power of two: modulo = mask
          uint32_t word = 0;
#pragma unroll
          for (uint32_t j = 0; j < 4; ++j) word |= (uint32_t)SQYB_W(op - offset + ((al - op + j) & om)) << (8 * j);
          const uint32_t head = al - op;                // < 4 <= mlen
          if ((uint32_t)lane < head) SQYB_W(op + lane) = SQYB_W(op - offset + (lane & om));
          const uint32_t body = (mlen - head) >> 2;     // whole words
          for (uint32_t wb = 0; wb < body; wb += 32) {
            const uint32_t w = wb + lane;
            if (w < body) *reinterpret_cast<uint32_t*>(O.win + ((al + 4u * w) & (kWin - 1))) = word;
            const uint32_t stepw = body - wb < 32u ? body - wb : 32u;
            O.flush_to(al + 4u * (wb + stepw));
          }
          const uint32_t donew = head + (body << 2);
          if ((uint32_t)lane < mlen - donew) {
            const uint32_t k = donew + lane;
            SQYB_W(op + k) = (uint8_t)(word >> (8 * ((k - head) & 3u)));
          }
        } else if ((offset & (offset - 1u)) == 0u && mlen < 1024u) {
          // period 1, 2, 4, 8 or 16: k mod offset is a mask (the common case: byte runs and 16/32-bit periodic data)
          const uint32_t base = op - offset, om = offset - 1u;
          for (uint32_t kb = 0; kb < mlen; kb += 32) {
            const uint32_t k = kb + lane;
            if (k < mlen) SQYB_W(op + k) = SQYB_W(base + (k & om));
            if (kb + 32u < mlen) O.flush_to(op + kb + 32u);
          }
        } else {
          // any other short period (or a long match with period 8/16). The pattern [op-offset, op) repeats; the first D bytes
          // (D = smallest multiple of the period >= 32) are taken from it, everything after that is a copy from D bytes
          // back, i.e. from an earlier 32-byte step — the ring may wrap over the original pattern on long matches.
          const uint32_t base = op - offset;
          const uint32_t D = offset * ((31u + offset) / offset);
          const float inv = __frcp_rn((float)offset);
          for (uint32_t kb = 0; kb < mlen; kb += 32) {
            const uint32_t k = kb + lane;
            if (k < mlen) {
              uint32_t src = op + k - D;
              if (k < D) src = base + (k - offset * (uint32_t)__float2int_rz(((float)k + 0.5f) * inv));   // k < 62: exact
              SQYB_W(op + k) = SQYB_W(src);
            }
            const uint32_t step = mlen - kb < 32u ? mlen - kb : 32u;
            O.flush_to(op + kb + step);
            __syncwarp();
          }
        }
      } else {
        // ---- far source (already flushed) or bytes in front of a linked block: L1-bypassing global loads ----
        O.flush_to(op);   // make sure everything up to the last complete chunk is in global memory
        for (uint32_t kb = 0; kb < mlen; kb += 32) {
          const uint32_t k = kb + lane;
          if (k < mlen) {
            // may be negative in a linked frame; a short period (only possible when the match starts in front of
            // the block) repeats the pattern [op-offset, op) so that no lane reads a byte written in this step
            uint32_t kk = k;
            if (offset < 32u) kk = k % offset;
            const long long sp = (long long)op - offset + kk;
            uint8_t v;
            if (sp >= (long long)O.flushed) v = SQYB_W((uint32_t)sp);   // unflushed tail
            else v = __ldcg(O.d + sp);
            SQYB_W(op + k) = v;
          }
          const uint32_t step = mlen - kb < 32u ? mlen - kb : 32u;
          O.flush_to(op + kb + step);
          __syncwarp();
        }
      }
    return true;
  };
  while (ip < end) {
    ensure(ip);
    // ---- batch of sequences. The token chain is serial, but a sequence header is only a few bytes: lane j parses the
    // bytes at ip+j AS IF a token started there (token, one optional length byte each, offset), all 32 candidates in
    // parallel; the real chain is then followed from lane 0 with one shuffle per sequence (next token = candidate
    // lane `qrel`), which also hands every sequence its output position. Then the owners copy their literals in
    // parallel and the matches are replayed in order. A sequence is "simple" (batchable) when its length chains have
    // at most one byte (lengths < 270) and it lies inside the resident compressed window;
    // everything else — and any batch that would write more than kBatchOut bytes, which keeps near sources inside the
    // output ring without a flush — goes through the single-sequence path below.
    const uint32_t ringend = (cur + 2u) * 512u;
    uint32_t my_lits, my_lit, my_mlen, my_off, my_q, my_mo = 0;
    bool my_simple = true, my_fin;
    {
      const uint32_t pos = ip + lane;
      const uint32_t token = SQYB_RB(pos);
      uint32_t q = pos + 1u;
      my_lit = token >> 4;
      uint32_t ml = token & 15u;
      if (my_lit == 15u) { const uint32_t x = SQYB_RB(q); q++; my_lit += x; my_simple = x != 255u; }
      my_lits = q;
      q += my_lit;
      my_fin = q == end;
      my_off = SQYB_RB(q) | (SQYB_RB(q + 1u) << 8);
      if (!my_fin) {
        q += 2u;
        if (ml == 15u) { const uint32_t x = SQYB_RB(q); q++; ml += x; my_simple = my_simple && x != 255u; }
        ml += 4u;
      } else {
        ml = 0u;
      }
      my_mlen = ml;
      my_q = q - ip;                                   // where the next token starts, relative to ip (simple: < 31+2+269+2+2)
      my_simple = my_simple && q <= ringend && (my_fin || q < end);
    }
    // chain word: next-token lane (511 for the final sequence: ends the chain) | output bytes (2047 when not simple:
    // fails the batch-size test); match word: offset | length
    const uint32_t my_chain = (my_fin ? 511u : (my_q & 0x1ffu)) | ((my_simple ? my_lit + my_mlen : 2047u) << 9);
    const uint32_t my_match = my_off | (my_mlen << 16);
    uint32_t c = 0, o = op, owners = 0;
    while (c < 32u) {
      const uint32_t pk = __shfl_sync(0xffffffffu, my_chain, c);
      const uint32_t tot = pk >> 9;
      if (o - op + tot > kBatchOut) break;
      if ((uint32_t)lane == c) my_mo = o + my_lit;
      owners |= 1u << c;
      o += tot;
      c = pk & 0x1ffu;
    }
    if (owners) {
      if (o > O.dcap) { err = kErrBadBlock; return op; }
      const int hi = 31 - __clz(owners);               // the batch's last sequence
      const uint32_t pnext = __shfl_sync(0xffffffffu, my_q, hi);
      const bool last = __shfl_sync(0xffffffffu, my_fin ? 1u : 0u, hi) != 0u;
      // literals: the owner lane of every sequence copies up to four of them itself (the lanes of a warp wait for the longest
      // run, and most runs of bit-plane data have one to three bytes); longer runs are copied by the whole warp,
      // 32 bytes per step (measured: owner copies of up to 16 / 8 / 4 literals: cfg2 decode 6.01 / 5.93 / 5.79 ms)
      const bool mine = (owners >> lane) & 1u;
      if (mine && my_lit <= kLitOwn) {
        const uint32_t dst0 = my_mo - my_lit;
        for (uint32_t k = 0; k < my_lit; ++k) SQYB_W(dst0 + k) = (uint8_t)SQYB_RB(my_lits + k);
      }
      uint32_t big = __ballot_sync(0xffffffffu, mine && my_lit > kLitOwn);
      while (big) {
        const int i = __ffs(big) - 1;
        big &= big - 1u;
        const uint32_t lit = __shfl_sync(0xffffffffu, my_lit, i), from = __shfl_sync(0xffffffffu, my_lits, i),
                       to = __shfl_sync(0xffffffffu, my_mo, i) - lit;
        for (uint32_t k = lane; k < lit; k += 32u) SQYB_W(to + k) = (uint8_t)SQYB_RB(from + k);
      }
      __syncwarp();
      // matches, in stream order (= lane order of the owners). Inside a batch no flush is needed and a match has at
      // most 273 bytes, so the near copies are plain loops over the output ring.
      uint32_t todo = last ? owners & ~(1u << hi) : owners;   // the block's final sequence has no match
      // Far matches first, four at a time: their sources (more than kNear bytes back, inside this block) were flushed before
      // this batch began, so they depend on nothing the batch writes and on no order among themselves — while a near match
      // behind them may read what they produce. A group of eight lanes copies one of them (most have 5..16 bytes: one or two
      // steps), where the loop below spends a whole warp and ~40 instructions on each. An encoder that points at the FIRST
      // occurrence of a pattern (lz4_encode.cu) makes these the majority of the matches of a sparse bit plane.
      {
        const bool is_far = ((todo >> lane) & 1u) && my_off > kNear && my_off <= my_mo && my_mlen <= kFarMax;
        uint32_t far = __ballot_sync(0xffffffffu, is_far);
        todo &= ~far;
        const int g = lane / kFarW;
        const uint32_t l8 = (uint32_t)lane % kFarW;
        while (far) {
          int sel = -1;
#pragma unroll
          for (int t = 0; t < 32 / kFarW; ++t) {
            const int i = __ffs(far) - 1;          // (-1 when the batch has no further far match)
            if (t == g) sel = i;
            far &= far - 1u;
          }
          const uint32_t mw = __shfl_sync(0xffffffffu, my_match, sel & 31), mo = __shfl_sync(0xffffffffu, my_mo, sel & 31);
          if (sel >= 0) {
            const uint32_t offset = mw & 0xffffu, mlen = mw >> 16;
            const uint8_t* from = O.d + (mo - offset);
            if (O.line_aligned) {
#pragma unroll 1
              for (uint32_t k = l8; k < mlen; k += kFarW) SQYB_W(mo + k) = ld_l1_u8(from + k);
            } else {
#pragma unroll 1
              for (uint32_t k = l8; k < mlen; k += kFarW) SQYB_W(mo + k) = __ldcg(from + k);
            }
          }
        }
        __syncwarp();
      }
      while (todo) {
        const int i = __ffs(todo) - 1;
        todo &= todo - 1u;
        const uint32_t mw = __shfl_sync(0xffffffffu, my_match, i), mo = __shfl_sync(0xffffffffu, my_mo, i);
        const uint32_t offset = mw & 0xffffu, mlen = mw >> 16;
        bad |= offset == 0u;
        if (offset <= kNear && offset <= mo) {
          const uint32_t base = mo - offset;
          if (offset >= mlen || offset >= 32u) {
            // a 32-byte step never reads a byte it writes; later steps may read what earlier ones wrote
            if ((uint32_t)lane < mlen) SQYB_W(mo + lane) = SQYB_W(base + lane);
#pragma unroll 1
            for (uint32_t k = lane + 32u; k < mlen + lane; k += 32u) {   // (same trip count on every lane)
              __syncwarp();
              if (k < mlen) SQYB_W(mo + k) = SQYB_W(base + k);
            }
          } else if ((offset & (offset - 1u)) == 0u) {
            // period 1, 2, 4, 8, 16: every byte comes from the pattern in front of the match
            // (first step peeled, the rest not unrolled: most matches have at most 32 bytes, and an unrolled loop pays its
            //  remainder logic on every one of them)
            const uint32_t om = offset - 1u;
            if ((uint32_t)lane < mlen) SQYB_W(mo + lane) = SQYB_W(base + (lane & om));
            if (mlen > 32u) {
#pragma unroll 1
              for (uint32_t k = lane + 32u; k < mlen; k += 32u) SQYB_W(mo + k) = SQYB_W(base + (k & om));
            }
          } else {
            const float inv = __frcp_rn((float)offset);
#pragma unroll 1
            for (uint32_t k = lane; k < mlen; k += 32u)   // k < 512: the quotient is exact
              SQYB_W(mo + k) = SQYB_W(base + (k - offset * (uint32_t)__float2int_rz(((float)k + 0.5f) * inv)));
          }
        } else if (offset <= mo) {
          // far source inside this block: it ends at least 1199 bytes in front of the match (offset > kNear, mlen <= 273)
          // while everything up to 1023 bytes in front of it was flushed after the previous batch, so it is read back
          // from global memory (L2) without any window bookkeeping
          // The flushed part ends on a 512-byte boundary of the block: with a 128-byte aligned block a cache line is either
          // final or untouched when it is first read, so the reads may stay in L1 — an encoder that points at the first
          // occurrence of a pattern (lz4_encode.cu) reads the same early lines of the block over and over.
          const uint8_t* from = O.d + (mo - offset);
          if (O.line_aligned) {
            if ((uint32_t)lane < mlen) SQYB_W(mo + lane) = ld_l1_u8(from + lane);
            if (mlen > 32u) {
#pragma unroll 1
              for (uint32_t k = lane + 32u; k < mlen; k += 32u) SQYB_W(mo + k) = ld_l1_u8(from + k);
            }
          } else {
#pragma unroll 1
            for (uint32_t k = lane; k < mlen; k += 32u) SQYB_W(mo + k) = __ldcg(from + k);
          }
        } else if (!do_match(mo, offset, mlen)) {   // reaches in front of a linked block
          return op;
        }
        __syncwarp();
      }
      op = o;
      ip += pnext;
      O.flush_to(op);
      if (O.overflow) { err = kErrBadBlock; return op; }
      continue;
    }
    // ---- single sequence (long literal run, long match, or a sequence that crosses the resident window) ----
    uint32_t token = SQYB_RB(ip);
    ip++;
    uint32_t lit = token >> 4;
    if (lit == 15) {
      uint32_t b;
      do {
        if (ip >= end) { err = kErrBadBlock; return op; }
        ensure(ip);   // 256 KiB blocks can carry > 1000 length bytes
        b = SQYB_RB(ip);
        ip++;
        lit += b;
      } while (b == 255);
    }
    if (lit) {
      if (ip + lit > end || op + lit > O.dcap) { err = kErrBadBlock; return op; }
      const bool in_ring = ip + lit <= (cur + 2) * 512u;
      for (uint32_t kb = 0; kb < lit; kb += 32) {
        const uint32_t k = kb + lane;
        if (k < lit) SQYB_W(op + k) = in_ring ? (uint8_t)SQYB_RB(ip + k) : __ldg(A + ip + k);
        const uint32_t step = lit - kb < 32u ? lit - kb : 32u;
        O.flush_to(op + kb + step);
      }
      op += lit;
      ip += lit;
    }
    if (ip >= end) break;
    ensure(ip);
    const uint32_t offset = SQYB_RB(ip) | (SQYB_RB(ip + 1) << 8);
    ip += 2;
    uint32_t mlen = token & 15u;
    if (mlen == 15) {
      uint32_t b;
      do {
        if (ip >= end) { err = kErrBadBlock; return op; }
        ensure(ip);
        b = SQYB_RB(ip);
        ip++;
        mlen += b;
      } while (b == 255);
    }
    mlen += 4;
    bad |= offset == 0;
    if (op + mlen > O.dcap) { err = kErrBadBlock; return op; }
    __syncwarp();
    if (!do_match(op, offset, mlen)) return op;
    op += mlen;
    __syncwarp();
    O.flush_to(op);
    if (O.overflow) { err = kErrBadBlock; return op; }
  }
#undef SQYB_RB
#undef SQYB_W
  if (bad || ip != end) err = kErrBadBlock;
  return op;
}

// measures the decoded size of the blocks the directory could not infer
__global__ void __launch_bounds__(kDecThreads) lz4_sizes_kernel(const uint8_t* __restrict__ src, DecCtl* ctl, DecTables T) {
  if (ctl->error || ctl->need_sizes == 0) return;
  const int lane = threadIdx.x & 31;
  const uint32_t nblocks = ctl->nblocks;
  while (true) {
    uint32_t b = 0;
    if (lane == 0) b = atomicAdd(&ctl->ticket_size, 1u);
    b = __shfl_sync(0xffffffffu, b, 0);
    if (b >= nblocks) return;
    if (T.dsize[b] != 0 || (T.word[b] & kLz4StoredFlag)) continue;
    uint32_t err = 0;
    const uint32_t sz = measure_block_warp(src + T.src_off[b], T.word[b] & 0x7FFFFFFFu, err, lane);
    if (lane == 0) {
      T.dsize[b] = sz;
      if (err) atomicMax(&ctl->error, err);
    }
  }
}

// ---- fast table build for a stream that is one frame of this library (everything the encoder writes) ----
// A single CTA spends ~1 ms on the prefix sum + table stores of a 4 GiB frame (262144 blocks: one SM's store
// bandwidth); two small multi-CTA kernels do it in a few microseconds: per-tile sums, then every tile adds the sums
// in front of it, scans its 4096 block sizes in shared memory and writes its table rows with coalesced stores.
__device__ __forceinline__ uint32_t index_word(const uint8_t* idx, bool aligned, uint32_t i) {
  return aligned ? __ldg(reinterpret_cast<const uint32_t*>(idx) + i) : rd32(idx + 4ull * i);
}

__global__ void __launch_bounds__(256) lz4_tile_sums_kernel(const uint8_t* __restrict__ src, DecCtl* ctl,
                                                            unsigned long long* __restrict__ tile_sums) {
  __shared__ uint32_t wsum[8];
  if (ctl->error || !ctl->fast) return;
  const uint32_t nblk = ctl->fast_nblk, bb = ctl->fast_bb, ntiles = (nblk + kTile - 1) / kTile;
  const uint8_t* idx = src + ctl->fast_idx;
  const bool aligned = (((uintptr_t)idx) & 3) == 0;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (uint32_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
    uint32_t s = 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const uint32_t i = t * kTile + k * 256 + tid;
      if (i < nblk) {
        const uint32_t sz = index_word(idx, aligned, i) & 0x7FFFFFFFu;
        // untrusted index: no block is larger than the block size (bb <= 65536 keeps the 32-bit tile sums exact)
        if (sz > bb) atomicMax(&ctl->error, (uint32_t)kErrBadBlock);
        s += 4u + (sz > bb ? bb : sz);
      }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_down_sync(0xffffffffu, s, d);
    __syncthreads();
    if (lane == 0) wsum[warp] = s;
    __syncthreads();
    if (tid == 0) {
      uint32_t x = 0;
      for (int w = 0; w < 8; ++w) x += wsum[w];
      tile_sums[t] = x;
    }
  }
}

__global__ void __launch_bounds__(256) lz4_expand_kernel(const uint8_t* __restrict__ src, DecCtl* ctl, DecTables T,
                                                         const unsigned long long* __restrict__ tile_sums, uint64_t dst_bytes) {
  __shared__ uint32_t words[kTile];
  __shared__ uint32_t pre[kTile];            // exclusive prefix of (4 + size) inside the tile
  __shared__ unsigned long long red[8];
  __shared__ uint32_t tsum[256];
  if (ctl->error || !ctl->fast) return;
  const uint32_t nblk = ctl->fast_nblk, bb = ctl->fast_bb, ntiles = (nblk + kTile - 1) / kTile;
  const unsigned long long raw = ctl->fast_raw, first = ctl->fast_first;
  const uint8_t* idx = src + ctl->fast_idx;
  const bool aligned = (((uintptr_t)idx) & 3) == 0;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (blockIdx.x == 0 && tid == 0) {
    ctl->total_decoded = raw;
    if (raw > dst_bytes || (raw == 0 && dst_bytes != 0)) ctl->error = kErrSizeMismatch;
  }
  for (uint32_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
    // bytes in front of this tile
    unsigned long long b = 0;
    for (uint32_t u = tid; u < t; u += 256) b += tile_sums[u];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) b += __shfl_down_sync(0xffffffffu, b, d);
    __syncthreads();
    if (lane == 0) red[warp] = b;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const uint32_t i = t * kTile + k * 256 + tid;
      words[k * 256 + tid] = i < nblk ? index_word(idx, aligned, i) : 0u;
    }
    __syncthreads();
    unsigned long long base = first;
    for (int w = 0; w < 8; ++w) base += red[w];
    // thread-local scan over 16 consecutive blocks, then a scan of the 256 thread totals
    uint32_t loc[16], s = 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const uint32_t i = t * kTile + tid * 16 + k;
      loc[k] = s;
      s += i < nblk ? 4u + (words[tid * 16 + k] & 0x7FFFFFFFu) : 0u;
    }
    uint32_t incl = s;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t x = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += x;
    }
    if (lane == 31) tsum[warp] = incl;
    __syncthreads();
    uint32_t wbase = 0;
    for (int w = 0; w < warp; ++w) wbase += tsum[w];
    const uint32_t tbase = wbase + incl - s;
#pragma unroll
    for (int k = 0; k < 16; ++k) pre[tid * 16 + k] = tbase + loc[k];
    // the offsets are only good when the sizes of the (untrusted) index add up to exactly the frame its header promised:
    // the thread that ends the last tile checks it, the decoders look at ctl->error before they touch the table
    if (t == ntiles - 1 && tid == 255 && base + tbase + s + kLz4EndMarkBytes != ctl->fast_end)
      atomicMax(&ctl->error, (uint32_t)kErrBadBlock);
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const uint32_t j = k * 256 + tid, i = t * kTile + j;
      if (i < nblk) {
        T.src_off[i] = base + pre[j] + 4u;
        T.word[i] = words[j];
        const unsigned long long rem = raw - (unsigned long long)i * bb;
        T.dsize[i] = (uint32_t)(rem < bb ? rem : bb);
        T.link[i] = kNoLink;
        T.dst_off[i] = (unsigned long long)i * bb;
        T.done[i] = 0u;
        T.range[i] = 0u;
      }
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(kDirThreads) lz4_offsets_kernel(DecCtl* ctl, DecTables T, uint64_t dst_bytes) {
  __shared__ unsigned long long warp_sums[32];
  if (ctl->error || ctl->fast) return;
  const uint32_t nblk = ctl->nblocks;
  const int tid = threadIdx.x;
  unsigned long long running = 0;
  for (uint32_t base = 0; base < nblk; base += kDirThreads * kPerThread) {
    uint32_t d[kPerThread];
    unsigned long long local = 0;
#pragma unroll
    for (int k = 0; k < kPerThread; ++k) {
      const uint32_t i = base + tid * kPerThread + k;
      d[k] = i < nblk ? T.dsize[i] : 0u;
      local += d[k];
    }
    unsigned long long total;
    const unsigned long long incl = block_scan_incl(local, warp_sums, total);
    unsigned long long off = running + incl - local;
#pragma unroll
    for (int k = 0; k < kPerThread; ++k) {
      const uint32_t i = base + tid * kPerThread + k;
      if (i < nblk) {
        T.dst_off[i] = off;
        T.done[i] = 0;
        T.range[i] = 0;
        off += d[k];
      }
    }
    running += total;
    __syncthreads();
  }
  // the window of a linked block ends at the first byte of its frame (liblz4 refuses matches that reach further)
  for (uint32_t i = tid; i < nblk; i += kDirThreads) {
    const uint32_t link = T.link[i];
    if (link != kNoLink && link != kLinkHead) {
      const unsigned long long in_frame = T.dst_off[i] - T.dst_off[T.reach[i]];
      T.reach[i] = (uint32_t)(in_frame < 65535ull ? in_frame : 65535ull);
    }
  }
  if (tid == 0) {
    ctl->total_decoded = running;
    // the reference accepts 0 < decoded <= expected (encoders/lz4.hpp:334-338); we refuse overruns
    if (running > dst_bytes || (running == 0 && dst_bytes != 0)) ctl->error = kErrSizeMismatch;
  }
}

// fused transpose (lz4_decode_kernel, FW > 0): a range's voxels go back in pieces of kPieceChunks 32-voxel chunks (16384 voxels).
// The range counter holds the range's decoded blocks in its low half and the pieces claimed so far in its high half.
constexpr uint32_t kPieceChunks = 512;
constexpr int kListMode = -1;   // lz4_decode_kernel's FW for the blocks of a list (k_lz4_decode_list)

// transposes the still unclaimed pieces of a complete range (its planes were written by other warps of this launch: fence, then
// L2 loads). One chunk per lane at a time: a second one in flight costs the 48-register decoder spills.
template <int FW>
__device__ __forceinline__ void transpose_range(const uint16_t* planes, uint16_t* vox, uint32_t* counter, uint32_t range, uint64_t S,
                                                int lane) {
  constexpr uint32_t P = 16 / FW, kChunks = 8192u * P / 32u, kPieces = kChunks / kPieceChunks;
  __threadfence();
  while (true) {
    uint32_t piece = 0;
    if (lane == 0) piece = atomicAdd(counter, 1u << 16) >> 16;
    piece = __shfl_sync(0xffffffffu, piece, 0);
    if (piece >= kPieces) return;
    const uint64_t t0 = (uint64_t)range * kChunks + piece * kPieceChunks;
#pragma unroll 1
    for (uint32_t c = lane; c < kPieceChunks; c += 32u) bitswap_thread::decode_chunk<FW, true>(planes, vox, t0 + c, S);
  }
}

// Every block is taken here; the stored / closed-form blocks are handled inline: their 16-byte-store fills are
// memory-bound and hide under the issue-bound decoding of the other warps, whereas a separate classification pass in
// front of this kernel cost 0.63 ms per 4 GiB.
// CTAS = CTAs per SM the registers are budgeted for: 5 (48 registers, 40 warps per SM) for streams that fill the machine,
// 4 (64 registers, no spills) for small ones, which are bound by the serial chain of their slowest blocks and not by the
// number of warps in flight (512x512x256 stack: 1.00 -> 0.75 ms; 4 GiB: 5.80 -> 6.25 ms)
// FW > 0: the stream is one frame of this library holding the 16 KiB blocks of the P = 16/FW bit planes of a uint16 bitswapFW
// (plane-major, bpp blocks per plane), and the kernel also transposes the planes back into `vox`. A range = block r of every
// plane = voxels [r * 8192P, (r+1) * 8192P). Tickets are dealt range by range; the warp that finishes the last block of a
// range (per-range counter) transposes it while its planes are still in L2, so the transpose, which needs memory bandwidth,
// runs beside the decode of other blocks, which needs issue slots, instead of as a launch of its own behind them. Warps that find
// no block left help with the pieces of the last ranges dealt instead of leaving a range's transpose to one warp at the end.
// Two instantiations chosen at launch cost nothing; the plain one has no trace of the fused code.
// FW == kListMode: the blocks named by a list (a sub-volume's blocks, k_lz4_decode_list). Ticket t decodes block T.range[t] of
// `count` listed ones into dst + t * 16 KiB instead of its place in the stream; far matches read back from that compact place
// (WinOut::d), and every block adds its decoded bytes to ctl->total_decoded.
template <int CTAS, int FW>
__global__ void __launch_bounds__(kWinWarps * 32, CTAS) lz4_decode_kernel(const uint8_t* __restrict__ src, uint64_t src_bytes,
                                                                        uint8_t* __restrict__ dst, DecCtl* ctl, DecTables T,
                                                                        uint32_t first, uint32_t count,
                                                                        uint32_t nsets, uint32_t set_stride, uint32_t slot,
                                                                        uint16_t* __restrict__ vox, uint32_t bpp) {
  extern __shared__ __align__(16) unsigned char dsm[];
  if (ctl->error) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint8_t* win = dsm + (size_t)warp * kWinWarpSmem;
  uint8_t* ring8 = win + kWin;
  const uint32_t nblocks = ctl->nblocks;
  // count != 0: only `nsets` sets of `count` consecutive blocks, set j starting at first + j * set_stride (the blocks of all
  // bit planes that make up one z-slab), with a work counter of their own
  constexpr bool kList = FW == kListMode;
  const uint32_t total = kList ? count : count ? count * nsets : nblocks;
  uint32_t* ticket = count && !kList ? &ctl->set_ticket[slot & 31u] : &ctl->ticket_decode;
  constexpr uint32_t P = FW > 0 ? 16 / FW : 1;
  const uint64_t S = (uint64_t)bpp * (kLz4BlockBytes / 2);   // (fused only) 16-bit words per plane
  while (true) {
    uint32_t b = 0;
    if (lane == 0) b = atomicAdd(ticket, 1u);
    b = __shfl_sync(0xffffffffu, b, 0);
    if constexpr (FW > 0) {
      if (b >= total) {
        // every block is held by a running warp: wait for one of the last ranges dealt and take pieces of its transpose
        constexpr uint32_t kPieces = 8192u * P / 32u / kPieceChunks;
        const uint32_t nranges = total / P, h = b - total;
        const uint32_t helped = min(nranges, gridDim.x * (uint32_t)kWinWarps / P + 2u);
        if (h >= helped * kPieces) return;
        const uint32_t r = nranges - 1u - h / kPieces;
        if (lane == 0)
          while ((atomicAdd(T.range + r, 0u) & 0xffffu) < P) __nanosleep(256);
        __syncwarp();
        transpose_range<FW>(reinterpret_cast<const uint16_t*>(dst), vox, T.range + r, r, S, lane);
        continue;
      }
    }
    if (b >= total) return;
    const uint32_t range = b / P;                      // (fused only)
    if (FW > 0) b = (b % P) * bpp + range;
    const uint32_t listed = b;                         // (list mode only) the block's compact place
    if constexpr (kList) {
      b = T.range[listed];
      if (b >= nblocks) continue;
    } else if (count) {
      const uint32_t j = b / count;
      b = first + j * set_stride + (b - j * count);
      if (b >= nblocks) continue;
    }
    const uint32_t word = T.word[b];
    const uint32_t csize = word & 0x7FFFFFFFu;
    const uint32_t dsize = T.dsize[b];
    const unsigned long long doff = T.dst_off[b];
    uint32_t link = T.link[b];
    if (link != kNoLink && ctl->deferred) continue;   // block-linked frames: lz4_decode_deferred_kernel + resolve passes
    if (link == kLinkHead) link = kNoLink;
    const uint8_t* s = src + T.src_off[b];
    uint8_t* d = dst + (kList ? (unsigned long long)listed * kLz4BlockBytes : doff);
    bool waited = false;
    uint32_t err = 0;
    // closed-form run block (what the encoder emits for an all-equal block): token 0x1F, byte, offset 1, length
    // bytes, token 0x50, five bytes -> a 16-byte-store fill, no ring traffic
    bool filled = false;
    if (!(word & kLz4StoredFlag) && csize >= 12 && csize <= 96 && dsize >= 64 && link == kNoLink && (((uintptr_t)d) & 15) == 0) {
      const uint32_t t0 = __ldg(s), v = __ldg(s + 1), o0 = __ldg(s + 2), o1 = __ldg(s + 3);
      if (t0 == 0x1Fu && o0 == 1u && o1 == 0u) {
        uint32_t ip = 4, mlen = 15 + 4, b;
        do { b = ip < csize ? __ldg(s + ip) : 0u; ip++; mlen += b; } while (b == 255u && ip < csize);
        bool ok = ip + 6 == csize && 1u + mlen + 5u == dsize && __ldg(s + ip) == 0x50u;
        for (uint32_t k = 0; ok && k < 5; ++k) ok = __ldg(s + ip + 1 + k) == v;
        if (ok) {
          const uint32_t v4 = v * 0x01010101u;
          const uint4 fill = make_uint4(v4, v4, v4, v4);
          const uint32_t nv = dsize >> 4;
          for (uint32_t q = lane; q < nv; q += 32) st_stream(reinterpret_cast<uint4*>(d) + q, fill);
          for (uint32_t k = (nv << 4) + lane; k < dsize; k += 32) d[k] = (uint8_t)v;
          filled = true;
        }
      }
    }
    if (filled) {
      // nothing else to do
    } else if (word & kLz4StoredFlag) {
      if (csize != dsize) err = kErrSizeMismatch;
      else warp_copy_from_stream(d, s, csize, lane);
    } else {
      WinOut O;
      O.win = win;
      O.d = d;
      O.flushed = 0;
      O.dcap = dsize;
      O.aligned = (((uintptr_t)d) & 15) == 0;
      O.line_aligned = (((uintptr_t)d) & 127) == 0;
      O.overflow = false;
      O.lane = lane;
      // a linked block may reach back to the first byte of its frame (T.reach), never into the frame in front of it
      const uint32_t got = decode_block_window(s, csize, O, ring8, src, src + src_bytes, T.reach, link, T.done, waited, err, lane);
      if (!err) O.finish(got);
      if (!err && (O.overflow || got != dsize)) err = kErrSizeMismatch;
    }
    if (err && lane == 0) atomicMax(&ctl->error, err);
    if constexpr (kList) {
      if (!err && lane == 0) atomicAdd(&ctl->total_decoded, (unsigned long long)dsize);
      continue;
    }
    if constexpr (FW > 0) {
      // the planes of a complete range go back to voxels (a broken block sets ctl->error; the range is transposed all the same,
      // inside `vox`, and the caller reports the error)
      __syncwarp();
      uint32_t last = 0;
      if (lane == 0) {
        __threadfence();
        last = (atomicAdd(T.range + range, 1u) & 0xffffu) == P - 1u;
      }
      if (__shfl_sync(0xffffffffu, last, 0))
        transpose_range<FW>(reinterpret_cast<const uint16_t*>(dst), vox, T.range + range, range, S, lane);
      continue;
    }
    // publish completion (linked frames): a block is done when it and its predecessor are done
    __syncwarp();
    if (lane == 0) {
      if (link != kNoLink && !waited) {
        while (atomicAdd(T.done + link, 0u) == 0u) __nanosleep(100);
      }
      __threadfence();
      atomicExch(T.done + b, 1u);
    }
    __syncwarp();
  }
}


// ------------------------------------------------------------------------------------------------
// Block-linked frames (the reference's serial mode = the sqy CLI default, encoders/lz4_utils.hpp:99-173): a block may
// copy from the 64 KiB in front of it, i.e. from the tail of its predecessor, which exists only when the predecessor
// is finished: decoded as they come, the blocks run one after the other (0.15 GB/s for 8192 blocks of 256 KiB).
// Deferred cross-block references break that chain in three passes:
//   1. lz4_decode_deferred_kernel : every block is decoded at once, a warp per block, straight in global memory. A byte
//      that comes from in front of the block is not copied but REMEMBERED: origin[i] = its distance in front of the
//      block start (1..65535, the LZ4 offset range; 0 = the byte in dst[i] is real). Copies inside the block carry the
//      origin along, so after this pass every byte of every block is either real or names one byte of the 64 KiB window
//      in front of its block.
//   2. lz4_resolve_chain_kernel   : the only serial part — one CTA walks the blocks in order and resolves the last
//      65535 bytes of each (what the next block's origins can point at) from the already resolved bytes in front of it:
//      64 KiB of gathers per block instead of a whole block decode.
//   3. lz4_resolve_rest_kernel    : all remaining remembered bytes of all blocks, in parallel.
// A source pattern is always read in front of the match (k mod offset), so lanes never depend on each other inside a match.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) lz4_decode_deferred_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst,
                                                                  uint16_t* __restrict__ origin, DecCtl* ctl, DecTables T) {
  if (ctl->error || !ctl->deferred) return;
  const int lane = threadIdx.x & 31;
  const uint32_t nblocks = ctl->nblocks;
  while (true) {
    uint32_t b = 0;
    if (lane == 0) b = atomicAdd(&ctl->ticket_deferred, 1u);
    b = __shfl_sync(0xffffffffu, b, 0);
    if (b >= nblocks) return;
    const uint32_t link = T.link[b];
    if (link == kNoLink) continue;
    const uint32_t word = T.word[b];
    const uint32_t csize = word & 0x7FFFFFFFu, dsize = T.dsize[b];
    const unsigned long long doff = T.dst_off[b];
    const uint8_t* s = src + T.src_off[b];
    uint8_t* d = dst + doff;
    uint16_t* o = origin + doff;
    // bytes that exist in front of this block inside its frame's reach
    const unsigned long long before = link == kLinkHead ? 0ull : T.reach[b];
    uint32_t err = 0;
    if (word & kLz4StoredFlag) {
      if (csize != dsize) err = kErrSizeMismatch;
      else
        for (uint32_t k = lane; k < csize; k += 32) { d[k] = __ldg(s + k); o[k] = 0; }
    } else {
      uint32_t ip = 0, op = 0;
      // The last 32 output symbols (byte | origin << 8) stay in registers, lane l holding position op - 32 + l: a match with
      // an offset of at most 32 — runs and short periods, most of what bit planes consist of — takes its pattern from
      // there with one shuffle per 32 bytes and never waits for an L2 round trip. In front of the block: origins 32..1.
      uint32_t tail = (uint32_t)(32 - lane) << 8;
      auto push = [&](uint32_t L, uint32_t last) {   // L symbols were written at op; `last` = the last one this lane wrote
        // every one of the final 32 positions is the LAST write of its lane, (L + lane) mod 32; older ones slide down
        const uint32_t a = __shfl_sync(0xffffffffu, last, (L + lane) & 31);
        const uint32_t b = __shfl_sync(0xffffffffu, tail, (L + lane) & 31);
        tail = ((uint64_t)L + lane >= 32u) ? a : b;
      };
      while (ip < csize && !err) {
        const uint32_t token = __ldg(s + ip);
        ip++;
        uint32_t lit = token >> 4;
        if (lit == 15u) {
          uint32_t x;
          do {
            if (ip >= csize) { err = kErrBadBlock; break; }
            x = __ldg(s + ip);
            ip++;
            lit += x;
          } while (x == 255u);
        }
        if (err) break;
        if ((unsigned long long)ip + lit > csize || (unsigned long long)op + lit > dsize) { err = kErrBadBlock; break; }
        if (lit) {
          uint32_t last = 0;
          for (uint32_t k = lane; k < lit; k += 32) {
            last = __ldg(s + ip + k);
            d[op + k] = (uint8_t)last;
            o[op + k] = 0;
          }
          push(lit, last);
          ip += lit;
          op += lit;
        }
        if (ip >= csize) break;            // the last sequence has literals only
        if (ip + 2u > csize) { err = kErrBadBlock; break; }
        const uint32_t offset = __ldg(s + ip) | (__ldg(s + ip + 1) << 8);
        ip += 2;
        uint32_t mlen = token & 15u;
        if (mlen == 15u) {
          uint32_t x;
          do {
            if (ip >= csize) { err = kErrBadBlock; break; }
            x = __ldg(s + ip);
            ip++;
            mlen += x;
          } while (x == 255u);
        }
        if (err) break;
        mlen += 4u;
        if (offset == 0u || (unsigned long long)op + mlen > dsize) { err = kErrBadBlock; break; }
        if (offset > op && (unsigned long long)(offset - op) > before) { err = kErrBadBlock; break; }
        uint32_t last = 0;
        if (offset <= 32u) {
          // pattern = the last `offset` symbols = tail lanes 32-offset .. 31; output k takes pattern[k mod offset]
          uint32_t j = (uint32_t)lane % offset;
          const uint32_t step = 32u % offset;
          for (uint32_t kb = 0; kb < mlen; kb += 32) {   // (same trip count on every lane: the shuffle needs them all)
            const uint32_t sym = __shfl_sync(0xffffffffu, tail, (32u - offset + j) & 31u);
            const uint32_t k = kb + lane;
            if (k < mlen) {
              d[op + k] = (uint8_t)sym;
              o[op + k] = (uint16_t)(sym >> 8);
              last = sym;
            }
            j += step;
            if (j >= offset) j -= offset;
          }
        } else {
          __syncwarp();                    // everything written so far is visible to every lane
          const long long base = (long long)op - (long long)offset;   // start of the pattern, may lie in front of the block
          const bool wraps = offset < mlen, pow2 = (offset & (offset - 1u)) == 0u;
          for (uint32_t k = lane; k < mlen; k += 32) {
            uint32_t j = k;
            if (wraps) j = pow2 ? (k & (offset - 1u)) : (k % offset);
            const long long sp = base + (long long)j;
            uint32_t v = 0, g;
            if (sp < 0) {
              g = (uint32_t)(-sp);         // a byte of the window in front of the block: remember which one
            } else {
              v = __ldcg(d + sp);
              g = __ldcg(o + sp);
            }
            d[op + k] = (uint8_t)v;
            o[op + k] = (uint16_t)g;
            last = v | (g << 8);
          }
        }
        push(mlen, last);
        op += mlen;
      }
      __syncwarp();
      if (!err && (ip != csize || op != dsize)) err = kErrSizeMismatch;
    }
    // publish the block (the chain walk runs beside this kernel and picks the blocks up in order)
    __syncwarp();
    if (lane == 0) {
      if (err) atomicMax(&ctl->error, err);
      __threadfence();
      atomicExch(T.done + b, 1u);
    }
  }
}

constexpr uint32_t kChainThreads = 512;
constexpr uint32_t kChainTail = 65536;      // bytes resolved per regular block (one more than an origin can reach: keeps the vectors aligned)
constexpr size_t kChainSmem = 2 * (size_t)kChainTail;

__global__ void __launch_bounds__(kChainThreads) lz4_resolve_chain_kernel(uint8_t* __restrict__ dst, uint16_t* __restrict__ origin,
                                                                          const DecCtl* ctl, DecTables T) {
  extern __shared__ __align__(16) unsigned char chain_smem[];
  __shared__ uint32_t sh_abort;
  if (!ctl->deferred) return;
  const uint32_t nblocks = ctl->nblocks;
  const uint32_t tid = threadIdx.x;
  // The window in front of the current block = the resolved tail of its predecessor lives in shared memory (two 64 KiB
  // buffers, swapped every block), so the gathers of the chain cost shared-memory latency instead of an L2 round trip each.
  uint32_t cur = 0;                          // byte offset of the buffer this block writes (0 or 65536); the other one is `prev`
  bool have_prev = false;                    // `prev` holds the 65536 bytes in front of the block
  // the table row of the next block is fetched while this one is resolved
  uint32_t link = nblocks ? T.link[0] : kNoLink, dsize = nblocks ? T.dsize[0] : 0u;
  unsigned long long doff = nblocks ? T.dst_off[0] : 0ull;
  for (uint32_t b = 0; b < nblocks; ++b) {
    const uint32_t nb = b + 1 < nblocks ? b + 1 : b;
    const uint32_t link_n = T.link[nb], dsize_n = T.dsize[nb];
    const unsigned long long doff_n = T.dst_off[nb];
    if (link != kNoLink) {
      // This kernel runs BESIDE pass 1 (second stream): wait until the block has been decoded. Pass 1 publishes every
      // block it takes, also a broken one, and the blocks in front of this one were waited for in earlier iterations.
      if (tid == 0) {
        uint32_t abort = 0;
        unsigned long long t_start = 0;
        while (atomicAdd(T.done + b, 0u) == 0u) {
          if (atomicAdd(const_cast<uint32_t*>(&ctl->error), 0u) != 0u) { abort = 1; break; }
          // never spin for ever: ten seconds without the block (pass 1 was not started, or was killed) end the walk with an error
          unsigned long long now;
          asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
          if (t_start == 0) t_start = now;
          if (now - t_start > 10000000000ull) {
            atomicMax(const_cast<uint32_t*>(&ctl->error), (uint32_t)kErrBadBlock);
            abort = 1;
            break;
          }
          __nanosleep(200);
        }
        __threadfence();
        sh_abort = abort;
      }
      __syncthreads();
      if (sh_abort) return;
    }
    if (link == kNoLink || link == kLinkHead) {              // (the same for every thread) heads hold real bytes only
      have_prev = false;
    } else {
      const unsigned long long t0r = doff + dsize - kChainTail;
      const bool regular = dsize >= kChainTail && doff >= kChainTail && ((((uintptr_t)(dst + t0r)) | ((uintptr_t)(dst + doff))) & 15) == 0 &&
                           (((uintptr_t)(origin + t0r)) & 15) == 0;
      if (regular) {
        uint8_t* prev = chain_smem + (cur ^ kChainTail);
        if (!have_prev) {                    // first regular block behind a head / an irregular block: fetch the window once
          const uint4* w = reinterpret_cast<const uint4*>(dst + doff - kChainTail);
          for (uint32_t v = tid; v < kChainTail / 16; v += kChainThreads) reinterpret_cast<uint4*>(prev)[v] = __ldcg(w + v);
          __syncthreads();
        }
        // 8 consecutive bytes per step: their origins are one 16-byte vector, their real bytes one 8-byte vector
        constexpr int kVec = kChainTail / 8 / kChainThreads;   // 16 vectors per thread, all loads in flight at once
        uint4 g[kVec];
        uint2 v[kVec];
        const uint4* go = reinterpret_cast<const uint4*>(origin + t0r);
        const uint2* gv = reinterpret_cast<const uint2*>(dst + t0r);
#pragma unroll
        for (int q = 0; q < kVec; ++q) {
          g[q] = __ldcg(go + tid + q * kChainThreads);
          v[q] = __ldcg(gv + tid + q * kChainThreads);
        }
        uint8_t* mine = chain_smem + cur;
#pragma unroll
        for (int q = 0; q < kVec; ++q) {
          const uint32_t gw[4] = {g[q].x, g[q].y, g[q].z, g[q].w};
          uint32_t lo = v[q].x, hi = v[q].y;
          if (gw[0] | gw[1] | gw[2] | gw[3]) {
            uint32_t out[2] = {0u, 0u};
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const uint32_t ge = (gw[e >> 1] >> (16 * (e & 1))) & 0xffffu;
              const uint32_t real = ((e < 4 ? lo : hi) >> (8 * (e & 3))) & 0xffu;
              const uint32_t byte = ge ? (uint32_t)prev[kChainTail - ge] : real;
              out[e >> 2] |= byte << (8 * (e & 3));
            }
            lo = out[0];
            hi = out[1];
            reinterpret_cast<uint2*>(dst + t0r)[tid + q * kChainThreads] = make_uint2(lo, hi);
          }
          reinterpret_cast<uint2*>(mine)[tid + q * kChainThreads] = make_uint2(lo, hi);
        }
        __syncthreads();
        cur ^= kChainTail;
        have_prev = true;
      } else {
        // short or unaligned block (the last one of a frame): gathers through L2
        const uint32_t tail = dsize < 65535u ? dsize : 65535u;
        const unsigned long long t0 = doff + dsize - tail;
        constexpr int kBatch = 16;
        for (uint32_t base = tid; base < tail; base += kChainThreads * kBatch) {
          uint32_t gg[kBatch];
          uint8_t vv[kBatch];
#pragma unroll
          for (int q = 0; q < kBatch; ++q) {
            const uint32_t i = base + kChainThreads * q;
            gg[q] = i < tail ? (uint32_t)__ldcg(origin + t0 + i) : 0u;
          }
#pragma unroll
          for (int q = 0; q < kBatch; ++q) vv[q] = gg[q] ? __ldcg(dst + doff - gg[q]) : (uint8_t)0;
#pragma unroll
          for (int q = 0; q < kBatch; ++q) {
            const uint32_t i = base + kChainThreads * q;
            if (gg[q]) dst[t0 + i] = vv[q];
          }
        }
        __syncthreads();
        have_prev = false;
      }
    }
    link = link_n;
    dsize = dsize_n;
    doff = doff_n;
  }
}

__global__ void __launch_bounds__(256) lz4_resolve_rest_kernel(uint8_t* __restrict__ dst, const uint16_t* __restrict__ origin,
                                                               const DecCtl* ctl, DecTables T) {
  if (ctl->error || !ctl->deferred) return;
  const uint32_t nblocks = ctl->nblocks;
  for (uint32_t b = blockIdx.x; b < nblocks; b += gridDim.x) {
    const uint32_t link = T.link[b];
    if (link == kNoLink || link == kLinkHead) continue;
    const unsigned long long doff = T.dst_off[b];
    const uint32_t dsize = T.dsize[b];
    const uint32_t body = dsize < 65535u ? 0u : dsize - 65535u;   // everything in front of the tail
    for (uint32_t i = threadIdx.x; i < body; i += blockDim.x) {
      const uint32_t g = __ldcg(origin + doff + i);
      if (g) dst[doff + i] = __ldcg(dst + doff - g);
    }
  }
}

}  // namespace

// number of block-linked blocks from which a stream takes the deferred-reference path (0 = never: every linked block waits
// for its predecessor, the behaviour before that path existed). sqyx_set_lz4_defer_min() lets tests and benches run both.
static std::atomic<long> g_defer_min{(long)kDeferMin};
long k_lz4_set_defer_min(long nblocks) {
  const long prev = g_defer_min.load(std::memory_order_relaxed);
  if (nblocks >= 0) g_defer_min.store(nblocks, std::memory_order_relaxed);
  return prev;
}

size_t k_lz4_decode_capacity(uint64_t dst_bytes) { return (size_t)(dst_bytes / kLz4BlockBytes + 1024); }

size_t k_lz4_decode_workspace_bytes(uint64_t dst_bytes) {
  const size_t cap = k_lz4_decode_capacity(dst_bytes);
  return 256 + cap * (8 + 8 + 4 + 4 + 4 + 4 + 4 + 4) + 8 * (cap / kTile + 2) + 256;
}

// Enqueues the whole decode; the status lands in workspace (see k_lz4_decode_status).
static DecTables dec_tables(void* workspace, uint64_t dst_bytes, unsigned long long** tile_sums_out) {
  const size_t cap = k_lz4_decode_capacity(dst_bytes);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  DecTables T;
  uint8_t* p = ws + 256;
  T.src_off = reinterpret_cast<unsigned long long*>(p); p += 8 * cap;
  T.dst_off = reinterpret_cast<unsigned long long*>(p); p += 8 * cap;
  T.word = reinterpret_cast<uint32_t*>(p); p += 4 * cap;
  T.dsize = reinterpret_cast<uint32_t*>(p); p += 4 * cap;
  T.link = reinterpret_cast<uint32_t*>(p); p += 4 * cap;
  T.done = reinterpret_cast<uint32_t*>(p); p += 4 * cap;
  T.reach = reinterpret_cast<uint32_t*>(p); p += 4 * cap;
  T.range = reinterpret_cast<uint32_t*>(p); p += 4 * cap;
  if (tile_sums_out) *tile_sums_out = reinterpret_cast<unsigned long long*>((reinterpret_cast<uintptr_t>(p) + 7) & ~(uintptr_t)7);
  return T;
}

size_t k_lz4_decode_linked_workspace_bytes(uint64_t dst_bytes) { return 2 * (size_t)dst_bytes + 256; }

// second step for streams of block-linked frames (k_lz4_decode_status reported them as deferred): `workspace` still
// holds the block table of k_lz4_decode_tables, `origins` has room for one uint16 per output byte
int k_lz4_decode_linked(const uint8_t* src, uint64_t src_bytes, uint8_t* dst, uint64_t dst_bytes, void* workspace, void* origins,
                        cudaStream_t st) {
  (void)src_bytes;
  DecCtl* ctl = reinterpret_cast<DecCtl*>(workspace);
  const DecTables T = dec_tables(workspace, dst_bytes, nullptr);
  uint16_t* org = static_cast<uint16_t*>(origins);
  // The chain walk starts together with pass 1 on a stream of its own and follows it block by block (T.done): the blocks
  // come in plane order, the all-zero planes in front are decoded within a millisecond, and only the tail of the walk is
  // left when the last noisy block of pass 1 is through.
  cudaStream_t aux = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
  SQYB_CUDA_OK(cudaStreamCreateWithFlags(&aux, cudaStreamNonBlocking));
  cudaError_t e = cudaEventCreateWithFlags(&fork, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&join, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(lz4_resolve_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kChainSmem);
  if (e == cudaSuccess) e = cudaEventRecord(fork, st);
  if (e == cudaSuccess) e = cudaStreamWaitEvent(aux, fork, 0);
  if (e == cudaSuccess) {
    // pass 1 is launched first: where kernels of different streams are serialised (profilers), the walk then simply finds
    // every block published; side by side, it gets an SM as soon as the first CTAs of pass 1 (the all-zero planes) retire
    lz4_decode_deferred_kernel<<<kNumSMs * 8, 256, 0, st>>>(src, dst, org, ctl, T);
    e = cudaGetLastError();
    if (e == cudaSuccess) {              // (the walk waits for pass 1: it is only started when pass 1 was)
      lz4_resolve_chain_kernel<<<1, kChainThreads, kChainSmem, aux>>>(dst, org, ctl, T);
      e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaEventRecord(join, aux);
  }
  if (e == cudaSuccess) e = cudaStreamWaitEvent(st, join, 0);
  if (e == cudaSuccess) {
    lz4_resolve_rest_kernel<<<kNumSMs * 8, 256, 0, st>>>(dst, org, ctl, T);
    SQYB_COUNT_LAUNCH(3);
    e = cudaGetLastError();
  }
  if (fork) cudaEventDestroy(fork);     // (released when the work that uses them has finished)
  if (join) cudaEventDestroy(join);
  cudaStreamDestroy(aux);
  return (int)e;
}

int k_lz4_decode_tables(const uint8_t* src, uint64_t src_bytes, uint64_t dst_bytes, void* workspace, int measure_all,
                        int allow_deferred, cudaStream_t st) {
  const size_t cap = k_lz4_decode_capacity(dst_bytes);
  DecCtl* ctl = reinterpret_cast<DecCtl*>(workspace);
  unsigned long long* tile_sums = nullptr;
  const DecTables T = dec_tables(workspace, dst_bytes, &tile_sums);
  const uint32_t tiles = (uint32_t)(cap / kTile + 1), tile_grid = tiles < 1024u ? tiles : 1024u;
  SQYB_CUDA_OK(cudaMemsetAsync(ctl, 0, sizeof(DecCtl), st));
  lz4_directory_kernel<<<1, kDirThreads, 0, st>>>(src, src_bytes, ctl, T, (uint32_t)cap, measure_all,
                                                  allow_deferred ? (int)g_defer_min.load(std::memory_order_relaxed) : 0);
  lz4_tile_sums_kernel<<<tile_grid, 256, 0, st>>>(src, ctl, tile_sums);
  lz4_expand_kernel<<<tile_grid, 256, 0, st>>>(src, ctl, T, tile_sums, dst_bytes);
  lz4_sizes_kernel<<<kNumSMs * 4, kDecThreads, 0, st>>>(src, ctl, T);
  lz4_offsets_kernel<<<1, kDirThreads, 0, st>>>(ctl, T, dst_bytes);
  SQYB_COUNT_LAUNCH(5);
  return (int)cudaGetLastError();
}

// the block decoders over the table k_lz4_decode_tables left in `workspace`: the whole stream (count == 0), or `nsets` sets of
// `count` consecutive blocks, set j starting at block first + j * set_stride, with work counter `slot` (0..31, one per launch
// in flight)
int k_lz4_decode_run(const uint8_t* src, uint64_t src_bytes, uint8_t* dst, uint64_t dst_bytes, void* workspace, uint32_t first,
                     uint32_t count, uint32_t nsets, uint32_t set_stride, uint32_t slot, cudaStream_t st) {
  DecCtl* ctl = reinterpret_cast<DecCtl*>(workspace);
  const DecTables T = dec_tables(workspace, dst_bytes, nullptr);
  const size_t win_smem = kWinWarps * kWinWarpSmem;
  if (count == 0 && dst_bytes <= kSmallStreamBytes)
    lz4_decode_kernel<4, 0><<<kNumSMs * 4, kWinWarps * 32, win_smem, st>>>(src, src_bytes, dst, ctl, T, first, count, nsets, set_stride,
                                                                           slot, nullptr, 0);
  else
    lz4_decode_kernel<5, 0><<<kNumSMs * 5, kWinWarps * 32, win_smem, st>>>(src, src_bytes, dst, ctl, T, first, count, nsets, set_stride,
                                                                           slot, nullptr, 0);
  SQYB_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

// the blocks d_list[0 .. nlist) of the table k_lz4_decode_tables left in `workspace` (built for stream_bytes decoded bytes), block
// d_list[t] into compact + t * 16 KiB;
// ctl->total_decoded restarts at 0 and counts the bytes of the blocks that decoded. The list rides in the table's `range`
// array (the fused transpose's counters, unused here). Always the 48-register build: a list is as long as the box is large.
int k_lz4_decode_list(const uint8_t* src, uint64_t src_bytes, uint64_t stream_bytes, uint8_t* compact, void* workspace,
                      const uint32_t* d_list, uint32_t nlist, cudaStream_t st) {
  DecCtl* ctl = reinterpret_cast<DecCtl*>(workspace);
  DecTables T = dec_tables(workspace, stream_bytes, nullptr);
  T.range = const_cast<uint32_t*>(d_list);
  SQYB_CUDA_OK(cudaMemsetAsync(&ctl->total_decoded, 0, sizeof(ctl->total_decoded), st));
  lz4_decode_kernel<5, kListMode><<<kNumSMs * 5, kWinWarps * 32, kWinWarps * kWinWarpSmem, st>>>(src, src_bytes, compact, ctl, T, 0,
                                                                                                 nlist, 0, 0, 0, nullptr, 0);
  SQYB_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

// (the fused route is taken for stacks of 1 GiB and more, api.cu: kFuseMinBytes — always the 48-register build)
template <int FW>
static void launch_decode_fused(const uint8_t* src, uint64_t src_bytes, uint8_t* planes, DecCtl* ctl, const DecTables& T,
                                uint16_t* vox, uint32_t bpp, cudaStream_t st) {
  lz4_decode_kernel<5, FW><<<kNumSMs * 5, kWinWarps * 32, kWinWarps * kWinWarpSmem, st>>>(src, src_bytes, planes, ctl, T, 0, 0, 0, 0, 0,
                                                                                        vox, bpp);
}

int k_lz4_decode_fused(const uint8_t* src, uint64_t src_bytes, uint8_t* planes, uint64_t plane_bytes, void* workspace, int w,
                       uint16_t* vox, cudaStream_t st) {
  if (w != 1 && w != 2 && w != 4 && w != 8) return -1;
  const uint64_t range_bytes = (uint64_t)kLz4BlockBytes * (16 / w);
  if (plane_bytes == 0 || plane_bytes % range_bytes || ((((uintptr_t)planes) | ((uintptr_t)vox)) & 31)) return -3;
  DecCtl* ctl = reinterpret_cast<DecCtl*>(workspace);
  const DecTables T = dec_tables(workspace, plane_bytes, nullptr);
  const uint32_t bpp = (uint32_t)(plane_bytes / range_bytes);
  switch (w) {
    case 1: launch_decode_fused<1>(src, src_bytes, planes, ctl, T, vox, bpp, st); break;
    case 2: launch_decode_fused<2>(src, src_bytes, planes, ctl, T, vox, bpp, st); break;
    case 4: launch_decode_fused<4>(src, src_bytes, planes, ctl, T, vox, bpp, st); break;
    case 8: launch_decode_fused<8>(src, src_bytes, planes, ctl, T, vox, bpp, st); break;
  }
  SQYB_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

// whether the table describes one indexed frame of this library whose 16 KiB blocks hold exactly dst_bytes (synchronises the
// stream)
int k_lz4_decode_own_frame(void* workspace, uint64_t dst_bytes, bool* own_frame, cudaStream_t st) {
  DecCtl h;
  SQYB_CUDA_OK(cudaMemcpyAsync(&h, workspace, sizeof(DecCtl), cudaMemcpyDeviceToHost, st));
  SQYB_CUDA_OK(cudaStreamSynchronize(st));
  *own_frame = !h.error && h.own && h.fast_bb == (uint32_t)kLz4BlockBytes && (uint64_t)h.fast_nblk * h.fast_bb == dst_bytes;
  return 0;
}

// copies {error, total_decoded} back (synchronises the stream)
int k_lz4_decode_status(void* workspace, uint32_t* error, uint64_t* total_decoded, uint32_t* deferred_blocks, cudaStream_t st) {
  DecCtl h;
  SQYB_CUDA_OK(cudaMemcpyAsync(&h, workspace, sizeof(DecCtl), cudaMemcpyDeviceToHost, st));
  SQYB_CUDA_OK(cudaStreamSynchronize(st));
  *error = h.error;
  *total_decoded = h.total_decoded;
  if (deferred_blocks) *deferred_blocks = h.deferred ? h.nlinked : 0u;
  return 0;
}

}  // namespace sqyb
