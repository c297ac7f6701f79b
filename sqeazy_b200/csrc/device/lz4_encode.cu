// Chunked LZ4 block encoder for sm_100a — one CTA per 16 KiB block, everything in shared memory.
//
// Replaces the reference's per-chunk liblz4 calls + serial compaction
// (encoders/lz4.hpp:214-242, encoders/lz4_utils.hpp:99-173 encode_serial, :193-274 encode_parallel,
// :175-190 remove_blanks). Output = valid LZ4 frame bytes (see lz4_format.h); compressed-byte parity
// with liblz4 is not defined by the reference (SURVEY F5) — validity, round trip through the
// reference decoder and the compression ratio are. The output is a pure function of the input bytes
// (and the pitch hint): no result depends on the order in which threads run.
//
// Per block (16 KiB of input staged in shared memory by 512 threads):
//   load    : 128-bit coalesced loads -> smem; all-equal blocks take a closed-form path
//   phase A0: byte-equality bit masks E_q for two fixed offsets — 1 and the row pitch of the stack in this stream (a
//             2048-voxel row of a bit plane is 256 bytes: what differs from the row above is what the sample scattered
//             differently) — one bit per position, 32 positions per thread
//   phase A1: fixed-offset candidates (>= 5 equal bytes) and their 2-bit length codes by shifts / ANDs on the masks
//   phase A2: the positions without such a candidate (a few per cent of a sparse plane) are COMPACTED into a list and
//             looked up in ONE shared-memory hash table that holds the FIRST listed position of the block per hash:
//             all 512 threads insert their entries with atomicMin (=> deterministic), one barrier, all 512 threads look
//             theirs up — two sweeps over the list (the version before ran 16 waves of 2 barriers, one per 1 KiB sub-block)
//   phase B : every THREAD parses its own 32-byte segment greedily with bit operations only; the length of a run
//             (fixed-offset match) is read off the masks in O(1): ones to the end of the segment, whole segments by
//             a per-warp "all ones" bit set, the rest from one more mask word. Hash matches are extended the same way
//             where both sides sit in runs, 4 bytes at a time where not. A match may overshoot into later segments
//             of the warp's 1 KiB sub-block, whose entry points move until the warp's parse is stable
//   phase C : the selected matches of all segments are compacted into one list in stream order (position | length, offset)
//   phase D : from here on a SEQUENCE has a thread: literal count, size, output offset (block-wide scan), token, length bytes,
//             offset and the literals (runs of more than 32 bytes are queued and copied by whole warps) follow from a list
//             entry and its predecessor — evenly spread over the 512 threads, where a thread that sized and emitted the
//             sequences of its own segment kept 4-12 of 32 lanes busy
//   hand-off: size word into the index frame + compressed bytes into a per-block staging slot (no CTA waits for
//             another); lz4_tile_sums_kernel + lz4_block_offsets_kernel prefix-sum the sizes over many CTAs and
//             lz4_scatter_kernel moves every block to its final offset (replaces remove_blanks)
#include "common.cuh"
#include "kernels.h"
#include "lz4_format.h"

namespace sqyb {
namespace {

constexpr int kB = kLz4BlockBytes;
constexpr int kThreads = 512;
constexpr int kWarps = kThreads / 32;
constexpr int kSub = kB / kWarps;        // 1 KiB sub-block per warp: matches never cross it
constexpr int kSegs = kB / 32;           // 32-byte segments, one per thread
constexpr int kPad = 256;
constexpr int kHashLog = 12;
constexpr int kInf = 0x7FFFFFFF;
constexpr int kNumShort = 1;             // short fixed offsets, in priority order out of 1, 2, 4, 3 ...
constexpr int kNumOff = kNumShort + 1;   // ... and the row pitch. Offsets 2, 4 and 3 were tried as well until the hash table
                                         // held the first occurrences of the whole block: since then a periodic pattern finds
                                         // itself there, and on every stream of tools/lz4_model2.c's sample (bit, 2-bit, nibble
                                         // and byte planes with and without background removal, raw and diff'ed voxels, 8-bit
                                         // stacks) the three change the size by < 0.1 % either way — for 13 % of the kernel's time
                                         // (cfg2 planes 6.04 -> 5.26 ms at -0.08 % payload, plain planes 6.23 -> 5.83 ms at +0.02 %)
__host__ __device__ constexpr int short_offset(int q) { return q == 0 ? 1 : (q == 1 ? 2 : (q == 2 ? 4 : 3)); }
constexpr int kListMax = 15104;          // positions that may look up the hash table (more: the rest goes without; sized so that
                                         // three CTAs still fit an SM — only all-noise blocks list more, and those are stored)
constexpr int kEarlyBytes = 2048;        // early-store test on the hash candidates of the first 2 KiB (tools/lz4_model2.c EARLY=: 4096, 2048 and 1024 decide alike) ...
constexpr int kEarlyMin = 128;           // ... a block with fewer candidates than this is stored
constexpr uint32_t kNoCand = 0xFFFFu;
constexpr uint32_t kNoPos = 0xFFFFFFFFu;
constexpr uint32_t kPrefetchAhead = 3 * kNumSMs;   // blocks between a CTA's block and the one it requests into L2 (one residency wave)
constexpr int kLitSelf = 32;             // literal runs up to this length are copied by their sequence's thread

static_assert(kSegs == kThreads, "one segment per thread");
static_assert(kSub == 1024 && kSegs / kWarps == 32, "a warp's 32 segments are one sub-block = one hash wave");

struct __align__(16) EncSmem {
  uint32_t data[(kB + kPad) / 4];
  union {
    uint16_t list[kListMax];             // phase A2: positions that look up; then, in place: candidate | code << 14 (kNoCand: none)
    uint32_t out[(kB + 64) / 4];         // phase D: encoded bytes (every list read happens before the first out write)
  };
  uint32_t htab[1 << kHashLog];          // phase A2: FIRST listed position of the block with this hash (kNoPos: none)
                                         // phases C, D: the block's sequences, position | length << 14
  uint32_t E[4][kSegs + 4];              // rows q < kNumOff: E[q][t] bit j: data[32t+j] == data[32t+j-off(q)]
                                         // row 2, as uint16 lead[kNumOff][kSegs + 2] (lead_row): ones of E[q] from the first position of
                                         //   segment t on, to the end of the warp's sub-block at most; 0 for the first segment of a
                                         //   sub-block (what a run of the sub-block in front continues with)
                                         // row 3: the `wants` masks of the first 2 KiB for the early-store test
                                         // phases C, D: all four rows hold the sequences' offsets (uint16)
  uint32_t segHM[kSegs];                 // per segment: positions with a hash candidate (>= 5 bytes)
  uint32_t full[kNumOff][kWarps];        // per warp: segments whose E[q] word is all ones
  int w_size[kWarps], w_off[kWarps];     // per-warp totals of the scans
  int total;
  int nlong;                             // phase D: queued long literal runs
  int early;                             // candidates seen by the early-store test
};

static_assert(sizeof(EncSmem) <= (228 * 1024 - 3 * 1024) / 3, "three CTAs per SM (1 KiB of each CTA's share is the system's)");
static_assert(sizeof(uint16_t) * kNumOff * (kSegs + 2) <= sizeof(uint32_t) * (kSegs + 4), "the lead table fits row 2 of S.E");
static_assert(kEarlyBytes / 32 <= kSegs, "the early-store test's wants masks fit row 3 of S.E");

__device__ __forceinline__ int ext_bytes(int v) {
  if (v < 15) return 0;          // by far the common case: keep the division off the hot path
  if (v < 270) return 1;
  return 1 + (v - 15) / 255;
}

__device__ __forceinline__ uint32_t load4(const uint32_t* words, int byte_off) {
  const uint32_t w0 = words[byte_off >> 2], w1 = words[(byte_off >> 2) + 1];
  return __funnelshift_r(w0, w1, (byte_off & 3) * 8);
}

// one step of a byte-equality bit mask: the four bits "byte j of a == byte j of b" are shifted in at the top of e, so that
// after the eight words of a segment word k's bits sit at 4k..4k+3. (x has a zero byte where a and b agree; bit 7 of
// ((x & 0x7f..) + 0x7f..) | x is clear exactly in those bytes; one high-half multiply gathers the four flags — it runs in the
// FMA pipe, next to the logic pipe that bounds this kernel. Six instructions where __vcmpeq4 + mask + multiply + shifts take nine.)
__device__ __forceinline__ uint32_t eq4_shift_in(uint32_t e, uint32_t a, uint32_t b) {
  const uint32_t x = a ^ b;
  const uint32_t t = (x & 0x7f7f7f7fu) + 0x7f7f7f7fu;
  const uint32_t y = ~(t | x) & 0x80808080u;
  return __funnelshift_r(e, __umulhi(y, 0x02040810u), 4);   // bits 7, 15, 23, 31 of y -> bits 0..3 of the high word
}

// per-warp totals of a block-wide scan (one int per warp in shared memory, complete behind a barrier) -> what the warps in
// front of this one add up to, and the grand total: a 16-lane shuffle scan instead of sixteen loads and adds per thread
__device__ __forceinline__ void warp_totals(const int* totals, int warp, int lane, int& before, int& all) {
  int v = lane < kWarps ? totals[lane] : 0;
#pragma unroll
  for (int d = 1; d < kWarps; d <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= d) v += t;
  }
  all = __shfl_sync(0xffffffffu, v, kWarps - 1);
  const int prev = __shfl_sync(0xffffffffu, v, (warp + 31) & 31);
  before = warp ? prev : 0;
}

// writes the LZ4 length extension for `v` (nibble already holds 15) at p, returns bytes written
__device__ __forceinline__ int put_ext(uint8_t* p, int v) {
  int r = v - 15, k = 0;
  while (r >= 255) { p[k++] = 255; r -= 255; }
  p[k++] = (uint8_t)r;
  return k;
}

// number of consecutive ones of E[q] from position x on, inside the sub-block of x: the ones left in x's segment, then
// what the table says about the segments behind it (lead_row: computed once per segment with ballots and a shuffle, so that
// the few lanes that measure a run do not walk the masks themselves)
// (the table lives in row 2 of S.E, which is free until phase C: it is written before the hash table is — which it shared
//  its memory with before — and the barrier between the two went away)
__device__ __forceinline__ uint16_t* lead_row(EncSmem& S, int q) { return reinterpret_cast<uint16_t*>(&S.E[2][0]) + q * (kSegs + 2); }
__device__ __forceinline__ const uint16_t* lead_row(const EncSmem& S, int q) { return reinterpret_cast<const uint16_t*>(&S.E[2][0]) + q * (kSegs + 2); }
__device__ __forceinline__ int run_ones(const EncSmem& S, int q, int x) {
  const int t = x >> 5, b = x & 31;
  const uint32_t z = ~(S.E[q][t] >> b);          // zeros where the run goes on; the shifted-in bits end it at the segment border
  const int r = z ? __ffs(z) - 1 : 32;           // (z == 0 only for b == 0 and a full word); r <= 32 - b
  return r == 32 - b ? r + (int)lead_row(S, q)[t + 1] : r;   // (the entry of a sub-block's first segment is 0: runs end there)
}

// The general path of a block (phases A0..D on the bytes in S.data), kept out of line: the closed-form path of all-equal
// blocks — 56 % of a background-removed stack, bound by bytes in flight — then keeps the short prologue and the register
// allocation of a kernel that does nothing else. Returns the encoded size; `stored` when the block does not shrink.
// pitch_words: row pitch of the stack in this stream in 32-bit words (a multiple of 8), 0 = none.
template <bool kWait>
__device__ __noinline__ int encode_general(EncSmem& S, const int n, const int pitch_words, bool& stored_out) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint8_t* data8 = reinterpret_cast<uint8_t*>(S.data);
  uint8_t* out8 = reinterpret_cast<uint8_t*>(S.out);
  int csize = 0;
  bool stored = false;
  // (set here and not beside the block load: shared-memory stores in the prologue delay the loads of the closed-form path
  //  of all-equal blocks, which is bound by bytes in flight; barriers lie between these stores and their first use)
  if (tid == 0) S.early = 0;
#pragma unroll
  for (int k = 0; k < (1 << kHashLog) / kThreads; ++k) S.htab[tid + k * kThreads] = kNoPos;
  // ---------------- phase A0: byte-equality bit masks for the fixed offsets ----------------
  // In bit-plane data byte runs and the row above carry the long matches. A thread compares its 32-byte
  // segment with itself shifted by the offset (eq4_shift_in on 8 words) and keeps one bit per position; a match of length L
  // at i with offset off(q) is then simply L consecutive ones in E_q starting at bit i — found, measured and extended
  // with shifts, ANDs and ffs on registers, never touching the bytes again.
  const int seg_lo = tid * 32;
  uint32_t Ms = 0, D0 = 0, D1 = 0, D2 = 0, C0 = 0, C1 = 0;   // candidate mask, offset index planes, length code planes
  uint32_t wants = 0;                                        // positions that look up the hash table
  // Phases A0 and A1 of a warp's 1 KiB sub-block depend on nothing another warp computes (masks and candidates of a segment
  // look one segment ahead and one back, inside the sub-block), so a warp runs them on its own — which lets four SAMPLED
  // warps settle first whether the block is noise (early store, below) before the other twelve spend anything on it.
  auto analyse = [&]() {
    {
      uint32_t W[9];
      W[0] = tid > 0 ? S.data[8 * tid - 1] : 0u;
  #pragma unroll
      for (int k = 0; k < 8; ++k) W[k + 1] = S.data[8 * tid + k];
      const int lim = n - kLz4LastLiterals - seg_lo;     // match bytes never touch the last 5 bytes of the block
      const uint32_t tailmask = lim >= 32 ? 0xffffffffu : (lim <= 0 ? 0u : (1u << lim) - 1u);
  #pragma unroll
      for (int q = 0; q < kNumShort; ++q) {
        const int d = short_offset(q);
        uint32_t e = 0;
  #pragma unroll
        for (int k = 0; k < 8; ++k) {
          const uint32_t prev = d == 4 ? W[k] : __funnelshift_r(W[k], W[k + 1], 32 - 8 * d);   // bytes 4k-d .. 4k-d+3
          e = eq4_shift_in(e, W[k + 1], prev);
        }
        if (tid == 0) e &= ~((1u << d) - 1u);            // no source in front of the block
        S.E[q][tid] = e & tailmask;
      }
      {
        uint32_t e = 0;
        if (pitch_words > 0 && 8 * tid >= pitch_words) {   // (whole segments: the pitch is a multiple of 32 bytes)
  #pragma unroll
          for (int k = 0; k < 8; ++k) {
            e = eq4_shift_in(e, W[k + 1], S.data[8 * tid + k - pitch_words]);
          }
        }
        S.E[kNumShort][tid] = e & tailmask;
      }
      if (tid < kNumOff) S.E[tid][kSegs] = 0;
    }
    __syncwarp();

    // ---------------- phase A1: fixed-offset candidates of this thread's segment (registers only) ----------------
    {
      uint32_t L6 = 0, L7 = 0, L8 = 0;
      uint32_t tail4 = 0;                                  // positions inside a byte run with exactly four equal bytes ahead
  #pragma unroll
      for (int q = 0; q < kNumOff; ++q) {
        // matches never cross the warp's 1 KiB sub-block: the last segment sees no successor
        const uint32_t own = S.E[q][tid];
        const unsigned long long e = (unsigned long long)own | ((unsigned long long)(lane == 31 ? 0u : S.E[q][tid + 1]) << 32);
        const unsigned long long r5 = e & (e >> 1) & (e >> 2) & (e >> 3) & (e >> 4);
        const unsigned long long r6 = r5 & (e >> 5), r7 = r6 & (e >> 6), r8 = r7 & (e >> 7);
        if (q == 0) {
          // Inside a run of equal bytes, the position with exactly four of them ahead never pays for a lookup: a match from
          // there would have to carry the run's last four bytes AND what follows it, and the parse only lands there when a
          // hash match ends on that very byte (tools/lz4_model2.c NOINTERIOR=1 NIQ=1 KEEPTAIL=3: 12 % fewer lookups on
          // background-removed planes — the phase that dominates their sparse planes — at the same size; the three positions
          // behind it are worth 0.5 % of the size each and keep looking up)
          const uint32_t r4only = (uint32_t)(e & (e >> 1) & (e >> 2) & (e >> 3) & ~r5);
          const uint32_t before = (own << 1) | (lane ? S.E[0][tid - 1] >> 31 : 0u);   // the byte in front continues the run too
          tail4 = r4only & before;
        }
        const uint32_t sel = (uint32_t)r5 & ~Ms;         // at least 5 bytes and no better-ranked offset yet
        Ms |= sel;
        L6 |= sel & (uint32_t)r6;
        L7 |= sel & (uint32_t)r7;
        L8 |= sel & (uint32_t)r8;
        if (q & 1) D0 |= sel;
        if (q & 2) D1 |= sel;
        if (q & 4) D2 |= sel;
        const uint32_t fullset = __ballot_sync(0xffffffffu, own == 0xffffffffu);
        if (lane == 0) S.full[q][warp] = fullset;
      }
      const int lim = n - kLz4MFLimit + 1 - seg_lo;      // a match starts at most 12 bytes before the block end
      const uint32_t valid = lim >= 32 ? 0xffffffffu : (lim <= 0 ? 0u : (1u << lim) - 1u);
      Ms &= valid;
      C0 = (L6 ^ L7 ^ L8) & Ms;                          // code = number of the planes L6,L7,L8 that are set: 5,6,7,>=8 bytes
      C1 = L7 & Ms;
      wants = ~Ms & valid & ~tail4;
      S.segHM[tid] = 0;
    }
  };
  // Four warps analyse their sub-blocks first: 0 and 1 (the first 2 KiB: what the hash test below looks at), 6 and 11.
  const bool sampled = warp < kEarlyBytes / kSub || warp == 6 || warp == 11;
  // kWait: the other twelve wait for the verdict; otherwise (kLz4HintNoNoise) all sixteen analyse at once. Which warps
  // analyse first never reaches the output: the early-store test reads the sampled warps only.
  const bool eager = kWait ? sampled : true;
  int cnt = 0, incl = 0;               // positions of this segment that look up; inclusive scan over the warp
  auto count_wants = [&]() {
    cnt = __popc(wants);
    incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += t;
    }
    if (lane == 31) S.w_size[warp] = incl;
  };
  if (eager) {
    analyse();
    count_wants();
  }
  // (for the early-store test below: the `wants` masks of the first 2 KiB, in a row of S.E that is free until phase C)
  if (warp < kEarlyBytes / kSub) S.E[3][tid] = wants;
  const int ncand_short = sampled ? __reduce_add_sync(0xffffffffu, __popc(Ms)) : 0;   // (warp-uniform)
  // One barrier, two answers. Lanes 0..15 of a warp vote "rich": a sampled warp that is already rich in fixed-offset
  // candidates — every compressible bit-plane block — settles the early-store test for the CTA. Lane 16 votes "this warp has
  // not analysed its sub-block yet" (at most twelve such votes).
  const int votes = __syncthreads_count(lane < 16 ? ncand_short >= kEarlyMin : (lane == 16 && !eager));
  const bool rich = votes >= 16, all_eager = (votes & 15) == 0;
  const bool test_early = !rich && n > kEarlyBytes;

  int entry0 = 0;
  auto lead_table = [&]() {
#pragma unroll
    for (int q = 0; q < kNumOff; ++q) {
      const uint32_t own = S.E[q][tid];
      const int lead = own == 0xffffffffu ? 32 : __ffs(~own) - 1;
      const uint32_t nf = ~(S.full[q][warp] >> lane);          // zeros: full segments from this one on (shifted-in bits: the warp ends)
      const int k = min(nf ? __ffs(nf) - 1 : 32, 32 - lane);   // full segments in a row, this one included
      const int tail = __shfl_sync(0xffffffffu, lead, (lane + k) & 31);   // leading ones of the first segment that is not full
      lead_row(S, q)[tid] = lane ? (uint16_t)(32 * k + (lane + k < 32 ? tail : 0)) : (uint16_t)0;
      if (tid == 0) lead_row(S, q)[kSegs] = 0;
      // first guess of where the parse enters this segment (phase B), from the same words
      const uint32_t prevtop = __shfl_up_sync(0xffffffffu, own >> 27, 1);
      if (lane > 0 && prevtop == 31u) entry0 = max(entry0, lead);
    }
  };
  // ---------------- phase A2: hash candidates for the positions without a fixed-offset match ----------------
  // The wanting positions of the block are compacted, in order, into S.list (exclusive scan of the per-thread counts), all
  // of them are inserted into one hash table, then all of them are looked up. An entry is overwritten by its result.
  int mybase;
  {
    auto write_list = [&](int base) {
      uint32_t m = wants;
      int e = base;
      while (m && e < kListMax) {
        const int j = __ffs(m) - 1;
        m &= m - 1;
        S.list[e++] = (uint16_t)(seg_lo + j);
      }
    };
    // The table keeps the FIRST listed position of the block per hash (atomicMin: the same whatever the thread order),
    // filled before anything is looked up: a position finds the earliest occurrence of its four bytes — in its own
    // sub-block as well — and the whole phase is two sweeps over the list with all 512 threads instead of a wave per
    // sub-block (16 x 2 barriers, most threads idle). tools/lz4_model2.c (FIRST=1): ratio +0.1..0.5 % over the waves.
    auto insert = [&](int from, int to) {
      for (int e = from + tid; e < to; e += kThreads) {
        const int i = (int)S.list[e];
        const uint32_t h = (load4(S.data, i) * 2654435761u) >> (32 - kHashLog);
        atomicMin(&S.htab[h], (uint32_t)i);
      }
    };
    auto lookup = [&](int from, int to) {
      for (int e = from + tid; e < to; e += kThreads) {
        const int i = (int)S.list[e];
        // eight bytes at i and at the candidate from three aligned words each
        const uint32_t* wi = S.data + (i >> 2);
        const uint32_t shi = (i & 3) * 8;
        const uint32_t i0 = wi[0], i1 = wi[1], i2 = wi[2];
        const uint32_t v = __funnelshift_r(i0, i1, shi);
        const uint32_t c = S.htab[(v * 2654435761u) >> (32 - kHashLog)];
        uint32_t res = kNoCand;
        const uint32_t* wc = S.data + ((c & (kB - 1)) >> 2);
        const uint32_t shc = (c & 3) * 8;
        const uint32_t c0 = wc[0], c1 = wc[1];
        if (c < (uint32_t)i && __funnelshift_r(c0, c1, shc) == v) {
          const int maxlen = min((i & ~(kSub - 1)) + kSub, n - kLz4LastLiterals) - i;
          const uint32_t x = __funnelshift_r(i1, i2, shi) ^ __funnelshift_r(c1, wc[2], shc);
          int len = 4 + (x ? ((__ffs(x) - 1) >> 3) : 4);
          if (len > maxlen) len = maxlen;
          // 4-byte matches save one byte and cost a sequence on both ends of the codec: dropping them keeps the
          // ratio within ~1 % on bit planes, improves it on background-removed stacks and matches liblz4 on noisy
          // 8-bit codes (tools/lz4_model.c), while halving the number of sequences
          if (len >= 5) {
            res = c | ((uint32_t)(len - 5 < 3 ? len - 5 : 3) << 14);   // code 0,1,2: exactly 5,6,7 bytes; 3: >= 8
            atomicOr(&S.segHM[i >> 5], 1u << (i & 31));
          }
        }
        S.list[e] = (uint16_t)res;       // the entry is overwritten by its result
      }
    };
    // Early store: a block with fewer than kEarlyMin candidates — four times the fixed-offset ones of the sampled 4 KiB + the
    // hash ones of the first 2 KiB — is noise (camera-noise bit planes, 8-bit quantiser codes) and would shrink by < 3 %
    // (tools/lz4_model2.c EARLY=2048 SAMPLED=1 DUMP=1: noise blocks count <= 29, every compressible block of the sample sets
    // >= 243; the sampled count decides like the full one on all of them). It is stored without the masks of the other
    // twelve sub-blocks, the list, the parse and the emission, which is also what makes its decode a plain copy.
    // (Positions of the first 2 KiB find the same sources in a table that holds the first 2 KiB only as in the full one: a
    //  first occurrence lies in front of them.)
    if (test_early) {
      // The test needs no list: the 2048 positions are spread over the 512 threads as they are (four each, consecutive lanes
      // on consecutive bytes), the segments' owners have passed their `wants` masks through S.E[3]. Nothing is kept:
      // a block that goes on enters its first 2 KiB into the list below like the rest — the same first occurrences come out
      // (they lie in front of the position that looks them up) — so a noise block never pays for the serial list writes of
      // two warps (32 entries per thread) while fourteen wait.
      if (lane == 0 && ncand_short) atomicAdd(&S.early, 4 * ncand_short);
      static_assert(kEarlyBytes / kSub == 2 && kEarlyBytes % kThreads == 0, "the first two warps own the tested positions");
      uint32_t mine = 0;                 // bit k: position k * kThreads + tid looks up
#pragma unroll
      for (int k = 0; k < kEarlyBytes / kThreads; ++k) {
        const int i = k * kThreads + tid;
        if ((S.E[3][i >> 5] >> (i & 31)) & 1u) {
          mine |= 1u << k;
          atomicMin(&S.htab[(load4(S.data, i) * 2654435761u) >> (32 - kHashLog)], (uint32_t)i);
        }
      }
      __syncthreads();
      int nf = 0;
#pragma unroll
      for (int k = 0; k < kEarlyBytes / kThreads; ++k) {
        const int i = k * kThreads + tid;
        if ((mine >> k) & 1u) {
          const uint32_t v = load4(S.data, i);
          const uint32_t c = S.htab[(v * 2654435761u) >> (32 - kHashLog)];
          // a candidate counts when it gives a match of >= 5 bytes inside the sub-block (what the lookup below keeps)
          if (c < (uint32_t)i && load4(S.data, (int)c) == v && data8[i + 4] == data8[c + 4] &&
              min((i & ~(kSub - 1)) + kSub, n - kLz4LastLiterals) - i >= 5)
            ++nf;
        }
      }
      nf = __reduce_add_sync(0xffffffffu, nf);
      if (lane == 0 && nf) atomicAdd(&S.early, nf);
      __syncthreads();
      if (S.early < kEarlyMin) {
        stored_out = true;
        return 0;
      }
    }
    if (!all_eager) {
      if (!eager) {
        analyse();
        count_wants();
      }
      __syncthreads();
    }
    __syncwarp();                      // (S.full of this warp)
    lead_table();
    {
      int wbase, wall;
      warp_totals(S.w_size, warp, lane, wbase, wall);
      mybase = wbase + incl - cnt;
      write_list(mybase);
      const int total = min(wall, kListMax);
      __syncthreads();
      insert(0, total);
      __syncthreads();
      lookup(0, total);
      __syncthreads();
    }
  }
  const uint32_t HM = S.segHM[tid];
  // (no test for "no candidate at all" and no barrier here: such a block comes out of the parse with no sequence and is stored)
  {
    // ---------------- phase B: every thread parses its own 32-byte segment greedily ----------------
    // A match may overshoot into the following segments of the same warp; their entry point moves and
    // they re-parse until the warp's parse is stable (lane k is final after at most k+1 rounds).
    const int limit = min((warp + 1) * kSub, n - kLz4LastLiterals);
    const uint32_t M = Ms | HM;                        // hash candidates exist only where no fixed-offset one does
    uint32_t Sel = 0;
    unsigned long long lens = 0;       // lengths of the long matches of this segment, 11 bits each, in order
    // First guess of where the parse enters this segment: if the previous segment ends inside a run with period d
    // (its last five bytes continue one), the match that covers them runs on to the end of the ones of E_d here. A
    // segment in the middle of a long run then has nothing to parse, and half of the repair parses of the cascade
    // disappear. A wrong guess is corrected like any other moved entry point.
    int entry = entry0, exit_abs = seg_lo + 32;
    bool need = true;
    while (true) {                     // cascade rounds
      if (need) {
        // thread-serial parse: bit operations, the masks and (for hash matches) a few words of the block
        // (a repair parse — the entry point moved — runs only until it meets a match the parse before it had selected: from
        //  there on everything is what it was, lengths included)
        const uint32_t oldSel = Sel;
        const unsigned long long oldLens = lens;
        int pos = entry, nlong = 0;
        bool spliced = false;
        Sel = 0;
        lens = 0;
        while (pos < 32) {
          const uint32_t mm = M & (0xffffffffu << pos);
          if (!mm) break;
          const int j = __ffs(mm) - 1;
          if ((oldSel >> j) & 1u) {
            const int dropped = __popc(oldSel & C0 & C1 & ((1u << j) - 1u));   // long matches of the old parse in front of j
            Sel |= oldSel & (0xffffffffu << j);
            lens |= (oldLens >> (11 * dropped)) << (11 * nlong);
            spliced = true;
            break;
          }
          const int i = seg_lo + j, maxlen = limit - i;
          int code, len;
          if ((Ms >> j) & 1u) {
            code = ((C0 >> j) & 1) | (((C1 >> j) & 1) << 1);
            len = 5 + code;
            if (code == 3) {           // a run: its length is in the masks
              const int q = ((D0 >> j) & 1u) | (((D1 >> j) & 1u) << 1) | (((D2 >> j) & 1u) << 2);
              len = run_ones(S, q, i);
            }
          } else {
            const int e = mybase + __popc(wants & ((1u << j) - 1u));
            const uint32_t ce = S.list[e];
            const int c = (int)(ce & 0x3FFFu);
            code = (int)(ce >> 14);
            len = 5 + code;
            C0 = (C0 & ~(1u << j)) | ((uint32_t)(code & 1) << j);      // phases C and D read the code from the planes
            C1 = (C1 & ~(1u << j)) | ((uint32_t)(code >> 1) << j);
            if (code == 3) {
              // both sides inside runs (the zeros around an isolated byte of a sparse plane): equal as far as both runs go
              len = 8;
              while (len < maxlen) {
                const int k = min(run_ones(S, 0, i + len), run_ones(S, 0, c + len));
                len += k;
                if (len >= maxlen) break;
                const uint32_t x = load4(S.data, i + len) ^ load4(S.data, c + len);
                if (x) { len += (__ffs(x) - 1) >> 3; break; }
                len += 4;
              }
            }
          }
          if (len > maxlen) len = maxlen;
          if (code == 3) {
            lens |= (unsigned long long)len << (11 * nlong);
            nlong++;
          }
          Sel |= 1u << j;
          pos = j + len;
        }
        if (!spliced) exit_abs = seg_lo + (pos > 32 ? pos : 32);
      }
      int incl = exit_abs;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl = max(incl, t);
      }
      int prev = __shfl_up_sync(0xffffffffu, incl, 1);
      if (lane == 0) prev = seg_lo;
      const int ne = min(max(prev - seg_lo, 0), 32);
      need = ne != entry;
      entry = ne;
      if (!__any_sync(0xffffffffu, need)) break;
    }

    // ---------------- phase C: the selected matches of the block, compacted in stream order ----------------
    // Phases A and B give every 32-byte segment a thread; the sequences they select are spread unevenly (none inside a run,
    // five or six around the isolated bytes of a sparse plane), and a thread that sizes and emits the sequences of its own
    // segment one after the other keeps 4-12 of the 32 lanes busy. From here on a SEQUENCE has a thread: the matches are
    // written to a list (position | length, offset), everything else — literal counts, sizes, output offsets, tokens,
    // literal copies — follows from a list entry and its predecessor, evenly spread over the 512 threads.
    const int nm = __popc(Sel);
    int sincl = nm;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, sincl, d);
      if (lane >= d) sincl += t;
    }
    if (lane == 31) S.w_size[warp] = sincl;
    __syncthreads();                                   // every warp is through phase B as well: S.E (masks and lead table) is free
    int sbase, nseq;
    warp_totals(S.w_size, warp, lane, sbase, nseq);
    sbase += sincl - nm;
    uint32_t* seq_pl = S.htab;                                           // position | length << 14
    uint16_t* seq_off = reinterpret_cast<uint16_t*>(&S.E[0][0]);         // match offset
    static_assert(sizeof(S.htab) >= 4 * (kB / 5 + 2) && sizeof(S.E) >= 2 * (kB / 5 + 2), "room for every sequence of a block");
    {
      uint32_t m = Sel;
      unsigned long long q = lens;
      int k = sbase;
      while (m) {
        const int j = __ffs(m) - 1;
        m &= m - 1;
        const int code = ((C0 >> j) & 1) | (((C1 >> j) & 1) << 1);
        int len = 5 + code;
        if (code == 3) { len = (int)(q & 0x7FF); q >>= 11; }
        const int i = seg_lo + j;
        uint32_t off;
        if ((Ms >> j) & 1u) {
          const uint32_t qq = ((D0 >> j) & 1u) | (((D1 >> j) & 1u) << 1) | (((D2 >> j) & 1u) << 2);
          off = qq == (uint32_t)kNumShort ? 4u * (uint32_t)pitch_words : (uint32_t)short_offset((int)qq);
        } else {
          off = (uint32_t)(i - (int)(S.list[mybase + __popc(wants & ((1u << j) - 1u))] & 0x3FFFu));
        }
        seq_pl[k] = (uint32_t)i | ((uint32_t)len << 14);
        seq_off[k] = (uint16_t)off;
        ++k;
      }
    }
    if (tid == 0) S.nlong = 0;
    __syncthreads();                                   // the list is complete; S.list (candidates) is free from here on

    // ---- matches cut at a sub-block border are joined again ----
    // A run that goes on over a 1 KiB border was parsed as one match per sub-block, every piece with a token, an offset and
    // length bytes of its own. When the last match
    // of a sub-block ends on the border and the first one behind it starts there with the same offset, the two are one valid
    // match: the piece behind the border becomes a dummy (bit 31: sized and emitted as nothing) and its length goes to the
    // head of its chain. Lane w of warp 0 looks at border w; chains over whole sub-blocks are resolved with two ballots.
    // (cfg2 planes: payload -0.77 %, 5.31 -> 5.39 ms; a parse without the borders would save 2.2 %, tools/lz4_model2.c)
    constexpr uint32_t kJoined = 0x80000000u;
    if (warp == 0) {
      const int cntw = lane < kWarps ? S.w_size[lane] : 0;       // sequences of sub-block `lane`
      int wincl = cntw;
#pragma unroll
      for (int d = 1; d < kWarps; d <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, wincl, d);
        if (lane >= d) wincl += t;
      }
      const int k0 = wincl - cntw;                               // index of its first sequence
      bool joins = false;
      uint32_t cur = 0;
      if (lane >= 1 && lane < kWarps && cntw > 0 && k0 > 0) {
        cur = seq_pl[k0];
        const uint32_t prev = seq_pl[k0 - 1];
        const uint32_t border = (uint32_t)lane * kSub;
        joins = (cur & 0x3FFFu) == border && (prev & 0x3FFFu) + (prev >> 14) == border && seq_off[k0] == seq_off[k0 - 1];
      }
      const uint32_t J = __ballot_sync(0xffffffffu, joins);
      const uint32_t single = __ballot_sync(0xffffffffu, cntw == 1);
      // border w continues the chain of border w-1 when both join and sub-block w-1 consists of that one match
      const uint32_t cont = J & (J << 1) & (single << 1);
      const int first = 31 - __clz(~cont & ((2u << lane) - 1u));  // the chain's first border (bit 0 of cont is never set)
      const int head = __shfl_sync(0xffffffffu, k0, first) - 1;
      __syncwarp();                                              // every lane has read the lengths as the parse left them
      if (joins) {
        atomicAdd(&seq_pl[head], (cur >> 14) << 14);
        seq_pl[k0] = cur | kJoined;
      }
    }
    __syncthreads();
    // sequences [s0, s1) of this thread; entry nseq stands for the block's final literal run
    const int per = (nseq + kThreads) / kThreads;      // ceil((nseq + 1) / kThreads)
    const int s0 = min(tid * per, nseq + 1), s1 = min(s0 + per, nseq + 1);
    int mysize = 0;
    bool has_long = false;             // a literal run of this thread's sequences is copied by a whole warp (phase D)
    {
      int prev_end = 0;
      // (the sequence in front may be a joined piece or a head that has grown: the chain's pieces end where it ends, except
      //  for pieces in the middle of a chain — and those are followed by a piece, which reads nothing from prev_end)
      if (s0 > 0 && s0 <= nseq) { const uint32_t pp = seq_pl[s0 - 1]; prev_end = (int)(pp & 0x3FFFu) + (int)((pp & ~kJoined) >> 14); }
      for (int sq = s0; sq < s1; ++sq) {
        if (sq < nseq) {
          const uint32_t pl = seq_pl[sq];
          const int pos = (int)(pl & 0x3FFFu), len = (int)((pl & ~kJoined) >> 14), lit = pos - prev_end;
          if (!(pl & kJoined)) {
            mysize += 3 + ext_bytes(lit) + lit + ext_bytes(len - 4);
            has_long = has_long || lit > kLitSelf;
          }
          prev_end = pos + len;
        } else {
          const int lit = n - prev_end;
          mysize += 1 + ext_bytes(lit) + lit;
          has_long = has_long || lit > kLitSelf;
        }
      }
    }
    int oincl = mysize;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, oincl, d);
      if (lane >= d) oincl += t;
    }
    if (lane == 31) S.w_off[warp] = oincl;
    const int any_long = __syncthreads_or(has_long);
    int o;
    warp_totals(S.w_off, warp, lane, o, csize);
    o += oincl - mysize;
    if (csize >= n || nseq == 0) {
      stored = true;
    } else {
      // ---------------- phase D: emission, a thread per sequence ----------------
      // Literal runs of up to kLitSelf bytes are copied by the sequence's thread, longer ones (noise between runs) are queued
      // and copied by whole warps afterwards.
      uint32_t* longrec = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(S.list) + sizeof(S.out));   // behind `out`
      static_assert(sizeof(S.list) >= sizeof(S.out) + 8 * (kB / (kLitSelf + 1) + 2), "room for the long literal runs");
      int prev_end = 0;
      if (s0 > 0 && s0 <= nseq) { const uint32_t pp = seq_pl[s0 - 1]; prev_end = (int)(pp & 0x3FFFu) + (int)((pp & ~kJoined) >> 14); }
      for (int sq = s0; sq < s1; ++sq) {
        const bool fin = sq >= nseq;
        int pos = n, len = 4;
        if (!fin) {
          const uint32_t pl = seq_pl[sq];
          pos = (int)(pl & 0x3FFFu);
          len = (int)((pl & ~kJoined) >> 14);
          if (pl & kJoined) {                          // a joined piece: its bytes belong to the match of the chain's head
            prev_end = pos + len;
            continue;
          }
        }
        const int lit = pos - prev_end, ml = len - 4;
        out8[o] = (uint8_t)(((lit < 15 ? lit : 15) << 4) | (fin ? 0 : (ml < 15 ? ml : 15)));
        int d = o + 1;
        if (lit >= 15) d += put_ext(out8 + d, lit);
        if (lit <= kLitSelf) {
          for (int t = 0; t < lit; ++t) out8[d + t] = data8[prev_end + t];
        } else {
          const int r = atomicAdd(&S.nlong, 1);          // (the order of the queue does not reach the output)
          longrec[2 * r] = (uint32_t)prev_end | ((uint32_t)lit << 14);
          longrec[2 * r + 1] = (uint32_t)d;
        }
        d += lit;
        if (!fin) {
          const uint32_t off = seq_off[sq];
          out8[d] = (uint8_t)(off & 0xff);
          out8[d + 1] = (uint8_t)(off >> 8);
          d += 2;
          if (ml >= 15) d += put_ext(out8 + d, ml);
        }
        o = d;
        prev_end = pos + len;
      }
      if (any_long) {                  // (block-uniform: most blocks of a sparse plane have none and save the barrier)
        __syncthreads();
        const int nlong = S.nlong;
        for (int r = warp; r < nlong; r += kWarps) {
          const uint32_t r0 = longrec[2 * r], dst = longrec[2 * r + 1];
          const int from = (int)(r0 & 0x3FFFu), cnt = (int)(r0 >> 14);
          for (int t = lane; t < cnt; t += 32) out8[dst + t] = data8[from + t];
        }
      }
    }
  }
  stored_out = stored;
  return csize;
}

// kWait: see encode_general (the launch's kLz4HintNoNoise flag cleared)
template <bool kWait>
__global__ void __launch_bounds__(kThreads, 3)
lz4_encode_kernel(const uint8_t* __restrict__ src, uint64_t raw_bytes, uint8_t* __restrict__ dst, uint32_t nblocks,
                  uint8_t* __restrict__ staging, uint32_t* __restrict__ stats, uint32_t first, uint32_t set_stride, int pitch_words) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  EncSmem& S = *reinterpret_cast<EncSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  const uint32_t b = first + blockIdx.y * set_stride + blockIdx.x;   // (whole stream: first = 0, one set)
  if (b >= nblocks) return;
  const uint64_t boff = (uint64_t)b * kB;
  const int n = (int)((raw_bytes - boff) < (uint64_t)kB ? (raw_bytes - boff) : (uint64_t)kB);
  const uint8_t* bsrc = src + boff;
  uint8_t* data8 = reinterpret_cast<uint8_t*>(S.data);
  uint8_t* out8 = reinterpret_cast<uint8_t*>(S.out);
  // The block that the CTA one residency wave behind this one will load is requested into L2 now: an all-equal block is
  // bound by the bytes an SM has in flight (3 CTAs x 16 KiB), and a noise block holds its slot for the early-store test
  // without loading anything (measured: all-zero input 1.147 -> 1.068 ms per 4 GiB, cfg2 planes 5.35 -> 5.29 ms, plain planes
  // 5.73 -> 5.65 ms; three waves ahead: the same, ten: half of the gain).
  if (tid < kB / 128 && blockIdx.x + kPrefetchAhead < gridDim.x) {
    const uint64_t poff = boff + (uint64_t)kPrefetchAhead * kB + (uint64_t)tid * 128u;
    if (poff < raw_bytes) asm volatile("prefetch.global.L2 [%0];" ::"l"(src + poff));
  }

  // ---------------- load ----------------
  bool same = true;
  if ((((uintptr_t)bsrc) & 15) == 0) {
    const uint4* s4 = reinterpret_cast<const uint4*>(bsrc);
    const uint32_t pat = (uint32_t)bsrc[0] * 0x01010101u;
    uint4* d4 = reinterpret_cast<uint4*>(S.data);
#pragma unroll
    for (int k = 0; k < kB / 16 / kThreads; ++k) {
      const int v = tid + k * kThreads;
      uint4 x = make_uint4(0, 0, 0, 0);
      if ((v + 1) * 16 <= n) {
        x = ld_stream(s4 + v);
        same = same && (x.x == pat) && (x.y == pat) && (x.z == pat) && (x.w == pat);
      } else if (v * 16 < n) {
        uint32_t w[4] = {0, 0, 0, 0};
#pragma unroll
        for (int q = 0; q < 16; ++q) {
          const bool in = v * 16 + q < n;
          const uint32_t byte = in ? bsrc[v * 16 + q] : 0;
          same = same && (!in || byte == (pat & 0xffu));
          w[q >> 2] |= byte << (8 * (q & 3));
        }
        x = make_uint4(w[0], w[1], w[2], w[3]);
      }
      d4[v] = x;
    }
  } else {
    const uint8_t first = bsrc[0];
    for (int i = tid; i < kB; i += kThreads) {
      const uint8_t x = i < n ? bsrc[i] : 0;
      data8[i] = x;
      same = same && (i >= n || x == first);
    }
  }
  if (tid < kPad / 4) S.data[kB / 4 + tid] = 0;
  const int all_same = __syncthreads_and(same ? 1 : 0);

  int csize = 0;        // encoded bytes (without the 4-byte block header)
  bool stored = false;
  int kind = 0;         // stats: 0 general, 1 constant, 2 stored

  if (all_same && n >= 16) {
    // ---------------- closed form: 1 literal, match(offset 1, n-6), 5 literals ----------------
    kind = 1;
    if (warp == 0) {
      const uint8_t v = data8[0];
      const int mlen = n - 6;
      const int e = mlen - 4;
      const int nx = ext_bytes(e);
      if (lane == 0) {
        out8[0] = (uint8_t)((1 << 4) | (e < 15 ? e : 15));
        out8[1] = v;
        out8[2] = 1;
        out8[3] = 0;
      }
      if (e >= 15) {
        const int r = e - 15;
        for (int k = lane; k < nx; k += 32) out8[4 + k] = (k < nx - 1) ? 255 : (uint8_t)(r % 255);
      }
      if (lane < 6) out8[4 + nx + lane] = lane == 0 ? (uint8_t)(5 << 4) : v;
      if (lane == 0) S.total = 4 + nx + 6;
    }
    __syncthreads();
    csize = S.total;
  } else {
    csize = encode_general<kWait>(S, n, pitch_words, stored);
    if (stored) { csize = n; kind = 2; }
  }
  __syncthreads();

  // ---------------- hand-off: size word + staged bytes; no CTA ever waits for another ----------------
  // (a decoupled look-back here made fast CTAs — constant blocks — sit on their SM slot until slower predecessors had
  //  published their sizes: 30-60 % of the kernel's stall samples, profiles/. Offsets are now a separate tiny scan and
  //  the compressed blocks are moved once more by lz4_scatter_kernel; the extra traffic is 2x the compressed bytes.)
  const uint32_t word = stored ? ((uint32_t)n | kLz4StoredFlag) : (uint32_t)csize;
  if (!stored) {
    uint4* st4 = reinterpret_cast<uint4*>(staging + (uint64_t)b * kB);
    const uint4* o4 = reinterpret_cast<const uint4*>(S.out);
    for (int v = tid; v < (csize + 15) / 16; v += kThreads) st4[v] = o4[v];
  }
  if (tid == 0) {
    uint8_t* ip = dst + kSkippableHeaderBytes + sizeof(SqybIndexHeader) + 4ull * b;   // the block's entry in the index frame
    if ((((uintptr_t)ip) & 3) == 0) *reinterpret_cast<uint32_t*>(ip) = word;
    else { ip[0] = (uint8_t)word; ip[1] = (uint8_t)(word >> 8); ip[2] = (uint8_t)(word >> 16); ip[3] = (uint8_t)(word >> 24); }
    if (stats) atomicAdd(stats + kind, 1u);
  }
}

// Compaction (replaces remove_blanks, lz4_utils.hpp:175-190): the byte offset of a block is the prefix sum of
// (4 + block bytes) over the index words. A single-CTA scan of 262144 words costs 0.23 ms (one SM's latency), so the
// sum is split over many CTAs: lz4_tile_sums_kernel adds up tiles of 1024 blocks, lz4_block_offsets_kernel adds the
// tile sums in front of its tile and scans its own 1024 words.
constexpr int kEncTile = 1024;

__device__ __forceinline__ uint32_t enc_index_word(const uint8_t* idx, bool aligned, uint32_t i) {
  const uint8_t* p = idx + 4ull * i;
  return aligned ? reinterpret_cast<const uint32_t*>(idx)[i]
                 : (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}

__global__ void __launch_bounds__(256) lz4_tile_sums_kernel(const uint8_t* __restrict__ dst, uint32_t nblocks,
                                                            unsigned long long* __restrict__ tile_sums) {
  __shared__ uint32_t wsum[8];
  const uint8_t* idx = dst + kSkippableHeaderBytes + sizeof(SqybIndexHeader);
  const bool aligned = (((uintptr_t)idx) & 3) == 0;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t ntiles = (nblocks + kEncTile - 1) / kEncTile;
  for (uint32_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
    uint32_t s = 0;
#pragma unroll
    for (int k = 0; k < kEncTile / 256; ++k) {
      const uint32_t i = t * kEncTile + k * 256 + tid;
      if (i < nblocks) s += 4u + (enc_index_word(idx, aligned, i) & 0x7FFFFFFFu);
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

// byte offset of every block header (relative to the first one); the CTA of the last tile also writes the EndMark and
// the sizes
__global__ void __launch_bounds__(256) lz4_block_offsets_kernel(uint8_t* __restrict__ dst, uint32_t nblocks,
                                                                const unsigned long long* __restrict__ tile_sums,
                                                                unsigned long long* __restrict__ offsets,
                                                                unsigned long long* __restrict__ payload_bytes_out) {
  __shared__ unsigned long long red[8];
  __shared__ uint32_t tsum[8];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint8_t* idx = dst + kSkippableHeaderBytes + sizeof(SqybIndexHeader);
  const bool aligned = (((uintptr_t)idx) & 3) == 0;
  const uint32_t ntiles = (nblocks + kEncTile - 1) / kEncTile;
  for (uint32_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
    unsigned long long bsum = 0;
    for (uint32_t u = tid; u < t; u += 256) bsum += tile_sums[u];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) bsum += __shfl_down_sync(0xffffffffu, bsum, d);
    __syncthreads();
    if (lane == 0) red[warp] = bsum;
    // thread-local scan over 4 consecutive blocks + scan of the 256 thread totals
    uint32_t loc[4], s = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t i = t * kEncTile + tid * 4 + k;
      loc[k] = s;
      s += i < nblocks ? 4u + (enc_index_word(idx, aligned, i) & 0x7FFFFFFFu) : 0u;
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
    unsigned long long base = 0;
    for (int w = 0; w < 8; ++w) base += red[w];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t i = t * kEncTile + tid * 4 + k;
      if (i < nblocks) offsets[i] = base + wbase + incl - s + loc[k];
    }
    if (t == ntiles - 1 && tid == 0) {
      uint32_t tot = 0;
      for (int w = 0; w < 8; ++w) tot += tsum[w];
      const unsigned long long end = lz4_prefix_bytes(nblocks) + base + tot;
      for (int k = 0; k < 4; ++k) dst[end + k] = 0;  // EndMark
      *payload_bytes_out = end + 4;
      const unsigned long long frame_bytes = end + 4 - (lz4_prefix_bytes(nblocks) - kLz4FrameHeaderBytes);
      uint8_t* fp = dst + kSkippableHeaderBytes + 24;   // SqybIndexHeader::frame_bytes
      for (int k = 0; k < 8; ++k) fp[k] = (uint8_t)(frame_bytes >> (8 * k));
    }
    __syncthreads();
  }
}

// moves every block to its final place in the frame: header word + bytes (staged compressed bytes, or the raw input
// for stored blocks). A warp per block; 16-byte stores, source words funnel-shifted to the destination's alignment.
__global__ void __launch_bounds__(256) lz4_scatter_kernel(const uint8_t* __restrict__ src, uint64_t raw_bytes,
                                                          const uint8_t* __restrict__ staging, uint8_t* __restrict__ dst,
                                                          uint32_t nblocks, const unsigned long long* __restrict__ offsets) {
  const int lane = threadIdx.x & 31;
  const uint32_t wpb = blockDim.x >> 5;
  const uint8_t* idx = dst + kSkippableHeaderBytes + sizeof(SqybIndexHeader);
  const unsigned long long first = lz4_prefix_bytes(nblocks);
  for (uint32_t b = blockIdx.x * wpb + (threadIdx.x >> 5); b < nblocks; b += gridDim.x * wpb) {
    const uint8_t* p = idx + 4ull * b;
    const uint32_t word = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
    const uint32_t nbytes = word & 0x7FFFFFFFu;
    const uint8_t* from = (word & kLz4StoredFlag) ? src + (uint64_t)b * kB : staging + (uint64_t)b * kB;
    uint8_t* g = dst + first + offsets[b];
    if (lane < 4) g[lane] = (uint8_t)(word >> (8 * lane));
    g += 4;
    uint32_t head = (uint32_t)((16 - ((uintptr_t)g & 15)) & 15);
    if (head > nbytes) head = nbytes;
    if ((uint32_t)lane < head) g[lane] = __ldg(from + lane);
    const uint8_t* f = from + head;
    uint8_t* o = g + head;
    const uint32_t rest = nbytes - head;
    uint32_t nvec = rest >= 24 ? (rest - 8) >> 4 : 0;   // keeps the 5-word read inside the block's bytes
    const uint32_t sh = ((uintptr_t)f & 3) * 8;
    const uint32_t* fw = reinterpret_cast<const uint32_t*>((uintptr_t)f & ~(uintptr_t)3);
    if (reinterpret_cast<const uint8_t*>(fw) < from) nvec = 0;   // never read in front of the block's first byte
    for (uint32_t v = lane; v < nvec; v += 32) {
      const uint32_t* q = fw + v * 4;
      const uint32_t x0 = __ldg(q), x1 = __ldg(q + 1), x2 = __ldg(q + 2), x3 = __ldg(q + 3), x4 = __ldg(q + 4);
      uint4 val;
      val.x = __funnelshift_r(x0, x1, sh);
      val.y = __funnelshift_r(x1, x2, sh);
      val.z = __funnelshift_r(x2, x3, sh);
      val.w = __funnelshift_r(x3, x4, sh);
      reinterpret_cast<uint4*>(o)[v] = val;
    }
    for (uint32_t k = (nvec << 4) + lane; k < rest; k += 32) o[k] = __ldg(f + k);
  }
}

// static prefix: skippable header, index header (frame_bytes patched by the last block), frame header
__global__ void lz4_write_prefix_kernel(uint8_t* dst, uint64_t raw_bytes, uint32_t nblocks,
                                        unsigned long long* payload_bytes_out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const uint64_t end = lz4_write_prefix(dst, nblocks, raw_bytes, kLz4FrameHeaderBytes + kLz4EndMarkBytes);
  if (nblocks == 0) {
    lz4_put32(dst + end, 0);   // EndMark
    *payload_bytes_out = end + kLz4EndMarkBytes;
  }
}

}  // namespace

size_t k_lz4_encode_workspace_bytes(uint64_t raw_bytes) {
  const uint64_t nb = lz4_nblocks(raw_bytes);
  return 256 + 8 * nb + 8 * (nb / kEncTile + 2) + 256 + nb * (uint64_t)kB + 256;   // control | block offsets | tile sums | staging (one slot per block)
}

// workspace layout: [0,8) payload bytes (u64) | [16,28) block-kind counters | [256, 256+8*nblocks) offsets | staging
namespace {
struct EncWs {
  uint32_t nblocks;
  unsigned long long *payload, *offsets, *tile_sums;
  uint8_t* staging;
  uint32_t* stats;
};
int enc_ws(uint64_t raw_bytes, void* workspace, EncWs& W) {
  const uint64_t nb64 = lz4_nblocks(raw_bytes);
  if (nb64 > 0xFFFFFFF0ull) return -2;
  W.nblocks = (uint32_t)nb64;
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  W.payload = reinterpret_cast<unsigned long long*>(ws);
  W.stats = reinterpret_cast<uint32_t*>(ws + 16);
  W.offsets = reinterpret_cast<unsigned long long*>(ws + 256);
  W.tile_sums = W.offsets + W.nblocks;
  W.staging = ws + ((256 + 8ull * W.nblocks + 8ull * (W.nblocks / kEncTile + 2) + 255) & ~255ull);
  return 0;
}
}  // namespace

int k_lz4_encode_begin(uint64_t raw_bytes, uint8_t* dst, void* workspace, cudaStream_t st) {
  EncWs W;
  if (int e = enc_ws(raw_bytes, workspace, W)) return e;
  SQYB_CUDA_OK(cudaMemsetAsync(workspace, 0, 64, st));
  lz4_write_prefix_kernel<<<1, 32, 0, st>>>(dst, raw_bytes, W.nblocks, W.payload);
  SQYB_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

// pitch hint -> words; only multiples of 32 bytes well inside a block qualify (whole segments, sources inside the block)
static int pitch_words_of(uint32_t pitch_bytes) {
  return (pitch_bytes >= 32u && pitch_bytes <= (uint32_t)kB / 2 && pitch_bytes % 32u == 0u) ? (int)(pitch_bytes / 4u) : 0;
}

int k_lz4_encode_blocks(const uint8_t* src, uint64_t raw_bytes, uint8_t* dst, void* workspace, uint32_t first, uint32_t count,
                        uint32_t nsets, uint32_t set_stride, uint32_t pitch_bytes, cudaStream_t st) {
  EncWs W;
  if (int e = enc_ws(raw_bytes, workspace, W)) return e;
  if (!count || !nsets) return 0;
  if (nsets > 65535u || (uint64_t)first + (uint64_t)(nsets - 1) * set_stride + count > W.nblocks) return -2;
  const dim3 grid(count, nsets);
  const int pw = pitch_words_of(pitch_bytes & ~kLz4HintNoNoise);
  if (pitch_bytes & kLz4HintNoNoise) {
    SQYB_CUDA_OK(cudaFuncSetAttribute(lz4_encode_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(EncSmem)));
    lz4_encode_kernel<false><<<grid, kThreads, sizeof(EncSmem), st>>>(src, raw_bytes, dst, W.nblocks, W.staging, W.stats, first, set_stride, pw);
  } else {
    SQYB_CUDA_OK(cudaFuncSetAttribute(lz4_encode_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(EncSmem)));
    lz4_encode_kernel<true><<<grid, kThreads, sizeof(EncSmem), st>>>(src, raw_bytes, dst, W.nblocks, W.staging, W.stats, first, set_stride, pw);
  }
  SQYB_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

int k_lz4_encode_end(const uint8_t* src, uint64_t raw_bytes, uint8_t* dst, void* workspace, cudaStream_t st) {
  EncWs W;
  if (int e = enc_ws(raw_bytes, workspace, W)) return e;
  if (!W.nblocks) return 0;
  const uint32_t ntiles = (W.nblocks + kEncTile - 1) / kEncTile;
  const uint32_t tile_grid = ntiles < (uint32_t)kNumSMs * 8 ? ntiles : (uint32_t)kNumSMs * 8;
  lz4_tile_sums_kernel<<<tile_grid, 256, 0, st>>>(dst, W.nblocks, W.tile_sums);
  lz4_block_offsets_kernel<<<tile_grid, 256, 0, st>>>(dst, W.nblocks, W.tile_sums, W.offsets, W.payload);
  const uint32_t scatter_blocks = (W.nblocks + 7) / 8 < (uint32_t)kNumSMs * 8 ? (W.nblocks + 7) / 8 : (uint32_t)kNumSMs * 8;
  lz4_scatter_kernel<<<scatter_blocks, 256, 0, st>>>(src, raw_bytes, W.staging, dst, W.nblocks, W.offsets);
  SQYB_COUNT_LAUNCH(3);
  return (int)cudaGetLastError();
}

int k_lz4_encode(const uint8_t* src, uint64_t raw_bytes, uint8_t* dst, void* workspace, uint32_t pitch_bytes, cudaStream_t st) {
  EncWs W;
  if (int e = enc_ws(raw_bytes, workspace, W)) return e;
  if (int e = k_lz4_encode_begin(raw_bytes, dst, workspace, st)) return e;
  if (int e = k_lz4_encode_blocks(src, raw_bytes, dst, workspace, 0, W.nblocks, 1, 0, pitch_bytes, st)) return e;
  return k_lz4_encode_end(src, raw_bytes, dst, workspace, st);
}

}  // namespace sqyb
