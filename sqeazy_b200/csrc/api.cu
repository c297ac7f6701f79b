// C-ABI layer: SQY_* (include/sqeazy.h, host buffers, the reference's boundary) and sqyx_*
// (include/sqeazy_b200.h, device buffers). Sequences the sm_100a kernels the way
// dynamic_pipeline::detail_encode / detail_decode sequence the reference's stages
// (dynamic_pipeline.hpp:619-690, 772-846). No CPU compute path exists here: without a CUDA device
// every compute entry point fails with 1.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nvtx3/nvToolsExt.h>   // header-only: ranges cost nothing unless a profiler injects its library

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/sqeazy.h"
#include "../../include/sqeazy_b200.h"
#include "device/kernels.h"
#include "device/lz4_format.h"
#include "host/numerics.hpp"
#include "host/pipeline.hpp"
#include "host/text.hpp"
#include "staging.hpp"

using namespace sqyb;

namespace sqyb {
std::atomic<long> g_kernel_launches{0};
}

namespace {

constexpr int kVersionMajor = 0, kVersionMinor = 7, kVersionPatch = 2;

#define CK(expr)                                                                                          \
  do {                                                                                                    \
    cudaError_t _e = (expr);                                                                              \
    if (_e != cudaSuccess) {                                                                              \
      std::fprintf(stderr, "[sqeazy_b200] CUDA error %s at %s:%d\n", cudaGetErrorString(_e), __FILE__, __LINE__); \
      return 1;                                                                                           \
    }                                                                                                     \
  } while (0)

#define CKK(expr)                                                                             \
  do {                                                                                        \
    int _r = (expr);                                                                          \
    if (_r != 0) {                                                                            \
      std::fprintf(stderr, "[sqeazy_b200] kernel launch failed (%d) at %s:%d\n", _r, __FILE__, __LINE__); \
      return 1;                                                                               \
    }                                                                                         \
  } while (0)

// ---- cached device scratch, one arena per device, guarded by one lock (calls are serialised) ----
enum Slot { kSlotA = 0, kSlotB, kSlotIn, kSlotOut, kSlotWs, kSlotSmall, kSlotOrigins, kSlotRoi, kNumSlots };

struct Arena {
  void* ptr[kNumSlots] = {nullptr};
  size_t cap[kNumSlots] = {0};
  long last_stats[4] = {0, 0, 0, 0};
  int get(int slot, size_t bytes, void** out) {
    if (bytes == 0) bytes = 256;
    if (cap[slot] < bytes) {
      if (ptr[slot]) cudaFree(ptr[slot]);
      ptr[slot] = nullptr;
      cap[slot] = 0;
      const size_t want = (bytes + (size_t(1) << 20) - 1) & ~((size_t(1) << 20) - 1);
      cudaError_t e = cudaMalloc(&ptr[slot], want);
      if (e != cudaSuccess) {
        std::fprintf(stderr, "[sqeazy_b200] cudaMalloc(%zu) failed: %s\n", want, cudaGetErrorString(e));
        return 1;
      }
      cap[slot] = want;
    }
    *out = ptr[slot];
    return 0;
  }
  // host memory: the sub-frame that the indexed host route of the ROI calls assembles (roi_host). It is kept across calls: a buffer
  // of hundreds of MB (a batch of patches) would be mapped afresh by every allocation and have all its pages faulted in again
  std::unique_ptr<uint8_t[]> frame;
  size_t frame_cap = 0;
  uint8_t* host_frame(size_t bytes) {
    if (frame_cap < bytes) {
      frame.reset();
      frame.reset(new uint8_t[bytes]);   // uninitialised: the caller writes every byte it sends
      frame_cap = bytes;
    }
    return frame.get();
  }
  void release() {
    for (int i = 0; i < kNumSlots; ++i) {
      if (ptr[i]) cudaFree(ptr[i]);
      ptr[i] = nullptr;
      cap[i] = 0;
    }
    frame.reset();
    frame_cap = 0;
  }
};

// One context per device: scratch arena, copy stream, batch lanes, and the lock that serialises the calls that use this
// device. Calls on different devices run concurrently (round 1 had one process-wide lock).
// batch entry points (sqyx_*_batch_device_*): every lane of a batch has its own stream and scratch, so the kernels of
// different stacks share the SMs instead of queueing behind each other's tails
constexpr int kBatchLanes = 8;
constexpr int kMaxDevices = 16;
struct Dev {
  std::mutex mu;
  Arena arena;
  cudaStream_t copy_stream = nullptr;
  Arena batch_arena[kBatchLanes];
  cudaStream_t batch_stream[kBatchLanes] = {};
  long roi_info[4] = {-1, 0, 0, 0};   // the most recent sub-volume decode on this device (sqyx_last_roi_info)
};
Dev g_dev[kMaxDevices];
std::mutex g_timer_mu;   // g_stage_ms

// ---- optional per-stage CUDA-event timing (sqyx_enable_stage_timing) ----
enum StageTimer { kTFilterSwap = 0, kTLz4Enc, kTHist, kTLutApply, kTLz4Dec, kTLutDec, kTSwapDec, kNumTimers };
std::atomic<int> g_timing{0};
float g_stage_ms[kNumTimers] = {0};

// every stage of a call is also an NVTX range (SURVEY 5: the reference's tracing is wall-clock timers around the stage
// calls, verbs/bench.hpp:181-194): `nsys` / `ncu --nvtx` show filter+transpose, LZ4, histogram, LUT per call
const char* const kStageNames[kNumTimers] = {"sqy:filter+bitswap encode", "sqy:lz4 encode", "sqy:histogram", "sqy:lut apply",
                                             "sqy:lz4 decode", "sqy:lut decode", "sqy:bitswap decode"};
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

struct ScopedStageTimer {
  cudaEvent_t a = nullptr, b = nullptr;
  cudaStream_t st;
  int slot;
  bool on;
  NvtxRange range;
  ScopedStageTimer(int slot_, cudaStream_t st_) : st(st_), slot(slot_), on(g_timing.load() != 0), range(kStageNames[slot_]) {
    if (on) {
      cudaEventCreate(&a);
      cudaEventCreate(&b);
      cudaEventRecord(a, st);
    }
  }
  void stop() {
    if (on && a) {
      cudaEventRecord(b, st);
      cudaEventSynchronize(b);
      float ms = 0;
      cudaEventElapsedTime(&ms, a, b);
      {
        std::lock_guard<std::mutex> lk(g_timer_mu);
        g_stage_ms[slot] += ms;
      }
      cudaEventDestroy(a);
      cudaEventDestroy(b);
      a = b = nullptr;
    }
  }
  ~ScopedStageTimer() { stop(); }
};

std::mutex g_set_mu;
std::vector<int> g_set;          // set by sqyx_set_devices / sqyx_set_device; empty = not pinned by the caller

// the device a single-device call works on: SQY_CUDA_DEVICE, else a device set of one (sqyx_set_devices), else the calling
// thread's current device
int pick_device(int* out) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
    std::fprintf(stderr, "[sqeazy_b200] no CUDA device available (this build has no CPU path)\n");
    return 1;
  }
  int dev = 0;
  if (const char* env = std::getenv("SQY_CUDA_DEVICE")) {
    dev = std::atoi(env);
    if (dev < 0 || dev >= n) return 1;
    if (cudaSetDevice(dev) != cudaSuccess) return 1;
  } else {
    int pinned = -1;
    {
      std::lock_guard<std::mutex> lk(g_set_mu);
      if (g_set.size() == 1) pinned = g_set[0];
    }
    if (pinned >= 0) {
      dev = pinned;
      if (dev >= n || cudaSetDevice(dev) != cudaSuccess) return 1;
    } else if (cudaGetDevice(&dev) != cudaSuccess) {
      return 1;
    }
  }
  if (dev >= kMaxDevices) return 1;
  *out = dev;
  return 0;
}

// picks the call's device and holds its lock for the lifetime of the object
struct DevLock {
  Dev* dev = nullptr;
  int id = -1;
  std::unique_lock<std::mutex> lk;
  int acquire() {
    if (pick_device(&id)) return 1;
    dev = &g_dev[id];
    lk = std::unique_lock<std::mutex>(dev->mu);
    return 0;
  }
  int acquire(int device) {   // a given device; made current for the calling thread
    if (device < 0 || device >= kMaxDevices || cudaSetDevice(device) != cudaSuccess) return 1;
    id = device;
    dev = &g_dev[id];
    lk = std::unique_lock<std::mutex>(dev->mu);
    return 0;
  }
};

// LZ4 pitch hint (kernels.h): bytes between vertically adjacent voxels in the stream the `lz4` stage sees — a function of
// pipeline and shape only, so every route (device, streamed, sharded) writes the same bytes
uint32_t lz4_pitch_hint(const Pipeline& pl, const std::vector<uint64_t>& shape) {
  if (shape.size() < 2 || !pl.has_sink) return 0;
  const uint64_t X = shape.back();
  uint64_t pitch = 0;
  if (pl.sink.kind == StageKind::Quantiser && pl.has_tail && pl.head.empty()) pitch = X;                 // rows of 8-bit codes
  else if (pl.sink.kind == StageKind::Lz4 && !pl.head.empty() && pl.head.back().kind == StageKind::Bitswap) {
    const uint64_t bits = X * (uint64_t)pl.head.back().w;                                                 // bits of one row in one plane
    if (bits % 8 == 0) pitch = bits / 8;
  } else if (pl.sink.kind == StageKind::Lz4 && pl.head.empty()) pitch = X * (uint64_t)pl.elem;           // raw voxels
  uint32_t hint = pitch <= 8192 ? (uint32_t)pitch : 0u;
  // bit planes behind a background removal hold no noise planes: every warp of the encoder starts at once (kernels.h)
  if (pl.sink.kind == StageKind::Lz4)
    for (const Stage& s : pl.head)
      if (s.kind == StageKind::RemoveBackground || s.kind == StageKind::RmEstBkrd) hint |= kLz4HintNoNoise;
  return hint;
}

uint64_t shape_product(const std::vector<uint64_t>& shape) {
  uint64_t n = 1;
  for (uint64_t d : shape) n *= d;
  return shape.empty() ? 0 : n;
}

// the arena's small slot: what the histogram, quantiser and estimate steps keep on the device. Fields that overlap are never
// used by the same step.
struct SmallSlot {
  uint32_t* hist;      // four 65536-bin histograms (the quantiser uses the first)
  uint8_t* enc_lut;    // quantiser encode LUT, 65536 codes, over the second histogram
  uint16_t* dec_lut;   // quantiser decode LUT, 256 voxels, behind the histograms
  uint32_t* support;   // the estimate's 16 support indices, behind the histograms
};

int small_slot(Arena& A, SmallSlot* s) {
  void* p = nullptr;
  if (A.get(kSlotSmall, 4 * 65536 * sizeof(uint32_t) + 4096, &p)) return 1;
  uint32_t* h = static_cast<uint32_t*>(p);
  *s = SmallSlot{h, reinterpret_cast<uint8_t*>(h + 65536), reinterpret_cast<uint16_t*>(h + 4 * 65536), h + 4 * 65536};
  return 0;
}

// ---- rmestbkrd threshold: GPU histograms of the sampled faces/rows + host support formula ----
// what the estimate reads, as device pointers: the first `portion` voxels of the z = 0 and z = Z-1 faces and the rows y = 0 /
// y = Y-1 at z in {1, Z/2, Z-2} (nullptr: that z does not exist). The callers whose stack is not resident as a whole (streamed
// and sharded host paths) send just these pieces.
struct EstimateSamples {
  const uint16_t* face[2];
  const uint16_t* row[2][3];
  uint64_t portion, X;
};

EstimateSamples estimate_samples_of(const uint16_t* d_src, uint64_t Z, uint64_t Y, uint64_t X, size_t l2) {
  EstimateSamples S;
  const uint64_t frame = Y * X;
  S.portion = rmest_frame_portion(frame, l2);
  S.X = X;
  S.face[0] = d_src;
  S.face[1] = d_src + (Z - 1) * frame;
  // rows y = 0 and y = Y-1 at z in {1, Z/2, Z-2}, background_scheme_utils.hpp:79-103 (z indices are used as given, like the reference)
  const uint64_t zs[3] = {1, Z / 2, Z - 2};
  const uint64_t ys[2] = {0, Y - 1};
  for (int i = 0; i < 2; ++i)
    for (int k = 0; k < 3; ++k)   // Z < 3: the reference would read out of bounds; we skip those rows
      S.row[i][k] = zs[k] >= Z ? nullptr : d_src + zs[k] * frame + ys[i] * X;
  return S;
}

int estimate_background_samples(Arena& A, const EstimateSamples& S, float* supports, int* threshold, cudaStream_t st) {
  SmallSlot small;
  if (small_slot(A, &small)) return 1;
  uint32_t* d_h = small.hist;
  CK(cudaMemsetAsync(d_h, 0, 4 * 65536 * sizeof(uint32_t), st));
  // z = 0 and z = Z-1 faces (first `portion` elements), background_scheme_utils.hpp:57-77
  CKK(k_histogram_u16(S.face[0], S.portion, d_h, st));
  CKK(k_histogram_u16(S.face[1], S.portion, d_h + 65536, st));
  for (int i = 0; i < 2; ++i)
    for (int k = 0; k < 3; ++k)
      if (S.row[i][k]) CKK(k_histogram_u16(S.row[i][k], S.X, d_h + (2 + i) * 65536, st));
  // support index of the four histograms on the device; 64 bytes come back instead of 1 MiB of bins
  CKK(k_support_index(d_h, 4, 0.99f, small.support, st));
  uint32_t idx[16];
  CK(cudaMemcpyAsync(idx, small.support, sizeof(idx), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  float mn = 0.f;
  for (int i = 0; i < 4; ++i) {
    supports[i] = support_from_index(idx[4 * i], idx[4 * i + 1], idx[4 * i + 2]);
    if (i == 0 || supports[i] < mn) mn = supports[i];
  }
  *threshold = (int)(uint16_t)mn;  // remove_background_scheme(raw_type) ctor truncates
  return 0;
}

int estimate_background(Arena& A, const uint16_t* d_src, uint64_t Z, uint64_t Y, uint64_t X, long l2_bytes, float* supports,
                        int* threshold, cudaStream_t st) {
  if (Z == 0 || Y == 0 || X == 0) return 1;
  const size_t l2 = l2_bytes >= 0 ? (size_t)l2_bytes : host_l2_cache_bytes();
  return estimate_background_samples(A, estimate_samples_of(d_src, Z, Y, X, l2), supports, threshold, st);
}

// the same from a stack in HOST memory: only the sampled pieces cross the bus, packed into the arena's kSlotB (which the streamed
// and sharded host encoders have no other use for)
int estimate_background_host(Arena& A, const uint16_t* h_src, uint64_t Z, uint64_t Y, uint64_t X, int* threshold, cudaStream_t st) {
  if (Z == 0 || Y == 0 || X == 0) return 1;
  const EstimateSamples H = estimate_samples_of(h_src, Z, Y, X, host_l2_cache_bytes());
  EstimateSamples D = H;
  void* scratch = nullptr;
  if (A.get(kSlotB, 2 * (2 * H.portion + 6 * X), &scratch)) return 1;
  uint16_t* q = static_cast<uint16_t*>(scratch);
  for (int f = 0; f < 2; ++f) {
    CK(cudaMemcpyAsync(q, H.face[f], 2 * H.portion, cudaMemcpyHostToDevice, st));
    D.face[f] = q;
    q += H.portion;
  }
  for (int i = 0; i < 2; ++i)
    for (int k = 0; k < 3; ++k) {
      if (!H.row[i][k]) continue;
      CK(cudaMemcpyAsync(q, H.row[i][k], 2 * X, cudaMemcpyHostToDevice, st));
      D.row[i][k] = q;
      q += X;
    }
  float sup[4];
  return estimate_background_samples(A, D, sup, threshold, st);
}

// ---- encode ----
// payload size of the LZ4 encode whose workspace is `ws`, once `st` has drained; the block-kind counts go to A.last_stats
int lz4_encode_result(Arena& A, const void* ws, cudaStream_t st, uint64_t* payload_bytes) {
  unsigned long long hres[4] = {0, 0, 0, 0};
  CK(cudaMemcpyAsync(hres, ws, 32, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  *payload_bytes = hres[0];
  const uint32_t* stats = reinterpret_cast<const uint32_t*>(reinterpret_cast<const uint8_t*>(hres) + 16);
  A.last_stats[0] = stats[0]; A.last_stats[1] = stats[1]; A.last_stats[2] = stats[2]; A.last_stats[3] = (long)hres[0];
  return 0;
}

// the blob's text header, right-aligned in its `reserve`-byte slot (leading blanks are what header::pack itself pads with)
int header_slot(const Pipeline& pl, const std::vector<uint64_t>& shape, uint64_t payload_bytes, size_t reserve, std::string* slot) {
  const std::string hdr = pack_header(pl.type_name(), pl.elem, shape, pl.canonical(), payload_bytes);
  if (hdr.size() > reserve) {
    std::fprintf(stderr, "[sqeazy_b200] header (%zu B) exceeds its slot (%zu B)\n", hdr.size(), reserve);
    return 1;
  }
  *slot = std::string(reserve - hdr.size(), ' ') + hdr;
  return 0;
}

// the quantiser's LUTs for the histogram of a whole stack: the encode LUT into enc (65536 codes); the decode LUT travels in the
// header (quantiser_scheme_impl.hpp:200-204)
void quantiser_luts(Pipeline& pl, const uint32_t* hist, uint8_t* enc) {
  uint16_t dec[256];
  quantiser_luts_from_histogram(hist, enc, dec);
  pl.sink.kv["decode_lut_string"] = std::string(kVerbatimOpen) + base64_encode(dec, sizeof(dec)) + kVerbatimClose;
}

// Where a stage of a device call writes: the last stage that moves data writes the destination, every other one the arena slot
// (kSlotA / kSlotB) that does not hold its input (kSlotA when the input is in neither).
struct Scratch {
  Arena& A;
  uint64_t bytes;
  void* slot[2] = {nullptr, nullptr};
  int next(const void* in, void** out) {
    const int k = in == slot[0] ? 1 : 0;
    if (!slot[k] && A.get(k ? kSlotB : kSlotA, bytes, &slot[k])) return 1;
    *out = slot[k];
    return 0;
  }
};

int encode_device_impl(Arena& A, const Pipeline& pl_in, const void* d_src, const std::vector<uint64_t>& shape, uint8_t* d_dst,
                       uint64_t dst_cap, uint64_t* dst_bytes, const uint32_t* d_global_hist, cudaStream_t st) {
  Pipeline pl = pl_in;
  const uint64_t N = shape_product(shape);
  const uint64_t raw_bytes = (uint64_t)pl.elem * N;
  const size_t reserve = header_reserve_bytes(pl, shape);
  uint8_t* payload = d_dst + reserve;
  if (dst_cap < reserve) return 1;
  const uint64_t payload_cap = dst_cap - reserve;

  Scratch scratch{A, raw_bytes};
  const void* cur = d_src;
  for (size_t i = 0; i < pl.head.size(); ++i) {
    const Stage& s = pl.head[i];
    ScopedStageTimer tm(kTFilterSwap, st);
    int t = s.threshold;
    if (s.kind == StageKind::RmEstBkrd) {
      if (shape.size() != 3) {
        std::fprintf(stderr, "[sqeazy_b200] rmestbkrd needs a rank-3 shape\n");
        return 1;
      }
      float sup[4];
      if (estimate_background(A, static_cast<const uint16_t*>(cur), shape[0], shape[1], shape[2], -1, sup, &t, st)) return 1;
    }
    void* out = nullptr;
    if (scratch.next(cur, &out)) return 1;
    if (s.kind == StageKind::RemoveBackground || s.kind == StageKind::RmEstBkrd) {
      if (i + 1 < pl.head.size() && pl.head[i + 1].kind == StageKind::Bitswap && t > 0)   // filter fused into the transpose
        CKK(k_bitswap_encode(pl.elem, pl.head[++i].w, cur, out, N, t, st));
      else
        CKK(k_remove_background(pl.elem, cur, out, N, t, st));
    } else if (s.kind == StageKind::Bitshuffle) {
      if (k_bitshuffle_encode(pl.elem, cur, out, N, s.block_size, st)) {
        std::fprintf(stderr, "[sqeazy_b200] bitshuffle failed (block_size=%u must be a multiple of 8)\n", s.block_size);
        return 1;
      }
    } else if (s.kind == StageKind::Diff) {
      if (shape.size() != 3 || k_diff_encode(pl.elem, cur, out, shape[0], shape[1], shape[2], st)) {
        // diff_scheme_impl.hpp:84-87 needs rank 3; shapes on which the reference's own loops leave the plane are refused
        std::fprintf(stderr, "[sqeazy_b200] diff3x3x1: shape not supported\n");
        return 1;
      }
    } else {
      CKK(k_bitswap_encode(pl.elem, s.w, cur, out, N, 0, st));
    }
    cur = out;
  }

  // the sink's bytes: the head's output, or the quantiser's codes
  const void* bytes = cur;
  uint64_t nbytes = raw_bytes;
  const bool lz4 = pl.has_sink && (pl.sink.kind == StageKind::Lz4 || pl.has_tail);
  if (pl.has_sink && pl.sink.kind == StageKind::Quantiser) {
    if (pl.elem != 2) return 1;   // (the planner never builds it for uint8)
    SmallSlot small;
    if (small_slot(A, &small)) return 1;
    std::vector<uint32_t> h(65536);
    if (N > 0 || d_global_hist) {
      if (d_global_hist) {
        CK(cudaMemcpyAsync(h.data(), d_global_hist, 65536 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
      } else {
        CK(cudaMemsetAsync(small.hist, 0, 65536 * sizeof(uint32_t), st));
        ScopedStageTimer tm(kTHist, st);
        CKK(k_histogram_u16(static_cast<const uint16_t*>(cur), N, small.hist, st));
        tm.stop();
        CK(cudaMemcpyAsync(h.data(), small.hist, 65536 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
      }
      CK(cudaStreamSynchronize(st));
    }
    std::vector<uint8_t> enc(65536);
    quantiser_luts(pl, h.data(), enc.data());
    CK(cudaMemcpyAsync(small.enc_lut, enc.data(), 65536, cudaMemcpyHostToDevice, st));
    void* codes = payload;   // without an LZ4 tail the codes are the payload
    if (lz4 && scratch.next(cur, &codes)) return 1;
    if (!lz4 && payload_cap < N) return 1;
    {
      ScopedStageTimer tm(kTLutApply, st);
      CKK(k_lut_apply(static_cast<const uint16_t*>(cur), static_cast<uint8_t*>(codes), N, small.enc_lut, st));
    }
    if (!lz4) CK(cudaStreamSynchronize(st));  // enc (host vector) must outlive the H2D copy; the LZ4 encode waits for it below
    bytes = codes;
    nbytes = N;
  }

  // then LZ4 them (an `lz4` sink or an `lz4` tail), or copy them into the payload
  uint64_t payload_bytes = nbytes;
  if (lz4) {
    if (payload_cap < lz4_payload_bound(nbytes)) {
      std::fprintf(stderr, "[sqeazy_b200] destination too small for lz4 (%llu < %llu)\n", (unsigned long long)payload_cap,
                   (unsigned long long)lz4_payload_bound(nbytes));
      return 1;
    }
    void* ws = nullptr;
    if (A.get(kSlotWs, k_lz4_encode_workspace_bytes(nbytes), &ws)) return 1;
    {
      ScopedStageTimer tm(kTLz4Enc, st);
      CKK(k_lz4_encode(static_cast<const uint8_t*>(bytes), nbytes, payload, ws, lz4_pitch_hint(pl, shape), st));
    }
    if (lz4_encode_result(A, ws, st, &payload_bytes)) return 1;
  } else if (bytes != payload) {
    if (payload_cap < nbytes) return 1;
    if (nbytes) CK(cudaMemcpyAsync(payload, bytes, nbytes, cudaMemcpyDeviceToDevice, st));
  }

  std::string slot;
  if (header_slot(pl, shape, payload_bytes, reserve, &slot)) return 1;
  CK(cudaMemcpyAsync(d_dst, slot.data(), slot.size(), cudaMemcpyHostToDevice, st));
  CK(cudaStreamSynchronize(st));
  *dst_bytes = reserve + payload_bytes;
  return 0;
}

// ---- shared by the streamed host paths (host_encode_streamed below, the host sink of decode_device_impl) ----
constexpr uint64_t kStreamSlabBytes = uint64_t(256) << 20;
constexpr uint64_t kStreamMinBytes = uint64_t(512) << 20;
constexpr uint64_t kStreamGrainVoxels = 131072;   // a 16 KiB block of a 1-bit plane covers 131072 voxels (8192 * P for wider atoms)

// blocks [k0, k1) of an LZ4 stream
struct BlockRun {
  uint64_t k0, k1;
};

// The LZ4 stream of n voxels that the host entry points encode and decode slab by slab: `sets` streams of equal length one
// after the other, in 16 KiB blocks. Voxels [first, first + count) make up blocks [block(first), block(first + count)) of every
// set when first and count are multiples of the block's voxels in one set.
struct StreamGeom {
  uint64_t n;              // voxels
  uint32_t sets;           // the 16/w bit planes of a uint16 bitswapW, or the one stream of 8-bit quantiser codes
  uint32_t voxel_bytes;    // LZ4 bytes per voxel, over all sets
  static StreamGeom planes(uint64_t n, int w) { return {n, (uint32_t)(16 / w), 2}; }
  static StreamGeom codes(uint64_t n) { return {n, 1, 1}; }
  StreamGeom of(uint64_t voxels) const { return {voxels, sets, voxel_bytes}; }   // the same kind of stream over other voxels
  uint64_t bytes() const { return voxel_bytes * n; }
  uint64_t blocks() const { return bytes() / kLz4BlockBytes; }
  uint32_t block(uint64_t v) const { return (uint32_t)(voxel_bytes * v / sets / kLz4BlockBytes); }
  uint32_t set_blocks() const { return block(n); }   // blocks per set: the set stride
  // the blocks of one set that hold a voxel of the runs R (kernels.h): sorted disjoint block runs, the same in every set (a
  // sub-volume decode needs these blocks of every set and no others). While a run's step is at most the voxels of one block of
  // one set, every block from its first voxel's to its last voxel's holds one of its voxels; beyond that each voxel has a block
  // of its own, and the blocks between them hold nothing the run selects.
  std::vector<BlockRun> blocks_of(const RoiRuns& R) const {
    std::vector<BlockRun> out;
    const auto add = [&](uint64_t k0, uint64_t k1) {
      if (!out.empty() && k0 <= out.back().k1) out.back().k1 = std::max(out.back().k1, k1);
      else out.push_back({k0, k1});
    };
    const uint64_t block_voxels = (uint64_t)kLz4BlockBytes * sets / voxel_bytes;
    for (uint64_t r = 0; r < R.rows; ++r) {
      const uint64_t v0 = R.start(r);
      if (R.step <= block_voxels) {
        add(block(v0), (uint64_t)block(v0 + (R.len - 1) * R.step) + 1);
        continue;
      }
      for (uint64_t j = 0; j < R.len; ++j) {
        const uint64_t k = block(v0 + j * R.step);
        add(k, k + 1);
      }
    }
    return out;
  }
};

// The kinds of blob whose LZ4 blocks each hold a known piece of the stack, on uint16 (the decode of a piece of the stack needs
// just its blocks):
//   planes: `[filters ->] bitswapW -> lz4`, N a multiple of the 8192 * 16/W voxels that fill a 16 KiB block of every plane; the
//           filters decode as identity, so any number of them may stand anywhere in the head;
//   codes:  `quantiser -> lz4`, N a multiple of 16384.
// *w = W for planes, 0 for codes. Whether the payload is one frame of this library is for the caller to find out.
bool indexed_stream(const Pipeline& pl, uint64_t N, StreamGeom* geo, int* w) {
  if (pl.elem != 2 || !pl.has_sink) return false;
  if (pl.sink.kind == StageKind::Lz4 && !pl.has_tail) {
    int nswaps = 0;
    for (const Stage& s : pl.head) {
      if (s.kind == StageKind::Bitswap) { *w = s.w; nswaps++; }
      else if (s.kind == StageKind::Bitshuffle || s.kind == StageKind::Diff) return false;
    }
    if (nswaps != 1 || N % (8192ull * (16 / *w))) return false;
    *geo = StreamGeom::planes(N, *w);
    return true;
  }
  if (pl.sink.kind != StageKind::Quantiser || !pl.has_tail || !pl.head.empty() || !pl.sink.has_decode_lut || N % kLz4BlockBytes)
    return false;
  *w = 0;
  *geo = StreamGeom::codes(N);
  return true;
}

int copy_stream(cudaStream_t* cs) {   // of the current device; its lock is held
  int dev = 0;
  CK(cudaGetDevice(&dev));
  if (dev >= kMaxDevices) return 1;
  if (!g_dev[dev].copy_stream) CK(cudaStreamCreateWithFlags(&g_dev[dev].copy_stream, cudaStreamNonBlocking));
  *cs = g_dev[dev].copy_stream;
  return 0;
}

struct EventList {
  std::vector<cudaEvent_t> ev;
  ~EventList() { for (cudaEvent_t e : ev) cudaEventDestroy(e); }
  int next(cudaEvent_t* out) {
    cudaEvent_t e = nullptr;
    CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    ev.push_back(e);
    *out = e;
    return 0;
  }
};

// where decode_device_impl may deliver the volume slab by slab while the last inverse transpose is still running
struct HostSink {
  char* dst;
  int nthreads;
  bool done = false;
};

// ---- decode ----
// The transpose back of a uint16 bitswapW that directly follows the LZ4 stage can run inside the LZ4 block decoder
// (k_lz4_decode_fused). It pays from stacks of kFuseMinBytes on: there the 1.4 ms-per-4-GiB launch it replaces ran alone on the
// stream; below, the transposes the decoder's warps do at L2 latency and the tail of the last ranges cost more than that launch
// (measured, profiles/README.md round 3). SQYB_FUSE_TRANSPOSE=0 builds the two-launch route only (A/B: tools/ab_fused.py).
#ifndef SQYB_FUSE_TRANSPOSE
#define SQYB_FUSE_TRANSPOSE 1
#endif
#ifndef SQYB_FUSE_MIN_BYTES
#define SQYB_FUSE_MIN_BYTES (uint64_t(1) << 30)
#endif
constexpr uint64_t kFuseMinBytes = SQYB_FUSE_MIN_BYTES;

// where the fused decoder puts the voxels of the bit planes it decodes (lz4_decode_checked)
struct FusedTarget {
  int w;            // bits per plane of the bitswap
  uint16_t* vox;    // 32-byte aligned, dst_bytes / 2 voxels
};

// `fuse`: when the stream turns out to be one frame of this library whose 16 KiB blocks hold exactly the dst_bytes plane bytes,
// the planes are also transposed back into fuse->vox and *fused is set. The block table is built once either way: any other
// stream goes on to the block decoders over that table.
int lz4_decode_checked(Arena& A, const uint8_t* src, uint64_t nbytes, uint8_t* dst, uint64_t dst_bytes, uint64_t* decoded,
                       cudaStream_t st, const FusedTarget* fuse = nullptr, bool* fused = nullptr) {
  void* ws = nullptr;
  if (A.get(kSlotWs, k_lz4_decode_workspace_bytes(dst_bytes), &ws)) return 1;
  for (int attempt = 0; attempt < 2; ++attempt) {
    bool go_fused = false;
    {
      ScopedStageTimer tm(kTLz4Dec, st);
      CKK(k_lz4_decode_tables(src, nbytes, dst_bytes, ws, attempt, 1, st));
      if (fuse && attempt == 0 && k_lz4_decode_own_frame(ws, dst_bytes, &go_fused, st)) return 1;
      if (go_fused) CKK(k_lz4_decode_fused(src, nbytes, dst, dst_bytes, ws, fuse->w, fuse->vox, st));
      else CKK(k_lz4_decode_run(src, nbytes, dst, dst_bytes, ws, 0, 0, 0, 0, 0, st));
    }
    uint32_t err = 0, deferred = 0;
    uint64_t total = 0;
    if (k_lz4_decode_status(ws, &err, &total, &deferred, st)) return 1;
    if (go_fused) {
      // the index promised every block in full: a frame of this library that decodes to less is broken
      if (err || total != dst_bytes) {
        std::fprintf(stderr, "[sqeazy_b200] lz4 decode failed (code %u)\n", err ? err : 5u);
        return 1;
      }
      if (decoded) *decoded = total;
      *fused = true;
      return 0;
    }
    if (err == 0 && deferred) {
      // block-linked frames (reference serial mode / sqy CLI default): deferred cross-block references, lz4_decode.cu
      void* origins = nullptr;
      if (A.get(kSlotOrigins, k_lz4_decode_linked_workspace_bytes(dst_bytes), &origins)) return 1;
      {
        ScopedStageTimer tm(kTLz4Dec, st);
        CKK(k_lz4_decode_linked(src, nbytes, dst, dst_bytes, ws, origins, st));
      }
      uint32_t none = 0;
      if (k_lz4_decode_status(ws, &err, &total, &none, st)) return 1;
    }
    if (err == 0) {
      if (decoded) *decoded = total;
      return 0;
    }
    // 4 = bad block, 5 = size mismatch: foreign frames with short inner blocks -> measure every block and retry
    if (!(attempt == 0 && (err == 4 || err == 5))) {
      std::fprintf(stderr, "[sqeazy_b200] lz4 decode failed (code %u)\n", err);
      return 1;
    }
  }
  return 1;
}

// Runs make(first, count) on `st` for every slab of `slab` voxels of the N-voxel volume at d_vox; each slab leaves for the host on
// the device's copy stream as soon as the kernels that made it are done. Returns make's code, or 0 when every slab is there.
template <class Make>
int ship_slabs(HostSink* host, const uint16_t* d_vox, uint64_t N, uint64_t slab, cudaStream_t st, Make&& make) {
  cudaStream_t cs = nullptr;
  if (copy_stream(&cs)) return 1;
  EventList events;
  for (uint64_t first = 0; first < N; first += slab) {
    if (int rc = make(first, std::min(slab, N - first))) return rc;
    cudaEvent_t e = nullptr;
    if (events.next(&e)) return 1;
    CK(cudaEventRecord(e, st));
  }
  size_t i = 0;
  for (uint64_t first = 0; first < N; first += slab, ++i) {
    CK(cudaStreamWaitEvent(cs, events.ev[i], 0));
    CK((cudaError_t)staged_d2h(host->dst + 2 * first, d_vox + first, 2 * std::min(slab, N - first), host->nthreads, cs));
  }
  CK(cudaStreamSynchronize(cs));
  return 0;
}

// The mirror image of ship_slabs: sends the n voxels at h_src to d_vox slab by slab on the device's copy stream, and `st` runs
// make(first, count) on a slab as soon as it has arrived. ahead() runs once, when the first slab's copy has been issued and
// before `st` waits for it: the bus does not wait for what it puts on `st`, and that work does not wait for the bus.
template <class Ahead, class Make>
int take_slabs(const char* h_src, uint16_t* d_vox, uint64_t n, uint64_t slab, int nthreads, cudaStream_t st, Ahead&& ahead, Make&& make) {
  cudaStream_t cs = nullptr;
  if (copy_stream(&cs)) return 1;
  EventList events;
  for (uint64_t first = 0; first < n; first += slab) {
    const uint64_t count = std::min(slab, n - first);
    CK((cudaError_t)staged_h2d(d_vox + first, h_src + 2 * first, 2 * count, nthreads, cs));
    cudaEvent_t arrived = nullptr;
    if (events.next(&arrived)) return 1;
    CK(cudaEventRecord(arrived, cs));
    if (first == 0)
      if (int rc = ahead()) return rc;
    CK(cudaStreamWaitEvent(st, arrived, 0));
    if (int rc = make(first, count)) return rc;
  }
  return 0;
}

// LZ4 of the bit planes (bitswap w) of the geo.n uint16 voxels at h_src. The stack arrives in d_in slab by slab; each slab is
// filtered with the threshold and transposed into its place in the plane-major d_planes, and the blocks it completes in every
// plane are compressed into d_lz4 while the next slab is on the bus. threshold(&t) gives the threshold once the first slab is
// on its way (take_slabs' ahead).
template <class Threshold>
int encode_planes_slabs(const StreamGeom& geo, int w, Threshold&& threshold, uint32_t pitch_hint, uint64_t slab, const char* h_src,
                        uint16_t* d_in, uint16_t* d_planes, uint8_t* d_lz4, void* ws, int nthreads, cudaStream_t st) {
  const uint8_t* planes = reinterpret_cast<const uint8_t*>(d_planes);
  int thr = 0;
  CKK(k_lz4_encode_begin(geo.bytes(), d_lz4, ws, st));
  const int rc = take_slabs(h_src, d_in, geo.n, slab, nthreads, st, [&] { return threshold(&thr); },
                            [&](uint64_t first, uint64_t count) -> int {
                              CKK(k_bitswap_encode_range(w, d_in, d_planes, geo.n, first, count, thr, st));
                              CKK(k_lz4_encode_blocks(planes, geo.bytes(), d_lz4, ws, geo.block(first), geo.block(count), geo.sets,
                                                      geo.set_blocks(), pitch_hint, st));
                              return 0;
                            });
  if (rc) return rc;
  CKK(k_lz4_encode_end(planes, geo.bytes(), d_lz4, ws, st));
  return 0;
}

// Host decode of a blob of this library, >= min_bytes, of one of two kinds:
//   planes: `[filters ->] bitswapW -> lz4`. A slab's LZ4 blocks are those of all P = 16/W bit planes that make up its voxels (one
//           block-set launch of P sets), transposed back by k_bitswap_decode_range. The filters decode as identity, so any
//           number of them may stand anywhere in the head: wider on purpose than what the streamed encoders write (shard_kind).
//   codes:  `quantiser -> lz4`. A slab's LZ4 blocks are one run of the code stream, turned into voxels by k_lut_decode.
// Every slab leaves for the host while the next one is decoded; only the first slab's kernels run in front of the bus. Returns -1
// when the blob is not of these kinds (the caller takes the general route), 0 on success, an error code otherwise.
int decode_streamed(Arena& A, const Pipeline& pl, const uint8_t* d_payload, uint64_t payload_bytes, uint16_t* d_dst, uint64_t N,
                    cudaStream_t st, HostSink* host, uint64_t slab_voxels = kStreamSlabBytes / 2, uint64_t min_bytes = kStreamMinBytes) {
  if (g_timing.load() || 2 * N < min_bytes) return -1;
  StreamGeom geo{};
  int w = 0;
  if (!indexed_stream(pl, N, &geo, &w)) return -1;
  const bool planes = w != 0;
  if (planes && N % kStreamGrainVoxels) return -1;
  void *ws = nullptr, *dec_v = nullptr;
  if (A.get(kSlotWs, k_lz4_decode_workspace_bytes(geo.bytes()), &ws) || A.get(kSlotA, geo.bytes(), &dec_v)) return 1;
  uint8_t* dec = static_cast<uint8_t*>(dec_v);
  SmallSlot small{};
  if (planes) {
    if (((((uintptr_t)dec) | ((uintptr_t)d_dst)) & 31) != 0) return -1;
  } else {
    if (small_slot(A, &small)) return 1;
    CK(cudaMemcpyAsync(small.dec_lut, pl.sink.decode_lut, 512, cudaMemcpyHostToDevice, st));
  }
  CKK(k_lz4_decode_tables(d_payload, payload_bytes, geo.bytes(), ws, 0, 0, st));
  bool own = false;
  if (k_lz4_decode_own_frame(ws, geo.bytes(), &own, st)) return 1;
  if (!own) return -1;
  uint64_t slab = slab_voxels;
  while ((N + slab - 1) / slab > 32) slab *= 2;   // one work counter per block-set launch, 32 of them
  uint32_t slot = 0;
  const int rc = ship_slabs(host, d_dst, N, slab, st, [&](uint64_t first, uint64_t count) -> int {
    CKK(k_lz4_decode_run(d_payload, payload_bytes, dec, geo.bytes(), ws, geo.block(first), geo.block(count), geo.sets,
                         geo.set_blocks(), slot++, st));
    if (planes) return k_bitswap_decode_range(w, reinterpret_cast<const uint16_t*>(dec), d_dst, N, first, count, st) ? 101 : 0;
    CKK(k_lut_decode(dec + first, d_dst + first, count, small.dec_lut, st));
    return 0;
  });
  if (rc) return rc;
  uint32_t err = 0, none = 0;
  uint64_t total = 0;
  if (k_lz4_decode_status(ws, &err, &total, &none, st)) return 1;
  if (err || total != geo.bytes()) {
    std::fprintf(stderr, "[sqeazy_b200] lz4 decode failed (code %u)\n", err);
    return planes ? 11 : 101;   // what the general route returns for a broken `lz4` sink / `lz4` tail
  }
  host->done = true;
  return 0;
}

int decode_device_impl(Arena& A, const Header& hdr, const Pipeline& pl, const uint8_t* d_payload, uint64_t payload_bytes,
                       void* d_dst, uint64_t dst_cap, cudaStream_t st, HostSink* host = nullptr) {
  const uint64_t N = shape_product(hdr.shape);
  const uint64_t raw_bytes = (uint64_t)pl.elem * N;
  if (dst_cap < raw_bytes) return 1;
  if (N == 0) return 0;
  if (host) {
    const int rc = decode_streamed(A, pl, d_payload, payload_bytes, static_cast<uint16_t*>(d_dst), N, st, host);
    if (rc >= 0) return rc;
  }

  // the head stages that move data, decoded from the last one (`top`) down; the background filters decode as identity
  auto moves = [](const Stage& s) { return s.kind != StageKind::RemoveBackground && s.kind != StageKind::RmEstBkrd; };
  size_t left = 0;   // data-moving stages still to decode
  const Stage* top = nullptr;
  for (const Stage& s : pl.head) {
    if (!moves(s)) continue;
    if (s.kind == StageKind::Diff && (hdr.shape.size() != 3 || !diff_shape_supported(hdr.shape[0], hdr.shape[1], hdr.shape[2], pl.elem)))
      return 100 + 1;
    ++left;
    top = &s;
  }
  Scratch scratch{A, raw_bytes};
  // the output of a step that reads `in` and behind which `following` data-moving stages still decode
  auto out_for = [&](const void* in, size_t following, void** out) -> int {
    if (following == 0) {
      *out = d_dst;
      return 0;
    }
    return scratch.next(in, out);
  };

  // The transpose back of a uint16 bitswapW that directly follows the LZ4 stage may run inside the LZ4 block decoder when the
  // 16 KiB blocks hold whole groups of the P = 16/W planes (N a multiple of 8192P) and the stack is large enough to gain from it
  // (kFuseMinBytes). A host call that ships the volume slab by slab behind the last transpose keeps that.
  const bool try_fuse = SQYB_FUSE_TRANSPOSE && pl.elem == 2 && raw_bytes >= kFuseMinBytes && pl.has_sink &&
                        pl.sink.kind == StageKind::Lz4 && top && top->kind == StageKind::Bitswap &&
                        N % (8192ull * (16 / top->w)) == 0 && !(host && left == 1 && raw_bytes >= kStreamMinBytes);

  const void* cur = d_payload;   // the head's input
  size_t end = pl.head.size();   // the head decodes from pl.head[end - 1] down
  if (pl.has_sink) {
    const bool quantiser = pl.sink.kind == StageKind::Quantiser;
    void* out = nullptr;         // the sink's output
    if (out_for(d_payload, left, &out)) return 1;
    if (quantiser && pl.elem != 2) return 11;
    if (quantiser && !pl.sink.has_decode_lut) {
      std::fprintf(stderr, "[sqeazy_b200] quantiser stage without decode_lut_string in the header\n");
      return 11;
    }
    // LZ4 (an `lz4` sink or an `lz4` tail), or the payload as it is
    const uint64_t nbytes = quantiser ? N : raw_bytes;
    const void* bytes = d_payload;
    if (pl.sink.kind == StageKind::Lz4 || pl.has_tail) {
      void* lz4_out = out;
      if (quantiser && scratch.next(out, &lz4_out)) return 1;   // codes in the scratch slot that is not the LUT's output
      void* vox = nullptr;       // where the fused transpose puts the voxels
      if (try_fuse && out_for(out, left - 1, &vox)) return 1;
      FusedTarget target{try_fuse ? top->w : 0, static_cast<uint16_t*>(vox)};
      bool fused = false;
      if (lz4_decode_checked(A, d_payload, payload_bytes, static_cast<uint8_t*>(lz4_out), nbytes, nullptr, st,
                             try_fuse && (((uintptr_t)target.vox) & 31) == 0 ? &target : nullptr, &fused))
        return pl.has_tail ? 101 : 11;
      bytes = lz4_out;
      if (fused) {
        out = target.vox;
        bytes = out;
        end = size_t(top - pl.head.data());
        --left;
      }
    } else if (payload_bytes < nbytes) {
      return 11;
    }
    // then the quantiser's LUT, or the bytes as the head's input
    if (quantiser) {
      SmallSlot small;
      if (small_slot(A, &small)) return 1;
      CK(cudaMemcpyAsync(small.dec_lut, pl.sink.decode_lut, 512, cudaMemcpyHostToDevice, st));
      {
        ScopedStageTimer tm(kTLutDec, st);
        CKK(k_lut_decode(static_cast<const uint8_t*>(bytes), static_cast<uint16_t*>(out), N, small.dec_lut, st));
      }
      CK(cudaStreamSynchronize(st));
    } else if (bytes != out) {
      CK(cudaMemcpyAsync(out, bytes, raw_bytes, cudaMemcpyDeviceToDevice, st));
    }
    cur = out;
  } else {
    if (payload_bytes < raw_bytes) return 1;
    if (left == 0) {
      CK(cudaMemcpyAsync(d_dst, d_payload, raw_bytes, cudaMemcpyDeviceToDevice, st));
      cur = d_dst;
    }
  }

  for (size_t i = end; i-- > 0;) {
    const Stage& s = pl.head[i];
    if (!moves(s)) continue;
    void* out = nullptr;
    if (out_for(cur, --left, &out)) return 1;
    if (s.kind == StageKind::Diff) {
      if (k_diff_decode(pl.elem, cur, out, hdr.shape[0], hdr.shape[1], hdr.shape[2], st)) return 100 + 1;
    } else if (s.kind == StageKind::Bitshuffle) {
      if (k_bitshuffle_decode(pl.elem, cur, out, N, s.block_size, st)) return 100 + 1;
    } else if (left == 0 && host && pl.elem == 2 && raw_bytes >= kStreamMinBytes && N % 128 == 0 && !g_timing.load() &&
               ((((uintptr_t)cur) | ((uintptr_t)out)) & 31) == 0) {
      // last stage of a host call: transpose back slab by slab, every slab leaves for the host as soon as it is done
      const uint16_t* in16 = static_cast<const uint16_t*>(cur);
      uint16_t* out16 = static_cast<uint16_t*>(out);
      const int rc = ship_slabs(host, out16, N, kStreamSlabBytes / 2, st, [&](uint64_t first, uint64_t count) -> int {
        return k_bitswap_decode_range(s.w, in16, out16, N, first, count, st) ? 100 + 1 : 0;
      });
      if (rc) return rc;
      host->done = true;
    } else {
      ScopedStageTimer tm(kTSwapDec, st);
      if (k_bitswap_decode(pl.elem, s.w, cur, out, N, st)) return 100 + 1;
    }
    cur = out;
  }
  CK(cudaStreamSynchronize(st));
  return 0;
}

int parse_blob_header_device(const uint8_t* d_blob, uint64_t blob_bytes, Header& hdr, cudaStream_t st) {
  size_t peek = 16384;
  for (int attempt = 0; attempt < 2; ++attempt) {
    const size_t n = blob_bytes < peek ? (size_t)blob_bytes : peek;
    std::vector<char> h(n);
    CK(cudaMemcpyAsync(h.data(), d_blob, n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    hdr = unpack_header(h.data(), n);
    if (hdr.valid || n == blob_bytes) break;
    peek = 1 << 20;
  }
  return hdr.valid ? 0 : 1;
}

std::vector<uint64_t> to_shape(const long* shape, unsigned n) {
  std::vector<uint64_t> v;
  for (unsigned i = 0; i < n; ++i) v.push_back(shape[i] < 0 ? 0 : (uint64_t)shape[i]);
  return v;
}

// what the device entry points do around decode_device_impl: the blob's header, its element size and its pipeline
int decode_device_blob(Arena& A, int elem, const void* d_blob, long blob_bytes, void* d_dst, long dst_capacity, cudaStream_t st) {
  if (!d_blob || blob_bytes <= 0 || !d_dst || dst_capacity < 0) return 1;
  const uint8_t* blob = static_cast<const uint8_t*>(d_blob);
  Header hdr;
  if (parse_blob_header_device(blob, (uint64_t)blob_bytes, hdr, st)) return 1;
  if (sizeof_typename(hdr.raw_type) != (unsigned)elem) return 1;
  Pipeline pl;
  if (!(elem == 1 ? build_pipeline_u8(hdr.pipeline, pl) : build_pipeline_u16(hdr.pipeline, pl)) || pl.empty()) {
    std::fprintf(stderr, "[sqeazy]\t%s cannot be build with this version of sqeazy\n", hdr.pipeline.c_str());
    return 1;
  }
  return decode_device_impl(A, hdr, pl, blob + hdr.size, (uint64_t)blob_bytes - hdr.size, d_dst, (uint64_t)dst_capacity, st);
}

// ... and around encode_device_impl: the pipeline for the element size, the blob's size
int encode_device_blob(Arena& A, int elem, const char* pipeline, const void* d_src, const std::vector<uint64_t>& shape, void* d_dst,
                       long dst_capacity, long* dst_bytes, const void* d_global_hist, cudaStream_t st) {
  if (!pipeline || !d_dst || !dst_bytes || dst_capacity < 0) return 1;
  Pipeline pl;
  if (!(elem == 1 ? build_pipeline_u8(pipeline, pl) : build_pipeline_u16(pipeline, pl)) || pl.empty()) return 1;
  uint64_t out = 0;
  const int rc = encode_device_impl(A, pl, d_src, shape, static_cast<uint8_t*>(d_dst), (uint64_t)dst_capacity, &out,
                                    static_cast<const uint32_t*>(d_global_hist), st);
  if (rc == 0) *dst_bytes = (long)out;
  return rc;
}

// the bitshuffle entry points: one stage, synchronous
int bitshuffle_device(bool encode, int elem, const void* d_src, void* d_dst, long n, long block_size, void* stream) {
  if (n < 0 || block_size < 0 || block_size > (1l << 30)) return 1;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if ((encode ? k_bitshuffle_encode : k_bitshuffle_decode)(elem, d_src, d_dst, (uint64_t)n, (uint32_t)block_size, st)) return 1;
  return cudaStreamSynchronize(st) == cudaSuccess ? 0 : 1;
}

#include "sharded.inl"

// ---- sub-volume decode (sqyx_decode_roi_*, sqyx_decode_slice_*) ----
// A strided slice of the stack (a box when every step is 1): its runs (kernels.h: RoiRuns), its voxels, whether it selects
// every voxel of the stack.
struct Roi {
  RoiRuns runs{};
  uint64_t voxels = 0;
  bool whole = true;
};

// sel = ndims tuples of `width` longs, dimension 0 first: {lo, hi} (width 2: a box, step 1) or {lo, hi, step} (width 3), half-open,
// step >= 1; the slice takes ceil((hi - lo) / step) voxels of dimension k. 3 when it is malformed or leaves the shape.
int roi_of(const std::vector<uint64_t>& shape, const long* sel, unsigned width, unsigned ndims, Roi* out) {
  if (!sel || ndims == 0 || ndims != shape.size()) return 3;
  Roi roi;
  roi.voxels = 1;
  std::vector<uint64_t> stride(ndims, 1), lo(ndims), extent(ndims), step(ndims);
  for (unsigned k = ndims; k-- > 0;) {
    const long l = sel[width * k], h = sel[width * k + 1], s = width == 3 ? sel[width * k + 2] : 1;
    if (l < 0 || l > h || (uint64_t)h > shape[k] || s < 1) return 3;
    lo[k] = (uint64_t)l, step[k] = (uint64_t)s, extent[k] = ((uint64_t)(h - l) + step[k] - 1) / step[k];
    roi.voxels *= extent[k];
    roi.whole = roi.whole && l == 0 && extent[k] == shape[k];
    if (k + 1 < ndims) stride[k] = stride[k + 1] * shape[k + 1];
  }
  RoiRuns& R = roi.runs;
  if (roi.voxels) {
    // the trailing dimensions that the slice spans whole with step 1 go into the runs: one run per index tuple of the dimensions
    // in front of j. A step in j is the runs' inner step when j is the last dimension; otherwise j leads too, with its step in
    // its stride, and a run is the stride[j] voxels of the dimensions behind it.
    unsigned j = ndims - 1;
    while (j > 0 && lo[j] == 0 && extent[j] == shape[j]) --j;
    const bool inner = step[j] > 1 && extent[j] > 1;
    const bool lead_j = inner && j + 1 < ndims;
    R.len = lead_j ? stride[j] : inner ? extent[j] : extent[j] * stride[j];
    R.step = inner && !lead_j ? step[j] : 1;
    R.base = lo[j] * stride[j];
    R.rows = 1;
    for (unsigned k = 0; k < j + (lead_j ? 1 : 0); ++k) {
      R.base += k < j ? lo[k] * stride[k] : 0;
      if (extent[k] == 1) continue;
      if (R.nlead == kRoiMaxLead) return 1;
      R.extent[R.nlead] = extent[k];
      R.stride[R.nlead++] = stride[k] * step[k];
      R.rows *= extent[k];
    }
  }
  *out = roi;
  return 0;
}

// The selections of a call: nsel of them one after the other, ndims tuples of `width` longs each (roi_of), and their voxels in
// all. 3 when any is malformed, or nsel is 0 or above kMaxSelections.
constexpr unsigned kMaxSelections = 65536;
int rois_of(const std::vector<uint64_t>& shape, const long* sels, unsigned width, unsigned ndims, unsigned nsel, std::vector<Roi>* out,
            uint64_t* voxels) {
  if (!sels || nsel == 0 || nsel > kMaxSelections) return 3;
  out->assign(nsel, Roi{});
  *voxels = 0;
  for (unsigned i = 0; i < nsel; ++i) {
    if (int rc = roi_of(shape, sels + (size_t)width * ndims * i, width, ndims, &(*out)[i])) return rc;
    *voxels += (*out)[i].voxels;
  }
  return 0;
}

// The blocks of an indexed stream (indexed_stream) that hold a voxel of any of the selections: `runs` of every set (the union of
// every selection's blocks, sorted and disjoint), nsel blocks per set. Each block is decoded once, into compact places, set after
// set: list[t] = the stream's block at compact place t, pos[k] = the place of block k within its set (~0: not needed).
struct RoiPlan {
  std::vector<BlockRun> runs;
  uint64_t nsel = 0;
  std::vector<uint32_t> list, pos;
};

RoiPlan roi_plan(const StreamGeom& geo, const std::vector<Roi>& rois) {
  RoiPlan P;
  std::vector<BlockRun> all;
  for (const Roi& roi : rois) {
    if (!roi.voxels) continue;
    const std::vector<BlockRun> b = geo.blocks_of(roi.runs);
    all.insert(all.end(), b.begin(), b.end());
  }
  std::sort(all.begin(), all.end(), [](const BlockRun& a, const BlockRun& b) { return a.k0 < b.k0; });
  for (const BlockRun& b : all) {
    if (!P.runs.empty() && b.k0 <= P.runs.back().k1) P.runs.back().k1 = std::max(P.runs.back().k1, b.k1);
    else P.runs.push_back(b);
  }
  P.pos.assign(geo.set_blocks(), ~0u);
  for (const BlockRun& b : P.runs)
    for (uint64_t k = b.k0; k < b.k1; ++k) P.pos[k] = (uint32_t)P.nsel++;
  P.list.reserve(geo.sets * P.nsel);
  for (uint32_t j = 0; j < geo.sets; ++j)
    for (const BlockRun& b : P.runs)
      for (uint64_t k = b.k0; k < b.k1; ++k) P.list.push_back((uint32_t)((uint64_t)j * geo.set_blocks() + k));
  return P;
}

// The gather's selections (kernels.h: RoiSelections) and its tables on the device, in the arena's kSlotRoi: for a batch (the
// sqyx_decode_slice_batch_* calls) the descriptors of its selections (kernels.h: roi_batch; `host` holds what that copy reads until
// the caller synchronises), then P's pos, then P's list when the caller decodes by list, one copy each. A single call takes no
// descriptor: its runs go to roi_gather_kernel by value, which tools/ab_roi.py measured faster than a batch of one
// (profiles/README.md). So a single crop (P = nullptr) copies nothing and takes no slot.
struct RoiTables {
  RoiSelections sels;
  const uint32_t *d_pos, *d_list;
};

int roi_tables(Arena& A, RoiSource source, const std::vector<Roi>& rois, bool batch, const RoiPlan* P, bool with_list,
               std::vector<RoiSel>& host, RoiTables* T, cudaStream_t st) {
  T->sels = RoiSelections{rois[0].runs, nullptr, {}};
  if (batch) {
    std::vector<RoiRuns> runs;
    runs.reserve(rois.size());
    for (const Roi& roi : rois) runs.push_back(roi.runs);
    host.resize(rois.size());
    T->sels.batch = roi_batch(source, runs.data(), runs.size(), host.data());
  }
  const size_t sel_bytes = batch ? sizeof(RoiSel) * rois.size() : 0, pos_bytes = P ? 4 * P->pos.size() : 0;
  const size_t list_bytes = P && with_list ? 4 * P->list.size() : 0;
  if (sel_bytes + pos_bytes + list_bytes == 0) return 0;
  void* p = nullptr;
  if (A.get(kSlotRoi, sel_bytes + pos_bytes + list_bytes, &p)) return 1;
  uint8_t* d = static_cast<uint8_t*>(p);
  if (batch) T->sels.d_sels = reinterpret_cast<const RoiSel*>(d);
  T->d_pos = reinterpret_cast<const uint32_t*>(d + sel_bytes);
  T->d_list = reinterpret_cast<const uint32_t*>(d + sel_bytes + pos_bytes);
  if (sel_bytes) CK(cudaMemcpyAsync(d, host.data(), sel_bytes, cudaMemcpyHostToDevice, st));
  if (pos_bytes) CK(cudaMemcpyAsync(d + sel_bytes, P->pos.data(), pos_bytes, cudaMemcpyHostToDevice, st));
  if (list_bytes) CK(cudaMemcpyAsync(d + sel_bytes + pos_bytes, P->list.data(), list_bytes, cudaMemcpyHostToDevice, st));
  return 0;
}

// the gather behind the indexed route, from the compact blocks of P (`ws`: the block decode's workspace), then the block decode's
// status: 11 (planes) / 101 (codes), what the whole-stack decode returns, when a block that a selection needs did not decode
int roi_finish(Arena& A, const Pipeline& pl, int w, const RoiPlan& P, const RoiTables& T, const uint8_t* compact, void* ws,
               uint16_t* d_dst, cudaStream_t st) {
  if (w) {
    CKK(k_roi_gather_planes(w, compact, T.d_pos, P.nsel, T.sels, d_dst, st));
  } else {
    SmallSlot small;
    if (small_slot(A, &small)) return 1;
    CK(cudaMemcpyAsync(small.dec_lut, pl.sink.decode_lut, 512, cudaMemcpyHostToDevice, st));
    CKK(k_roi_gather_codes(compact, T.d_pos, small.dec_lut, T.sels, d_dst, st));
  }
  uint32_t err = 0, none = 0;
  uint64_t total = 0;
  if (k_lz4_decode_status(ws, &err, &total, &none, st)) return 1;   // (synchronises: the host tables have been consumed)
  if (err || total != (uint64_t)P.list.size() * kLz4BlockBytes) {
    std::fprintf(stderr, "[sqeazy_b200] lz4 decode failed (code %u)\n", err ? err : 5u);
    return w ? 11 : 101;
  }
  return 0;
}

// the crop behind the decode-whole route: every selection out of the whole decoded stack `full` of N voxels
int roi_crop(Arena& A, const Pipeline& pl, const void* full, uint64_t N, const std::vector<Roi>& rois, bool batch,
             std::vector<RoiSel>& host, void* d_dst, cudaStream_t st) {
  RoiTables T{};
  if (roi_tables(A, kRoiVolume, rois, batch, nullptr, false, host, &T, st)) return 1;
  CKK(k_roi_crop(pl.elem, full, N, T.sels, d_dst, st));
  return 0;
}

// Selections of a blob in device memory (not all empty; not one selection of the whole stack) into d_dst, one after the other.
// Indexed route (info[0] = 1): the block table of the whole payload, one launch for the blocks that hold a selected voxel of any
// selection, each once, and the gather. Every other blob (info[0] = 2): decoded whole into the arena once, then cropped.
int roi_device(Arena& A, const Header& hdr, const Pipeline& pl, const uint8_t* d_payload, uint64_t payload_bytes,
               const std::vector<Roi>& rois, bool batch, void* d_dst, cudaStream_t st, long* info) {
  const uint64_t N = shape_product(hdr.shape);
  StreamGeom geo{};
  int w = 0;
  std::vector<RoiSel> host;   // what the descriptor copy reads
  RoiTables T{};
  if (indexed_stream(pl, N, &geo, &w)) {
    void* ws = nullptr;
    if (A.get(kSlotWs, k_lz4_decode_workspace_bytes(geo.bytes()), &ws)) return 1;
    CKK(k_lz4_decode_tables(d_payload, payload_bytes, geo.bytes(), ws, 0, 0, st));
    bool own = false;
    if (k_lz4_decode_own_frame(ws, geo.bytes(), &own, st)) return 1;
    if (own) {
      const RoiPlan P = roi_plan(geo, rois);
      void* compact = nullptr;
      if (A.get(kSlotA, P.list.size() * kLz4BlockBytes, &compact) ||
          roi_tables(A, w ? kRoiPlanes : kRoiCodes, rois, batch, &P, true, host, &T, st))
        return 1;
      info[0] = 1;
      CKK(k_lz4_decode_list(d_payload, payload_bytes, geo.bytes(), static_cast<uint8_t*>(compact), ws, T.d_list, (uint32_t)P.list.size(), st));
      if (int rc = roi_finish(A, pl, w, P, T, static_cast<const uint8_t*>(compact), ws, static_cast<uint16_t*>(d_dst), st))
        return rc;
      info[1] = (long)P.list.size();
      return 0;
    }
  }
  info[0] = 2;
  void* full = nullptr;
  if (A.get(kSlotOut, pl.elem * N, &full)) return 1;
  if (int rc = decode_device_impl(A, hdr, pl, d_payload, payload_bytes, full, pl.elem * N, st)) return rc;
  if (int rc = roi_crop(A, pl, full, N, rois, batch, host, d_dst, st)) return rc;
  CK(cudaStreamSynchronize(st));
  return 0;
}

// The same for a blob in host memory, into the host buffer dst (`voxels` in all). Indexed route: the blocks the selections need,
// each once, are cut out of the blob on the host into a frame of their own (index frame, their blocks, EndMark), which alone crosses
// the bus in one copy and is decoded whole on the device: its blocks land at the compact places of the device route. Otherwise the
// payload goes to the device as the whole-stack host decode sends it, once, is decoded whole and cropped. info[2] = the bytes sent
// to the device.
int roi_host(Arena& A, const Header& hdr, const Pipeline& pl, const char* src, uint64_t srclength, const std::vector<Roi>& rois,
             bool batch, uint64_t voxels, char* dst, int nthreads, long* info) {
  const uint64_t N = shape_product(hdr.shape), box_bytes = pl.elem * voxels;
  const uint8_t* payload = reinterpret_cast<const uint8_t*>(src) + hdr.size;
  const uint64_t payload_bytes = srclength - hdr.size;
  cudaStream_t st = nullptr;
  StreamGeom geo{};
  int w = 0;
  SqybIndexHeader index;
  std::vector<RoiSel> host;   // what the descriptor copy reads
  RoiTables T{};
  if (indexed_stream(pl, N, &geo, &w) && lz4_read_prefix(payload, payload_bytes, &index) &&
      index.block_bytes == (uint32_t)kLz4BlockBytes && index.nblocks == geo.blocks() && index.raw_bytes == geo.bytes()) {
    info[0] = 1;
    const RoiPlan P = roi_plan(geo, rois);
    std::vector<BlockRun> runs;   // the needed blocks of every set, in stream order
    for (uint32_t j = 0; j < geo.sets; ++j)
      for (const BlockRun& b : P.runs) runs.push_back({(uint64_t)j * geo.set_blocks() + b.k0, (uint64_t)j * geo.set_blocks() + b.k1});
    const uint8_t* words = payload + kSkippableHeaderBytes + sizeof(SqybIndexHeader);
    std::vector<uint64_t> off;
    if (piece_offsets(words, geo.blocks(), runs, off) || kLz4FrameHeaderBytes + off.back() + kLz4EndMarkBytes != index.frame_bytes)
      return w ? 11 : 101;   // the sizes must add up to the frame
    const uint64_t nlist = P.list.size(), sub_raw = nlist * kLz4BlockBytes;
    uint64_t body = 0;
    for (size_t i = 0; i < runs.size(); ++i) body += off[2 * i + 1] - off[2 * i];
    const uint64_t prefix = lz4_prefix_bytes(nlist), sub_bytes = prefix + body + kLz4EndMarkBytes;
    uint8_t* const sub = A.host_frame(sub_bytes);   // every byte is written below
    lz4_write_prefix(sub, (uint32_t)nlist, sub_raw, kLz4FrameHeaderBytes + body + kLz4EndMarkBytes);
    for (uint64_t t = 0; t < nlist; ++t)
      std::memcpy(sub + kSkippableHeaderBytes + sizeof(SqybIndexHeader) + 4 * t, words + 4ull * P.list[t], 4);
    const uint8_t* blocks = payload + lz4_prefix_bytes(geo.blocks());
    uint64_t q = prefix;
    for (size_t i = 0; i < runs.size(); ++i) {
      std::memcpy(sub + q, blocks + off[2 * i], off[2 * i + 1] - off[2 * i]);
      q += off[2 * i + 1] - off[2 * i];
    }
    lz4_put32(sub + q, 0u);   // EndMark
    void *d_sub = nullptr, *ws = nullptr, *compact = nullptr, *d_box = nullptr;
    if (A.get(kSlotIn, sub_bytes, &d_sub) || A.get(kSlotWs, k_lz4_decode_workspace_bytes(sub_raw), &ws) ||
        A.get(kSlotA, sub_raw, &compact) || A.get(kSlotOut, box_bytes, &d_box) ||
        roi_tables(A, w ? kRoiPlanes : kRoiCodes, rois, batch, &P, false, host, &T, st))
      return 1;
    CK((cudaError_t)staged_h2d(d_sub, sub, sub_bytes, nthreads, st));
    info[2] = (long)sub_bytes;
    const uint8_t* d_frame = static_cast<const uint8_t*>(d_sub);
    CKK(k_lz4_decode_tables(d_frame, sub_bytes, sub_raw, ws, 0, 0, st));
    CKK(k_lz4_decode_run(d_frame, sub_bytes, static_cast<uint8_t*>(compact), sub_raw, ws, 0, 0, 0, 0, 0, st));
    if (int rc = roi_finish(A, pl, w, P, T, static_cast<const uint8_t*>(compact), ws, static_cast<uint16_t*>(d_box), st))
      return rc;
    info[1] = (long)nlist;
    CK((cudaError_t)staged_d2h(dst, d_box, box_bytes, nthreads, st));
    CK(cudaStreamSynchronize(st));
    return 0;
  }
  info[0] = 2;
  void *d_in = nullptr, *full = nullptr, *d_box = nullptr;
  // the payload is staged at a 256-byte aligned device address, whatever the header length was
  if (A.get(kSlotIn, payload_bytes + 256, &d_in) || A.get(kSlotOut, pl.elem * N, &full)) return 1;
  CK((cudaError_t)staged_h2d(d_in, payload, payload_bytes, nthreads, st));
  info[2] = (long)payload_bytes;
  if (int rc = decode_device_impl(A, hdr, pl, static_cast<const uint8_t*>(d_in), payload_bytes, full, pl.elem * N, st)) return rc;
  if (A.get(kSlotA, box_bytes, &d_box)) return 1;
  if (int rc = roi_crop(A, pl, full, N, rois, batch, host, d_box, st)) return rc;
  CK((cudaError_t)staged_d2h(dst, d_box, box_bytes, nthreads, st));
  CK(cudaStreamSynchronize(st));
  return 0;
}

}  // namespace

// =================================================================================================
// sqyx_* — device pointers
// =================================================================================================
extern "C" {

int sqyx_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int sqyx_set_device(int device) {
  if (cudaSetDevice(device) != cudaSuccess) return 1;
  std::lock_guard<std::mutex> lk(g_set_mu);
  g_set.assign(1, device);      // a caller that names its device (one process per GPU) is not sharded over the others
  return 0;
}

int sqyx_set_devices(int n, const int* devices) {
  int have = 0;
  if (n < 0 || (n > 0 && !devices) || cudaGetDeviceCount(&have) != cudaSuccess) return 1;
  std::vector<int> v;
  for (int i = 0; i < n; ++i) {
    if (devices[i] < 0 || devices[i] >= have || devices[i] >= kMaxDevices) return 1;
    if (std::find(v.begin(), v.end(), devices[i]) == v.end()) v.push_back(devices[i]);
  }
  std::sort(v.begin(), v.end());
  std::lock_guard<std::mutex> lk(g_set_mu);
  g_set = v;                    // empty: back to the default (SQY_CUDA_DEVICES / every visible device)
  return 0;
}

int sqyx_last_shard_info(long* out3) {
  if (!out3) return 1;
  std::lock_guard<std::mutex> lk(g_shard_stats_mu);
  out3[0] = g_shard_stats.gpus;
  out3[1] = g_shard_stats.nccl;
  out3[2] = g_shard_stats.pieces;
  return 0;
}

long sqyx_nccl_allreduces(void) { return g_nccl_allreduces.load(); }

long sqyx_kernel_launches(void) { return sqyb::g_kernel_launches.load(); }

int sqyx_enable_stage_timing(int on) {
  g_timing.store(on ? 1 : 0);
  return 0;
}

int sqyx_stage_ms(float* out7, int reset) {
  std::lock_guard<std::mutex> lk(g_timer_mu);
  for (int i = 0; i < kNumTimers; ++i) {
    if (out7) out7[i] = g_stage_ms[i];
    if (reset) g_stage_ms[i] = 0;
  }
  return 0;
}

long sqyx_host_l2_bytes(void) { return (long)host_l2_cache_bytes(); }

int sqyx_last_lz4_stats(long* out4) {
  DevLock dl;
  if (dl.acquire()) return 1;
  Arena* A = &dl.dev->arena;
  for (int i = 0; i < 4; ++i) out4[i] = A->last_stats[i];
  return 0;
}

long sqyx_set_lz4_defer_min(long nblocks) { return k_lz4_set_defer_min(nblocks); }

int sqyx_release_scratch(void) {
  DevLock dl;
  if (dl.acquire()) return 1;
  Arena* A = &dl.dev->arena;
  cudaDeviceSynchronize();
  A->release();
  for (int l = 0; l < kBatchLanes; ++l) dl.dev->batch_arena[l].release();
  staging_release();
  return 0;
}

int sqyx_encode_device_ex_UI16(const char* pipeline, const void* d_src, const long* shape, unsigned shape_size, void* d_dst,
                               long dst_capacity, long* dst_bytes, const void* d_global_hist, void* stream) {
  try {
    if (!shape) return 1;
    DevLock dl;
    if (dl.acquire()) return 1;
    return encode_device_blob(dl.dev->arena, 2, pipeline, d_src, to_shape(shape, shape_size), d_dst, dst_capacity, dst_bytes,
                              d_global_hist, static_cast<cudaStream_t>(stream));
  } catch (...) {
    return 1;
  }
}

int sqyx_encode_device_UI16(const char* pipeline, const void* d_src, const long* shape, unsigned shape_size, void* d_dst,
                            long dst_capacity, long* dst_bytes, void* stream) {
  return sqyx_encode_device_ex_UI16(pipeline, d_src, shape, shape_size, d_dst, dst_capacity, dst_bytes, nullptr, stream);
}

int sqyx_decode_device_UI16(const void* d_blob, long blob_bytes, void* d_dst, long dst_capacity, void* stream) {
  try {
    DevLock dl;
    if (dl.acquire()) return 1;
    return decode_device_blob(dl.dev->arena, 2, d_blob, blob_bytes, d_dst, dst_capacity, static_cast<cudaStream_t>(stream));
  } catch (...) {
    return 1;
  }
}

// ---- batches of independent stacks (time-lapse, cfg4/cfg5): lanes of one stack each, run concurrently ----
extern "C++" {
namespace {
template <class Fn>
int run_batch(int n, int* rcs, Fn&& one) {
  if (n < 0) return 1;
  if (n == 0) return 0;
  DevLock dl;
  if (dl.acquire()) return 1;
  const int dev = dl.id;
  Dev& D = *dl.dev;
  const int lanes = n < kBatchLanes ? n : kBatchLanes;
  for (int l = 0; l < lanes; ++l)
    if (!D.batch_stream[l] && cudaStreamCreateWithFlags(&D.batch_stream[l], cudaStreamNonBlocking) != cudaSuccess) return 1;
  const int timing = g_timing.exchange(0);   // the stage timers are per call, not per lane
  std::vector<int> rc((size_t)n, 1);
  std::vector<std::thread> th;
  for (int l = 0; l < lanes; ++l)
    th.emplace_back([&, l] {
      if (cudaSetDevice(dev) != cudaSuccess) return;
      for (int i = l; i < n; i += lanes) {
        try {
          rc[(size_t)i] = one(i, D.batch_arena[l], D.batch_stream[l]);
        } catch (...) {
          rc[(size_t)i] = 1;
        }
      }
    });
  for (auto& t : th) t.join();
  g_timing.store(timing);
  int bad = 0;
  for (int i = 0; i < n; ++i) {
    if (rcs) rcs[i] = rc[(size_t)i];
    bad |= rc[(size_t)i] != 0;
  }
  return bad ? 1 : 0;
}
}  // namespace
}  // extern "C++"

int sqyx_decode_batch_device_UI16(int n, const void* const* d_blobs, const long* blob_bytes, void* const* d_dsts,
                                  const long* dst_capacities, int* rcs) {
  if (n > 0 && (!d_blobs || !blob_bytes || !d_dsts || !dst_capacities)) return 1;
  return run_batch(n, rcs, [&](int i, Arena& A, cudaStream_t st) -> int {
    return decode_device_blob(A, 2, d_blobs[i], blob_bytes[i], d_dsts[i], dst_capacities[i], st);
  });
}

int sqyx_encode_batch_device_UI16(int n, const char* pipeline, const void* const* d_srcs, const long* shape, unsigned shape_size,
                                  void* const* d_dsts, const long* dst_capacities, long* dst_bytes, int* rcs) {
  if (!shape || (n > 0 && (!d_srcs || !d_dsts || !dst_capacities || !dst_bytes)) || !SQY_Pipeline_Possible_UI16(pipeline)) return 1;
  const std::vector<uint64_t> shp = to_shape(shape, shape_size);
  return run_batch(n, rcs, [&](int i, Arena& A, cudaStream_t st) -> int {
    return encode_device_blob(A, 2, pipeline, d_srcs[i], shp, d_dsts[i], dst_capacities[i], &dst_bytes[i], nullptr, st);
  });
}

int sqyx_encode_device_UI8(const char* pipeline, const void* d_src, const long* shape, unsigned shape_size, void* d_dst,
                           long dst_capacity, long* dst_bytes, void* stream) {
  try {
    if (!shape) return 1;
    DevLock dl;
    if (dl.acquire()) return 1;
    return encode_device_blob(dl.dev->arena, 1, pipeline, d_src, to_shape(shape, shape_size), d_dst, dst_capacity, dst_bytes, nullptr,
                              static_cast<cudaStream_t>(stream));
  } catch (...) {
    return 1;
  }
}

int sqyx_decode_device_UI8(const void* d_blob, long blob_bytes, void* d_dst, long dst_capacity, void* stream) {
  try {
    DevLock dl;
    if (dl.acquire()) return 1;
    return decode_device_blob(dl.dev->arena, 1, d_blob, blob_bytes, d_dst, dst_capacity, static_cast<cudaStream_t>(stream));
  } catch (...) {
    return 1;
  }
}

int sqyx_bitswap_encode_UI8(int w, const void* d_src, void* d_dst, long n, int threshold, void* stream) {
  if (n < 0) return 1;
  return k_bitswap_encode(1, w, d_src, d_dst, (uint64_t)n, threshold, static_cast<cudaStream_t>(stream)) ? 1 : 0;
}
int sqyx_bitswap_decode_UI8(int w, const void* d_src, void* d_dst, long n, void* stream) {
  if (n < 0) return 1;
  return k_bitswap_decode(1, w, d_src, d_dst, (uint64_t)n, static_cast<cudaStream_t>(stream)) ? 1 : 0;
}
int sqyx_remove_background_UI8(const void* d_src, void* d_dst, long n, int threshold, void* stream) {
  if (n < 0) return 1;
  return k_remove_background(1, d_src, d_dst, (uint64_t)n, threshold, static_cast<cudaStream_t>(stream)) ? 1 : 0;
}

int sqyx_bitshuffle_encode_UI16(const void* d_src, void* d_dst, long n, long block_size, void* stream) {
  return bitshuffle_device(true, 2, d_src, d_dst, n, block_size, stream);
}
int sqyx_bitshuffle_decode_UI16(const void* d_src, void* d_dst, long n, long block_size, void* stream) {
  return bitshuffle_device(false, 2, d_src, d_dst, n, block_size, stream);
}
int sqyx_bitshuffle_encode_UI8(const void* d_src, void* d_dst, long n, long block_size, void* stream) {
  return bitshuffle_device(true, 1, d_src, d_dst, n, block_size, stream);
}
int sqyx_bitshuffle_decode_UI8(const void* d_src, void* d_dst, long n, long block_size, void* stream) {
  return bitshuffle_device(false, 1, d_src, d_dst, n, block_size, stream);
}

int sqyx_diff_device(int decode, int sizeof_voxel, const void* d_src, void* d_dst, long z, long y, long x, void* stream) {
  if (z < 0 || y < 0 || x < 0 || (sizeof_voxel != 1 && sizeof_voxel != 2) || d_src == d_dst) return 1;
  if (!diff_shape_supported((uint64_t)z, (uint64_t)y, (uint64_t)x, sizeof_voxel)) return 2;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (decode ? k_diff_decode(sizeof_voxel, d_src, d_dst, (uint64_t)z, (uint64_t)y, (uint64_t)x, st)
             : k_diff_encode(sizeof_voxel, d_src, d_dst, (uint64_t)z, (uint64_t)y, (uint64_t)x, st))
    return 1;
  return cudaStreamSynchronize(st) == cudaSuccess ? 0 : 1;
}
int sqyx_diff_shape_supported(int sizeof_voxel, long z, long y, long x) {
  return z >= 0 && y >= 0 && x >= 0 && diff_shape_supported((uint64_t)z, (uint64_t)y, (uint64_t)x, sizeof_voxel) ? 1 : 0;
}

int sqyx_bitswap_encode_UI16(int w, const void* d_src, void* d_dst, long n, int threshold, void* stream) {
  if (n < 0) return 1;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (k_bitswap_encode(2, w, d_src, d_dst, (uint64_t)n, threshold, st)) return 1;
  return cudaStreamSynchronize(st) == cudaSuccess ? 0 : 1;
}

int sqyx_bitswap_decode_UI16(int w, const void* d_src, void* d_dst, long n, void* stream) {
  if (n < 0) return 1;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (k_bitswap_decode(2, w, d_src, d_dst, (uint64_t)n, st)) return 1;
  return cudaStreamSynchronize(st) == cudaSuccess ? 0 : 1;
}

int sqyx_remove_background_UI16(const void* d_src, void* d_dst, long n, int threshold, void* stream) {
  if (n < 0) return 1;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (k_remove_background(2, d_src, d_dst, (uint64_t)n, threshold, st)) return 1;
  return cudaStreamSynchronize(st) == cudaSuccess ? 0 : 1;
}

int sqyx_estimate_background_UI16(const void* d_src, const long* shape3, long l2_bytes, float* supports4, int* threshold,
                                  void* stream) {
  if (!d_src || !shape3 || !supports4 || !threshold) return 1;
  DevLock dl;
  if (dl.acquire()) return 1;
  Arena* A = &dl.dev->arena;
  return estimate_background(*A, static_cast<const uint16_t*>(d_src), (uint64_t)shape3[0], (uint64_t)shape3[1], (uint64_t)shape3[2],
                             l2_bytes, supports4, threshold, static_cast<cudaStream_t>(stream));
}

int sqyx_histogram_UI16(const void* d_src, long n, void* d_hist, void* stream) {
  if (n < 0 || !d_hist) return 1;
  return k_histogram_u16(static_cast<const uint16_t*>(d_src), (uint64_t)n, static_cast<uint32_t*>(d_hist),
                         static_cast<cudaStream_t>(stream)) ? 1 : 0;
}

float sqyx_histogram_support(const unsigned* hist, float threshold) { return hist ? histogram_support(hist, threshold) : 0.f; }

long sqyx_rmest_frame_portion(long frame_elems, long l2_bytes) {
  const size_t l2 = l2_bytes >= 0 ? (size_t)l2_bytes : host_l2_cache_bytes();
  return (long)rmest_frame_portion((uint64_t)frame_elems, l2);
}

int sqyx_quantiser_luts(const unsigned* hist, unsigned char* enc, unsigned short* dec) {
  if (!hist || !enc || !dec) return 1;
  quantiser_luts_from_histogram(hist, enc, dec);
  return 0;
}

int sqyx_lut_apply_UI16(const void* d_src, void* d_codes, long n, const unsigned char* enc_host, void* stream) {
  if (n < 0 || !enc_host) return 1;
  DevLock dl;
  if (dl.acquire()) return 1;
  Arena* A = &dl.dev->arena;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  SmallSlot small;
  if (small_slot(*A, &small)) return 1;
  CK(cudaMemcpyAsync(small.enc_lut, enc_host, 65536, cudaMemcpyHostToDevice, st));
  CKK(k_lut_apply(static_cast<const uint16_t*>(d_src), static_cast<uint8_t*>(d_codes), (uint64_t)n, small.enc_lut, st));
  CK(cudaStreamSynchronize(st));
  return 0;
}

int sqyx_lut_decode_UI16(const void* d_codes, void* d_dst, long n, const unsigned short* dec_host, void* stream) {
  if (n < 0 || !dec_host) return 1;
  DevLock dl;
  if (dl.acquire()) return 1;
  Arena* A = &dl.dev->arena;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  SmallSlot small;
  if (small_slot(*A, &small)) return 1;
  CK(cudaMemcpyAsync(small.dec_lut, dec_host, 512, cudaMemcpyHostToDevice, st));
  CKK(k_lut_decode(static_cast<const uint8_t*>(d_codes), static_cast<uint16_t*>(d_dst), (uint64_t)n, small.dec_lut, st));
  CK(cudaStreamSynchronize(st));
  return 0;
}

long sqyx_lz4_bound(long nbytes) { return nbytes < 0 ? -1 : (long)lz4_payload_bound((uint64_t)nbytes); }

int sqyx_lz4_encode_ex(const void* d_src, long nbytes, void* d_dst, long dst_capacity, long* payload_bytes, long pitch_bytes, void* stream) {
  if (nbytes < 0 || !d_dst || !payload_bytes) return 1;
  if ((uint64_t)dst_capacity < lz4_payload_bound((uint64_t)nbytes)) return 1;
  DevLock dl;
  if (dl.acquire()) return 1;
  Arena* A = &dl.dev->arena;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  void* ws = nullptr;
  if (A->get(kSlotWs, k_lz4_encode_workspace_bytes((uint64_t)nbytes), &ws)) return 1;
  // (pitch_bytes may carry kLz4HintNoNoise, kernels.h)
  const long pitch = pitch_bytes & ~(long)kLz4HintNoNoise;
  const uint32_t hint = (pitch > 0 && pitch <= 8192 ? (uint32_t)pitch : 0u) | (uint32_t)(pitch_bytes & (long)kLz4HintNoNoise);
  CKK(k_lz4_encode(static_cast<const uint8_t*>(d_src), (uint64_t)nbytes, static_cast<uint8_t*>(d_dst), ws, hint, st));
  uint64_t got = 0;
  if (lz4_encode_result(*A, ws, st, &got)) return 1;
  *payload_bytes = (long)got;
  return 0;
}

int sqyx_lz4_encode(const void* d_src, long nbytes, void* d_dst, long dst_capacity, long* payload_bytes, void* stream) {
  return sqyx_lz4_encode_ex(d_src, nbytes, d_dst, dst_capacity, payload_bytes, 0, stream);
}

int sqyx_lz4_decode(const void* d_src, long nbytes, void* d_dst, long dst_bytes, long* decoded_bytes, void* stream) {
  if (nbytes < 0 || dst_bytes < 0 || !d_src || !d_dst) return 1;
  DevLock dl;
  if (dl.acquire()) return 1;
  Arena* A = &dl.dev->arena;
  uint64_t got = 0;
  const int rc = lz4_decode_checked(*A, static_cast<const uint8_t*>(d_src), (uint64_t)nbytes, static_cast<uint8_t*>(d_dst),
                                    (uint64_t)dst_bytes, &got, static_cast<cudaStream_t>(stream));
  if (decoded_bytes) *decoded_bytes = (long)got;
  return rc;
}

// =================================================================================================
// SQY_* — the reference's boundary (host buffers)
// =================================================================================================

int SQY_Header_Size(const char* src, long* length) {
  if (!src || !length) return 1;
  const Header h = unpack_header(src, (size_t)(*length < 0 ? 0 : *length));
  *length = (long)h.size;  // 0 when no valid header is found (the reference's empty header)
  return 0;
}

int SQY_Decompressed_NDims(const char* src, long* num) {
  if (!src || !num) return 1;
  const Header h = unpack_header(src, (size_t)(*num < 0 ? 0 : *num));
  *num = (long)h.shape.size();
  return 0;
}

int SQY_Decompressed_Shape(const char* src, long* shape) {
  if (!src || !shape) return 1;
  const Header h = unpack_header(src, (size_t)(shape[0] < 0 ? 0 : shape[0]));
  for (size_t i = 0; i < h.shape.size(); ++i) shape[i] = (long)h.shape[i];
  return 0;
}

int SQY_Decompressed_Sizeof(const char* src, long* Sizeof) {
  if (!src || !Sizeof) return 1;
  const Header h = unpack_header(src, (size_t)(*Sizeof < 0 ? 0 : *Sizeof));
  *Sizeof = h.valid ? (long)sizeof_typename(h.raw_type) : 0;
  return 0;
}

int SQY_Decompressed_Length(const char* src, long* length) {
  if (!src || !length) return 1;
  const Header h = unpack_header(src, (size_t)(*length < 0 ? 0 : *length));
  // header::raw_size_byte (sqeazy_header.hpp:467-477); an empty shape multiplies out to 1 element in the reference
  uint64_t n = 1;
  for (uint64_t d : h.shape) n *= d;
  *length = (long)(n * sizeof_typename(h.raw_type));
  return 0;
}

int SQY_Version_Triple(int* version) {
  if (!version) return 1;
  version[0] = kVersionMajor;
  version[1] = kVersionMinor;
  version[2] = kVersionPatch;
  return 0;
}

bool SQY_Pipeline_Possible_UI16(const char* pipeline) {
  try {
    return pipeline ? pipeline_possible_u16(pipeline) : false;
  } catch (...) {
    return false;
  }
}
bool SQY_Pipeline_Possible_UI8(const char* pipeline) {
  try {
    return pipeline ? pipeline_possible_u8(pipeline) : false;
  } catch (...) {
    return false;
  }
}
bool SQY_Pipeline_Possible(const char* pipeline, int sizeofpixel) {   // src/sqeazy.cpp:254-268
  return sizeofpixel == 2 ? SQY_Pipeline_Possible_UI16(pipeline) : (sizeofpixel == 1 ? SQY_Pipeline_Possible_UI8(pipeline) : false);
}

int SQY_Pipeline_Max_Compressed_Length_UI16(const char* pipeline, long pipeline_length, long* length) {
  try {
    if (!pipeline || !length || pipeline_length < 0 || *length < 0) return 1;
    Pipeline pl;
    if (!build_pipeline_u16(std::string(pipeline, (size_t)pipeline_length), pl) || pl.empty()) return 1;
    *length = (long)max_encoded_size(pl, (uint64_t)*length);
    return 0;
  } catch (...) {
    return 1;
  }
}

int SQY_Pipeline_Max_Compressed_Length_3D_UI16(const char* pipeline, long* shape, unsigned shape_size, long* length) {
  try {
    if (!pipeline || !length || !shape || *length < 0) return 1;
    Pipeline pl;
    if (!build_pipeline_u16(std::string(pipeline, (size_t)*length), pl) || pl.empty()) return 1;
    uint64_t n = 1;
    for (unsigned i = 0; i < shape_size; ++i) n *= (uint64_t)shape[i];  // 64-bit, unlike the reference (SURVEY F7)
    *length = (long)max_encoded_size(pl, 2 * n);
    return 0;
  } catch (...) {
    return 1;
  }
}

int SQY_Pipeline_Max_Compressed_Length_UI8(const char* pipeline, long pipeline_length, long* length) {   // src/sqeazy.cpp:144-163
  try {
    if (!pipeline || !length || pipeline_length < 0 || *length < 0) return 1;
    Pipeline pl;
    if (!build_pipeline_u8(std::string(pipeline, (size_t)pipeline_length), pl) || pl.empty()) return 1;
    *length = (long)max_encoded_size(pl, (uint64_t)*length);
    return 0;
  } catch (...) {
    return 1;
  }
}
int SQY_Pipeline_Max_Compressed_Length_3D_UI8(const char* pipeline, long* shape, unsigned shape_size, long* length) {   // :209-231
  try {
    if (!pipeline || !length || !shape || *length < 0) return 1;
    Pipeline pl;
    if (!build_pipeline_u8(std::string(pipeline, (size_t)*length), pl) || pl.empty()) return 1;
    uint64_t n = 1;
    for (unsigned i = 0; i < shape_size; ++i) n *= (uint64_t)shape[i];
    *length = (long)max_encoded_size(pl, n);
    return 0;
  } catch (...) {
    return 1;
  }
}

// ---- streamed host paths: the PCIe hop of a large stack overlaps the kernels ----
// `[remove_background | rmestbkrd ->] bitswapN -> lz4` on uint16 (the headline pipelines): the stack arrives in 256 MiB z-slabs
// and each slab is filtered, transposed and LZ4-compressed while the next one is still on the bus (encode_planes_slabs).
// Only the last slab's kernels, the offset scan and the compaction remain after the last byte has arrived. Decode: the final
// inverse transpose runs slab by slab and every slab leaves for the host as soon as it is done.
// returns 0 and the blob size, or an error; the caller has checked that the pipeline is one of these (shard_kind: PlanesLz4),
// that the stack has at least kStreamMinBytes and that N is a multiple of kStreamGrainVoxels
int host_encode_streamed(Arena& A, const Pipeline& pl, const char* src, const std::vector<uint64_t>& shape, uint64_t N, char* dst,
                         uint64_t cap, uint64_t* out_bytes, int nthreads) {
  const StreamGeom geo = StreamGeom::planes(N, pl.head.back().w);
  cudaStream_t st = nullptr;
  void *d_in = nullptr, *d_out_v = nullptr, *d_planes = nullptr, *ws = nullptr;
  if (A.get(kSlotIn, 2 * N, &d_in) || A.get(kSlotOut, cap, &d_out_v) || A.get(kSlotA, geo.bytes(), &d_planes) ||
      A.get(kSlotWs, k_lz4_encode_workspace_bytes(geo.bytes()), &ws))
    return 1;
  uint8_t* d_out = static_cast<uint8_t*>(d_out_v);
  const size_t reserve = header_reserve_bytes(pl, shape);
  if (cap < reserve || cap - reserve < lz4_payload_bound(geo.bytes())) return 1;
  // rmestbkrd: the estimate's two z faces and six border rows are sent on their own behind the first slab, which is already on
  // its way: the bus never waits for the estimate, and the threshold is there before the first kernel.
  auto threshold = [&](int* t) -> int {
    *t = pl.head.size() == 2 ? pl.head[0].threshold : 0;
    if (pl.head.size() != 2 || pl.head[0].kind != StageKind::RmEstBkrd) return 0;
    return estimate_background_host(A, reinterpret_cast<const uint16_t*>(src), shape[0], shape[1], shape[2], t, st);
  };
  if (encode_planes_slabs(geo, pl.head.back().w, threshold, lz4_pitch_hint(pl, shape), kStreamSlabBytes / 2, src,
                          static_cast<uint16_t*>(d_in), static_cast<uint16_t*>(d_planes), d_out + reserve, ws, nthreads, st))
    return 1;
  uint64_t payload_bytes = 0;
  std::string slot;
  if (lz4_encode_result(A, ws, st, &payload_bytes) || header_slot(pl, shape, payload_bytes, reserve, &slot)) return 1;
  CK(cudaMemcpyAsync(d_out, slot.data(), slot.size(), cudaMemcpyHostToDevice, st));
  CK((cudaError_t)staged_d2h(dst, d_out, reserve + payload_bytes, nthreads, st));
  CK(cudaStreamSynchronize(st));
  *out_bytes = reserve + payload_bytes;
  return 0;
}

static int host_encode(int elem, const char* pipeline, const char* src, long* shape, unsigned shape_size, char* dst, long* dstlength,
                       int nthreads) {
  NvtxRange range(elem == 1 ? "SQY_PipelineEncode_UI8" : "SQY_PipelineEncode_UI16");
  try {
    if (!pipeline || !src || !shape || !dst || !dstlength) return 1;
    Pipeline pl;
    if (!(elem == 1 ? build_pipeline_u8(pipeline, pl) : build_pipeline_u16(pipeline, pl))) return 1;
    if (pl.empty()) {
      std::fprintf(stderr, "[sqeazy]\t received pipeline of size 0, cannot encode buffer\n");
      return 1;
    }
    const std::vector<uint64_t> shp = to_shape(shape, shape_size);
    const uint64_t N = shape_product(shp), raw_bytes = (uint64_t)elem * N;
    const uint64_t cap = max_encoded_size(pl, raw_bytes);
    if (elem == 2) {
      // one stack over several GPUs (and the streamed quantiser path on one): sharded.inl
      {
        std::lock_guard<std::mutex> lk(g_shard_stats_mu);
        g_shard_stats = ShardStats();
      }
      uint64_t out = 0;
      const int rc = host_encode_sharded(pl, src, shp, N, dst, cap, &out, nthreads);
      if (rc > 0) return 1;
      if (rc == 0) {
        *dstlength = (long)out;
        return 0;
      }
    }
    DevLock dl;
    if (dl.acquire()) return 1;
    Arena* A = &dl.dev->arena;
    if (shard_kind(pl, shp) == ShardKind::PlanesLz4 && 2 * N >= kStreamMinBytes && N % kStreamGrainVoxels == 0 && !g_timing.load()) {
      uint64_t out = 0;
      if (host_encode_streamed(*A, pl, src, shp, N, dst, cap, &out, nthreads)) return 1;
      *dstlength = (long)out;
      return 0;
    }
    void *d_in = nullptr, *d_out = nullptr;
    if (A->get(kSlotIn, raw_bytes, &d_in) || A->get(kSlotOut, cap, &d_out)) return 1;
    cudaStream_t st = nullptr;
    CK((cudaError_t)staged_h2d(d_in, src, raw_bytes, nthreads, st));   // pageable buffers: nthreads host threads feed a pinned ring
    uint64_t out = 0;
    const int rc = encode_device_impl(*A, pl, d_in, shp, static_cast<uint8_t*>(d_out), cap, &out,
                                      nullptr, st);
    if (rc) return 1;
    CK((cudaError_t)staged_d2h(dst, d_out, out, nthreads, st));
    CK(cudaStreamSynchronize(st));
    *dstlength = (long)out;
    return 0;
  } catch (...) {
    return 1;
  }
}

static int host_decode(int elem, const char* src, long srclength, char* dst, int nthreads) {
  NvtxRange range(elem == 1 ? "SQY_Decode_UI8" : "SQY_Decode_UI16");
  try {
    if (!src || !dst || srclength <= 0) return 1;
    const Header hdr = unpack_header(src, (size_t)srclength);
    if (!hdr.valid) return 1;
    Pipeline pl;
    if (!(elem == 1 ? build_pipeline_u8(hdr.pipeline, pl) : build_pipeline_u16(hdr.pipeline, pl))) {
      std::fprintf(stderr, "[sqeazy]\t%s cannot be build with this version of sqeazy\n", hdr.pipeline.c_str());
      return 1;
    }
    if (pl.empty()) {
      std::fprintf(stderr, "[sqeazy]\t received pipeline of size 0, no decoding possible\n");
      return 1;
    }
    if (sizeof_typename(hdr.raw_type) != (unsigned)elem) return 1;
    const uint64_t raw_bytes = (uint64_t)elem * shape_product(hdr.shape);
    if (elem == 2) {
      {
        std::lock_guard<std::mutex> lk(g_shard_stats_mu);
        g_shard_stats = ShardStats();
      }
      const int rc = host_decode_sharded(hdr, pl, src, (uint64_t)srclength, dst, nthreads);
      if (rc >= 0) return rc;
    }
    DevLock dl;
    if (dl.acquire()) return 1;
    Arena* A = &dl.dev->arena;
    void *d_in = nullptr, *d_out = nullptr;
    const uint64_t payload_bytes = (uint64_t)srclength - hdr.size;
    // the payload is staged at a 256-byte aligned device address, whatever the header length was
    if (A->get(kSlotIn, payload_bytes + 256, &d_in) || A->get(kSlotOut, raw_bytes, &d_out)) return 1;
    cudaStream_t st = nullptr;
    CK((cudaError_t)staged_h2d(d_in, src + hdr.size, payload_bytes, nthreads, st));
    HostSink sink{dst, nthreads};
    const int rc = decode_device_impl(*A, hdr, pl, static_cast<const uint8_t*>(d_in), payload_bytes, d_out,
                                      raw_bytes, st, &sink);
    if (rc) return rc;
    if (!sink.done) CK((cudaError_t)staged_d2h(dst, d_out, raw_bytes, nthreads, st));
    CK(cudaStreamSynchronize(st));
    return 0;
  } catch (...) {
    return 1;
  }
}

int SQY_PipelineEncode_UI16(const char* pipeline, const char* src, long* shape, unsigned shape_size, char* dst, long* dstlength,
                            int nthreads) {
  // nthreads: host threads that stage a pageable caller buffer (staging.hpp); the kernels have no thread knob
  return host_encode(2, pipeline, src, shape, shape_size, dst, dstlength, nthreads);
}

int SQY_Decode_UI16(const char* src, long srclength, char* dst, int nthreads) {
  return host_decode(2, src, srclength, dst, nthreads);
}

int SQY_PipelineDecode_UI16(const char* src, long srclength, char* dst, int nthreads) {
  return SQY_Decode_UI16(src, srclength, dst, nthreads);
}

// uint8 volumes (src/sqeazy.cpp:72-106, 309-335)
int SQY_PipelineEncode_UI8(const char* pipeline, const char* src, long* shape, unsigned shape_size, char* dst, long* dstlength,
                           int nthreads) {
  return host_encode(1, pipeline, src, shape, shape_size, dst, dstlength, nthreads);
}
int SQY_Decode_UI8(const char* src, long srclength, char* dst, int nthreads) {
  return host_decode(1, src, srclength, dst, nthreads);
}

// ---- sub-volume decode: the twelve entry points share the planner, the checks and the whole-stack route. sel: nsel selections
// one after the other, each ndims tuples of `width` longs, boxes (width 2) or strided slices (width 3); rois_of. The selections
// are written one after the other. A batch (the sqyx_decode_slice_batch_* calls) never takes route 0: its union then holds every
// block ----
static int decode_roi_device(int elem, const void* d_blob, long blob_bytes, const long* sel, unsigned width, unsigned ndims,
                             unsigned nsel, bool batch, void* d_dst, long dst_capacity, void* stream) {
  try {
    if (!d_blob || blob_bytes <= 0 || dst_capacity < 0) return 1;
    DevLock dl;
    if (dl.acquire()) return 1;
    Arena& A = dl.dev->arena;
    long* info = dl.dev->roi_info;
    info[0] = -1, info[1] = info[2] = info[3] = 0;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const uint8_t* blob = static_cast<const uint8_t*>(d_blob);
    Header hdr;
    if (parse_blob_header_device(blob, (uint64_t)blob_bytes, hdr, st) || sizeof_typename(hdr.raw_type) != (unsigned)elem) return 1;
    Pipeline pl;
    if (!(elem == 1 ? build_pipeline_u8(hdr.pipeline, pl) : build_pipeline_u16(hdr.pipeline, pl)) || pl.empty()) return 1;
    std::vector<Roi> rois;
    uint64_t voxels = 0;
    if (int rc = rois_of(hdr.shape, sel, width, ndims, nsel, &rois, &voxels)) return rc;
    if ((uint64_t)dst_capacity < (uint64_t)elem * voxels || (voxels && !d_dst)) return 1;
    if (voxels == 0) return 0;
    int rc = 0;
    if (!batch && rois[0].whole) {
      info[0] = 0;
      rc = decode_device_blob(A, elem, d_blob, blob_bytes, d_dst, dst_capacity, st);
    } else {
      rc = roi_device(A, hdr, pl, blob + hdr.size, (uint64_t)blob_bytes - hdr.size, rois, batch, d_dst, st, info);
    }
    if (rc == 0) info[3] = (long)voxels;
    return rc;
  } catch (...) {
    return 1;
  }
}

static int decode_roi_host(const char* name, int elem, const char* src, long srclength, const long* sel, unsigned width, unsigned ndims,
                           unsigned nsel, bool batch, char* dst, long dst_capacity, int nthreads) {
  NvtxRange range(name);
  try {
    if (!src || srclength <= 0 || dst_capacity < 0) return 1;
    const Header hdr = unpack_header(src, (size_t)srclength);
    if (!hdr.valid || sizeof_typename(hdr.raw_type) != (unsigned)elem) return 1;
    Pipeline pl;
    if (!(elem == 1 ? build_pipeline_u8(hdr.pipeline, pl) : build_pipeline_u16(hdr.pipeline, pl)) || pl.empty()) return 1;
    std::vector<Roi> rois;
    uint64_t voxels = 0;
    if (int rc = rois_of(hdr.shape, sel, width, ndims, nsel, &rois, &voxels)) return rc;
    if ((uint64_t)dst_capacity < (uint64_t)elem * voxels || (voxels && !dst)) return 1;
    long info[4] = {-1, 0, 0, 0};
    int rc = 0;
    const bool whole = !batch && rois[0].whole;
    if (voxels && whole) {
      info[0] = 0;
      info[2] = srclength - (long)hdr.size;
      rc = host_decode(elem, src, srclength, dst, nthreads);   // takes the device locks it needs itself
    }
    DevLock dl;
    if (dl.acquire()) return 1;
    if (voxels && !whole) rc = roi_host(dl.dev->arena, hdr, pl, src, (uint64_t)srclength, rois, batch, voxels, dst, nthreads, info);
    if (rc == 0) info[3] = (long)voxels;
    std::copy(info, info + 4, dl.dev->roi_info);
    return rc;
  } catch (...) {
    return 1;
  }
}

int sqyx_decode_roi_device_UI16(const void* d_blob, long blob_bytes, const long* box, unsigned ndims, void* d_dst, long dst_capacity,
                                void* stream) {
  return decode_roi_device(2, d_blob, blob_bytes, box, 2, ndims, 1, false, d_dst, dst_capacity, stream);
}
int sqyx_decode_roi_device_UI8(const void* d_blob, long blob_bytes, const long* box, unsigned ndims, void* d_dst, long dst_capacity,
                               void* stream) {
  return decode_roi_device(1, d_blob, blob_bytes, box, 2, ndims, 1, false, d_dst, dst_capacity, stream);
}
int sqyx_decode_roi_UI16(const char* src, long srclength, const long* box, unsigned ndims, char* dst, long dst_capacity, int nthreads) {
  return decode_roi_host("sqyx_decode_roi_UI16", 2, src, srclength, box, 2, ndims, 1, false, dst, dst_capacity, nthreads);
}
int sqyx_decode_roi_UI8(const char* src, long srclength, const long* box, unsigned ndims, char* dst, long dst_capacity, int nthreads) {
  return decode_roi_host("sqyx_decode_roi_UI8", 1, src, srclength, box, 2, ndims, 1, false, dst, dst_capacity, nthreads);
}
int sqyx_decode_slice_device_UI16(const void* d_blob, long blob_bytes, const long* slices, unsigned ndims, void* d_dst,
                                  long dst_capacity, void* stream) {
  return decode_roi_device(2, d_blob, blob_bytes, slices, 3, ndims, 1, false, d_dst, dst_capacity, stream);
}
int sqyx_decode_slice_device_UI8(const void* d_blob, long blob_bytes, const long* slices, unsigned ndims, void* d_dst,
                                 long dst_capacity, void* stream) {
  return decode_roi_device(1, d_blob, blob_bytes, slices, 3, ndims, 1, false, d_dst, dst_capacity, stream);
}
int sqyx_decode_slice_UI16(const char* src, long srclength, const long* slices, unsigned ndims, char* dst, long dst_capacity,
                           int nthreads) {
  return decode_roi_host("sqyx_decode_slice_UI16", 2, src, srclength, slices, 3, ndims, 1, false, dst, dst_capacity, nthreads);
}
int sqyx_decode_slice_UI8(const char* src, long srclength, const long* slices, unsigned ndims, char* dst, long dst_capacity,
                          int nthreads) {
  return decode_roi_host("sqyx_decode_slice_UI8", 1, src, srclength, slices, 3, ndims, 1, false, dst, dst_capacity, nthreads);
}
int sqyx_decode_slice_batch_device_UI16(const void* d_blob, long blob_bytes, const long* slices, unsigned nsel, unsigned ndims,
                                        void* d_dst, long dst_capacity, void* stream) {
  return decode_roi_device(2, d_blob, blob_bytes, slices, 3, ndims, nsel, true, d_dst, dst_capacity, stream);
}
int sqyx_decode_slice_batch_device_UI8(const void* d_blob, long blob_bytes, const long* slices, unsigned nsel, unsigned ndims,
                                       void* d_dst, long dst_capacity, void* stream) {
  return decode_roi_device(1, d_blob, blob_bytes, slices, 3, ndims, nsel, true, d_dst, dst_capacity, stream);
}
int sqyx_decode_slice_batch_UI16(const char* src, long srclength, const long* slices, unsigned nsel, unsigned ndims, char* dst,
                                 long dst_capacity, int nthreads) {
  return decode_roi_host("sqyx_decode_slice_batch_UI16", 2, src, srclength, slices, 3, ndims, nsel, true, dst, dst_capacity, nthreads);
}
int sqyx_decode_slice_batch_UI8(const char* src, long srclength, const long* slices, unsigned nsel, unsigned ndims, char* dst,
                                long dst_capacity, int nthreads) {
  return decode_roi_host("sqyx_decode_slice_batch_UI8", 1, src, srclength, slices, 3, ndims, nsel, true, dst, dst_capacity, nthreads);
}

int sqyx_last_roi_info(long* out4) {
  if (!out4) return 1;
  DevLock dl;
  if (dl.acquire()) return 1;
  std::copy(dl.dev->roi_info, dl.dev->roi_info + 4, out4);
  return 0;
}

int SQY_h5_query_sizeof(const char*, const char*, unsigned*) { return 1; }
int SQY_h5_query_dtype(const char*, const char*, unsigned*) { return 1; }
int SQY_h5_query_ndims(const char*, const char*, unsigned*) { return 1; }
int SQY_h5_query_shape(const char*, const char*, unsigned*) { return 1; }
int SQY_h5_read_UI16(const char*, const char*, unsigned short*) { return 1; }
int SQY_h5_write_UI16(const char*, const char*, const unsigned short*, unsigned, const unsigned*, const char*) { return 1; }
int SQY_h5_write(const char*, const char*, const char*, unsigned long) { return 1; }
int SQY_h5_link(const char*, const char*, const char*, const char*, const char*, const char*) { return 1; }

}  // extern "C"
