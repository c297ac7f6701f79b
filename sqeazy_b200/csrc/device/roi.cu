// Sub-volume gather (api.cu: the sqyx_decode_roi_* and sqyx_decode_slice_* entry points): the voxels of a strided slice of a
// stack (a box when every step is 1), densely in C order, out of
//   planes: the compact 16 KiB blocks of the bit planes of a uint16 bitswapW that hold the box (k_lz4_decode_list, or a
//           sub-frame decoded whole), transposed back by the thread program of bitswap_thread.h;
//   codes:  the compact 16 KiB blocks of 8-bit quantiser codes that hold the box, through the 256-entry decode LUT;
//   raw:    a whole decoded stack (the crop behind the decode-whole route).
// One thread program (gather_item), templated on the source and on one of three programs chosen by the runs' inner step, run by
// two kernels: roi_gather_kernel for one selection, its runs by value (the single calls; its gather measured faster than that of
// a batch of one, profiles/README.md), and roi_gather_batch_kernel for many, written one after the other, their descriptors in
// device memory (the batch calls). The k_roi_* entry points take either (RoiSelections) and make one launch per program that a
// selection takes:
//   run   (step 1): a thread takes one aligned group of G voxels of the stack (32, or 16 codes: one 16-byte load) that meets a
//                   run and writes the voxels of the group that lie in the run to their dense place: whole groups with 16-byte
//                   stores where the destination allows it, the groups at the ends of a run voxel by voxel;
//   group (1 < step < G/2): the same groups, of which a thread writes the selected voxels, at least three of each whole group;
//   voxel (step >= G/2, when a group holds at most two selected voxels): a thread reads one selected voxel straight from its
//                   source (its bits of the P planes, its code, or the voxel) and writes it; nothing is transposed.
#include "bitswap_thread.h"
#include "common.cuh"
#include "kernels.h"
#include "lz4_format.h"

namespace sqyb {
namespace {

constexpr int kRoiThreads = 256;

template <int W>
struct FromPlanes {
  using T = uint16_t;
  static constexpr int G = 32;
  static constexpr uint32_t kWords = G * sizeof(T) / 4;
  const uint8_t* compact;
  const uint32_t* pos;
  uint64_t nsel;
  __device__ void prologue() const {}
  // group g = voxels [32g, 32g + 32): 4W bytes at offset 4W g of every plane segment, inside one 16 KiB block of each
  __device__ void load(uint64_t g, uint32_t (&L)[kWords]) const {
    const uint64_t o = g * (4 * W);
    const uint64_t k = o / kLz4BlockBytes;
    const uint16_t* block = reinterpret_cast<const uint16_t*>(compact + (uint64_t)__ldg(pos + k) * kLz4BlockBytes);
    uint32_t reg[16];
    bitswap_thread::load_planes<W, false>(block, (o % kLz4BlockBytes) / (4 * W), nsel * (kLz4BlockBytes / 2), reg);
    bitswap_thread::voxels_of<W>(reg, L);
  }
  // voxel v alone: W bits of it from each of the P planes (the layout of bitswap_thread.h's encode_chunk: in the words of
  // group v / 32, voxel m = v % 32 is atom P-1 - m % P of half (m / P) & 1 of word m / 2P; plane p is segment P-1-p)
  __device__ T voxel(uint64_t v) const {
    constexpr int P = 16 / W;
    const uint64_t o = (v / G) * (4 * W);
    const uint32_t* seg = reinterpret_cast<const uint32_t*>(compact + (uint64_t)__ldg(pos + o / kLz4BlockBytes) * kLz4BlockBytes +
                                                            o % kLz4BlockBytes);
    const uint32_t m = (uint32_t)(v % G);
    const int shift = 16 * ((m / P) & 1) + W * (P - 1 - m % P);
    const uint64_t S = nsel * (kLz4BlockBytes / 4);
    seg += m / (2 * P);
    uint32_t x = 0;
#pragma unroll
    for (int p = 0; p < P; ++p) x |= ((__ldg(seg + (uint64_t)(P - 1 - p) * S) >> shift) & ((1u << W) - 1u)) << (p * W);
    return (T)x;
  }
};

struct FromCodes {
  using T = uint16_t;
  static constexpr int G = 16;
  static constexpr uint32_t kWords = G * sizeof(T) / 4;
  const uint8_t* compact;
  const uint32_t* pos;
  const uint16_t* lut;
  __device__ void prologue() const {
    extern __shared__ uint16_t roi_lut[];
    if (threadIdx.x < 256) roi_lut[threadIdx.x] = lut[threadIdx.x];
    __syncthreads();
  }
  __device__ void load(uint64_t g, uint32_t (&L)[kWords]) const {
    extern __shared__ uint16_t roi_lut[];
    const uint64_t v = g * G;
    const uint64_t k = v / kLz4BlockBytes;
    const uint4 c = __ldg(reinterpret_cast<const uint4*>(compact + (uint64_t)__ldg(pos + k) * kLz4BlockBytes + v % kLz4BlockBytes));
    const uint32_t w[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      L[2 * i] = roi_lut[w[i] & 0xff] | ((uint32_t)roi_lut[(w[i] >> 8) & 0xff] << 16);
      L[2 * i + 1] = roi_lut[(w[i] >> 16) & 0xff] | ((uint32_t)roi_lut[w[i] >> 24] << 16);
    }
  }
  __device__ T voxel(uint64_t v) const {
    extern __shared__ uint16_t roi_lut[];
    return roi_lut[__ldg(compact + (uint64_t)__ldg(pos + v / kLz4BlockBytes) * kLz4BlockBytes + v % kLz4BlockBytes)];
  }
};

template <class E>
struct FromVolume {
  using T = E;
  static constexpr int G = 32;
  static constexpr uint32_t kWords = G * sizeof(T) / 4;
  const T* vol;   // 16-byte aligned
  uint64_t n;
  __device__ void prologue() const {}
  __device__ void load(uint64_t g, uint32_t (&L)[kWords]) const {
    if ((g + 1) * G <= n) {
      const uint4* p = reinterpret_cast<const uint4*>(vol + g * G);
#pragma unroll
      for (uint32_t i = 0; i < kWords / 4; ++i) {
        const uint4 v = __ldg(p + i);
        L[4 * i] = v.x; L[4 * i + 1] = v.y; L[4 * i + 2] = v.z; L[4 * i + 3] = v.w;
      }
      return;
    }
    // the last group of a ragged stack
    constexpr int kPer = 4 / sizeof(T);
#pragma unroll
    for (uint32_t i = 0; i < kWords; ++i) {
      uint32_t w = 0;
#pragma unroll
      for (int j = 0; j < kPer; ++j) {
        const uint64_t v = g * G + i * kPer + j;
        if (v < n) w |= (uint32_t)vol[v] << (8 * sizeof(T) * j);
      }
      L[i] = w;
    }
  }
  __device__ T voxel(uint64_t v) const { return __ldg(vol + v); }
};

// R.start(r) with its loop kept rolled: unrolled, the chain of 64-bit divisions makes the batch gather spill
__device__ __forceinline__ uint64_t run_start(const RoiRuns& R, uint64_t r) {
  uint64_t v = R.base;
#pragma unroll 1
  for (int k = R.nlead - 1; k >= 0; --k) {
    v += (r % R.extent[k]) * R.stride[k];
    r /= R.extent[k];
  }
  return v;
}

// The thread program of a selection by its runs' inner step, and the most groups of G voxels that the span of one run meets
__host__ __device__ inline int roi_program(const RoiRuns& R, int G) {
  return R.step >= (uint64_t)G / 2 ? kRoiVoxel : R.step == 1 ? kRoiRun : kRoiGroup;
}
__host__ __device__ inline uint64_t roi_groups(const RoiRuns& R, int G) { return ((R.len - 1) * R.step + 1 + G - 1) / G + 1; }

// Work item `it` of program kProgram for the selection R, written into dst; start(r) is R.start(r). run / group: items =
// R.rows * groups, item (r, q) is the q-th group that meets the span of run r; voxel: items = R.rows * R.len, one per selected voxel
template <int kProgram, class Src, class Start>
__device__ __forceinline__ void gather_item(const Src& src, const RoiRuns& R, uint64_t groups, uint64_t it, Start start,
                                            typename Src::T* dst) {
  using T = typename Src::T;
  constexpr int G = Src::G;
  constexpr int kPer = 4 / sizeof(T);
  if (kProgram == kRoiVoxel) {
    const uint64_t r = it / R.len;
    dst[it] = src.voxel(start(r) + (it - r * R.len) * R.step);
    return;
  }
  const uint64_t r = it / groups, v0 = start(r), v1 = v0 + (kProgram == kRoiRun ? R.len : (R.len - 1) * R.step + 1);
  const uint64_t g = v0 / G + (it - r * groups);
  if (g * G >= v1) return;
  uint32_t L[Src::kWords];
  src.load(g, L);
  T* out = dst + r * R.len;   // run: voxel v of the run lands at out[v - v0]; group: at out[(v - v0) / step]
  if (kProgram == kRoiGroup) {
    // the group's first selected voxel, at offset `next` in the group (G or more: none)
    const uint64_t j0 = g * G > v0 ? (g * G - v0 + R.step - 1) / R.step : 0;
    uint32_t next = (uint32_t)(v0 + j0 * R.step - g * G);
    const uint32_t step = (uint32_t)R.step;
    T* o = out + j0;
#pragma unroll
    for (int k = 0; k < G; ++k) {
      if (k == next && g * G + k < v1) {
        *o++ = (T)(L[k / kPer] >> (8 * sizeof(T) * (k % kPer)));
        next += step;
      }
    }
    return;
  }
  // packed selections start anywhere: whole groups take 16-byte stores only where the destination is aligned
  if (g * G >= v0 && (g + 1) * G <= v1 && (((uintptr_t)(out + (g * G - v0))) & 15) == 0) {
    uint4* o = reinterpret_cast<uint4*>(out + (g * G - v0));
#pragma unroll
    for (uint32_t i = 0; i < Src::kWords / 4; ++i) o[i] = make_uint4(L[4 * i], L[4 * i + 1], L[4 * i + 2], L[4 * i + 3]);
    return;
  }
#pragma unroll
  for (int k = 0; k < G; ++k) {
    const uint64_t v = g * G + k;
    if (v >= v0 && v < v1) out[v - v0] = (T)(L[k / kPer] >> (8 * sizeof(T) * (k % kPer)));
  }
}

// one selection, its runs by value
template <class Src, int kProgram>
__global__ void __launch_bounds__(kRoiThreads) roi_gather_kernel(Src src, RoiRuns R, uint64_t groups, typename Src::T* __restrict__ dst) {
  src.prologue();
  const uint64_t items = R.rows * (kProgram == kRoiVoxel ? R.len : groups);
  for (uint64_t it = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; it < items; it += (uint64_t)gridDim.x * blockDim.x)
    gather_item<kProgram>(src, R, groups, it, [&](uint64_t r) { return R.start(r); }, dst);
}

// The batch: one launch per thread program serves every selection of the call that takes it. sels[0 .. nsel) hold the prefix sums
// of their items (`before`); a thread finds the selection of its item by a binary search over them and runs the program for it,
// into dst + sels[s].first.
template <class Src, int kProgram>
__global__ void __launch_bounds__(kRoiThreads) roi_gather_batch_kernel(Src src, const RoiSel* __restrict__ sels, uint32_t nsel,
                                                                       uint64_t items, typename Src::T* __restrict__ dst) {
  src.prologue();
  for (uint64_t it = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; it < items; it += (uint64_t)gridDim.x * blockDim.x) {
    uint32_t s = 0, hi = nsel;   // sels[s].before <= it < sels[hi].before (hi = nsel: items)
    while (hi - s > 1) {
      const uint32_t mid = (s + hi) / 2;
      if (__ldg(&sels[mid].before) <= it) s = mid;
      else hi = mid;
    }
    const RoiRuns& R = sels[s].runs;
    const uint64_t groups = kProgram == kRoiVoxel ? 0 : roi_groups(R, Src::G);
    gather_item<kProgram>(src, R, groups, it - __ldg(&sels[s].before), [&](uint64_t r) { return run_start(R, r); },
                          dst + __ldg(&sels[s].first));
  }
}

// The launch of program kProgram: for one selection when it takes that program, for a batch when any of its selections does
template <class Src, int kProgram>
void launch_program(const Src& src, const RoiSelections& S, typename Src::T* dst, size_t smem, cudaStream_t st) {
  if (S.d_sels) {
    const RoiBatch& B = S.batch;
    if (!B.count[kProgram]) return;
    roi_gather_batch_kernel<Src, kProgram><<<grid_for(B.items[kProgram], kRoiThreads), kRoiThreads, smem, st>>>(
        src, S.d_sels + B.begin[kProgram], B.count[kProgram], B.items[kProgram], dst);
  } else {
    const RoiRuns& R = S.runs;
    if (!R.rows || !R.len || roi_program(R, Src::G) != kProgram) return;
    const uint64_t groups = roi_groups(R, Src::G), items = R.rows * (kProgram == kRoiVoxel ? R.len : groups);
    roi_gather_kernel<Src, kProgram><<<grid_for(items, kRoiThreads), kRoiThreads, smem, st>>>(src, R, groups, dst);
  }
  SQYB_COUNT_LAUNCH(1);
}

template <class Src>
int launch_gather(const Src& src, const RoiSelections& S, typename Src::T* dst, size_t smem, cudaStream_t st) {
  launch_program<Src, kRoiRun>(src, S, dst, smem, st);
  launch_program<Src, kRoiGroup>(src, S, dst, smem, st);
  launch_program<Src, kRoiVoxel>(src, S, dst, smem, st);
  return (int)cudaGetLastError();
}

}  // namespace

int k_roi_gather_planes(int w, const uint8_t* compact, const uint32_t* pos, uint64_t nsel, const RoiSelections& S, uint16_t* dst,
                        cudaStream_t st) {
  if ((((uintptr_t)compact) & 31) != 0) return -3;
  switch (w) {
    case 1: return launch_gather(FromPlanes<1>{compact, pos, nsel}, S, dst, 0, st);
    case 2: return launch_gather(FromPlanes<2>{compact, pos, nsel}, S, dst, 0, st);
    case 4: return launch_gather(FromPlanes<4>{compact, pos, nsel}, S, dst, 0, st);
    case 8: return launch_gather(FromPlanes<8>{compact, pos, nsel}, S, dst, 0, st);
  }
  return -1;
}

int k_roi_gather_codes(const uint8_t* compact, const uint32_t* pos, const uint16_t* lut_dev, const RoiSelections& S, uint16_t* dst,
                       cudaStream_t st) {
  if ((((uintptr_t)compact) & 15) != 0) return -3;
  return launch_gather(FromCodes{compact, pos, lut_dev}, S, dst, 256 * sizeof(uint16_t), st);
}

int k_roi_crop(int elem, const void* vol, uint64_t n, const RoiSelections& S, void* dst, cudaStream_t st) {
  if ((((uintptr_t)vol) & 15) != 0) return -3;
  if (elem == 2)
    return launch_gather(FromVolume<uint16_t>{static_cast<const uint16_t*>(vol), n}, S, static_cast<uint16_t*>(dst), 0, st);
  if (elem == 1)
    return launch_gather(FromVolume<uint8_t>{static_cast<const uint8_t*>(vol), n}, S, static_cast<uint8_t*>(dst), 0, st);
  return -1;
}

RoiBatch roi_batch(RoiSource source, const RoiRuns* R, size_t n, RoiSel* sels) {
  static_assert(FromPlanes<1>::G == FromVolume<uint16_t>::G && FromPlanes<1>::G == FromVolume<uint8_t>::G, "one group size");
  const int G = source == kRoiCodes ? FromCodes::G : FromPlanes<1>::G;
  RoiBatch B{};
  for (size_t i = 0; i < n; ++i)
    if (R[i].rows && R[i].len) B.count[roi_program(R[i], G)]++;
  B.begin[kRoiGroup] = B.count[kRoiRun];
  B.begin[kRoiVoxel] = B.begin[kRoiGroup] + B.count[kRoiGroup];
  uint32_t at[3] = {B.begin[0], B.begin[1], B.begin[2]};
  uint64_t first = 0;
  for (size_t i = 0; i < n; ++i) {
    const uint64_t voxels = R[i].rows * R[i].len;
    if (voxels) {
      const int p = roi_program(R[i], G);
      sels[at[p]++] = RoiSel{R[i], first, B.items[p]};
      B.items[p] += R[i].rows * (p == kRoiVoxel ? R[i].len : roi_groups(R[i], G));
    }
    first += voxels;
  }
  return B;
}

}  // namespace sqyb
