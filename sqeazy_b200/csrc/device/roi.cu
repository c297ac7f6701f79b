// Sub-volume gather (api.cu: the sqyx_decode_roi_* entry points): the voxels of a box of a stack, densely in C order, out of
//   planes: the compact 16 KiB blocks of the bit planes of a uint16 bitswapW that hold the box (k_lz4_decode_list, or a
//           sub-frame decoded whole), transposed back by the thread program of bitswap_thread.h;
//   codes:  the compact 16 KiB blocks of 8-bit quantiser codes that hold the box, through the 256-entry decode LUT;
//   raw:    a whole decoded stack (the crop behind the decode-whole route).
// One kernel, templated on the source. A thread takes one aligned group of G voxels of the stack (32, or 16 codes: one 16-byte
// load) that meets a row run and writes the voxels of the group that lie in the run to their dense place in the box: whole
// groups with 16-byte stores where the destination allows it, the groups at the ends of a run voxel by voxel.
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
};

// items = R.rows * groups: item (r, q) is the q-th group that meets run r (groups = the most a run of R.len voxels meets)
template <class Src>
__global__ void __launch_bounds__(kRoiThreads) roi_gather_kernel(Src src, RoiRuns R, uint64_t groups, typename Src::T* __restrict__ dst) {
  using T = typename Src::T;
  constexpr int G = Src::G;
  constexpr int kPer = 4 / sizeof(T);
  src.prologue();
  const uint64_t items = R.rows * groups;
  for (uint64_t it = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; it < items; it += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t r = it / groups, v0 = R.start(r), v1 = v0 + R.len;
    const uint64_t g = v0 / G + (it - r * groups);
    if (g * G >= v1) continue;
    uint32_t L[Src::kWords];
    src.load(g, L);
    T* out = dst + r * R.len;   // voxel v of the run lands at out[v - v0]
    if (g * G >= v0 && (g + 1) * G <= v1 && (((uintptr_t)(out + (g * G - v0))) & 15) == 0) {
      uint4* o = reinterpret_cast<uint4*>(out + (g * G - v0));
#pragma unroll
      for (uint32_t i = 0; i < Src::kWords / 4; ++i) o[i] = make_uint4(L[4 * i], L[4 * i + 1], L[4 * i + 2], L[4 * i + 3]);
      continue;
    }
#pragma unroll
    for (int k = 0; k < G; ++k) {
      const uint64_t v = g * G + k;
      if (v >= v0 && v < v1) out[v - v0] = (T)(L[k / kPer] >> (8 * sizeof(T) * (k % kPer)));
    }
  }
}

template <class Src>
int launch_gather(const Src& src, const RoiRuns& R, typename Src::T* dst, size_t smem, cudaStream_t st) {
  if (R.rows == 0 || R.len == 0) return 0;
  const uint64_t groups = (R.len + Src::G - 1) / Src::G + 1;
  roi_gather_kernel<Src><<<grid_for(R.rows * groups, kRoiThreads), kRoiThreads, smem, st>>>(src, R, groups, dst);
  SQYB_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

}  // namespace

int k_roi_gather_planes(int w, const uint8_t* compact, const uint32_t* pos, uint64_t nsel, const RoiRuns& R, uint16_t* dst,
                        cudaStream_t st) {
  if ((((uintptr_t)compact) & 31) != 0) return -3;
  switch (w) {
    case 1: return launch_gather(FromPlanes<1>{compact, pos, nsel}, R, dst, 0, st);
    case 2: return launch_gather(FromPlanes<2>{compact, pos, nsel}, R, dst, 0, st);
    case 4: return launch_gather(FromPlanes<4>{compact, pos, nsel}, R, dst, 0, st);
    case 8: return launch_gather(FromPlanes<8>{compact, pos, nsel}, R, dst, 0, st);
  }
  return -1;
}

int k_roi_gather_codes(const uint8_t* compact, const uint32_t* pos, const uint16_t* lut_dev, const RoiRuns& R, uint16_t* dst,
                       cudaStream_t st) {
  if ((((uintptr_t)compact) & 15) != 0) return -3;
  return launch_gather(FromCodes{compact, pos, lut_dev}, R, dst, 256 * sizeof(uint16_t), st);
}

int k_roi_crop(int elem, const void* vol, uint64_t n, const RoiRuns& R, void* dst, cudaStream_t st) {
  if ((((uintptr_t)vol) & 15) != 0) return -3;
  if (elem == 2)
    return launch_gather(FromVolume<uint16_t>{static_cast<const uint16_t*>(vol), n}, R, static_cast<uint16_t*>(dst), 0, st);
  if (elem == 1)
    return launch_gather(FromVolume<uint8_t>{static_cast<const uint8_t*>(vol), n}, R, static_cast<uint8_t*>(dst), 0, st);
  return -1;
}

}  // namespace sqyb
