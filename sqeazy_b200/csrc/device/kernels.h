// Internal launch interface of the sm_100a kernels (device pointers, explicit stream).
// Every function enqueues work on `st` and returns 0 or a cudaError_t / negative library code.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <atomic>

namespace sqyb {

// cumulative count of kernels launched by this library (reported as gpu_launches by bench.py)
extern std::atomic<long> g_kernel_launches;
#define SQYB_COUNT_LAUNCH(n) ::sqyb::g_kernel_launches.fetch_add((n), std::memory_order_relaxed)

// The head stages take elem = bytes per voxel: 1 (uint8 volumes, the *_UI8 entry points) or 2 (uint16).
// bitswap.cu: w = 1, 2, 4 (uint8) or 1, 2, 4, 8 (uint16); the threshold is taken as a voxel value
int k_bitswap_encode(int elem, int w, const void* in, void* out, uint64_t n, int threshold, cudaStream_t st);
int k_bitswap_decode(int elem, int w, const void* in, void* out, uint64_t n, cudaStream_t st);
int k_remove_background(int elem, const void* in, void* out, uint64_t n, int threshold, cudaStream_t st);
// uint16 only: voxels [first, first+count) of an n-voxel volume (in/out = whole-volume base pointers; multiples of 128 voxels): lets the
// host entry points transpose a z-slab as soon as it has arrived / ship a slab as soon as it is transposed back
int k_bitswap_encode_range(int w, const uint16_t* in, uint16_t* out, uint64_t n, uint64_t first, uint64_t count, int threshold,
                           cudaStream_t st);
int k_bitswap_decode_range(int w, const uint16_t* in, uint16_t* out, uint64_t n, uint64_t first, uint64_t count, cudaStream_t st);

// bitshuffle.cu: the bitshuffle library's blocked bit transpose (encoders/bitshuffle_scheme_impl.hpp:91-160).
// block_size in elements, 0 = the library's default (4096 for uint16, 8192 for uint8); -81 (the library's own code) when it
// is not a multiple of 8
int k_bitshuffle_encode(int elem, const void* in, void* out, uint64_t n, uint32_t block_size, cudaStream_t st);
int k_bitshuffle_decode(int elem, const void* in, void* out, uint64_t n, uint32_t block_size, cudaStream_t st);
uint32_t bitshuffle_block_elems(uint32_t block_size, int elem_size);

// diff.cu: diff3x3x1 (encoders/diff_scheme_impl.hpp:78-199); in != out; 1 = shape refused
bool diff_shape_supported(uint64_t Z, uint64_t Y, uint64_t X, int elem);
int k_diff_encode(int elem, const void* in, void* out, uint64_t Z, uint64_t Y, uint64_t X, cudaStream_t st);
int k_diff_decode(int elem, const void* in, void* out, uint64_t Z, uint64_t Y, uint64_t X, cudaStream_t st);

// quantise.cu
int k_histogram_u16(const uint16_t* in, uint64_t n, uint32_t* hist /* 65536 x u32, accumulated into */, cudaStream_t st);
// per histogram h: out[4h] = first bin whose cumulative share exceeds `threshold` (65536: none), out[4h+1] = bins[m],
// out[4h+2] = bins[m-1] (hist_impl.hpp:63-84,359-381)
int k_support_index(const uint32_t* hist_dev, int nhist, float threshold, uint32_t* out_dev, cudaStream_t st);
int k_lut_apply(const uint16_t* in, uint8_t* out, uint64_t n, const uint8_t* lut_dev /* 65536 */, cudaStream_t st);
int k_lut_decode(const uint8_t* in, uint16_t* out, uint64_t n, const uint16_t* lut_dev /* 256 */, cudaStream_t st);

// lz4_encode.cu
size_t k_lz4_encode_workspace_bytes(uint64_t raw_bytes);
// workspace[0..8) receives the payload size (u64) when the stream has drained; [16,28) block-kind counters
// pitch_bytes: distance in the stream between vertically adjacent voxels (a row of a bit plane: X * w / 8 bytes; a row of
// 8-bit codes: X bytes), tried as a fixed match offset like offset 1; 0 (or not a multiple of 32): none. The
// compressed bytes are a pure function of (input bytes, pitch_bytes).
// kLz4HintNoNoise OR-ed into pitch_bytes: the caller expects no incompressible blocks (bit planes behind a background
// removal). It changes only the order of work inside a block — without it twelve of a block's sixteen warps wait until four
// sampled ones have settled whether the block is noise and is stored as it is, which is what makes noise cheap (8-bit
// quantiser codes, the low planes of an unfiltered stack) and costs a compressible block a few per cent — never a byte.
constexpr uint32_t kLz4HintNoNoise = 0x80000000u;
int k_lz4_encode(const uint8_t* src, uint64_t raw_bytes, uint8_t* dst, void* workspace, uint32_t pitch_bytes, cudaStream_t st);
// the same in three steps, for input that becomes available piece by piece: begin (frame prefix), any number of block
// sets — `nsets` sets of `count` consecutive 16 KiB blocks, set j starting at block first + j * set_stride (the pieces of
// the 16/w bit planes that one z-slab contributes) —, end (offsets + compaction). Every block exactly once.
int k_lz4_encode_begin(uint64_t raw_bytes, uint8_t* dst, void* workspace, cudaStream_t st);
int k_lz4_encode_blocks(const uint8_t* src, uint64_t raw_bytes, uint8_t* dst, void* workspace, uint32_t first, uint32_t count,
                        uint32_t nsets, uint32_t set_stride, uint32_t pitch_bytes, cudaStream_t st);
int k_lz4_encode_end(const uint8_t* src, uint64_t raw_bytes, uint8_t* dst, void* workspace, cudaStream_t st);

// lz4_decode.cu
size_t k_lz4_decode_workspace_bytes(uint64_t dst_bytes);
// A decode in two steps, so that callers can take the blocks of one z-slab at a time (the host entry points ship a slab while
// the next one is decoded): the block table, then any number of block-set launches over it (count == 0: the whole stream).
// allow_deferred: streams with many block-LINKED blocks (the reference's serial mode) only get their block table here; their
// blocks are decoded by k_lz4_decode_linked (deferred cross-block references) once the caller has seen deferred_blocks > 0
// in the status and provided the origin buffer.
int k_lz4_decode_tables(const uint8_t* src, uint64_t src_bytes, uint64_t dst_bytes, void* workspace, int measure_all, int allow_deferred,
                        cudaStream_t st);
int k_lz4_decode_run(const uint8_t* src, uint64_t src_bytes, uint8_t* dst, uint64_t dst_bytes, void* workspace, uint32_t first,
                     uint32_t count, uint32_t nsets, uint32_t set_stride, uint32_t slot, cudaStream_t st);
// whether the table k_lz4_decode_tables left in `workspace` describes one frame of this library whose 16 KiB blocks hold exactly
// dst_bytes: the geometry that the slab-by-slab host decode and the fused decoder rely on. Synchronises `st`.
int k_lz4_decode_own_frame(void* workspace, uint64_t dst_bytes, bool* own_frame, cudaStream_t st);
// the block-decode launch for a stream that k_lz4_decode_own_frame found to be one frame of this library with
// 16 KiB blocks that hold the bit planes of a uint16 bitswap`w` (w = 1, 2, 4, 8; plane_bytes = the volume's bytes, a multiple
// of 16 KiB * 16/w): the planes are decoded into `planes` and transposed back into `vox` (32-byte aligned, plane_bytes / 2
// voxels) by the same launch. Always the 48-register build of the decoder: the caller takes this route for stacks of 1 GiB and more
int k_lz4_decode_fused(const uint8_t* src, uint64_t src_bytes, uint8_t* planes, uint64_t plane_bytes, void* workspace, int w,
                       uint16_t* vox, cudaStream_t st);
size_t k_lz4_decode_linked_workspace_bytes(uint64_t dst_bytes);
int k_lz4_decode_linked(const uint8_t* src, uint64_t src_bytes, uint8_t* dst, uint64_t dst_bytes, void* workspace, void* origins,
                        cudaStream_t st);
// linked blocks from which a stream takes the deferred-reference path (default 8, 0 = never); returns the previous value
long k_lz4_set_defer_min(long nblocks);
int k_lz4_decode_status(void* workspace, uint32_t* error, uint64_t* total_decoded, uint32_t* deferred_blocks, cudaStream_t st);
// the blocks a list names, d_list[0 .. nlist) (indices into the table k_lz4_decode_tables built for stream_bytes decoded bytes; a
// stream that k_lz4_decode_own_frame found to be one frame of this library): block d_list[t] is decoded into compact + t * 16 KiB.
// Afterwards the status holds the bytes of the listed blocks that decoded as total_decoded.
int k_lz4_decode_list(const uint8_t* src, uint64_t src_bytes, uint64_t stream_bytes, uint8_t* compact, void* workspace,
                      const uint32_t* d_list, uint32_t nlist, cudaStream_t st);

// roi.cu: the voxels of a strided slice of a stack (a box when every step is 1), written densely in C order. The slice is `rows`
// runs of `len` voxels: run r holds voxels start(r) + j * step (0 <= j < len) of the stack and lands at dst + r * len;
// start(r) = base + sum_k i_k * stride[k], where (i_0 .. i_{nlead-1}) is r in mixed radix over extent[] (the last one fastest).
// Trailing dimensions that the slice spans whole with step 1 are folded into the runs, leading ones of extent 1 into base; a step
// in a leading dimension is part of its stride.
constexpr int kRoiMaxLead = 8;
struct RoiRuns {
  uint64_t base, len, rows, step;
  int nlead;
  uint64_t extent[kRoiMaxLead], stride[kRoiMaxLead];
  __host__ __device__ uint64_t start(uint64_t r) const {
    uint64_t v = base;
    for (int k = nlead - 1; k >= 0; --k) {
      v += (r % extent[k]) * stride[k];
      r /= extent[k];
    }
    return v;
  }
};
// The gathers write one selection, or a batch of them densely one after the other. Each takes one launch per thread program that
// a selection takes (roi.cu). RoiSel describes a non-empty selection of a batch in device memory: its runs, its first voxel in the
// packed destination, and the work items of the selections in front of it in its program's launch.
enum RoiProgram { kRoiRun, kRoiGroup, kRoiVoxel };
struct RoiSel {
  RoiRuns runs;
  uint64_t first, before;
};
// the launches: program p takes descriptors [begin[p], begin[p] + count[p]) and items[p] work items
struct RoiBatch {
  uint32_t begin[3], count[3];
  uint64_t items[3];
};
// the selections of a gather: one selection's runs, passed to the kernel by value (d_sels = nullptr), or a batch's descriptors in
// device memory and their launches (roi_batch)
struct RoiSelections {
  RoiRuns runs;
  const RoiSel* d_sels;
  RoiBatch batch;
};
enum RoiSource { kRoiPlanes, kRoiCodes, kRoiVolume };
// host: the descriptors of selections R[0 .. n) in the order the launches take them, into sels (room for n; an empty selection
// takes no descriptor and no room in the destination), for a gather from `source`
RoiBatch roi_batch(RoiSource source, const RoiRuns* R, size_t n, RoiSel* sels);
// from the compact 16 KiB blocks of the P = 16/w bit planes of a uint16 bitswap`w` that hold the selections: block k of plane
// segment j (the stream's set j) is compact block j * nsel + pos[k] (pos[k] = ~0: not there, never read)
int k_roi_gather_planes(int w, const uint8_t* compact, const uint32_t* pos, uint64_t nsel, const RoiSelections& S, uint16_t* dst,
                        cudaStream_t st);
// from the compact 16 KiB blocks of 8-bit quantiser codes (block k is compact block pos[k]) through the 256-entry decode LUT
int k_roi_gather_codes(const uint8_t* compact, const uint32_t* pos, const uint16_t* lut_dev, const RoiSelections& S, uint16_t* dst,
                       cudaStream_t st);
// from a whole decoded stack of n voxels of elem bytes (the crop)
int k_roi_crop(int elem, const void* vol, uint64_t n, const RoiSelections& S, void* dst, cudaStream_t st);

}  // namespace sqyb
