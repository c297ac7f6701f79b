/* sqeazy_b200 device-pointer extension of the sqeazy C API (new; not in the reference).
 *
 * The reference's boundary (include/sqeazy.h) takes HOST buffers, so every call pays two PCIe
 * crossings. These entry points take DEVICE pointers and a CUDA stream handle (cudaStream_t passed
 * as void*; NULL = legacy default stream) so that callers holding data in HBM — and the roofline
 * measurements in bench.py — reach the same kernels without the copies. Plain C ABI: pointers and
 * sizes only. The SQY_* host entry points are thin wrappers over these.
 *
 * Return value: 0 on success, non-zero on failure (same convention as sqeazy.h).
 * All functions synchronise `stream` before returning unless stated otherwise.
 */
#ifndef SQEAZY_B200_EXT_H
#define SQEAZY_B200_EXT_H

#ifdef __cplusplus
extern "C" {
#endif

/* ---- whole pipelines (replace dynamic_pipeline::encode/decode, dynamic_pipeline.hpp:560-690,740-846) ---- */

/* d_src: shape-product uint16 voxels in device memory. d_dst: device buffer of dst_capacity bytes
 * (>= SQY_Pipeline_Max_Compressed_Length_UI16). Writes [header][payload]; *dst_bytes = blob bytes. */
int sqyx_encode_device_UI16(const char* pipeline, const void* d_src, const long* shape, unsigned shape_size, void* d_dst,
                            long dst_capacity, long* dst_bytes, void* stream);

/* as above; d_global_hist (device, 65536 x uint32) replaces the local histogram of a `quantiser` stage.
 * Multi-GPU: every rank fills its histogram with sqyx_histogram_UI16, all-reduces it (NCCL, sum) and
 * passes the result here, so all ranks derive the identical LUT. NULL = histogram d_src locally. */
int sqyx_encode_device_ex_UI16(const char* pipeline, const void* d_src, const long* shape, unsigned shape_size, void* d_dst,
                               long dst_capacity, long* dst_bytes, const void* d_global_hist, void* stream);

/* d_blob: [header][payload] in device memory; d_dst: device buffer of dst_capacity bytes (>= raw bytes). */
int sqyx_decode_device_UI16(const void* d_blob, long blob_bytes, void* d_dst, long dst_capacity, void* stream);

/* ---- sub-volumes: a box of a stack, decoded from the LZ4 blocks that hold it ----
 * box: 2*ndims longs {lo_0, hi_0, lo_1, hi_1, ...}, half-open, in the order SQY_Decompressed_Shape reports (C order: the last
 * dimension is contiguous in the stack); ndims must equal the blob's. The box's voxels are written densely in C order:
 * prod(hi_k - lo_k) * sizeof(voxel) bytes at dst, nothing past them. An empty box (some hi_k == lo_k) returns 0 and writes
 * nothing. 3 = box malformed or outside the shape (lo_k > hi_k, hi_k > shape_k, ndims mismatch), 1 = dst_capacity too small or
 * any other failure, 11 / 101 = a broken LZ4 block the box needs (the codes of the whole-stack decode).
 * Routes: the whole stack is the ordinary decode. Blobs of `[filters ->] bitswapW -> lz4` (uint16) and `quantiser -> lz4` whose
 * payload is one frame of this library in full 16 KiB blocks (N a multiple of 8192 * 16/W voxels, or of 16384) decode only the
 * blocks that hold the box; every other blob is decoded whole and cropped. The calls run on the calling thread's device, also
 * when a device set is configured (sqyx_set_devices). */
int sqyx_decode_roi_device_UI16(const void* d_blob, long blob_bytes, const long* box, unsigned ndims, void* d_dst, long dst_capacity,
                                void* stream);
int sqyx_decode_roi_device_UI8(const void* d_blob, long blob_bytes, const long* box, unsigned ndims, void* d_dst, long dst_capacity,
                               void* stream);
/* host buffers (the blob and dst in host memory, pageable or pinned; nthreads as for SQY_Decode_UI16). Only the header, the index
 * frame and the compressed bytes of the blocks the box needs go to the device when the blob takes the indexed route. */
int sqyx_decode_roi_UI16(const char* src, long srclength, const long* box, unsigned ndims, char* dst, long dst_capacity, int nthreads);
int sqyx_decode_roi_UI8(const char* src, long srclength, const long* box, unsigned ndims, char* dst, long dst_capacity, int nthreads);
/* strided slices: slices holds 3*ndims longs {lo_0, hi_0, step_0, lo_1, hi_1, step_1, ...}, half-open, step_k >= 1, in the order
 * SQY_Decompressed_Shape reports; the slice takes ceil((hi_k - lo_k) / step_k) voxels of dimension k (numpy's lo:hi:step) and
 * writes them densely in C order, nothing past them. Return codes and routes as for the boxes above, with 3 also for a step < 1;
 * the indexed route decodes only the blocks that hold a selected voxel. An all-steps-1 slice is the box; a slice of every voxel
 * is the ordinary decode, a whole range with a step is not. */
int sqyx_decode_slice_device_UI16(const void* d_blob, long blob_bytes, const long* slices, unsigned ndims, void* d_dst,
                                  long dst_capacity, void* stream);
int sqyx_decode_slice_device_UI8(const void* d_blob, long blob_bytes, const long* slices, unsigned ndims, void* d_dst,
                                 long dst_capacity, void* stream);
int sqyx_decode_slice_UI16(const char* src, long srclength, const long* slices, unsigned ndims, char* dst, long dst_capacity,
                           int nthreads);
int sqyx_decode_slice_UI8(const char* src, long srclength, const long* slices, unsigned ndims, char* dst, long dst_capacity,
                          int nthreads);
/* many strided slices of one stack in one call: slices holds nsel * ndims * 3 longs, selection i's {lo_0, hi_0, step_0, lo_1, ...}
 * at slices + 3 * ndims * i (a box is step 1). The selections are written densely in C order, one after the other with no gaps:
 * selection i starts sizeof(voxel) * (voxels of selections 0 .. i-1) bytes into dst. Nothing is written past the last one.
 * Selections may overlap, repeat or be empty; an empty one writes nothing and takes no space. Return codes as for one slice, with
 * 3 also for nsel == 0 or nsel > 65536; every selection is checked before anything is decoded, so a refused call writes nothing.
 * The indexed route plans the union of the selections' blocks once: one block table, one decode of the union (each block once;
 * the host calls send the union in one copy), one gather launch per thread program the selections take (7 launches for a batch
 * of boxes, at most 9). Every other blob is decoded whole once and every selection cropped out of it. A batch never takes
 * route 0; a batch of empty selections reports route -1. */
int sqyx_decode_slice_batch_device_UI16(const void* d_blob, long blob_bytes, const long* slices, unsigned nsel, unsigned ndims,
                                        void* d_dst, long dst_capacity, void* stream);
int sqyx_decode_slice_batch_device_UI8(const void* d_blob, long blob_bytes, const long* slices, unsigned nsel, unsigned ndims,
                                       void* d_dst, long dst_capacity, void* stream);
int sqyx_decode_slice_batch_UI16(const char* src, long srclength, const long* slices, unsigned nsel, unsigned ndims, char* dst,
                                 long dst_capacity, int nthreads);
int sqyx_decode_slice_batch_UI8(const char* src, long srclength, const long* slices, unsigned nsel, unsigned ndims, char* dst,
                                long dst_capacity, int nthreads);
/* out4 = {route of the most recent ROI, slice or slice-batch call on this thread's device (0 = box is the whole stack: the ordinary
 * decode, 1 = indexed, 2 = decode whole + crop, -1 = an empty box: nothing decoded), LZ4 blocks decoded by the indexed route (0 on
 * the others; a batch counts each block of the union once), bytes sent host->device (0 for device calls; the blob's payload on
 * routes 0 and 2), voxels written (a batch: summed over its selections)}.
 * Route 0 of a host call is SQY_Decode_UI16 / _UI8 itself: like them it may stream the stack slab by slab or shard it over a
 * configured device set, and its byte count is then the payload the GPUs received together, not one device's share. */
int sqyx_last_roi_info(long* out4);

/* ---- batches of independent stacks: a time-lapse or a set of stacks (BASELINE cfg4, cfg5; the reference loops over files,
 * src/cpp/src/verbs/compress.hpp:204-338, one stack after the other). Up to 8 stacks are in flight on streams and scratch
 * of their own, so the block decoders / encoders of different stacks share the SMs (a single stack of few large LZ4
 * blocks is bound by the serial chain of its slowest block). All stacks of an encode batch share pipeline and shape.
 * rcs (may be NULL) receives the per-stack return codes; the call returns 0 when all of them are 0. Synchronous. */
int sqyx_decode_batch_device_UI16(int n, const void* const* d_blobs, const long* blob_bytes, void* const* d_dsts,
                                  const long* dst_capacities, int* rcs);
int sqyx_encode_batch_device_UI16(int n, const char* pipeline, const void* const* d_srcs, const long* shape, unsigned shape_size,
                                  void* const* d_dsts, const long* dst_capacities, long* dst_bytes, int* rcs);

/* ---- single stages (what the parity tests drive) ---- */

/* bitswapN, w in {1,2,4,8}; threshold > 0 fuses remove_background(threshold) into the load.
 * reference: encoders/bitswap_scheme_impl.hpp:97-197 */
int sqyx_bitswap_encode_UI16(int w, const void* d_src, void* d_dst, long n, int threshold, void* stream);
int sqyx_bitswap_decode_UI16(int w, const void* d_src, void* d_dst, long n, void* stream);

/* bitshuffle head filter (SURVEY §8f-4): the blocked bit transpose of the bitshuffle library that
 * encoders/bitshuffle_scheme_impl.hpp:91-160 calls (bshuf_bitshuffle / bshuf_bitunshuffle, element size 2).
 * block_size in elements, 0 = the library's default (4096 for uint16); must be a multiple of 8. */
int sqyx_bitshuffle_encode_UI16(const void* d_src, void* d_dst, long n, long block_size, void* stream);
int sqyx_bitshuffle_decode_UI16(const void* d_src, void* d_dst, long n, long block_size, void* stream);
/* the same for uint8 stacks (element size 1: 8 bit rows per block, default block 8192 elements) */
int sqyx_bitshuffle_encode_UI8(const void* d_src, void* d_dst, long n, long block_size, void* stream);
int sqyx_bitshuffle_decode_UI8(const void* d_src, void* d_dst, long n, long block_size, void* stream);

/* diff3x3x1 head filter (SURVEY §8f-4), reference: encoders/diff_scheme_impl.hpp:78-199 with last_plane_neighborhood<3>
 * (neighborhood_utils.hpp:72-92, :186-226; diff_scheme_utils.hpp:75-103): voxel minus (sum of the 3x3 voxels around it in
 * the previous z plane, wrapped in the voxel type) / 9 on the rows the reference visits; decode = the inverse recurrence
 * along z. Device buffers of z*y*x voxels (C order), d_src != d_dst, sizeof_voxel 1 or 2. Returns 2 for a shape on which
 * the reference's own loops leave the plane or the buffer, or an extent exceeds the int16 / int8 coordinates the reference
 * keeps for uint16 / uint8 stacks (32767 / 128) (sqyx_diff_shape_supported tells), 1 for any other failure. */
int sqyx_diff_device(int decode, int sizeof_voxel, const void* d_src, void* d_dst, long z, long y, long x, void* stream);
int sqyx_diff_shape_supported(int sizeof_voxel, long z, long y, long x);

/* out = in > t ? in - t : 0. reference: encoders/remove_background_scheme_impl.hpp:73-95 */
int sqyx_remove_background_UI16(const void* d_src, void* d_dst, long n, int threshold, void* stream);

/* rmestbkrd threshold: four 99 % supports (z=0 face, z=Z-1 face, rows y=0 / y=Y-1 at z in {1,Z/2,Z-2}) and
 * threshold = (uint16)min. l2_bytes < 0 = use this host's L2 size the way the reference does (SQY_L2_BYTES
 * overrides). reference: encoders/background_scheme_utils.hpp:35-105, remove_estimated_background_scheme_impl.hpp:71-112 */
int sqyx_estimate_background_UI16(const void* d_src, const long* shape3, long l2_bytes, float* supports4, int* threshold,
                                  void* stream);

/* host-side pieces of the threshold estimate, for callers that histogram the sampled faces/rows themselves (z-slabs
 * spread over several GPUs: partial histograms are summed with an all-reduce, then every rank evaluates the support):
 * calc_support(threshold) of a 65536-bin histogram (hist_impl.hpp:63-84,359-381) and the number of leading frame
 * elements the reference samples (background_scheme_utils.hpp:44-45; l2_bytes < 0 = this host's L2). */
float sqyx_histogram_support(const unsigned* hist, float threshold);
long sqyx_rmest_frame_portion(long frame_elems, long l2_bytes);

/* 65536-bin uint32 histogram, ACCUMULATED into d_hist (zero it first). Does not synchronise.
 * reference: encoders/histogram_utils.hpp:41-55,98-154 */
int sqyx_histogram_UI16(const void* d_src, long n, void* d_hist, void* stream);

/* host-side LUT construction from a histogram (host pointers): enc 65536 x u8, dec 256 x u16.
 * reference: encoders/quantiser_utils.hpp:227-306,386-418 */
int sqyx_quantiser_luts(const unsigned* hist, unsigned char* enc, unsigned short* dec);

/* LUT gathers; the tables are HOST pointers (copied to the device inside).
 * reference: encoders/quantiser_scheme_impl.hpp:206-223 (apply), :245-282 (decode) */
int sqyx_lut_apply_UI16(const void* d_src, void* d_codes, long n, const unsigned char* enc_host, void* stream);
int sqyx_lut_decode_UI16(const void* d_codes, void* d_dst, long n, const unsigned short* dec_host, void* stream);

/* LZ4 frames. sqyx_lz4_bound(n) = capacity the encoder may need for n input bytes.
 * reference: encoders/lz4.hpp:214-242 (encode), :257-339 (decode), :166-188 (bound) */
long sqyx_lz4_bound(long nbytes);
int sqyx_lz4_encode(const void* d_src, long nbytes, void* d_dst, long dst_capacity, long* payload_bytes, void* stream);
/* pitch_bytes: distance in the stream between vertically adjacent voxels (a row of a bit plane of 2048-voxel rows: 256),
 * offered to the match finder as a fixed offset beside 1; must be a multiple of 32, 0 = none. The pipelines pass
 * X * w / 8 (bit planes) or X (8-bit codes). Output bytes are a pure function of (input, pitch_bytes).
 * SQYX_LZ4_HINT_NO_NOISE OR-ed into pitch_bytes: the stream is expected to hold no incompressible 16 KiB blocks (bit planes
 * behind a background removal, as the pipelines pass it): a few per cent faster on such streams, slower on noise, and never a
 * different byte. */
#define SQYX_LZ4_HINT_NO_NOISE 0x80000000L
int sqyx_lz4_encode_ex(const void* d_src, long nbytes, void* d_dst, long dst_capacity, long* payload_bytes, long pitch_bytes, void* stream);
int sqyx_lz4_decode(const void* d_src, long nbytes, void* d_dst, long dst_bytes, long* decoded_bytes, void* stream);

/* ---- uint8 volumes (the *_UI8 entry points of sqeazy.h on device pointers) ----
 * pipelines: bitswap1|2|4, remove_background(threshold=N) (alias rmbkrd) -> lz4 | pass_through [-> lz4]
 * reference: src/sqeazy.cpp:72-106 (encode), :309-335 (decode); encoders/bitplane_reorder_scalar.hpp:27-116 with
 * raw_type = uint8_t; encoders/remove_background_scheme_impl.hpp:73-95 */
int sqyx_encode_device_UI8(const char* pipeline, const void* d_src, const long* shape, unsigned shape_size, void* d_dst,
                           long dst_capacity, long* dst_bytes, void* stream);
int sqyx_decode_device_UI8(const void* d_blob, long blob_bytes, void* d_dst, long dst_capacity, void* stream);
int sqyx_bitswap_encode_UI8(int w, const void* d_src, void* d_dst, long n, int threshold, void* stream);
int sqyx_bitswap_decode_UI8(int w, const void* d_src, void* d_dst, long n, void* stream);
int sqyx_remove_background_UI8(const void* d_src, void* d_dst, long n, int threshold, void* stream);

/* ---- bookkeeping ---- */
int sqyx_device_count(void);
/* makes `device` current for the calling thread inside this library's CUDA runtime instance (one process
 * per GPU callers set it once; all sqyx_ and SQY_ calls then use that device) */
int sqyx_set_device(int device);
/* Multi-GPU inside ONE call (SURVEY 8e). The host-buffer entry points of sqeazy.h (SQY_PipelineEncode_UI16 /
 * SQY_Decode_UI16; reference: src/cpp/src/sqeazy.cpp:108-142, 281-307) shard one stack of
 * `[remove_background | rmestbkrd ->] bitswapN -> lz4` or `quantiser -> lz4` over a set of GPUs: contiguous z-slabs
 * (boundaries at multiples of 131072 voxels, >= 128 MiB of LZ4 input per GPU), every GPU fed over its own PCIe link,
 * ONE blob out — byte-identical to the single-GPU blob. The quantiser's 65536-bin histogram is summed with
 * ncclAllReduce (libnccl.so.2 bound at run time; SQY_NO_NCCL=1 or no NCCL: summed on the host).
 * The set: sqyx_set_devices(n, ids) (n = 0: back to the default), else the environment variable SQY_CUDA_DEVICES
 * ("all" or "0,1,2"), else SQY_CUDA_DEVICE, else every visible device. sqyx_set_device(d) pins all calls to d. */
int sqyx_set_devices(int n, const int* devices);
/* out3 = {GPUs the most recent SQY_ host call was sharded over (0: single-device route), 1 if its histogram all-reduce went
 * through NCCL, number of (plane, GPU) pieces merged} */
int sqyx_last_shard_info(long* out3);
/* cumulative number of in-library NCCL histogram all-reduces */
long sqyx_nccl_allreduces(void);
/* cumulative number of CUDA kernels launched by this library in this process */
long sqyx_kernel_launches(void);
/* block statistics of the most recent LZ4 encode on this thread's device:
 * out[0] general-path blocks, out[1] constant (closed-form) blocks, out[2] stored blocks, out[3] payload bytes */
int sqyx_last_lz4_stats(long* out4);
/* per-stage device time (CUDA events on the caller's stream, accumulated over calls while enabled):
 * out7 = {filter+bitswap encode, lz4 encode, histogram, LUT apply, lz4 decode, LUT decode, bitswap decode} in ms.
 * Enabling adds an event synchronisation per stage; leave it off for throughput runs. */
int sqyx_enable_stage_timing(int on);
int sqyx_stage_ms(float* out7, int reset);
/* value of compass-style L2 probe used by rmestbkrd on this host */
long sqyx_host_l2_bytes(void);
/* block-LINKED LZ4 frames (the reference's serial mode, the sqy CLI default): streams with at least `nblocks` linked blocks
 * are decoded with deferred cross-block references (all blocks at once; default 8), smaller ones block after block.
 * 0 = never defer, < 0 = query. Returns the previous value. */
long sqyx_set_lz4_defer_min(long nblocks);
/* releases the cached device scratch of the current device */
int sqyx_release_scratch(void);

#ifdef __cplusplus
}
#endif
#endif
