"""sqeazy_b200 — B200-native sqeazy volume pipeline (bitswapN, remove_background/rmestbkrd, quantiser, LZ4).

This package is a thin ctypes mirror of the C ABI in include/sqeazy.h (the reference's boundary,
src/cpp/inc/sqeazy.h) and include/sqeazy_b200.h (device-pointer extension). All compute happens in
the hand-written sm_100a kernels inside sqeazy_b200/libsqeazy.so; there is no Python or CPU
fallback: if the shared library is missing, importing `lib()` raises.

Host-buffer calls (numpy) map 1:1 to SQY_*; device-buffer calls (torch CUDA tensors) map to sqyx_*.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_bool, c_char_p, c_float, c_int, c_long, c_uint, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsqeazy.so")

# every symbol declared in include/sqeazy.h and include/sqeazy_b200.h
SQY_SYMBOLS = [
    "SQY_Header_Size", "SQY_Decompressed_NDims", "SQY_Decompressed_Shape", "SQY_Decompressed_Sizeof",
    "SQY_Decompressed_Length", "SQY_Version_Triple", "SQY_PipelineEncode_UI16", "SQY_PipelineEncode_UI8",
    "SQY_Pipeline_Max_Compressed_Length_UI16", "SQY_Pipeline_Max_Compressed_Length_UI8",
    "SQY_Pipeline_Max_Compressed_Length_3D_UI16", "SQY_Pipeline_Max_Compressed_Length_3D_UI8",
    "SQY_Pipeline_Possible_UI16", "SQY_Pipeline_Possible_UI8", "SQY_Pipeline_Possible", "SQY_Decode_UI16",
    "SQY_PipelineDecode_UI16", "SQY_Decode_UI8", "SQY_h5_query_sizeof", "SQY_h5_query_dtype", "SQY_h5_query_ndims",
    "SQY_h5_query_shape", "SQY_h5_read_UI16", "SQY_h5_write_UI16", "SQY_h5_write", "SQY_h5_link",
]
SQYX_SYMBOLS = [
    "sqyx_encode_device_UI16", "sqyx_encode_device_ex_UI16", "sqyx_decode_device_UI16", "sqyx_bitswap_encode_UI16",
    "sqyx_bitswap_decode_UI16", "sqyx_remove_background_UI16", "sqyx_estimate_background_UI16", "sqyx_histogram_UI16",
    "sqyx_quantiser_luts", "sqyx_lut_apply_UI16", "sqyx_lut_decode_UI16", "sqyx_lz4_bound", "sqyx_lz4_encode",
    "sqyx_lz4_decode", "sqyx_device_count", "sqyx_kernel_launches", "sqyx_last_lz4_stats", "sqyx_host_l2_bytes",
    "sqyx_release_scratch", "sqyx_set_device", "sqyx_enable_stage_timing", "sqyx_stage_ms", "sqyx_histogram_support",
    "sqyx_rmest_frame_portion", "sqyx_encode_device_UI8", "sqyx_decode_device_UI8", "sqyx_bitswap_encode_UI8",
    "sqyx_bitswap_decode_UI8", "sqyx_remove_background_UI8", "sqyx_decode_batch_device_UI16", "sqyx_encode_batch_device_UI16",
    "sqyx_bitshuffle_encode_UI16", "sqyx_bitshuffle_decode_UI16", "sqyx_bitshuffle_encode_UI8", "sqyx_bitshuffle_decode_UI8", "sqyx_set_lz4_defer_min",
    "sqyx_diff_device", "sqyx_diff_shape_supported", "sqyx_set_devices", "sqyx_last_shard_info", "sqyx_nccl_allreduces", "sqyx_lz4_encode_ex",
    "sqyx_decode_roi_device_UI16", "sqyx_decode_roi_device_UI8", "sqyx_decode_roi_UI16", "sqyx_decode_roi_UI8", "sqyx_last_roi_info",
    "sqyx_decode_slice_device_UI16", "sqyx_decode_slice_device_UI8", "sqyx_decode_slice_UI16", "sqyx_decode_slice_UI8",
    "sqyx_decode_slice_batch_device_UI16", "sqyx_decode_slice_batch_device_UI8", "sqyx_decode_slice_batch_UI16",
    "sqyx_decode_slice_batch_UI8",
]

# include/sqeazy_h5_filter.h: what HDF5 looks up in a filter plugin
H5_SYMBOLS = ["H5Z_filter_sqy", "H5PLget_plugin_type", "H5PLget_plugin_info"]

_lib = None


def lib() -> ctypes.CDLL:
    """Loads libsqeazy.so (built by `make` / __graft_entry__.build()). Fails loudly when absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: run `make` (or __graft_entry__.build()). sqeazy_b200 has no fallback path.")
        L = ctypes.CDLL(LIB_PATH)
        L.SQY_Pipeline_Possible_UI16.restype = c_bool
        L.SQY_Pipeline_Possible_UI8.restype = c_bool
        L.SQY_Pipeline_Possible.restype = c_bool
        for name in ("sqyx_lz4_bound", "sqyx_kernel_launches", "sqyx_host_l2_bytes", "sqyx_rmest_frame_portion", "sqyx_nccl_allreduces"):
            getattr(L, name).restype = c_long
        L.sqyx_histogram_support.restype = c_float
        L.sqyx_histogram_support.argtypes = [c_void_p, c_float]
        _lib = L
    return _lib


class SqeazyError(RuntimeError):
    pass


def _vp(a: np.ndarray):
    return a.ctypes.data_as(c_void_p)


# ------------------------------------------------------------------------------------------------
# SQY_* : host buffers (numpy)
# ------------------------------------------------------------------------------------------------
def pipeline_possible(pipeline: str, sizeof_pixel: int = 2) -> bool:
    return bool(lib().SQY_Pipeline_Possible(pipeline.encode("latin-1"), c_int(sizeof_pixel)))


def max_compressed_length(pipeline: str, raw_bytes: int) -> int:
    p = pipeline.encode("latin-1")
    n = c_long(raw_bytes)
    if lib().SQY_Pipeline_Max_Compressed_Length_UI16(p, c_long(len(p)), ctypes.byref(n)) != 0:
        raise SqeazyError(f"invalid pipeline {pipeline!r}")
    return n.value


def max_compressed_length_3d(pipeline: str, shape) -> int:
    p = pipeline.encode("latin-1")
    shp = (c_long * len(shape))(*shape)
    n = c_long(len(p))
    if lib().SQY_Pipeline_Max_Compressed_Length_3D_UI16(p, shp, c_uint(len(shape)), ctypes.byref(n)) != 0:
        raise SqeazyError(f"invalid pipeline {pipeline!r}")
    return n.value


def _check_out(out: np.ndarray, dtype, need_bytes: int, what: str):
    """a caller-supplied destination goes to the C API as a bare pointer: refuse anything it could overrun"""
    if not isinstance(out, np.ndarray) or out.dtype != np.dtype(dtype) or not out.flags["C_CONTIGUOUS"] or not out.flags["WRITEABLE"]:
        raise SqeazyError(f"{what}: `out` must be a writeable C-contiguous {np.dtype(dtype).name} array")
    if out.nbytes < need_bytes:
        raise SqeazyError(f"{what}: `out` holds {out.nbytes} bytes, {need_bytes} are needed")


def encode(pipeline: str, volume: np.ndarray, nthreads: int = 1, out: np.ndarray | None = None) -> np.ndarray:
    """SQY_PipelineEncode_UI16: uint16 volume (any rank, C order) -> blob bytes (uint8 array)."""
    vol = np.ascontiguousarray(volume, dtype=np.uint16)
    cap = max_compressed_length(pipeline, vol.nbytes)
    if out is None:
        out = np.empty(cap, dtype=np.uint8)
    _check_out(out, np.uint8, cap, "encode")
    shp = (c_long * vol.ndim)(*vol.shape)
    n = c_long(0)
    rc = lib().SQY_PipelineEncode_UI16(pipeline.encode("latin-1"), _vp(vol), shp, c_uint(vol.ndim), _vp(out), ctypes.byref(n),
                                       c_int(nthreads))
    if rc != 0:
        raise SqeazyError(f"SQY_PipelineEncode_UI16({pipeline!r}) returned {rc}")
    return out[: n.value]


def max_compressed_length_u8(pipeline: str, raw_bytes: int) -> int:
    p = pipeline.encode("latin-1")
    n = c_long(raw_bytes)
    if lib().SQY_Pipeline_Max_Compressed_Length_UI8(p, c_long(len(p)), ctypes.byref(n)) != 0:
        raise SqeazyError(f"invalid uint8 pipeline {pipeline!r}")
    return n.value


def max_compressed_length_3d_u8(pipeline: str, shape) -> int:
    p = pipeline.encode("latin-1")
    shp = (c_long * len(shape))(*shape)
    n = c_long(len(p))
    if lib().SQY_Pipeline_Max_Compressed_Length_3D_UI8(p, shp, c_uint(len(shape)), ctypes.byref(n)) != 0:
        raise SqeazyError(f"invalid uint8 pipeline {pipeline!r}")
    return n.value


def encode_u8(pipeline: str, volume: np.ndarray, nthreads: int = 1) -> np.ndarray:
    """SQY_PipelineEncode_UI8: uint8 volume (any rank, C order) -> blob bytes (uint8 array)."""
    vol = np.ascontiguousarray(volume, dtype=np.uint8)
    out = np.empty(max_compressed_length_u8(pipeline, vol.nbytes), dtype=np.uint8)
    shp = (c_long * vol.ndim)(*vol.shape)
    n = c_long(0)
    rc = lib().SQY_PipelineEncode_UI8(pipeline.encode("latin-1"), _vp(vol), shp, c_uint(vol.ndim), _vp(out), ctypes.byref(n),
                                      c_int(nthreads))
    if rc != 0:
        raise SqeazyError(f"SQY_PipelineEncode_UI8({pipeline!r}) returned {rc}")
    return out[: n.value]


def decode_u8(blob: np.ndarray, nthreads: int = 1) -> np.ndarray:
    """SQY_Decode_UI8: blob -> uint8 volume of the shape stored in the header."""
    blob = np.ascontiguousarray(blob, dtype=np.uint8)
    shape = decompressed_shape(blob)
    out = np.empty(decompressed_length(blob), dtype=np.uint8)
    rc = lib().SQY_Decode_UI8(_vp(blob), c_long(blob.size), _vp(out), c_int(nthreads))
    if rc != 0:
        raise SqeazyError(f"SQY_Decode_UI8 returned {rc}")
    return out.reshape(shape) if shape else out


def header_size(blob: np.ndarray) -> int:
    n = c_long(blob.size)
    lib().SQY_Header_Size(_vp(blob), ctypes.byref(n))
    return n.value


def decompressed_shape(blob: np.ndarray):
    nd = c_long(blob.size)
    lib().SQY_Decompressed_NDims(_vp(blob), ctypes.byref(nd))
    shp = (c_long * max(nd.value, 1))()
    shp[0] = blob.size
    lib().SQY_Decompressed_Shape(_vp(blob), shp)
    return tuple(shp[i] for i in range(nd.value))


def decompressed_length(blob: np.ndarray) -> int:
    n = c_long(blob.size)
    lib().SQY_Decompressed_Length(_vp(blob), ctypes.byref(n))
    return n.value


def decompressed_sizeof(blob: np.ndarray) -> int:
    n = c_long(blob.size)
    lib().SQY_Decompressed_Sizeof(_vp(blob), ctypes.byref(n))
    return n.value


def version_triple():
    v = (c_int * 3)()
    lib().SQY_Version_Triple(v)
    return tuple(v)


def decode(blob: np.ndarray, nthreads: int = 1, out: np.ndarray | None = None) -> np.ndarray:
    """SQY_Decode_UI16: blob -> uint16 volume of the shape stored in the header."""
    blob = np.ascontiguousarray(blob, dtype=np.uint8)
    shape = decompressed_shape(blob)
    nbytes = decompressed_length(blob)
    if out is None:
        out = np.empty(nbytes // 2, dtype=np.uint16)
    _check_out(out, np.uint16, nbytes, "decode")
    rc = lib().SQY_Decode_UI16(_vp(blob), c_long(blob.size), _vp(out), c_int(nthreads))
    if rc != 0:
        raise SqeazyError(f"SQY_Decode_UI16 returned {rc}")
    return out.reshape(shape) if shape else out


def _roi_box(box):
    """box: one (lo, hi) pair or (lo, hi, step) triple per dimension of the stack -> (the C array of 2 * ndims longs, or of
    3 * ndims when any triple is given, ndims, the selection's shape: ceil((hi - lo) / step) per dimension, whether it is
    strided). A selection that the library refuses (3) is passed on as it is."""
    tuples = [tuple(int(v) for v in t) for t in box]
    strided = any(len(t) == 3 for t in tuples)
    if strided:
        tuples = [t if len(t) == 3 else (*t, 1) for t in tuples]
    arr = (c_long * max(sum(len(t) for t in tuples), 1))(*[v for t in tuples for v in t])
    step = [t[2] if strided else 1 for t in tuples]
    shape = tuple(max(-(-(t[1] - t[0]) // s), 0) if s > 0 else 0 for t, s in zip(tuples, step))
    return arr, len(tuples), shape, strided


def _decode_roi(fns, names, dtype, blob, box, nthreads, out):
    blob = np.ascontiguousarray(blob, dtype=np.uint8)
    arr, nd, shape, strided = _roi_box(box)
    fn, name = fns[strided], names[strided]
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    if out is None:
        out = np.empty(shape, dtype=dtype)
    _check_out(out, dtype, nbytes, name)
    rc = fn(_vp(blob), c_long(blob.size), arr, c_uint(nd), _vp(out), c_long(out.nbytes), c_int(nthreads))
    if rc != 0:
        raise SqeazyError(f"{name} returned {rc}")
    return out


def decode_roi(blob: np.ndarray, box, nthreads: int = 1, out: np.ndarray | None = None) -> np.ndarray:
    """sqyx_decode_roi_UI16: the box [(lo, hi), ...] (half-open, one pair per dimension of the stack) of a uint16 blob, as an
    array of the box's shape. Only the blocks that hold the box cross the bus when the blob allows it (last_roi_info).
    With any (lo, hi, step) triple among the pairs it is the strided slice lo:hi:step (sqyx_decode_slice_UI16; a pair is step 1),
    as an array of the slice's shape, ceil((hi - lo) / step) per dimension."""
    L = lib()
    return _decode_roi((L.sqyx_decode_roi_UI16, L.sqyx_decode_slice_UI16), ("sqyx_decode_roi_UI16", "sqyx_decode_slice_UI16"),
                       np.uint16, blob, box, nthreads, out)


def decode_roi_u8(blob: np.ndarray, box, nthreads: int = 1, out: np.ndarray | None = None) -> np.ndarray:
    """sqyx_decode_roi_UI8 / sqyx_decode_slice_UI8: the same for uint8 stacks"""
    L = lib()
    return _decode_roi((L.sqyx_decode_roi_UI8, L.sqyx_decode_slice_UI8), ("sqyx_decode_roi_UI8", "sqyx_decode_slice_UI8"),
                       np.uint8, blob, box, nthreads, out)


def _roi_batch(sels):
    """sels: selections in the form decode_roi takes -> (the C array of nsel * ndims * 3 longs, nsel, ndims, the selections'
    shapes). Every selection must have as many dimensions as the first; the library checks that number against the stack."""
    triples = [[(int(t[0]), int(t[1]), int(t[2]) if len(t) == 3 else 1) for t in sel] for sel in sels]
    nd = len(triples[0]) if triples else 0
    if any(len(sel) != nd for sel in triples):
        raise SqeazyError("decode_roi_batch: the selections differ in their number of dimensions")
    flat = [v for sel in triples for t in sel for v in t]
    shapes = [_roi_box(sel)[2] for sel in triples]
    return (c_long * max(len(flat), 1))(*flat), len(triples), nd, shapes


def _views(flat, shapes):
    """the selections' arrays (or tensors), one after the other in the packed buffer `flat`"""
    out, at = [], 0
    for shape in shapes:
        n = int(np.prod(shape))
        out.append(flat[at : at + n].reshape(shape))
        at += n
    return out


def _decode_roi_batch(fn, name, dtype, blob, sels, nthreads, out):
    blob = np.ascontiguousarray(blob, dtype=np.uint8)
    arr, nsel, nd, shapes = _roi_batch(sels)
    total = sum(int(np.prod(s)) for s in shapes)
    if out is None:
        out = np.empty(total, dtype=dtype)
    _check_out(out, dtype, total * np.dtype(dtype).itemsize, name)
    rc = fn(_vp(blob), c_long(blob.size), arr, c_uint(nsel), c_uint(nd), _vp(out), c_long(out.nbytes), c_int(nthreads))
    if rc != 0:
        raise SqeazyError(f"{name} returned {rc}")
    return _views(out.reshape(-1), shapes)


def decode_roi_batch(blob: np.ndarray, sels, nthreads: int = 1, out: np.ndarray | None = None) -> list:
    """sqyx_decode_slice_batch_UI16: many selections of one uint16 blob in one call, each a list of (lo, hi) pairs or (lo, hi, step)
    triples as decode_roi takes them (a pair is step 1). Every LZ4 block that they need is decoded once. Returns one array per
    selection, in its own shape; all of them are views into one packed buffer (`out`, if given: room for the voxels of every
    selection), the selections one after the other in C order."""
    return _decode_roi_batch(lib().sqyx_decode_slice_batch_UI16, "sqyx_decode_slice_batch_UI16", np.uint16, blob, sels, nthreads, out)


def decode_roi_batch_u8(blob: np.ndarray, sels, nthreads: int = 1, out: np.ndarray | None = None) -> list:
    """sqyx_decode_slice_batch_UI8: the same for uint8 stacks"""
    return _decode_roi_batch(lib().sqyx_decode_slice_batch_UI8, "sqyx_decode_slice_batch_UI8", np.uint8, blob, sels, nthreads, out)


def last_roi_info():
    """the most recent sub-volume decode on this thread's device: route (0 = the whole stack, 1 = indexed, 2 = decoded whole and
    cropped, -1 = empty box), LZ4 blocks the indexed route decoded, bytes sent host -> device, voxels written"""
    o = (c_long * 4)()
    if lib().sqyx_last_roi_info(o) != 0:
        raise SqeazyError("sqyx_last_roi_info failed")
    return {"route": int(o[0]), "blocks": int(o[1]), "h2d_bytes": int(o[2]), "voxels": int(o[3])}


# ------------------------------------------------------------------------------------------------
# sqyx_* : device buffers (torch CUDA tensors). torch is plumbing only: memory, streams, distributed.
# ------------------------------------------------------------------------------------------------
def _stream_handle(stream=None):
    import torch
    s = stream if stream is not None else torch.cuda.current_stream()
    return c_void_p(s.cuda_stream)


def _dp(t):
    return c_void_p(t.data_ptr())


def set_device(index: int):
    """binds the library's CUDA runtime to `index` for this thread (torch.cuda.set_device does not reach it)"""
    if lib().sqyx_set_device(c_int(index)) != 0:
        raise SqeazyError(f"sqyx_set_device({index}) failed")


def set_devices(indices=None):
    """GPUs over which the host-buffer calls (`encode` / `decode`) may shard ONE stack (z-slabs, one blob). None or [] = the
    default again: SQY_CUDA_DEVICES, else every visible device. `set_device(i)` pins the calls to GPU i."""
    ids = list(indices or [])
    arr = (c_int * max(len(ids), 1))(*ids)
    if lib().sqyx_set_devices(c_int(len(ids)), arr) != 0:
        raise SqeazyError(f"sqyx_set_devices({ids}) failed")


def last_shard_info():
    """how the most recent host-buffer call on this process was spread: GPUs used (0 = single-device route), whether the
    histogram all-reduce went through NCCL, number of (plane, GPU) pieces merged"""
    out = (c_long * 3)()
    lib().sqyx_last_shard_info(out)
    return {"gpus": int(out[0]), "nccl": bool(out[1]), "pieces": int(out[2])}


def nccl_allreduces() -> int:
    """cumulative number of in-library NCCL histogram all-reduces"""
    return int(lib().sqyx_nccl_allreduces())


def encode_device(pipeline: str, volume, out=None, global_hist=None, stream=None):
    """sqyx_encode_device[_ex]_UI16. volume: CUDA tensor of 16-bit voxels (any rank); returns a uint8 CUDA view of the blob."""
    import torch
    assert volume.is_cuda and volume.element_size() == 2 and volume.is_contiguous()
    cap = max_compressed_length(pipeline, volume.numel() * 2)
    if out is None or out.numel() < cap:
        out = torch.empty(cap, dtype=torch.uint8, device=volume.device)
    shp = (c_long * volume.dim())(*volume.shape)
    n = c_long(0)
    gh = _dp(global_hist) if global_hist is not None else c_void_p(0)
    with torch.cuda.device(volume.device):
        rc = lib().sqyx_encode_device_ex_UI16(pipeline.encode("latin-1"), _dp(volume), shp, c_uint(volume.dim()), _dp(out),
                                              c_long(out.numel()), ctypes.byref(n), gh, _stream_handle(stream))
    if rc != 0:
        raise SqeazyError(f"sqyx_encode_device_UI16({pipeline!r}) returned {rc}")
    return out[: n.value]


def decode_device(blob, out, stream=None):
    """sqyx_decode_device_UI16. blob: uint8 CUDA tensor; out: CUDA tensor with room for the raw volume."""
    import torch
    assert blob.is_cuda and out.is_cuda and blob.is_contiguous() and out.is_contiguous()
    with torch.cuda.device(blob.device):
        rc = lib().sqyx_decode_device_UI16(_dp(blob), c_long(blob.numel()), _dp(out), c_long(out.numel() * out.element_size()),
                                           _stream_handle(stream))
    if rc != 0:
        raise SqeazyError(f"sqyx_decode_device_UI16 returned {rc}")
    return out


def _decode_roi_device(fns, names, blob, box, out, stream):
    import torch
    assert blob.is_cuda and out.is_cuda and blob.is_contiguous() and out.is_contiguous()
    arr, nd, _, strided = _roi_box(box)
    fn, name = fns[strided], names[strided]
    with torch.cuda.device(blob.device):
        rc = fn(_dp(blob), c_long(blob.numel()), arr, c_uint(nd), _dp(out), c_long(out.numel() * out.element_size()), _stream_handle(stream))
    if rc != 0:
        raise SqeazyError(f"{name} returned {rc}")
    return out


def decode_roi_device(blob, box, out, stream=None):
    """sqyx_decode_roi_device_UI16. blob: uint8 CUDA tensor; box: (lo, hi) pairs; out: CUDA tensor with room for the box's
    voxels, written densely in C order. With any (lo, hi, step) triple among the pairs: sqyx_decode_slice_device_UI16, the
    strided slice's voxels"""
    L = lib()
    return _decode_roi_device((L.sqyx_decode_roi_device_UI16, L.sqyx_decode_slice_device_UI16),
                              ("sqyx_decode_roi_device_UI16", "sqyx_decode_slice_device_UI16"), blob, box, out, stream)


def decode_roi_device_u8(blob, box, out, stream=None):
    L = lib()
    return _decode_roi_device((L.sqyx_decode_roi_device_UI8, L.sqyx_decode_slice_device_UI8),
                              ("sqyx_decode_roi_device_UI8", "sqyx_decode_slice_device_UI8"), blob, box, out, stream)


def _decode_roi_batch_device(fn, name, blob, sels, out, stream):
    import torch
    assert blob.is_cuda and out.is_cuda and blob.is_contiguous() and out.is_contiguous()
    arr, nsel, nd, shapes = _roi_batch(sels)
    with torch.cuda.device(blob.device):
        rc = fn(_dp(blob), c_long(blob.numel()), arr, c_uint(nsel), c_uint(nd), _dp(out), c_long(out.numel() * out.element_size()),
                _stream_handle(stream))
    if rc != 0:
        raise SqeazyError(f"{name} returned {rc}")
    return _views(out.view(-1), shapes)


def decode_roi_batch_device(blob, sels, out, stream=None):
    """sqyx_decode_slice_batch_device_UI16. blob: uint8 CUDA tensor; sels: selections as decode_roi_batch takes them; out: CUDA
    tensor with room for the voxels of every selection, written one after the other. Returns one view of `out` per selection, in
    its shape. For K patches of one shape, out.view(K, *shape) is the batch."""
    return _decode_roi_batch_device(lib().sqyx_decode_slice_batch_device_UI16, "sqyx_decode_slice_batch_device_UI16", blob, sels, out,
                                    stream)


def decode_roi_batch_device_u8(blob, sels, out, stream=None):
    return _decode_roi_batch_device(lib().sqyx_decode_slice_batch_device_UI8, "sqyx_decode_slice_batch_device_UI8", blob, sels, out,
                                    stream)


def decode_batch_device(blobs, outs):
    """sqyx_decode_batch_device_UI16: a batch of independent stacks (time-lapse, cfg4) decoded concurrently, up to 8 in
    flight on streams and scratch of their own. blobs / outs: lists of CUDA tensors. Synchronous."""
    import torch
    n = len(blobs)
    assert n == len(outs) and all(b.is_cuda and b.is_contiguous() for b in blobs) and all(o.is_cuda and o.is_contiguous() for o in outs)
    torch.cuda.current_stream().synchronize()   # the batch runs on the library's own streams
    bp = (c_void_p * n)(*[b.data_ptr() for b in blobs])
    bn = (c_long * n)(*[b.numel() for b in blobs])
    op = (c_void_p * n)(*[o.data_ptr() for o in outs])
    on = (c_long * n)(*[o.numel() * o.element_size() for o in outs])
    rcs = (c_int * n)()
    rc = lib().sqyx_decode_batch_device_UI16(c_int(n), bp, bn, op, on, rcs)
    if rc != 0:
        raise SqeazyError(f"sqyx_decode_batch_device_UI16 returned {list(rcs)}")
    return outs


def encode_batch_device(pipeline: str, volumes, outs=None):
    """sqyx_encode_batch_device_UI16: stacks of one shape through one pipeline, up to 8 in flight. Returns uint8 CUDA views."""
    import torch
    n = len(volumes)
    if n == 0:
        return []
    v0 = volumes[0]
    assert all(v.is_cuda and v.element_size() == 2 and v.is_contiguous() and v.shape == v0.shape for v in volumes)
    cap = max_compressed_length(pipeline, v0.numel() * 2)
    if outs is None:
        outs = [torch.empty(cap, dtype=torch.uint8, device=v0.device) for _ in range(n)]
    assert len(outs) == n and all(o.numel() >= cap for o in outs)
    torch.cuda.current_stream().synchronize()
    shp = (c_long * v0.dim())(*v0.shape)
    sp = (c_void_p * n)(*[v.data_ptr() for v in volumes])
    op = (c_void_p * n)(*[o.data_ptr() for o in outs])
    on = (c_long * n)(*[o.numel() for o in outs])
    nb = (c_long * n)()
    rcs = (c_int * n)()
    rc = lib().sqyx_encode_batch_device_UI16(c_int(n), pipeline.encode("latin-1"), sp, shp, c_uint(v0.dim()), op, on, nb, rcs)
    if rc != 0:
        raise SqeazyError(f"sqyx_encode_batch_device_UI16({pipeline!r}) returned {list(rcs)}")
    return [o[: nb[i]] for i, o in enumerate(outs)]


def bitswap_encode_device(w: int, src, dst, threshold: int = 0, stream=None):
    rc = lib().sqyx_bitswap_encode_UI16(c_int(w), _dp(src), _dp(dst), c_long(src.numel()), c_int(threshold), _stream_handle(stream))
    if rc != 0:
        raise SqeazyError("sqyx_bitswap_encode_UI16 failed")
    return dst


def bitswap_decode_device(w: int, src, dst, stream=None):
    rc = lib().sqyx_bitswap_decode_UI16(c_int(w), _dp(src), _dp(dst), c_long(src.numel()), _stream_handle(stream))
    if rc != 0:
        raise SqeazyError("sqyx_bitswap_decode_UI16 failed")
    return dst


def bitshuffle_encode_device(src, dst, block_size: int = 0, stream=None):
    """uint16 or uint8 elements by the tensor's element size"""
    fn = lib().sqyx_bitshuffle_encode_UI16 if src.element_size() == 2 else lib().sqyx_bitshuffle_encode_UI8
    rc = fn(_dp(src), _dp(dst), c_long(src.numel()), c_long(block_size), _stream_handle(stream))
    if rc != 0:
        raise SqeazyError("sqyx_bitshuffle_encode_UI16 failed")
    return dst


def bitshuffle_decode_device(src, dst, block_size: int = 0, stream=None):
    fn = lib().sqyx_bitshuffle_decode_UI16 if src.element_size() == 2 else lib().sqyx_bitshuffle_decode_UI8
    rc = fn(_dp(src), _dp(dst), c_long(src.numel()), c_long(block_size), _stream_handle(stream))
    if rc != 0:
        raise SqeazyError("sqyx_bitshuffle_decode_UI16 failed")
    return dst


def diff_device(src, dst, decode: bool = False, stream=None):
    """diff3x3x1 (encoders/diff_scheme_impl.hpp:78-199) of a rank-3 uint16 / uint8 device tensor into `dst` (another buffer)"""
    if src.dim() != 3:
        raise SqeazyError("diff3x3x1 needs a rank-3 stack")
    z, y, x = (int(v) for v in src.shape)
    rc = lib().sqyx_diff_device(c_int(1 if decode else 0), c_int(src.element_size()), _dp(src), _dp(dst), c_long(z), c_long(y),
                                c_long(x), _stream_handle(stream))
    if rc != 0:
        raise SqeazyError(f"sqyx_diff_device failed ({rc}: {'shape not supported' if rc == 2 else 'error'})")
    return dst


def diff_shape_supported(z: int, y: int, x: int, sizeof_voxel: int = 2) -> bool:
    return bool(lib().sqyx_diff_shape_supported(c_int(sizeof_voxel), c_long(z), c_long(y), c_long(x)))


H5Z_FILTER_SQY = 0o1307            # sqeazy_h5_filter.hpp:211 writes the id as the octal literal 01307 = 711
H5Z_FLAG_REVERSE = 0x0100


class H5ZClass2(ctypes.Structure):
    """H5Z_class2_t as H5PLget_plugin_info() returns it (include/sqeazy_h5_filter.h)"""
    _fields_ = [("version", c_int), ("id", c_int), ("encoder_present", c_uint), ("decoder_present", c_uint), ("name", c_char_p),
                ("can_apply", c_void_p), ("set_local", c_void_p), ("filter", c_void_p)]


def h5_plugin_info() -> H5ZClass2:
    L = lib()
    L.H5PLget_plugin_info.restype = POINTER(H5ZClass2)
    return L.H5PLget_plugin_info().contents


def h5_filter(chunk: np.ndarray, cd_header: bytes = b"", reverse: bool = False):
    """Calls H5Z_filter_sqy the way HDF5 does: the chunk lives in a malloc()ed buffer that the filter replaces.
    cd_header = the sqeazy header text the dataset was created with (hdf5_utils.hpp:728-737 packs it into cd_values).
    Returns the new chunk as a uint8 array, or None when the filter reports failure (returns 0)."""
    L = lib()
    libc = ctypes.CDLL(None)
    libc.malloc.restype = c_void_p
    libc.malloc.argtypes = [ctypes.c_size_t]
    libc.free.argtypes = [c_void_p]
    L.H5Z_filter_sqy.restype = ctypes.c_size_t
    L.H5Z_filter_sqy.argtypes = [c_uint, ctypes.c_size_t, c_void_p, ctypes.c_size_t, POINTER(ctypes.c_size_t), POINTER(c_void_p)]
    raw = np.ascontiguousarray(chunk).view(np.uint8).ravel()
    buf = c_void_p(libc.malloc(max(raw.size, 1)))
    ctypes.memmove(buf, raw.ctypes.data, raw.size)
    size = ctypes.c_size_t(raw.size)
    cd = np.zeros((len(cd_header) + 3) // 4, dtype=np.uint32)
    cd.view(np.uint8)[: len(cd_header)] = np.frombuffer(cd_header, dtype=np.uint8)
    n = L.H5Z_filter_sqy(c_uint(H5Z_FLAG_REVERSE if reverse else 0), cd.size, cd.ctypes.data_as(c_void_p) if cd.size else None,
                         raw.size, ctypes.byref(size), ctypes.byref(buf))
    out = None
    if n:
        assert size.value == n
        out = np.ctypeslib.as_array(ctypes.cast(buf, POINTER(ctypes.c_uint8)), shape=(n,)).copy()
    libc.free(buf)
    return out


def remove_background_device(src, dst, threshold: int, stream=None):
    rc = lib().sqyx_remove_background_UI16(_dp(src), _dp(dst), c_long(src.numel()), c_int(threshold), _stream_handle(stream))
    if rc != 0:
        raise SqeazyError("sqyx_remove_background_UI16 failed")
    return dst


def encode_device_u8(pipeline: str, volume, out=None, stream=None):
    """sqyx_encode_device_UI8. volume: CUDA tensor of 8-bit voxels (any rank); returns a uint8 CUDA view of the blob."""
    import torch
    assert volume.is_cuda and volume.element_size() == 1 and volume.is_contiguous()
    cap = max_compressed_length_u8(pipeline, volume.numel())
    if out is None or out.numel() < cap:
        out = torch.empty(cap, dtype=torch.uint8, device=volume.device)
    shp = (c_long * volume.dim())(*volume.shape)
    n = c_long(0)
    with torch.cuda.device(volume.device):
        rc = lib().sqyx_encode_device_UI8(pipeline.encode("latin-1"), _dp(volume), shp, c_uint(volume.dim()), _dp(out),
                                          c_long(out.numel()), ctypes.byref(n), _stream_handle(stream))
    if rc != 0:
        raise SqeazyError(f"sqyx_encode_device_UI8({pipeline!r}) returned {rc}")
    return out[: n.value]


def decode_device_u8(blob, out, stream=None):
    import torch
    assert blob.is_cuda and out.is_cuda and blob.is_contiguous() and out.is_contiguous()
    with torch.cuda.device(blob.device):
        rc = lib().sqyx_decode_device_UI8(_dp(blob), c_long(blob.numel()), _dp(out), c_long(out.numel() * out.element_size()),
                                          _stream_handle(stream))
    if rc != 0:
        raise SqeazyError(f"sqyx_decode_device_UI8 returned {rc}")
    return out


def bitswap_encode_device_u8(w: int, src, dst, threshold: int = 0, stream=None):
    rc = lib().sqyx_bitswap_encode_UI8(c_int(w), _dp(src), _dp(dst), c_long(src.numel()), c_int(threshold), _stream_handle(stream))
    if rc != 0:
        raise SqeazyError("sqyx_bitswap_encode_UI8 failed")
    return dst


def bitswap_decode_device_u8(w: int, src, dst, stream=None):
    rc = lib().sqyx_bitswap_decode_UI8(c_int(w), _dp(src), _dp(dst), c_long(src.numel()), _stream_handle(stream))
    if rc != 0:
        raise SqeazyError("sqyx_bitswap_decode_UI8 failed")
    return dst


def remove_background_device_u8(src, dst, threshold: int, stream=None):
    rc = lib().sqyx_remove_background_UI8(_dp(src), _dp(dst), c_long(src.numel()), c_int(threshold), _stream_handle(stream))
    if rc != 0:
        raise SqeazyError("sqyx_remove_background_UI8 failed")
    return dst


def estimate_background_device(volume, l2_bytes: int = -1, stream=None):
    """returns (supports[4] float32, threshold) of rmestbkrd for a rank-3 CUDA volume"""
    shp = (c_long * 3)(*volume.shape)
    sup = (c_float * 4)()
    t = c_int(0)
    rc = lib().sqyx_estimate_background_UI16(_dp(volume), shp, c_long(l2_bytes), sup, ctypes.byref(t), _stream_handle(stream))
    if rc != 0:
        raise SqeazyError("sqyx_estimate_background_UI16 failed")
    return np.array(list(sup), dtype=np.float32), t.value


def histogram_device(src, hist, stream=None):
    """accumulates the 65536-bin histogram of src into hist (int32/uint32 CUDA tensor of 65536); asynchronous"""
    rc = lib().sqyx_histogram_UI16(_dp(src), c_long(src.numel()), _dp(hist), _stream_handle(stream))
    if rc != 0:
        raise SqeazyError("sqyx_histogram_UI16 failed")
    return hist


def quantiser_luts(hist: np.ndarray):
    hist = np.ascontiguousarray(hist, dtype=np.uint32)
    enc = np.zeros(65536, dtype=np.uint8)
    dec = np.zeros(256, dtype=np.uint16)
    if lib().sqyx_quantiser_luts(_vp(hist), _vp(enc), _vp(dec)) != 0:
        raise SqeazyError("sqyx_quantiser_luts failed")
    return enc, dec


def histogram_support(hist: np.ndarray, threshold: float = 0.99) -> float:
    hist = np.ascontiguousarray(hist, dtype=np.uint32)
    return float(lib().sqyx_histogram_support(_vp(hist), c_float(threshold)))


def rmest_frame_portion(frame_elems: int, l2_bytes: int = -1) -> int:
    return int(lib().sqyx_rmest_frame_portion(c_long(frame_elems), c_long(l2_bytes)))


def lut_apply_device(src, codes, enc: np.ndarray, stream=None):
    enc = np.ascontiguousarray(enc, dtype=np.uint8)
    rc = lib().sqyx_lut_apply_UI16(_dp(src), _dp(codes), c_long(src.numel()), _vp(enc), _stream_handle(stream))
    if rc != 0:
        raise SqeazyError("sqyx_lut_apply_UI16 failed")
    return codes


def lut_decode_device(codes, dst, dec: np.ndarray, stream=None):
    dec = np.ascontiguousarray(dec, dtype=np.uint16)
    rc = lib().sqyx_lut_decode_UI16(_dp(codes), _dp(dst), c_long(codes.numel()), _vp(dec), _stream_handle(stream))
    if rc != 0:
        raise SqeazyError("sqyx_lut_decode_UI16 failed")
    return dst


def lz4_bound(nbytes: int) -> int:
    return int(lib().sqyx_lz4_bound(c_long(nbytes)))


def lz4_encode_device(src, out=None, stream=None, pitch: int = 0):
    """src: CUDA tensor (any dtype, contiguous) -> uint8 CUDA view of the LZ4 frame stream. pitch: bytes between vertically
    adjacent voxels in the stream (multiple of 32; 0 = no hint), see sqyx_lz4_encode_ex"""
    import torch
    nbytes = src.numel() * src.element_size()
    cap = lz4_bound(nbytes)
    if out is None or out.numel() < cap:
        out = torch.empty(cap, dtype=torch.uint8, device=src.device)
    n = c_long(0)
    rc = lib().sqyx_lz4_encode_ex(_dp(src), c_long(nbytes), _dp(out), c_long(out.numel()), ctypes.byref(n), c_long(pitch), _stream_handle(stream))
    if rc != 0:
        raise SqeazyError("sqyx_lz4_encode failed")
    return out[: n.value]


def lz4_decode_device(payload, out, stream=None):
    """payload: uint8 CUDA tensor of LZ4 frames; out: CUDA tensor receiving the decoded bytes. Returns decoded byte count."""
    n = c_long(0)
    rc = lib().sqyx_lz4_decode(_dp(payload), c_long(payload.numel()), _dp(out), c_long(out.numel() * out.element_size()),
                               ctypes.byref(n), _stream_handle(stream))
    if rc != 0:
        raise SqeazyError("sqyx_lz4_decode failed")
    return n.value


def kernel_launches() -> int:
    return int(lib().sqyx_kernel_launches())


def last_lz4_stats():
    o = (c_long * 4)()
    lib().sqyx_last_lz4_stats(o)
    return {"general_blocks": o[0], "constant_blocks": o[1], "stored_blocks": o[2], "payload_bytes": o[3]}


def set_lz4_defer_min(nblocks: int) -> int:
    """linked blocks from which a stream takes the deferred-reference decoder (default 8, 0 = never); returns the previous value"""
    f = lib().sqyx_set_lz4_defer_min
    f.restype = c_long
    return f(c_long(nblocks))


def host_l2_bytes() -> int:
    return int(lib().sqyx_host_l2_bytes())


STAGE_NAMES = ("filter_bitswap_encode", "lz4_encode", "histogram", "lut_apply", "lz4_decode", "lut_decode", "bitswap_decode")


def release_scratch():
    """frees the library's cached device scratch on the current device"""
    lib().sqyx_release_scratch()


def enable_stage_timing(on: bool = True):
    lib().sqyx_enable_stage_timing(c_int(1 if on else 0))


def stage_ms(reset: bool = True):
    """accumulated device milliseconds per stage since the last reset (needs enable_stage_timing(True))"""
    o = (c_float * 7)()
    lib().sqyx_stage_ms(o, c_int(1 if reset else 0))
    return dict(zip(STAGE_NAMES, [float(v) for v in o]))
