"""CPU oracle for the sqeazy hot path — TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference leg may import
this module; the product package (sqeazy_b200/) never does.

Two layers:
  * `port`  — oracle/sqy_oracle.c, a plain-C restatement of the reference's algorithms (always
              available; compiled by `make oracle` / __graft_entry__.build()).
  * `ref`   — oracle/_ref/libsqyref.so, the reference's own stage headers compiled from
              /root/reference (only buildable where /root/reference exists; the built .so travels
              to the GPU box). Used to pin the port and as the "reference" CPU baseline.
Pure-Python restatements of the control layer (pipeline grammar, header) live here too:
  string_parsers.hpp:355-395,434-467 ; sqeazy_header.hpp:147-193,295-344 ; dynamic_pipeline.hpp:177-226
"""
from __future__ import annotations

import base64
import ctypes
import os
import re
import subprocess
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_long, c_uint16, c_uint32, c_uint64, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_PORT_SO = os.path.join(_HERE, "_build", "libsqyoracle.so")
_REF_SO = os.path.join(_HERE, "_ref", "libsqyref.so")

VERBATIM_OPEN, VERBATIM_CLOSE = "<verbatim>", "</verbatim>"
HEADER_DELIM = "|01307#!"


def _p(a: np.ndarray):
    return a.ctypes.data_as(c_void_p)


def build_port() -> str:
    if not os.path.exists(_PORT_SO) or os.path.getmtime(_PORT_SO) < os.path.getmtime(os.path.join(_HERE, "sqy_oracle.c")):
        subprocess.check_call(["make", "-C", _ROOT, "oracle/_build/libsqyoracle.so"], stdout=subprocess.DEVNULL)
    return _PORT_SO


class Port:
    """ctypes view of oracle/sqy_oracle.c"""

    def __init__(self):
        self.lib = ctypes.CDLL(build_port())
        L = self.lib
        L.orc_support.restype = c_float
        L.orc_support.argtypes = [c_void_p, c_float]
        L.orc_lz4_frames_encode.restype = ctypes.c_int64
        L.orc_lz4_closest_blocksize_kb.restype = c_uint32
        L.orc_base64_encode.restype = c_uint64

    def bitswap_encode(self, w: int, a: np.ndarray) -> np.ndarray:
        a = np.ascontiguousarray(a, dtype=np.uint16).ravel()
        out = np.empty_like(a)
        assert self.lib.orc_bitswap_encode(c_int(w), _p(a), _p(out), c_uint64(a.size)) == 0
        return out

    def bitswap_decode(self, w: int, a: np.ndarray) -> np.ndarray:
        a = np.ascontiguousarray(a, dtype=np.uint16).ravel()
        out = np.empty_like(a)
        assert self.lib.orc_bitswap_decode(c_int(w), _p(a), _p(out), c_uint64(a.size)) == 0
        return out

    def bitshuffle(self, a: np.ndarray, block_size: int = 0, decode: bool = False) -> np.ndarray:
        """bshuf_bitshuffle / bshuf_bitunshuffle of the third-party bitshuffle library, restated (parity unpinned, see the C file)"""
        a = np.ascontiguousarray(a).ravel()
        out = np.empty_like(a)
        rc = self.lib.orc_bitshuffle(c_int(1 if decode else 0), _p(a), _p(out), c_uint64(a.size), c_uint32(a.itemsize), c_uint32(block_size))
        if rc != 0:
            raise ValueError(f"bitshuffle: error {rc}")
        return out

    def remove_background(self, a: np.ndarray, threshold: int) -> np.ndarray:
        a = np.ascontiguousarray(a, dtype=np.uint16)
        out = np.empty_like(a)
        self.lib.orc_remove_background(_p(a), _p(out), c_uint64(a.size), c_uint16(threshold & 0xFFFF))
        return out

    def bitswap8_encode(self, w: int, a: np.ndarray) -> np.ndarray:
        a = np.ascontiguousarray(a, dtype=np.uint8).ravel()
        out = np.empty_like(a)
        assert self.lib.orc_bitswap8_encode(c_int(w), _p(a), _p(out), c_uint64(a.size)) == 0
        return out

    def bitswap8_decode(self, w: int, a: np.ndarray) -> np.ndarray:
        a = np.ascontiguousarray(a, dtype=np.uint8).ravel()
        out = np.empty_like(a)
        assert self.lib.orc_bitswap8_decode(c_int(w), _p(a), _p(out), c_uint64(a.size)) == 0
        return out

    def remove_background8(self, a: np.ndarray, threshold: int) -> np.ndarray:
        a = np.ascontiguousarray(a, dtype=np.uint8)
        out = np.empty_like(a)
        self.lib.orc_remove_background8(_p(a), _p(out), c_uint64(a.size), ctypes.c_uint8(threshold & 0xFF))
        return out

    def histogram(self, a: np.ndarray) -> np.ndarray:
        a = np.ascontiguousarray(a, dtype=np.uint16)
        h = np.zeros(65536, dtype=np.uint32)
        self.lib.orc_histogram(_p(a), c_uint64(a.size), _p(h))
        return h

    def support(self, bins: np.ndarray, thr: float = 0.99) -> float:
        bins = np.ascontiguousarray(bins, dtype=np.uint32)
        return float(self.lib.orc_support(_p(bins), c_float(thr)))

    def darkest_face_supports(self, vol: np.ndarray, l2_bytes: int) -> np.ndarray:
        vol = np.ascontiguousarray(vol, dtype=np.uint16)
        Z, Y, X = vol.shape
        out = np.zeros(4, dtype=np.float32)
        self.lib.orc_darkest_face_supports(_p(vol), c_uint64(Z), c_uint64(Y), c_uint64(X), c_uint64(l2_bytes), _p(out))
        return out

    def rmestbkrd(self, vol: np.ndarray, l2_bytes: int):
        vol = np.ascontiguousarray(vol, dtype=np.uint16)
        Z, Y, X = vol.shape
        out = np.empty_like(vol)
        t = c_int(0)
        self.lib.orc_rmestbkrd(_p(vol), _p(out), c_uint64(Z), c_uint64(Y), c_uint64(X), c_uint64(l2_bytes), ctypes.byref(t))
        return out, t.value

    def diff_supported(self, shape, elem: int = 2) -> bool:
        Z, Y, X = (int(v) for v in shape)
        return bool(self.lib.orc_diff_supported(c_uint64(Z), c_uint64(Y), c_uint64(X), c_int(elem)))

    def diff(self, vol: np.ndarray, decode: bool = False) -> np.ndarray:
        """diff3x3x1 (encoders/diff_scheme_impl.hpp:78-199), uint16 or uint8 by the array's dtype; ValueError for a refused shape"""
        vol = np.ascontiguousarray(vol)
        assert vol.dtype in (np.uint16, np.uint8) and vol.ndim == 3
        Z, Y, X = vol.shape
        out = np.empty_like(vol)
        rc = self.lib.orc_diff(c_int(1 if decode else 0), _p(vol), _p(out), c_uint64(Z), c_uint64(Y), c_uint64(X), c_int(vol.itemsize))
        if rc != 0:
            raise ValueError(f"diff3x3x1: shape {vol.shape} not supported")
        return out

    def quantiser_luts(self, hist: np.ndarray):
        hist = np.ascontiguousarray(hist, dtype=np.uint32)
        enc = np.zeros(65536, dtype=np.uint8)
        dec = np.zeros(256, dtype=np.uint16)
        self.lib.orc_quantiser_luts(_p(hist), _p(enc), _p(dec))
        return enc, dec

    def lut_apply(self, a: np.ndarray, enc: np.ndarray) -> np.ndarray:
        a = np.ascontiguousarray(a, dtype=np.uint16)
        out = np.empty(a.shape, dtype=np.uint8)
        self.lib.orc_lut_apply(_p(a), _p(out), c_uint64(a.size), _p(np.ascontiguousarray(enc, dtype=np.uint8)))
        return out

    def lut_decode(self, codes: np.ndarray, dec: np.ndarray) -> np.ndarray:
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        out = np.empty(codes.shape, dtype=np.uint16)
        self.lib.orc_lut_decode(_p(codes), _p(out), c_uint64(codes.size), _p(np.ascontiguousarray(dec, dtype=np.uint16)))
        return out

    def lz4_frames_decode(self, payload: np.ndarray, raw_bytes: int) -> np.ndarray:
        payload = np.ascontiguousarray(payload, dtype=np.uint8)
        out = np.zeros(raw_bytes, dtype=np.uint8)
        got = c_uint64(0)
        rc = self.lib.orc_lz4_frames_decode(_p(payload), c_uint64(payload.size), _p(out), c_uint64(raw_bytes), ctypes.byref(got))
        if rc != 0:
            raise ValueError("oracle: invalid LZ4 frame stream")
        return out[: got.value]

    def lz4_frames_encode(self, raw: np.ndarray, chunk: int = 262144) -> np.ndarray:
        raw = np.ascontiguousarray(raw).view(np.uint8).ravel()
        cap = raw.size + raw.size // 200 + 64 * (raw.size // max(chunk, 1) + 2) + 64
        out = np.zeros(cap, dtype=np.uint8)
        n = self.lib.orc_lz4_frames_encode(_p(raw), c_uint64(raw.size), _p(out), c_uint64(cap), c_uint64(chunk))
        assert n >= 0
        return out[:n].copy()

    def closest_blocksize_kb(self, kb: int) -> int:
        return int(self.lib.orc_lz4_closest_blocksize_kb(c_uint32(kb)))


class Ref:
    """ctypes view of oracle/_ref/libsqyref.so (the reference's own code). `available` may be False."""

    def __init__(self):
        self.available = os.path.exists(_REF_SO)
        self.lib = None
        if self.available:
            try:
                self.lib = ctypes.CDLL(_REF_SO)
            except OSError:
                self.available = False
        if self.available:
            L = self.lib
            L.ref_l2_cache_bytes.restype = c_long
            for f in ("ref_lz4_max_encoded_size", "ref_lz4_encode_u16", "ref_lz4_encode_bytes", "ref_quantiser_lut_string",
                      "ref_lz4_config", "ref_pipeline_encode_stages"):
                getattr(L, f).restype = c_long

    def l2_cache_bytes(self) -> int:
        return int(self.lib.ref_l2_cache_bytes())

    def bitswap_encode(self, w, a, nthreads=1, scalar=False):
        a = np.ascontiguousarray(a, dtype=np.uint16).ravel()
        out = np.zeros_like(a)
        if scalar:
            rc = self.lib.ref_bitswap_encode_scalar(c_int(w), _p(a), _p(out), c_long(a.size))
        else:
            rc = self.lib.ref_bitswap_encode(c_int(w), _p(a), _p(out), c_long(a.size), c_int(nthreads))
        assert rc == 0
        return out

    def bitswap_decode(self, w, a):
        a = np.ascontiguousarray(a, dtype=np.uint16).ravel()
        out = np.zeros_like(a)
        assert self.lib.ref_bitswap_decode(c_int(w), _p(a), _p(out), c_long(a.size)) == 0
        return out

    def remove_background(self, a, threshold, nthreads=1):
        a = np.ascontiguousarray(a, dtype=np.uint16)
        out = np.zeros_like(a)
        assert self.lib.ref_remove_background(c_int(threshold), _p(a), _p(out), c_long(a.size), c_int(nthreads)) == 0
        return out

    def bitswap8_encode(self, w, a):
        a = np.ascontiguousarray(a, dtype=np.uint8).ravel()
        out = np.zeros_like(a)
        assert self.lib.ref_bitswap8_encode(c_int(w), _p(a), _p(out), c_long(a.size)) == 0
        return out

    def bitswap8_decode(self, w, a):
        a = np.ascontiguousarray(a, dtype=np.uint8).ravel()
        out = np.zeros_like(a)
        assert self.lib.ref_bitswap8_decode(c_int(w), _p(a), _p(out), c_long(a.size)) == 0
        return out

    def remove_background8(self, a, threshold):
        a = np.ascontiguousarray(a, dtype=np.uint8)
        out = np.zeros_like(a)
        assert self.lib.ref_remove_background8(c_int(threshold), _p(a), _p(out), c_long(a.size)) == 0
        return out

    def darkest_face_supports(self, vol):
        vol = np.ascontiguousarray(vol, dtype=np.uint16)
        Z, Y, X = vol.shape
        out = np.zeros(4, dtype=np.float32)
        self.lib.ref_darkest_face_supports(_p(vol), c_long(Z), c_long(Y), c_long(X), _p(out))
        return out

    def rmestbkrd(self, vol, nthreads=1):
        vol = np.ascontiguousarray(vol, dtype=np.uint16)
        Z, Y, X = vol.shape
        out = np.zeros_like(vol)
        assert self.lib.ref_rmestbkrd_encode(_p(vol), _p(out), c_long(Z), c_long(Y), c_long(X), c_int(nthreads)) == 0
        return out

    def diff(self, vol, decode=False, nthreads=1):
        """diff_scheme<uint16_t> / <uint8_t> of the reference (encode with nthreads, decode always serial)"""
        vol = np.ascontiguousarray(vol)
        assert vol.dtype in (np.uint16, np.uint8) and vol.ndim == 3
        Z, Y, X = vol.shape
        out = np.zeros_like(vol)
        if vol.dtype == np.uint16:
            rc = (self.lib.ref_diff_decode(_p(vol), _p(out), c_long(Z), c_long(Y), c_long(X)) if decode
                  else self.lib.ref_diff_encode(_p(vol), _p(out), c_long(Z), c_long(Y), c_long(X), c_int(nthreads)))
        else:
            fn = self.lib.ref_diff8_decode if decode else self.lib.ref_diff8_encode
            rc = fn(_p(vol), _p(out), c_long(Z), c_long(Y), c_long(X))
        assert rc == 0
        return out

    def diff_name(self) -> str:
        buf = ctypes.create_string_buffer(64)
        assert self.lib.ref_diff_name(buf, c_int(64)) == 0
        return buf.value.decode()

    def quantiser_setup(self, a):
        a = np.ascontiguousarray(a, dtype=np.uint16)
        hist = np.zeros(65536, dtype=np.uint32)
        enc = np.zeros(65536, dtype=np.uint8)
        dec = np.zeros(256, dtype=np.uint16)
        self.lib.ref_quantiser_setup(_p(a), c_long(a.size), _p(hist), _p(enc), _p(dec))
        return hist, enc, dec

    def quantiser_luts_from_hist(self, hist):
        hist = np.ascontiguousarray(hist, dtype=np.uint32)
        enc = np.zeros(65536, dtype=np.uint8)
        dec = np.zeros(256, dtype=np.uint16)
        self.lib.ref_quantiser_luts_from_hist(_p(hist), _p(enc), _p(dec))
        return enc, dec

    def quantiser_encode(self, a):
        a = np.ascontiguousarray(a, dtype=np.uint16)
        out = np.zeros(a.shape, dtype=np.uint8)
        dec = np.zeros(256, dtype=np.uint16)
        self.lib.ref_quantiser_encode(_p(a), c_long(a.size), _p(out), _p(dec), c_int(1))
        return out, dec

    def quantiser_lut_string(self, dec) -> str:
        dec = np.ascontiguousarray(dec, dtype=np.uint16)
        buf = ctypes.create_string_buffer(4096)
        n = self.lib.ref_quantiser_lut_string(_p(dec), buf, c_long(4096))
        assert n >= 0
        return buf.value.decode("latin-1")

    def lz4_max_encoded_size(self, nbytes, nthreads=1, config=b""):
        return int(self.lib.ref_lz4_max_encoded_size(c_char_p(config), c_long(nbytes), c_int(nthreads)))

    def lz4_config(self, config=b"") -> str:
        buf = ctypes.create_string_buffer(1024)
        n = self.lib.ref_lz4_config(c_char_p(config), buf, c_long(1024))
        assert n >= 0
        return buf.value.decode()

    def lz4_encode(self, a, nthreads=1, config=b""):
        """payload exactly as lz4_scheme<T>::encode writes it (T = uint16 or char by dtype)"""
        a = np.ascontiguousarray(a)
        nbytes = a.nbytes
        cap = self.lz4_max_encoded_size(nbytes, max(nthreads, 1), config) + 1024
        out = np.zeros(cap, dtype=np.uint8)
        if a.dtype == np.uint16:
            n = self.lib.ref_lz4_encode_u16(c_char_p(config), _p(a), c_long(a.size), _p(out), c_int(nthreads))
        else:
            b = a.view(np.uint8)
            n = self.lib.ref_lz4_encode_bytes(c_char_p(config), _p(b), c_long(b.size), _p(out), c_int(nthreads))
        if n < 0:
            raise RuntimeError("reference lz4 encode failed")
        return out[:n].copy()

    def lz4_decode_u16(self, payload, n_voxels):
        payload = np.ascontiguousarray(payload, dtype=np.uint8)
        out = np.zeros(n_voxels, dtype=np.uint16)
        rc = self.lib.ref_lz4_decode_u16(_p(payload), c_long(payload.size), _p(out), c_long(n_voxels))
        return rc, out

    def lz4_decode_bytes(self, payload, nbytes):
        payload = np.ascontiguousarray(payload, dtype=np.uint8)
        out = np.zeros(nbytes, dtype=np.uint8)
        rc = self.lib.ref_lz4_decode_bytes(_p(payload), c_long(payload.size), _p(out), c_long(nbytes))
        return rc, out

    def pipeline_encode_stages(self, pipeline_id, vol, nthreads, w=1, threshold=0):
        """stage chain in detail_encode order; returns (payload, seconds)"""
        vol = np.ascontiguousarray(vol, dtype=np.uint16)
        Z, Y, X = vol.shape
        cap = self.lz4_max_encoded_size(vol.nbytes, max(nthreads, 1)) + 4096
        out = np.zeros(cap, dtype=np.uint8)
        sa = np.empty(vol.size, dtype=np.uint16)
        sb = np.empty(vol.size, dtype=np.uint16)
        secs = c_double(0)
        n = self.lib.ref_pipeline_encode_stages(c_int(pipeline_id), _p(vol), c_long(Z), c_long(Y), c_long(X), _p(out), _p(sa), _p(sb),
                                                c_int(nthreads), c_int(w), c_int(threshold), ctypes.byref(secs))
        if n < 0:
            raise RuntimeError("reference stage chain failed")
        return out[:n], secs.value

    def pipeline_decode_stages(self, w, payload, n_voxels):
        payload = np.ascontiguousarray(payload, dtype=np.uint8)
        out = np.zeros(n_voxels, dtype=np.uint16)
        scratch = np.zeros(n_voxels, dtype=np.uint16)
        secs = c_double(0)
        rc = self.lib.ref_pipeline_decode_stages(c_int(w), _p(payload), c_long(payload.size), _p(out), _p(scratch), c_long(n_voxels),
                                                 ctypes.byref(secs))
        return rc, out, secs.value


class _LZ4FFrameInfo(ctypes.Structure):
    _fields_ = [("blockSizeID", c_int), ("blockMode", c_int), ("contentChecksumFlag", c_int), ("frameType", c_int),
                ("contentSize", ctypes.c_ulonglong), ("dictID", ctypes.c_uint), ("blockChecksumFlag", c_int)]


class _LZ4FPreferences(ctypes.Structure):
    _fields_ = [("frameInfo", _LZ4FFrameInfo), ("compressionLevel", c_int), ("autoFlush", ctypes.c_uint),
                ("favorDecSpeed", ctypes.c_uint), ("reserved", ctypes.c_uint * 3)]


class Standin:
    """Stand-in for `Ref` where oracle/_ref cannot be built (the reference's sources are not in the repository), reached
    through the `ref_or_standin` test fixture only. It is NOT the reference's code:
      * LZ4 encode: the reference's lz4_scheme encode (SURVEY.md A.5) restated over liblz4, the library the reference
        calls; byte-identical to the reference-made payloads of tests/golden (tests/test_oracle.py);
      * LZ4 decode: the reference's decode loop (lz4.hpp:257-339) restated over liblz4's LZ4F_decompress; rc 0 only when
        exactly the expected bytes come out;
      * filters, diff, quantiser: the C port (oracle/sqy_oracle.c), pinned to the reference by the golden vectors;
      * L2 size (rmestbkrd): the kernel's sysfs record of the host, independent of the library under test.
    `available` is False without liblz4. Tests that pin the C port itself need the reference (`live_ref`)."""

    LZ4_LIB = "liblz4.so.1"

    def __init__(self):
        self.port = port()
        try:
            self.lz4 = ctypes.CDLL(self.LZ4_LIB)
            self.available = True
        except OSError:
            self.lz4, self.available = None, False
            return
        L = self.lz4
        L.LZ4F_isError.argtypes = [ctypes.c_size_t]
        for f in ("LZ4F_compressBound", "LZ4F_compressBegin", "LZ4F_compressUpdate", "LZ4F_compressEnd"):
            getattr(L, f).restype = ctypes.c_size_t
        L.LZ4F_compressBound.argtypes = [ctypes.c_size_t, c_void_p]
        L.LZ4F_createCompressionContext.argtypes = [POINTER(c_void_p), ctypes.c_uint]
        L.LZ4F_freeCompressionContext.argtypes = [c_void_p]
        L.LZ4F_compressBegin.argtypes = [c_void_p, c_void_p, ctypes.c_size_t, c_void_p]
        L.LZ4F_compressUpdate.argtypes = [c_void_p, c_void_p, ctypes.c_size_t, c_void_p, ctypes.c_size_t, c_void_p]
        L.LZ4F_compressEnd.argtypes = [c_void_p, c_void_p, ctypes.c_size_t, c_void_p]
        L.LZ4F_decompress.restype = ctypes.c_size_t
        L.LZ4F_decompress.argtypes = [c_void_p, c_void_p, POINTER(ctypes.c_size_t), c_void_p, POINTER(ctypes.c_size_t), c_void_p]
        L.LZ4F_createDecompressionContext.argtypes = [POINTER(c_void_p), ctypes.c_uint]
        L.LZ4F_freeDecompressionContext.argtypes = [c_void_p]

    # ---- lz4_scheme (encoders/lz4.hpp:58-274, lz4_utils.hpp:99-173 as summarised in SURVEY.md A.5) ----
    def _lz4_args(self, config: bytes):
        args = {"accel": 1, "blocksize_kb": 256, "framestep_kb": 256, "n_chunks_of_input": 0}
        for k, v in minors(config.decode()).items():
            if k in args:
                args[k] = int(v)
        bs = self.port.closest_blocksize_kb(args["blocksize_kb"])
        fs = bs if args["framestep_kb"] < bs else bs * max(1, round(args["framestep_kb"] / bs))
        if args["n_chunks_of_input"]:
            fs = 0
        return args["accel"], bs, fs, args["n_chunks_of_input"]

    def _prefs(self, accel, bs_kb):
        p = _LZ4FPreferences()
        p.frameInfo.blockSizeID = {64: 4, 256: 5, 1024: 6, 4096: 7}[bs_kb]   # linked blocks, no checksums, no content size
        p.compressionLevel = accel
        return p

    def _encode_serial(self, raw: np.ndarray, chunk: int, prefs) -> bytes:
        """one frame: compressBegin, one compressUpdate per chunk, compressEnd"""
        L = self.lz4
        cap = L.LZ4F_compressBound(chunk, ctypes.byref(prefs)) + 64
        buf = np.zeros(max(cap, 64), dtype=np.uint8)
        ctx = c_void_p()
        assert not L.LZ4F_isError(L.LZ4F_createCompressionContext(ctypes.byref(ctx), 100))
        parts = []
        try:
            def put(n):
                assert not L.LZ4F_isError(n), "liblz4 frame compression failed"
                parts.append(buf[:n].tobytes())
            put(L.LZ4F_compressBegin(ctx, _p(buf), buf.size, ctypes.byref(prefs)))
            for s in range(0, raw.size, chunk):
                piece = np.ascontiguousarray(raw[s:s + chunk])
                put(L.LZ4F_compressUpdate(ctx, _p(buf), buf.size, _p(piece), piece.size, None))
            put(L.LZ4F_compressEnd(ctx, _p(buf), buf.size, None))
        finally:
            L.LZ4F_freeCompressionContext(ctx)
        return b"".join(parts)

    def lz4_config(self, config=b"") -> str:
        accel, bs, fs, n = self._lz4_args(config)
        return f"accel={accel},blocksize_kb={bs},framestep_kb={fs},n_chunks_of_input={n}"

    def lz4_encode(self, a, nthreads=1, config=b""):
        """payload exactly as lz4_scheme<T>::encode writes it: one frame (nthreads = 1 or one chunk), else a frame per chunk"""
        raw = np.ascontiguousarray(a).view(np.uint8).ravel()
        accel, bs, fs, n = self._lz4_args(config)
        chunk = min(raw.size // n if n else fs << 10, raw.size) or raw.size or 1
        prefs = self._prefs(accel, bs)
        if nthreads <= 1 or raw.size <= chunk:
            out = self._encode_serial(raw, chunk, prefs)
        else:
            out = b"".join(self._encode_serial(raw[s:s + chunk], chunk, prefs) for s in range(0, raw.size, chunk))
        return np.frombuffer(out, dtype=np.uint8).copy()

    def _lz4_decode(self, payload, nbytes):
        """frames one after the other (skippable ones skipped by liblz4) until the input is used up"""
        L = self.lz4
        src = np.ascontiguousarray(payload, dtype=np.uint8)
        out = np.zeros(nbytes, dtype=np.uint8)
        ctx = c_void_p()
        assert not L.LZ4F_isError(L.LZ4F_createDecompressionContext(ctypes.byref(ctx), 100))
        pos = got = hint = 0
        try:
            while pos < src.size:
                dst_n, src_n = ctypes.c_size_t(nbytes - got), ctypes.c_size_t(src.size - pos)
                hint = L.LZ4F_decompress(ctx, c_void_p(out.ctypes.data + got), ctypes.byref(dst_n),
                                         c_void_p(src.ctypes.data + pos), ctypes.byref(src_n), None)
                if L.LZ4F_isError(hint) or (src_n.value == 0 and dst_n.value == 0):
                    return 1, out
                pos += src_n.value
                got += dst_n.value
        finally:
            L.LZ4F_freeDecompressionContext(ctx)
        return (0 if hint == 0 and got == nbytes else 1), out

    def lz4_decode_u16(self, payload, n_voxels):
        rc, out = self._lz4_decode(payload, 2 * n_voxels)
        return rc, out.view(np.uint16)

    def lz4_decode_bytes(self, payload, nbytes):
        return self._lz4_decode(payload, nbytes)

    # ---- filters and quantiser: the C port ----
    def l2_cache_bytes(self) -> int:
        base = "/sys/devices/system/cpu/cpu0/cache"
        for idx in sorted(os.listdir(base)):
            with open(os.path.join(base, idx, "level")) as f:
                if f.read().strip() != "2":
                    continue
            with open(os.path.join(base, idx, "size")) as f:
                size = f.read().strip()
            return int(size[:-1]) << {"K": 10, "M": 20}[size[-1]] if size[-1] in "KM" else int(size)
        raise RuntimeError("no L2 cache record under " + base)

    def bitswap_encode(self, w, a, nthreads=1, scalar=False):
        return self.port.bitswap_encode(w, a)

    def bitswap_decode(self, w, a):
        return self.port.bitswap_decode(w, a)

    def bitswap8_encode(self, w, a):
        return self.port.bitswap8_encode(w, a)

    def bitswap8_decode(self, w, a):
        return self.port.bitswap8_decode(w, a)

    def remove_background(self, a, threshold, nthreads=1):
        return self.port.remove_background(a, threshold)

    def remove_background8(self, a, threshold):
        return self.port.remove_background8(a, threshold)

    def rmestbkrd(self, vol, nthreads=1):
        return self.port.rmestbkrd(vol, self.l2_cache_bytes())[0]

    def diff(self, vol, decode=False, nthreads=1):
        return self.port.diff(vol, decode=decode)

    def quantiser_setup(self, a):
        hist = self.port.histogram(np.ascontiguousarray(a, dtype=np.uint16))
        enc, dec = self.port.quantiser_luts(hist)
        return hist, enc, dec

    def quantiser_encode(self, a):
        _, enc, dec = self.quantiser_setup(a)
        return self.port.lut_apply(a, enc), dec

    def quantiser_lut_string(self, dec) -> str:
        return lut_to_verbatim(dec)

    # ---- stage chains of oracle/ref_harness.cpp ----
    def pipeline_encode_stages(self, pipeline_id, vol, nthreads, w=1, threshold=0):
        import time

        vol = np.ascontiguousarray(vol, dtype=np.uint16)
        t0 = time.perf_counter()
        if pipeline_id == 0:
            data = self.port.bitswap_encode(1, vol)
        elif pipeline_id == 1:
            data = self.port.bitswap_encode(1, self.rmestbkrd(vol))
        elif pipeline_id == 2:
            data = self.quantiser_encode(vol)[0]
        elif pipeline_id == 3:
            data = self.port.bitswap_encode(w, self.port.remove_background(vol, threshold))
        else:
            data = vol
        payload = self.lz4_encode(data, nthreads=nthreads)
        return payload, time.perf_counter() - t0

    def pipeline_decode_stages(self, w, payload, n_voxels):
        import time

        t0 = time.perf_counter()
        rc, out = self.lz4_decode_u16(payload, n_voxels)
        if rc == 0 and w:
            out = self.port.bitswap_decode(w, out)
        return rc, out, time.perf_counter() - t0


_port = None
_ref = None
_standin = None


def port() -> Port:
    global _port
    if _port is None:
        _port = Port()
    return _port


def ref() -> Ref:
    global _ref
    if _ref is None:
        _ref = Ref()
    return _ref


def standin() -> Standin:
    global _standin
    if _standin is None:
        _standin = Standin()
    return _standin


# ------------------------------------------------------------------------------------------------
# control layer restated in Python
# ------------------------------------------------------------------------------------------------
def split_outside_verbatim(s: str, sep: str):
    """string_parsers.hpp:124-147 (informed_split): separators inside <verbatim>..</verbatim> are literal"""
    if not s or not sep:
        return []
    out, start, i, inside = [], 0, 0, False
    while i < len(s):
        if not inside and s.startswith(VERBATIM_OPEN, i):
            inside = True
            i += len(VERBATIM_OPEN)
        elif inside and s.startswith(VERBATIM_CLOSE, i):
            inside = False
            i += len(VERBATIM_CLOSE)
        elif not inside and s.startswith(sep, i):
            out.append(s[start:i])
            i += len(sep)
            start = i
        else:
            i += 1
    out.append(s[start:])
    return out


def to_pairs(pipeline: str):
    """pipeline_parser::to_pairs, string_parsers.hpp:355-395"""
    pairs = []
    for major in split_outside_verbatim(pipeline, "->"):
        dist = major.find("(")
        if dist < 0:
            dist = len(major)
        key = major[:dist]
        args = major[dist + 1 : len(major) - 1] if len(key) < len(major) else ""
        pairs.append((key, args))
    return pairs


def minors(args: str):
    """pipeline_parser::minors, string_parsers.hpp:434-467"""
    out = {}
    for item in split_outside_verbatim(args, ","):
        dist = item.find("=")
        if dist < 0:
            dist = len(item)
        key = item[:dist]
        out[key] = item[dist + 1 :] if dist + 1 < len(item) else item
    return out


HEAD_U16 = {"bitswap1", "bitshuffle", "diff3x3x1", "remove_background", "rmestbkrd"}   # sqeazy_pipelines.hpp:31-45 (hot-path subset)
SINK_U16 = {"pass_through", "quantiser", "lz4"}                    # :47-56
TAIL_CHAR = {"lz4"}                                                # :58-74 (hot-path subset)


def can_be_built_from(pipeline: str, head=HEAD_U16, sink=SINK_U16, tail=TAIL_CHAR) -> bool:
    """dynamic_pipeline.hpp:177-226 restricted to the hot-path registry"""
    if not pipeline:
        return False
    pairs = to_pairs(pipeline)
    found, sink_matched = 0, False
    for name, _ in pairs:
        if not sink_matched and name in head:
            found += 1
            continue
        if name in sink:
            found += 1
            sink_matched = True
            continue
        if name in tail:
            found += 1
    rebuilt = 2 * (len(pairs) - 1) + sum(len(n) + (2 + len(a) if a else 0) for n, a in pairs)
    return found == len(pairs) and rebuilt == len(pipeline)


def json_escape(s: str) -> str:
    """Boost.PropertyTree json create_escapes (as used by write_json in sqeazy_header.hpp:185)"""
    out = []
    for ch in s:
        c = ord(ch)
        if c == 0x20 or c == 0x21 or 0x23 <= c <= 0x2E or 0x30 <= c <= 0x5B or c >= 0x5D:
            out.append(ch)
        elif ch == "\b":
            out.append("\\b")
        elif ch == "\f":
            out.append("\\f")
        elif ch == "\n":
            out.append("\\n")
        elif ch == "\r":
            out.append("\\r")
        elif ch == "\t":
            out.append("\\t")
        elif ch == "/":
            out.append("\\/")
        elif ch == '"':
            out.append('\\"')
        elif ch == "\\":
            out.append("\\\\")
        else:
            out.append("\\u%04X" % c)
    return "".join(out)


def pack_header(shape, pipeline: str, payload_bytes: int, raw_type="uint16", sizeof_raw=2, version="0.7.2", headref="b200") -> str:
    """header::pack, sqeazy_header.hpp:147-193"""
    dims = ",\n".join('            "dim": "%d"' % d for d in shape)
    js = (
        "{\n"
        '    "pipename": "%s",\n'
        '    "raw": {\n'
        '        "type": "%s",\n'
        '        "rank": "%d",\n'
        '        "shape": {\n%s\n        }\n'
        "    },\n"
        '    "encoded": {\n'
        '        "bytes": "%d"\n'
        "    },\n"
        '    "sqy": {\n'
        '        "version": "%s",\n'
        '        "headref": "%s"\n'
        "    }\n"
        "}\n" % (json_escape(pipeline), raw_type, len(shape), dims, payload_bytes, version, headref)
    ) + HEADER_DELIM
    if len(js) % sizeof_raw:
        js = " " * (sizeof_raw - len(js) % sizeof_raw) + js
    return js


def unpack_header(blob: bytes):
    """header::unpack, sqeazy_header.hpp:295-344 ; returns dict or None"""
    end = blob.find(HEADER_DELIM.encode())
    if end < 0:
        return None
    text = blob[:end].decode("latin-1")
    if text.count("{") != text.count("}") or text.count("}") == 0 or text.count(":") < 2:
        return None
    def grab(key):
        m = re.search(r'"%s"\s*:\s*"((?:[^"\\]|\\.)*)"' % key, text)
        return m.group(1) if m else None
    unesc = lambda s: re.sub(r"\\(.)", lambda m: {"n": "\n", "t": "\t", "b": "\b", "f": "\f", "r": "\r"}.get(m.group(1), m.group(1)), s)
    return {
        "pipeline": unesc(grab("pipename") or ""),
        "raw_type": grab("type"),
        "rank": int(grab("rank") or 0),
        "shape": [int(v) for v in re.findall(r'"dim"\s*:\s*"(\d+)"', text)],
        "bytes": int(grab("bytes") or 0),
        "size": end + len(HEADER_DELIM),
    }


def lut_to_verbatim(dec: np.ndarray) -> str:
    """parsing::range_to_verbatim, string_parsers.hpp:508-535"""
    return VERBATIM_OPEN + base64.b64encode(np.ascontiguousarray(dec, dtype="<u2").tobytes()).decode() + VERBATIM_CLOSE
