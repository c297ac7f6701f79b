"""uint8 volumes through the *_UI8 entry points (src/sqeazy.cpp:72-106, 144-163, 209-231, 309-335): stage kernels bit-exact
against the oracle (which equals the reference's own uint8 instantiation, tests/test_oracle.py), whole pipelines round
trip through the host and the device API, reference-style uint8 blobs decode on the GPU."""
import numpy as np
import pytest

from oracle import oracle as orc
from test_gpu_parity import dev

pytestmark = pytest.mark.gpu


def vol8(shape, seed=0):
    """8-bit light-sheet-like volume: background 20 +- 2, a bright slab, a few saturated voxels"""
    rng = np.random.default_rng(seed)
    v = np.clip(np.rint(20 + 2 * rng.standard_normal(shape)), 0, 255)
    v[shape[0] // 3: shape[0] // 2, shape[1] // 4: shape[1] // 2] += 90
    v.ravel()[rng.integers(0, v.size, 50)] = 255
    return v.astype(np.uint8)


@pytest.mark.parametrize("w", [1, 2, 4])
@pytest.mark.parametrize("n", [0, 1, 7, 8, 9, 127, 128, 129, 128 * 33, 128 * 4099, (1 << 21) + 5])
def test_bitswap8_parity(sq, cuda, port, w, n):
    a = np.random.default_rng(n + w).integers(0, 256, size=n, dtype=np.uint8)
    d_in = dev(cuda, a) if n else cuda.empty(0, dtype=cuda.uint8, device="cuda")
    d_out = cuda.full((n + 16,), 0xEE, dtype=cuda.uint8, device="cuda")
    sq.bitswap_encode_device_u8(w, d_in, d_out[:n])
    got = d_out.cpu().numpy()
    assert np.array_equal(got[:n], port.bitswap8_encode(w, a))
    assert np.all(got[n:] == 0xEE)
    back = cuda.empty(n, dtype=cuda.uint8, device="cuda")
    sq.bitswap_decode_device_u8(w, d_out[:n], back)
    assert np.array_equal(back.cpu().numpy(), a)


def test_bitswap8_unaligned_pointers(sq, cuda, port):
    a = np.random.default_rng(1).integers(0, 256, size=128 * 40 + 32, dtype=np.uint8)
    d = dev(cuda, a)
    for off in (1, 3, 16):
        src = d[off: off + 128 * 40]
        out = cuda.empty(128 * 40 + 32, dtype=cuda.uint8, device="cuda")[off: off + 128 * 40]
        sq.bitswap_encode_device_u8(1, src, out)
        assert np.array_equal(out.cpu().numpy(), port.bitswap8_encode(1, a[off: off + 128 * 40]))


@pytest.mark.parametrize("w,thr", [(1, 19), (2, 1), (4, 21), (1, 255), (1, 300)])
def test_fused_threshold_bitswap8(sq, cuda, port, w, thr):
    a = vol8((16, 64, 128), seed=thr).ravel()
    d_out = cuda.empty(a.size, dtype=cuda.uint8, device="cuda")
    sq.bitswap_encode_device_u8(w, dev(cuda, a), d_out, threshold=thr & 0xFF)
    assert np.array_equal(d_out.cpu().numpy(), port.bitswap8_encode(w, port.remove_background8(a, thr)))


@pytest.mark.parametrize("n", [0, 5, 16, 1000 + 3, 1 << 20])
def test_remove_background8(sq, cuda, port, n):
    a = np.random.default_rng(n).integers(0, 256, size=n, dtype=np.uint8)
    d_in = dev(cuda, a) if n else cuda.empty(0, dtype=cuda.uint8, device="cuda")
    d_out = cuda.empty(n, dtype=cuda.uint8, device="cuda")
    sq.remove_background_device_u8(d_in, d_out, 37)
    assert np.array_equal(d_out.cpu().numpy(), port.remove_background8(a, 37))


@pytest.mark.parametrize("pipeline", ["bitswap1->lz4", "lz4", "bitswap4->lz4", "bitswap2", "pass_through", "pass_through->lz4",
                                      "remove_background(threshold=19)->bitswap1->lz4", "rmbkrd(threshold=19)->lz4"])
@pytest.mark.parametrize("shape", [(24, 64, 128), (5, 7, 11), (4099,)])
def test_pipeline_roundtrip_u8(sq, cuda, port, pipeline, shape):
    vol = vol8(shape, seed=len(pipeline)) if len(shape) == 3 else np.random.default_rng(2).integers(0, 40, shape, dtype=np.uint8)
    expect = port.remove_background8(vol, 19) if "threshold=19" in pipeline else vol
    blob = sq.encode_u8(pipeline, vol)
    assert blob.size <= sq.max_compressed_length_u8(pipeline, vol.nbytes)
    assert sq.decompressed_sizeof(blob) == 1 and sq.decompressed_shape(blob) == tuple(shape) and sq.decompressed_length(blob) == vol.size
    hdr = orc.unpack_header(blob.tobytes())
    assert hdr["raw_type"] == "uint8"
    back = sq.decode_u8(blob)
    assert back.dtype == np.uint8 and np.array_equal(back, expect)
    # device API writes the same blob modulo LZ4's racy match choice: it must decode to the same voxels
    dblob = sq.encode_device_u8(pipeline, dev(cuda, vol))
    out = cuda.empty(vol.size, dtype=cuda.uint8, device="cuda")
    sq.decode_device_u8(dblob, out)
    assert np.array_equal(out.cpu().numpy().reshape(shape), expect)
    # the uint16 entry points refuse a uint8 blob
    with pytest.raises(sq.SqeazyError):
        sq.decode(blob)


def test_u8_payload_is_the_oracles_bit_planes(sq, cuda, port):
    """bitswap1->lz4 on uint8: the LZ4 stream decodes (oracle frame decoder, reference decoder) to the oracle's planes"""
    vol = vol8((16, 128, 128), seed=3)
    blob = sq.encode_u8("bitswap1->lz4", vol)
    payload = blob[sq.header_size(blob):]
    planes = port.bitswap8_encode(1, vol)
    assert np.array_equal(port.lz4_frames_decode(payload, vol.size), planes)
    r = orc.ref()
    if r.available:
        rc, out = r.lz4_decode_bytes(payload, vol.size)
        assert rc == 0 and np.array_equal(out, planes)
    assert vol.size / blob.size > 1.5


def test_reference_style_u8_blob_decodes_on_gpu(sq, cuda, ref_or_standin):
    """a blob put together from the reference's own uint8 stage code (bitswap_scheme<uint8_t>, lz4_scheme) + header"""
    vol = vol8((12, 96, 160), seed=4)
    planes = ref_or_standin.bitswap8_encode(1, vol)
    payload = ref_or_standin.lz4_encode(planes, nthreads=4)
    name = "bitswap1(num_bits_per_plane=1)->lz4(accel=1,blocksize_kb=256,framestep_kb=256,n_chunks_of_input=0)"
    h = orc.pack_header(vol.shape, name, payload.size, raw_type="uint8", sizeof_raw=1, version="0.5.2", headref="4c45a9b")
    blob = np.concatenate([np.frombuffer(h.encode(), dtype=np.uint8), payload])
    assert np.array_equal(sq.decode_u8(blob), vol)
