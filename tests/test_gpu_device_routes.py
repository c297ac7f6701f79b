"""Which kernels the device entry points (`sqyx_encode_device_*` / `sqyx_decode_device_*`) launch, and which code each refusal
of the device decoder returns. The pipeline suites compare voxels only; a stage that silently ran a different sequence of
kernels (an extra copy, a filter no longer fused into the transpose after it, a lost fused LZ4 transpose) would pass them.
The counts are derived from the launchers in csrc/device and the sequencing of api.cu:

- bitswap, remove_background, diff3x3x1 encode, LUT apply and LUT decode: one launch each; a threshold filter directly in front
  of a bitswap, with a threshold above 0, runs inside the bitswap's launch;
- bitshuffle: one launch each for the whole blocks, the last partial block (a multiple of 8 elements) and the < 8 left over;
- diff3x3x1 decode: plane 0, one launch per coded plane 1 .. min(X, Z)-1, one for the planes behind them;
- LZ4 encode: begin + blocks + end (3) = 5; LZ4 decode: the block table (5) + the block decoder;
- rmestbkrd's estimate: 2 face histograms, 6 row histograms, the support index; the quantiser's histogram: one.
"""
import numpy as np
import pytest

from oracle import oracle as orc
from sqeazy_b200.synth import numpy_volume, torch_volume
from test_gpu_host_routes import counted_device, first_compressed_block
from test_gpu_parity import dev, expected_roundtrip, host16
from test_gpu_uint8 import vol8

pytestmark = pytest.mark.gpu

LZ4_ENCODE = 5
LZ4_DECODE = 5 + 1
ESTIMATE = 9
FILTERS = ("remove_background", "rmbkrd", "rmestbkrd")
SINKS = ("lz4", "quantiser", "pass_through")

# every pipeline of test_gpu_parity.py::PIPES, test_gpu_bitshuffle.py and test_gpu_diff.py
PIPES16 = ["bitswap1->lz4", "rmestbkrd->bitswap1->lz4", "quantiser->lz4", "remove_background(threshold=110)->bitswap4->lz4",
           "rmbkrd(threshold=105)->bitswap1->lz4", "lz4", "bitswap1", "bitswap2->lz4", "bitswap8", "quantiser", "pass_through",
           "remove_background(threshold=100)", "rmestbkrd", "bitswap1->pass_through->lz4", "rmestbkrd->lz4",
           "bitshuffle->lz4", "bitshuffle", "bitshuffle(block_size=512)->lz4", "rmestbkrd->bitshuffle->lz4",
           "remove_background(threshold=105)->bitshuffle->lz4", "bitshuffle->pass_through->lz4",
           "diff3x3x1->lz4", "diff3x3x1", "diff3x3x1->bitswap1->lz4", "rmestbkrd->diff3x3x1->bitswap1->lz4",
           "remove_background(threshold=105)->diff3x3x1->lz4", "diff3x3x1->pass_through->lz4", "bitswap1->diff3x3x1->lz4"]
# ... and of test_gpu_uint8.py, test_gpu_bitshuffle.py and test_gpu_diff.py on uint8
PIPES8 = ["bitswap1->lz4", "lz4", "bitswap4->lz4", "bitswap2", "pass_through", "pass_through->lz4",
          "remove_background(threshold=19)->bitswap1->lz4", "rmbkrd(threshold=19)->lz4",
          "bitshuffle->lz4", "bitshuffle", "remove_background(threshold=19)->bitshuffle(block_size=256)->lz4",
          "diff3x3x1->lz4", "diff3x3x1", "diff3x3x1->bitswap1->lz4"]
# whole 32-voxel chunks on aligned buffers (the fast kernels), and a ragged stack (generic bitswap, bitshuffle tails)
SHAPES = [(16, 64, 128), (5, 33, 47)]
SHAPES8 = [(24, 64, 128), (5, 7, 11)]


def split(pipeline):
    pairs = orc.to_pairs(pipeline)
    k = next((i for i, (name, _) in enumerate(pairs) if name in SINKS), len(pairs))
    return pairs[:k], (pairs[k][0] if k < len(pairs) else None), k + 1 < len(pairs)


def bitshuffle_launches(n, args, elem):
    bs = int(orc.minors(args).get("block_size", 0)) or max(128, 8192 // elem // 8 * 8)
    full = n // bs * bs
    last = (n - full) // 8 * 8
    return (full > 0) + (last > 0) + (n - full - last > 0)


def threshold(name, args, vol, sq, port):
    if name == "rmestbkrd":
        return port.rmestbkrd(vol, sq.host_l2_bytes())[1]
    return int(orc.minors(args).get("threshold", 0)) & (0xFF if vol.dtype == np.uint8 else 0xFFFF)


def encode_launches(pipeline, vol, sq, port):
    head, sink, tail = split(pipeline)
    n = 0
    i = 0
    while i < len(head):
        name, args = head[i]
        if name in FILTERS:
            n += (ESTIMATE if name == "rmestbkrd" else 0) + 1
            if i + 1 < len(head) and head[i + 1][0].startswith("bitswap") and threshold(name, args, vol, sq, port) > 0:
                i += 1
        elif name == "bitshuffle":
            n += bitshuffle_launches(vol.size, args, vol.itemsize)
        else:
            n += 1
        i += 1
    if sink == "lz4" or tail:
        n += LZ4_ENCODE
    if sink == "quantiser":
        n += 2
    return n


def decode_launches(pipeline, vol):
    head, sink, tail = split(pipeline)
    n = (LZ4_DECODE if sink == "lz4" or tail else 0) + (sink == "quantiser")
    for name, args in head:
        if name == "bitshuffle":
            n += bitshuffle_launches(vol.size, args, vol.itemsize)
        elif name == "diff3x3x1":
            Z, _, X = vol.shape
            zend = min(X, Z)
            n += zend + (zend < Z)
        elif name not in FILTERS:
            n += 1
    return n


def expected_u8(port, pipeline, vol):
    for name, args in orc.to_pairs(pipeline):
        if name in FILTERS:
            vol = port.remove_background8(vol.reshape(-1), int(orc.minors(args)["threshold"])).reshape(vol.shape)
    return vol


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("pipeline", PIPES16)
def test_device_routes_u16(sq, cuda, port, pipeline, shape):
    vol = numpy_volume(shape, "scmos", index=8)
    d_vol = dev(cuda, vol).reshape(shape)
    blob = None

    def enc():
        nonlocal blob
        blob = sq.encode_device(pipeline, d_vol)

    assert counted_device(sq, cuda, enc) == encode_launches(pipeline, vol, sq, port)
    out = cuda.empty(shape, dtype=cuda.int16, device="cuda")
    assert counted_device(sq, cuda, sq.decode_device, blob, out) == decode_launches(pipeline, vol)
    assert np.array_equal(host16(out), expected_roundtrip(port, sq, pipeline, vol))


@pytest.mark.parametrize("shape", SHAPES8)
@pytest.mark.parametrize("pipeline", PIPES8)
def test_device_routes_u8(sq, cuda, port, pipeline, shape):
    vol = vol8(shape, seed=len(pipeline))
    d_vol = dev(cuda, vol)
    blob = None

    def enc():
        nonlocal blob
        blob = sq.encode_device_u8(pipeline, d_vol)

    assert counted_device(sq, cuda, enc) == encode_launches(pipeline, vol, sq, port)
    out = cuda.empty(shape, dtype=cuda.uint8, device="cuda")
    assert counted_device(sq, cuda, sq.decode_device_u8, blob, out) == decode_launches(pipeline, vol)
    assert np.array_equal(out.cpu().numpy(), expected_u8(port, pipeline, vol))


def test_one_gib_bitswap1_lz4_fuses_the_transpose_into_the_decoder(sq, cuda):
    """1 GiB of 16/1 planes in whole 16 KiB blocks: the LZ4 block decoder also transposes back, no bitswap launch of its own"""
    shape = (128, 2048, 2048)
    vol = torch_volume(shape, "scmos", index=45)
    blob = None

    def enc():
        nonlocal blob
        blob = sq.encode_device("bitswap1->lz4", vol)

    assert counted_device(sq, cuda, enc) == 1 + LZ4_ENCODE
    out = cuda.empty(shape, dtype=cuda.int16, device="cuda")
    assert counted_device(sq, cuda, sq.decode_device, blob, out) == LZ4_DECODE
    assert cuda.equal(out, vol)


# ---------------------------------------------------------------------------------------------------------------- refusals
SMALL = (16, 64, 128)


def compressible(shape=SMALL):
    v = numpy_volume(shape, "scmos", index=9)
    v[: shape[0] // 2] = 100
    return v


def encoded(sq, cuda, pipeline, vol):
    return sq.encode_device(pipeline, dev(cuda, vol)).cpu().numpy()


def forged(vol, pipeline, payload):
    h = orc.pack_header(vol.shape, pipeline, payload.size)
    return np.concatenate([np.frombuffer(h.encode(), dtype=np.uint8), payload])


def corrupt_first_block(sq, blob):
    blob = blob.copy()
    hsz = sq.header_size(blob)
    off, size = first_compressed_block(blob[hsz:])
    blob[hsz + off : hsz + off + size] = 0xFF
    return blob


def refused(sq, cuda, blob, shape, code, voxels=None):
    out = cuda.empty(voxels if voxels is not None else int(np.prod(shape)), dtype=cuda.int16, device="cuda")
    with pytest.raises(sq.SqeazyError, match=rf"returned {code}$"):
        sq.decode_device(dev(cuda, blob), out)


def test_destination_too_small_is_1(sq, cuda):
    vol = compressible()
    refused(sq, cuda, encoded(sq, cuda, "bitswap1->lz4", vol), SMALL, 1, voxels=vol.size - 1)


def test_short_payload_without_sink_is_1(sq, cuda):
    refused(sq, cuda, encoded(sq, cuda, "bitswap1", compressible())[:-2], SMALL, 1)


@pytest.mark.parametrize("pipeline", ["pass_through", "quantiser"])
def test_short_payload_of_a_sink_without_tail_is_11(sq, cuda, pipeline):
    refused(sq, cuda, encoded(sq, cuda, pipeline, compressible())[:-1], SMALL, 11)


def test_corrupt_lz4_sink_is_11(sq, cuda):
    refused(sq, cuda, corrupt_first_block(sq, encoded(sq, cuda, "bitswap1->lz4", compressible())), SMALL, 11)


@pytest.mark.parametrize("pipeline", ["pass_through->lz4", "quantiser->lz4"])
def test_corrupt_lz4_tail_is_101(sq, cuda, pipeline):
    refused(sq, cuda, corrupt_first_block(sq, encoded(sq, cuda, pipeline, compressible())), SMALL, 101)


def test_quantiser_without_decode_lut_is_11(sq, cuda):
    vol = compressible()
    blob = encoded(sq, cuda, "quantiser", vol)
    refused(sq, cuda, forged(vol, "quantiser", blob[sq.header_size(blob):]), SMALL, 11)


def test_quantiser_blob_of_uint8_is_refused(sq, cuda):
    """the uint8 pipelines have no quantiser: the entry point refuses the header before the decoder sees it"""
    vol = compressible()
    blob = encoded(sq, cuda, "quantiser", vol)
    payload = blob[sq.header_size(blob):]
    h = orc.pack_header(vol.shape, "quantiser", payload.size, raw_type="uint8", sizeof_raw=1)
    out = cuda.empty(vol.size, dtype=cuda.uint8, device="cuda")
    with pytest.raises(sq.SqeazyError, match=r"returned 1$"):
        sq.decode_device_u8(dev(cuda, np.concatenate([np.frombuffer(h.encode(), dtype=np.uint8), payload])), out)


def test_diff_shape_refused_is_101(sq, cuda):
    vol = compressible((2, 64, 128))
    refused(sq, cuda, forged(vol, "diff3x3x1", vol.view(np.uint8).ravel()), vol.shape, 101)


def test_bitshuffle_launch_refused_is_101(sq, cuda):
    """a block size that is not a multiple of 8: the bitshuffle launcher refuses it"""
    vol = compressible((4, 32, 32))
    refused(sq, cuda, forged(vol, "bitshuffle(block_size=12)", vol.view(np.uint8).ravel()), vol.shape, 101)
