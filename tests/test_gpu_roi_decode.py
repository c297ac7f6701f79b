"""Sub-volume decode (`sqyx_decode_roi_*`): a box of a stack, decoded from the LZ4 blocks that hold it.

Every box of every pipeline must equal the whole-stack decode sliced with numpy, through the device and the host entry points,
and write nothing behind the box. Blobs of `[filters ->] bitswapW -> lz4` and `quantiser -> lz4` in full 16 KiB blocks take the
indexed route (1): the block table (5 launches), the listed blocks (1), the gather (1), and only the blocks the box needs; the
test restates from the shape and W which blocks those are and, from the blob's index words, what the host route sends to the
device. The whole stack is the ordinary decode (route 0); every other blob is decoded whole and cropped (route 2).
"""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle as orc
from sqeazy_b200.synth import numpy_volume, torch_volume
from test_gpu_device_routes import PIPES16, PIPES8, SHAPES, SHAPES8, compressible, counted_device
from test_gpu_host_routes import first_compressed_block
from test_gpu_parity import dev, host16
from test_gpu_uint8 import vol8
from tiff_helper import read_tiff

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BLOCK = 16384
TABLES = 5
ROI_LAUNCHES = TABLES + 1 + 1
GUARD = 64
SENTINEL = 0xA5


def boxes(shape):
    """the whole stack, a voxel at each extreme corner, one z-plane, one row of every plane, an unaligned interior box, an
    empty box"""
    Z, Y, X = shape
    return {
        "whole": [(0, Z), (0, Y), (0, X)],
        "first_voxel": [(0, 1), (0, 1), (0, 1)],
        "last_voxel": [(Z - 1, Z), (Y - 1, Y), (X - 1, X)],
        "z_plane": [(Z // 2, Z // 2 + 1), (0, Y), (0, X)],
        "row_per_plane": [(0, Z), (Y // 3, Y // 3 + 1), (0, X)],
        "interior": [(1, Z - 1), (Y // 4 + 1, Y // 2 + 3), (X // 5, X - X // 5 - 1)],
        "empty": [(2, 2), (0, Y), (0, X)],
    }


def crop(vol, box):
    return vol[tuple(slice(lo, hi) for lo, hi in box)]


def roi_device(sq, cuda, d_blob, box, elem=2):
    """the device ROI decode into a buffer with GUARD sentinel elements behind the box; returns (box voxels, guard intact)"""
    n = int(np.prod([hi - lo for lo, hi in box]))
    out = cuda.full((n + GUARD,), SENTINEL, dtype=cuda.int16 if elem == 2 else cuda.uint8, device="cuda")
    (sq.decode_roi_device if elem == 2 else sq.decode_roi_device_u8)(d_blob, box, out)
    h = out.cpu().numpy().view(np.uint16 if elem == 2 else np.uint8)
    return h[:n], bool(np.all(h[n:] == (np.uint16(SENTINEL) if elem == 2 else np.uint8(SENTINEL))))


def roi_host(sq, blob, box, elem=2):
    n = int(np.prod([hi - lo for lo, hi in box]))
    dtype = np.uint16 if elem == 2 else np.uint8
    out = np.full(n + GUARD, SENTINEL, dtype=dtype)
    (sq.decode_roi if elem == 2 else sq.decode_roi_u8)(blob, box, nthreads=4, out=out)
    return out[:n], bool(np.all(out[n:] == SENTINEL))


def check_all_boxes(sq, cuda, blob, full, elem):
    d_blob = dev(cuda, blob)
    for name, box in boxes(full.shape).items():
        want = crop(full, box).ravel()
        got, guard = roi_device(sq, cuda, d_blob, box, elem)
        assert guard and np.array_equal(got, want), ("device", name)
        got, guard = roi_host(sq, blob, box, elem)
        assert guard and np.array_equal(got, want), ("host", name)


# ---------------------------------------------------------------------------------------------------------------- every pipeline
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("pipeline", PIPES16)
def test_every_box_of_every_u16_pipeline(sq, cuda, pipeline, shape):
    vol = numpy_volume(shape, "scmos", index=8)
    blob = sq.encode_device(pipeline, dev(cuda, vol).reshape(shape))
    full = cuda.empty(shape, dtype=cuda.int16, device="cuda")
    sq.decode_device(blob, full)
    check_all_boxes(sq, cuda, blob.cpu().numpy(), host16(full), 2)


@pytest.mark.parametrize("shape", SHAPES8)
@pytest.mark.parametrize("pipeline", PIPES8)
def test_every_box_of_every_u8_pipeline(sq, cuda, pipeline, shape):
    vol = vol8(shape, seed=len(pipeline))
    blob = sq.encode_device_u8(pipeline, dev(cuda, vol))
    full = cuda.empty(shape, dtype=cuda.uint8, device="cuda")
    sq.decode_device_u8(blob, full)
    check_all_boxes(sq, cuda, blob.cpu().numpy(), full.cpu().numpy(), 1)
    roi_host(sq, blob.cpu().numpy(), boxes(shape)["interior"], 1)
    assert sq.last_roi_info()["route"] == 2   # (no indexed route for uint8)


# ---------------------------------------------------------------------------------------------------------------- indexed route
BIG = (16, 1024, 2048)   # 64 MiB, whole 16 KiB blocks of every plane for every W
INDEXED = ["bitswap1->lz4", "rmestbkrd->bitswap1->lz4", "remove_background(threshold=110)->bitswap4->lz4", "bitswap8->lz4",
           "quantiser->lz4"]


def geometry(pipeline):
    """(sets, voxels per 16 KiB block of one set) of the LZ4 stream the pipeline writes"""
    if pipeline.startswith("quantiser"):
        return 1, BLOCK
    w = int(pipeline.split("->lz4")[0].split("bitswap")[1].split("(")[0])
    return 16 // w, BLOCK * 8 // w


def needed_blocks(shape, box, pipeline):
    """the stream's blocks (global indices, ascending) that hold the box's voxels: block v // vpb of every set"""
    sets, vpb = geometry(pipeline)
    set_blocks = int(np.prod(shape)) // vpb
    idx = np.ravel_multi_index(np.meshgrid(*[np.arange(lo, hi) for lo, hi in box], indexing="ij"), shape).ravel()
    per_set = np.unique(idx // vpb)
    return np.concatenate([j * set_blocks + per_set for j in range(sets)])


def index_words(payload):
    nblocks = int(payload[20:24].view(np.uint32)[0])
    return payload[40 : 40 + 4 * nblocks].view(np.uint32)


def sub_frame_bytes(blob, hsz, blocks):
    """what the host route sends: index frame of the listed blocks, their headers and data, EndMark"""
    words = index_words(blob[hsz:])[blocks] & 0x7FFFFFFF
    return 8 + 32 + 4 * len(blocks) + 7 + int(np.sum(4 + words.astype(np.int64))) + 4


@pytest.fixture(scope="module")
def big_vol():
    v = torch_volume(BIG, "scmos", index=46)
    v[: BIG[0] // 4] = 100
    return v.cpu().numpy().view(np.uint16)


@pytest.mark.parametrize("pipeline", INDEXED)
def test_indexed_route_decodes_just_the_blocks_of_the_box(sq, cuda, big_vol, pipeline):
    blob = sq.encode(pipeline, big_vol, nthreads=4)
    hsz = sq.header_size(blob)
    d_blob = dev(cuda, blob)
    full = sq.decode(blob, nthreads=4)
    for name, box in boxes(BIG).items():
        if name == "empty":
            continue
        want = crop(full, box).ravel()
        n = want.size
        out = cuda.full((n + GUARD,), SENTINEL, dtype=cuda.int16, device="cuda")
        launches = counted_device(sq, cuda, sq.decode_roi_device, d_blob, box, out)
        got = host16(out)
        assert np.array_equal(got[:n], want) and np.all(got[n:] == SENTINEL), name
        info = sq.last_roi_info()
        if name == "whole":
            assert info == {"route": 0, "blocks": 0, "h2d_bytes": 0, "voxels": n}
            ordinary = cuda.empty(BIG, dtype=cuda.int16, device="cuda")
            assert launches == counted_device(sq, cuda, sq.decode_device, d_blob, ordinary)
            continue
        blocks = needed_blocks(BIG, box, pipeline)
        assert info == {"route": 1, "blocks": blocks.size, "h2d_bytes": 0, "voxels": n}, name
        assert launches == ROI_LAUNCHES, name
        k0 = sq.kernel_launches()
        host, guard = roi_host(sq, blob, box)
        assert sq.kernel_launches() - k0 == ROI_LAUNCHES, name
        assert guard and np.array_equal(host, want), name
        assert sq.last_roi_info() == {"route": 1, "blocks": blocks.size, "h2d_bytes": sub_frame_bytes(blob, hsz, blocks), "voxels": n}


def test_one_plane_sends_a_small_share_of_the_blob(sq, cuda, big_vol):
    blob = sq.encode("bitswap1->lz4", big_vol, nthreads=4)
    box = [(BIG[0] - 1, BIG[0]), (0, BIG[1]), (0, BIG[2])]
    got, _ = roi_host(sq, blob, box)
    assert np.array_equal(got, big_vol[-1].ravel())
    assert sq.last_roi_info()["h2d_bytes"] < blob.size // 8


# ---------------------------------------------------------------------------------------------------------------- random access
def compressed_block(payload):
    """(index, data offset, size) of the first compressed block behind the index frame and the LZ4 frame header"""
    off, size = first_compressed_block(payload)
    p = 8 + int(payload[4:8].view(np.uint32)[0]) + 7
    k = 0
    while p + 4 != off:
        p += 4 + (int(payload[p : p + 4].view(np.uint32)[0]) & 0x7FFFFFFF)
        k += 1
    return k, off, size


@pytest.mark.parametrize("pipeline, code", [("bitswap1->lz4", 11), ("quantiser->lz4", 101)])
def test_a_broken_block_outside_the_box_does_not_matter(sq, cuda, big_vol, pipeline, code):
    blob = sq.encode(pipeline, big_vol, nthreads=4).copy()
    good = sq.decode(blob, nthreads=4)
    hsz = sq.header_size(blob)
    k, off, size = compressed_block(blob[hsz:])
    blob[hsz + off : hsz + off + size] = 0xFF
    sets, vpb = geometry(pipeline)
    set_blocks = int(np.prod(BIG)) // vpb
    z_broken = (k % set_blocks) * vpb // (BIG[1] * BIG[2])          # a z-plane the broken block holds voxels of
    z_clean = BIG[0] - 1 if z_broken < BIG[0] // 2 else 0
    assert z_clean * BIG[1] * BIG[2] // vpb != k % set_blocks
    d_blob = dev(cuda, blob)
    with pytest.raises(sq.SqeazyError, match=rf"returned {code}$"):
        sq.decode_device(d_blob, cuda.empty(BIG, dtype=cuda.int16, device="cuda"))
    with pytest.raises(sq.SqeazyError, match=rf"returned {code}$"):
        sq.decode(blob, nthreads=4)
    clean = [(z_clean, z_clean + 1), (0, BIG[1]), (0, BIG[2])]
    got_d, guard_d = roi_device(sq, cuda, d_blob, clean)
    assert sq.last_roi_info()["route"] == 1
    got_h, guard_h = roi_host(sq, blob, clean)
    assert sq.last_roi_info()["route"] == 1
    assert guard_d and guard_h and np.array_equal(got_d, good[z_clean].ravel()) and np.array_equal(got_h, good[z_clean].ravel())
    broken = [(z_broken, z_broken + 1), (0, BIG[1]), (0, BIG[2])]
    for fn in (lambda: roi_device(sq, cuda, d_blob, broken), lambda: roi_host(sq, blob, broken)):
        with pytest.raises(sq.SqeazyError, match=rf"returned {code}$"):
            fn()
    n = BIG[1] * BIG[2]
    out = cuda.full((n + GUARD,), SENTINEL, dtype=cuda.int16, device="cuda")
    with pytest.raises(sq.SqeazyError):
        sq.decode_roi_device(d_blob, broken, out)
    assert np.all(host16(out)[n:] == SENTINEL)
    h = np.full(n + GUARD, SENTINEL, dtype=np.uint16)
    with pytest.raises(sq.SqeazyError):
        sq.decode_roi(blob, broken, out=h)
    assert np.all(h[n:] == SENTINEL)


# ---------------------------------------------------------------------------------------------------------------- refusals
SMALL = (16, 64, 128)


@pytest.mark.parametrize("box", [[(3, 2), (0, 64), (0, 128)], [(0, 16), (0, 65), (0, 128)], [(0, 16), (0, 64)],
                                 [(0, 16), (0, 64), (0, 128), (0, 1)], [(-1, 2), (0, 64), (0, 128)]])
def test_malformed_box_is_3(sq, cuda, box):
    blob = sq.encode_device("bitswap1->lz4", dev(cuda, compressible()))
    out = cuda.empty(int(np.prod(SMALL)), dtype=cuda.int16, device="cuda")
    with pytest.raises(sq.SqeazyError, match=r"returned 3$"):
        sq.decode_roi_device(blob, box, out)
    with pytest.raises(sq.SqeazyError, match=r"returned 3$"):
        sq.decode_roi(blob.cpu().numpy(), box, out=np.empty(2 * int(np.prod(SMALL)), dtype=np.uint16))


def test_short_destination_is_1_and_a_truncated_blob_is_refused(sq, cuda):
    vol = compressible()
    blob = sq.encode_device("bitswap1->lz4", dev(cuda, vol))
    box = [(1, 3), (5, 9), (0, 128)]
    n = 2 * 4 * 128
    out = cuda.empty(n - 1, dtype=cuda.int16, device="cuda")
    with pytest.raises(sq.SqeazyError, match=r"returned 1$"):
        sq.decode_roi_device(blob, box, out)
    lib = sq.lib()
    arr = (ctypes.c_long * 6)(*[v for p in box for v in p])
    h = np.empty(n, dtype=np.uint16)
    b = blob.cpu().numpy()
    assert lib.sqyx_decode_roi_UI16(b.ctypes.data_as(ctypes.c_void_p), ctypes.c_long(b.size), arr, ctypes.c_uint(3),
                                    h.ctypes.data_as(ctypes.c_void_p), ctypes.c_long(2 * n - 1), ctypes.c_int(1)) == 1
    cut = b[: b.size - 100]
    with pytest.raises(sq.SqeazyError):
        sq.decode_roi_device(dev(cuda, cut), box, cuda.empty(n, dtype=cuda.int16, device="cuda"))
    with pytest.raises(sq.SqeazyError):
        sq.decode_roi(cut, box)
    got, guard = roi_device(sq, cuda, blob, box)
    assert guard and np.array_equal(got, crop(vol, box).ravel())
    assert np.array_equal(sq.decode_roi(b, box), crop(vol, box))


# ---------------------------------------------------------------------------------------------------------------- other blobs
def test_reference_style_blob_is_decoded_whole_and_cropped(sq, cuda, ref_or_standin):
    vol = numpy_volume((16, 128, 256), "scmos", index=10)
    name = "bitswap1(num_bits_per_plane=1)->lz4(accel=1,blocksize_kb=256,framestep_kb=256,n_chunks_of_input=0)"
    payload, _ = ref_or_standin.pipeline_encode_stages(0, vol, 8)
    h = orc.pack_header(vol.shape, name, payload.size, version="0.5.2", headref="4c45a9b")
    blob = np.concatenate([np.frombuffer(h.encode(), dtype=np.uint8), payload])
    check_all_boxes(sq, cuda, blob, vol, 2)
    box = boxes(vol.shape)["interior"]
    roi_host(sq, blob, box)
    assert sq.last_roi_info()["route"] == 2
    roi_device(sq, cuda, dev(cuda, blob), box)
    assert sq.last_roi_info()["route"] == 2


def test_ragged_stack_is_decoded_whole_and_cropped(sq, cuda):
    shape = (5, 33, 47)
    vol = numpy_volume(shape, "scmos", index=11)
    blob = sq.encode("bitswap1->lz4", vol)
    check_all_boxes(sq, cuda, blob, vol, 2)
    roi_host(sq, blob, boxes(shape)["interior"])
    assert sq.last_roi_info()["route"] == 2


def test_one_gib_stack_takes_the_indexed_route(sq, cuda):
    shape = (128, 2048, 2048)
    vol = torch_volume(shape, "scmos", index=45)
    blob = sq.encode_device("bitswap1->lz4", vol)
    box = [(60, 70), (100, 612), (1000, 1900)]
    n = 10 * 512 * 900
    out = cuda.empty(n, dtype=cuda.int16, device="cuda")
    assert counted_device(sq, cuda, sq.decode_roi_device, blob, box, out) == ROI_LAUNCHES
    assert cuda.equal(out.view(10, 512, 900), vol[60:70, 100:612, 1000:1900])
    assert sq.last_roi_info()["route"] == 1
    plane = [(127, 128), (0, 2048), (0, 2048)]
    out = cuda.empty(2048 * 2048, dtype=cuda.int16, device="cuda")
    sq.decode_roi_device(blob, plane, out)
    assert cuda.equal(out.view(2048, 2048), vol[127])
    del vol, blob


# ---------------------------------------------------------------------------------------------------------------- CLI
def test_cli_decompress_roi_writes_the_box(sq, cuda, tmp_path):
    sqy = os.path.join(ROOT, "sqeazy_b200", "bin", "sqy")
    vol = numpy_volume((12, 64, 96), "scmos", index=2)
    f = tmp_path / "stack.sqy"
    sq.encode("bitswap1->lz4", vol).tofile(str(f))
    out = str(tmp_path / "box.tif")
    r = subprocess.run([sqy, "decompress", "--roi", "2:7,10:50,3:90", str(f), "-o", out], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert np.array_equal(read_tiff(out), vol[2:7, 10:50, 3:90])
    r = subprocess.run([sqy, "decompress", "--roi", "2:7,10:50", str(f), "-o", out], capture_output=True, text=True, timeout=300)
    assert r.returncode == 1
    r = subprocess.run([sqy, "decompress", "--roi", "2:2,10:50,3:90", str(f), "-o", out], capture_output=True, text=True, timeout=300)
    assert r.returncode == 1 and "non-empty" in r.stderr
