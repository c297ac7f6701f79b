"""Strided-slice decode (`sqyx_decode_slice_*`): lo:hi:step per dimension of a stack, decoded from the LZ4 blocks that hold it.

Every slice of every pipeline must equal numpy's slicing of the whole-stack decode, through the device and the host entry points,
and write nothing behind the slice. Blobs of `[filters ->] bitswapW -> lz4` and `quantiser -> lz4` in full 16 KiB blocks take the
indexed route (1) with the launches of the box calls, and decode only the blocks that hold a selected voxel: the test restates
them with numpy from the selected voxels' linear indices, and what the host route sends from the blob's index words. Every other
blob is decoded whole and cropped with the step (route 2).
"""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle as orc
from sqeazy_b200.synth import numpy_volume, torch_volume
from test_gpu_device_routes import PIPES16, PIPES8, SHAPES, SHAPES8, compressible, counted_device
from test_gpu_parity import dev, host16
from test_gpu_roi_decode import BIG, GUARD, INDEXED, ROI_LAUNCHES, SENTINEL, compressed_block, geometry, sub_frame_bytes
from test_gpu_uint8 import vol8
from tiff_helper import read_tiff

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SQY = os.path.join(ROOT, "sqeazy_b200", "bin", "sqy")


def slices(shape):
    """steps in each dimension alone and all at once, steps of every gather program (the group of 16 or 32 voxels holds many,
    two or one selected voxels), a step beyond and equal to the extent, steps that do not divide the range, lo > 0, one voxel,
    the whole range with step 2"""
    Z, Y, X = shape
    return {
        "z_step": [(0, Z, 2), (0, Y), (0, X)],
        "y_step": [(0, Z), (0, Y, 3), (0, X)],
        "x_step_2": [(0, Z), (0, Y), (0, X, 2)],
        "x_step_5": [(0, Z), (1, Y - 1), (1, X, 5)],
        "x_step_8": [(1, Z), (0, Y), (0, X, 8)],
        "x_step_16": [(0, Z), (0, Y, 2), (3, X, 16)],
        "x_step_33": [(0, Z), (0, Y), (X // 4, X, 33)],
        "all_steps": [(0, Z, 2), (0, Y, 3), (0, X, 4)],
        "step_beyond_extent": [(1, Z, Z + 3), (0, Y, 2 * Y), (2, X, X)],
        "step_equal_extent": [(0, Z, Z), (0, Y, Y), (0, X, X)],
        "non_dividing": [(0, Z, 3), (1, Y, 4), (0, X - 1, 6)],
        "lo_with_step": [(2, Z, 3), (Y // 3, Y, 5), (X // 2 + 1, X, 7)],
        "one_voxel": [(Z - 1, Z, 4), (Y // 2, Y // 2 + 1, 3), (X - 1, X, 9)],
        "whole_step_2": [(0, Z, 2), (0, Y, 2), (0, X, 2)],
    }


def triples(sel):
    return [t if len(t) == 3 else (*t, 1) for t in sel]


def cut(vol, sel):
    return vol[tuple(slice(lo, hi, step) for lo, hi, step in triples(sel))]


def count(sel):
    return int(np.prod([len(range(lo, hi, step)) for lo, hi, step in triples(sel)]))


def slice_device(sq, cuda, d_blob, sel, elem=2):
    """the device slice decode into a buffer with GUARD sentinel elements behind it; returns (voxels, guard intact)"""
    n = count(sel)
    out = cuda.full((n + GUARD,), SENTINEL, dtype=cuda.int16 if elem == 2 else cuda.uint8, device="cuda")
    (sq.decode_roi_device if elem == 2 else sq.decode_roi_device_u8)(d_blob, sel, out)
    h = out.cpu().numpy().view(np.uint16 if elem == 2 else np.uint8)
    return h[:n], bool(np.all(h[n:] == (np.uint16(SENTINEL) if elem == 2 else np.uint8(SENTINEL))))


def slice_host(sq, blob, sel, elem=2):
    n = count(sel)
    out = np.full(n + GUARD, SENTINEL, dtype=np.uint16 if elem == 2 else np.uint8)
    (sq.decode_roi if elem == 2 else sq.decode_roi_u8)(blob, sel, nthreads=4, out=out)
    return out[:n], bool(np.all(out[n:] == SENTINEL))


def check_all_slices(sq, cuda, blob, full, elem):
    d_blob = dev(cuda, blob)
    for name, sel in slices(full.shape).items():
        want = cut(full, sel).ravel()
        got, guard = slice_device(sq, cuda, d_blob, sel, elem)
        assert guard and np.array_equal(got, want), ("device", name)
        assert sq.last_roi_info()["voxels"] == want.size, ("device", name)
        got, guard = slice_host(sq, blob, sel, elem)
        assert guard and np.array_equal(got, want), ("host", name)
        assert sq.last_roi_info()["voxels"] == want.size, ("host", name)


# ---------------------------------------------------------------------------------------------------------------- every pipeline
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("pipeline", PIPES16)
def test_every_slice_of_every_u16_pipeline(sq, cuda, pipeline, shape):
    vol = numpy_volume(shape, "scmos", index=8)
    blob = sq.encode_device(pipeline, dev(cuda, vol).reshape(shape))
    full = cuda.empty(shape, dtype=cuda.int16, device="cuda")
    sq.decode_device(blob, full)
    check_all_slices(sq, cuda, blob.cpu().numpy(), host16(full), 2)


@pytest.mark.parametrize("shape", SHAPES8)
@pytest.mark.parametrize("pipeline", PIPES8)
def test_every_slice_of_every_u8_pipeline(sq, cuda, pipeline, shape):
    vol = vol8(shape, seed=len(pipeline))
    blob = sq.encode_device_u8(pipeline, dev(cuda, vol))
    full = cuda.empty(shape, dtype=cuda.uint8, device="cuda")
    sq.decode_device_u8(blob, full)
    check_all_slices(sq, cuda, blob.cpu().numpy(), full.cpu().numpy(), 1)
    slice_host(sq, blob.cpu().numpy(), slices(shape)["all_steps"], 1)
    assert sq.last_roi_info()["route"] == 2   # (no indexed route for uint8)


def test_whole_stack_with_steps_1_is_the_ordinary_decode_and_with_a_step_is_not(sq, cuda):
    vol = compressible()
    blob = sq.encode("bitswap1->lz4", vol)
    Z, Y, X = vol.shape
    got, guard = slice_host(sq, blob, [(0, Z, 1), (0, Y, 1), (0, X, 1)])
    assert guard and np.array_equal(got, vol.ravel()) and sq.last_roi_info()["route"] == 0
    got, guard = slice_host(sq, blob, [(0, Z, 1), (0, Y, 1), (0, X, 2)])
    assert guard and np.array_equal(got, vol[:, :, ::2].ravel()) and sq.last_roi_info()["route"] == 1


# ---------------------------------------------------------------------------------------------------------------- indexed route
def needed_blocks(shape, sel, pipeline):
    """the stream's blocks (global indices, ascending) that hold a selected voxel: block idx // vpb of every set"""
    sets, vpb = geometry(pipeline)
    set_blocks = int(np.prod(shape)) // vpb
    axes = [np.arange(lo, hi, step) for lo, hi, step in triples(sel)]
    idx = np.ravel_multi_index(np.meshgrid(*axes, indexing="ij"), shape).ravel()
    per_set = np.unique(idx // vpb)
    return np.concatenate([j * set_blocks + per_set for j in range(sets)])


def big_slices():
    Z, Y, X = BIG
    return {
        "overview": [(0, Z, 8), (0, Y, 4), (0, X, 4)],
        "z_step_4": [(0, Z, 4), (0, Y), (0, X)],
        "x_step_of_one_plane": [(Z // 2, Z // 2 + 1), (0, Y), (0, X, 4)],
        "rows_far_apart": [(1, Z, 3), (5, Y, 100), (0, X, 3)],
        "whole_step_2": [(0, Z, 2), (0, Y, 2), (0, X, 2)],
        "x_step_beyond_a_group": [(3, 9), (10, Y - 10, 7), (1, X, 40)],
    }


@pytest.fixture(scope="module")
def big_vol():
    v = torch_volume(BIG, "scmos", index=46)
    v[: BIG[0] // 4] = 100
    return v.cpu().numpy().view(np.uint16)


@pytest.mark.parametrize("pipeline", INDEXED)
def test_indexed_route_decodes_just_the_blocks_of_selected_voxels(sq, cuda, big_vol, pipeline):
    blob = sq.encode(pipeline, big_vol, nthreads=4)
    hsz = sq.header_size(blob)
    d_blob = dev(cuda, blob)
    full = sq.decode(blob, nthreads=4)
    sets, vpb = geometry(pipeline)
    all_blocks = sets * int(np.prod(BIG)) // vpb
    for name, sel in big_slices().items():
        want = cut(full, sel).ravel()
        n = want.size
        out = cuda.full((n + GUARD,), SENTINEL, dtype=cuda.int16, device="cuda")
        launches = counted_device(sq, cuda, sq.decode_roi_device, d_blob, sel, out)
        got = host16(out)
        assert np.array_equal(got[:n], want) and np.all(got[n:] == SENTINEL), name
        blocks = needed_blocks(BIG, sel, pipeline)
        assert sq.last_roi_info() == {"route": 1, "blocks": blocks.size, "h2d_bytes": 0, "voxels": n}, name
        assert launches == ROI_LAUNCHES, name
        if name == "z_step_4":
            assert blocks.size * 4 == all_blocks
        k0 = sq.kernel_launches()
        host, guard = slice_host(sq, blob, sel)
        assert sq.kernel_launches() - k0 == ROI_LAUNCHES, name
        assert guard and np.array_equal(host, want), name
        assert sq.last_roi_info() == {"route": 1, "blocks": blocks.size, "h2d_bytes": sub_frame_bytes(blob, hsz, blocks), "voxels": n}


@pytest.mark.parametrize("pipeline", ["bitswap1->lz4", "bitswap8->lz4", "quantiser->lz4"])
def test_a_step_beyond_a_block_decodes_no_block_without_a_selected_voxel(sq, cuda, big_vol, pipeline):
    """rows longer than a block of one set, so that the runs' own step skips whole blocks"""
    shape = (4, 4, int(np.prod(BIG)) // 16)
    vol = big_vol.reshape(shape)
    blob = sq.encode(pipeline, vol, nthreads=4)
    full = sq.decode(blob, nthreads=4).reshape(shape)
    _, vpb = geometry(pipeline)
    for sel in ([(0, 4, 3), (1, 4), (5, shape[2], 3 * vpb + 11)], [(2, 3), (0, 4, 2), (vpb - 1, shape[2], vpb + 1)]):
        want = cut(full, sel).ravel()
        got, guard = slice_device(sq, cuda, dev(cuda, blob), sel)
        assert guard and np.array_equal(got, want)
        blocks = needed_blocks(shape, sel, pipeline)
        assert sq.last_roi_info()["blocks"] == blocks.size
        sets, _ = geometry(pipeline)
        assert blocks.size == sets * want.size   # every selected voxel in a block of its own
        got, guard = slice_host(sq, blob, sel)
        assert guard and np.array_equal(got, want)
        assert sq.last_roi_info()["route"] == 1 and sq.last_roi_info()["blocks"] == blocks.size


# ---------------------------------------------------------------------------------------------------------------- random access
@pytest.mark.parametrize("pipeline, code", [("bitswap1->lz4", 11), ("quantiser->lz4", 101)])
def test_a_broken_block_matters_only_when_it_holds_a_selected_voxel(sq, cuda, big_vol, pipeline, code):
    blob = sq.encode(pipeline, big_vol, nthreads=4).copy()
    good = sq.decode(blob, nthreads=4)
    hsz = sq.header_size(blob)
    k, off, size = compressed_block(blob[hsz:])
    blob[hsz + off : hsz + off + size] = 0xFF
    _, vpb = geometry(pipeline)
    set_blocks = int(np.prod(BIG)) // vpb
    z_broken = (k % set_blocks) * vpb // (BIG[1] * BIG[2])           # the z-plane the broken block holds voxels of
    skip = [(1 - z_broken % 2, BIG[0], 2), (0, BIG[1], 3), (0, BIG[2], 2)]   # every other plane, not z_broken
    d_blob = dev(cuda, blob)
    got_d, guard_d = slice_device(sq, cuda, d_blob, skip)
    assert sq.last_roi_info()["route"] == 1
    got_h, guard_h = slice_host(sq, blob, skip)
    assert sq.last_roi_info()["route"] == 1
    want = cut(good, skip).ravel()
    assert guard_d and guard_h and np.array_equal(got_d, want) and np.array_equal(got_h, want)
    hit = [(z_broken, BIG[0], BIG[0]), (0, BIG[1], 2), (0, BIG[2], 5)]
    n = count(hit)
    out = cuda.full((n + GUARD,), SENTINEL, dtype=cuda.int16, device="cuda")
    with pytest.raises(sq.SqeazyError, match=rf"returned {code}$"):
        sq.decode_roi_device(d_blob, hit, out)
    assert np.all(host16(out)[n:] == SENTINEL)
    h = np.full(n + GUARD, SENTINEL, dtype=np.uint16)
    with pytest.raises(sq.SqeazyError, match=rf"returned {code}$"):
        sq.decode_roi(blob, hit, out=h)
    assert np.all(h[n:] == SENTINEL)


# ---------------------------------------------------------------------------------------------------------------- refusals
@pytest.mark.parametrize("sel", [[(0, 16, 0), (0, 64), (0, 128)], [(0, 16), (0, 64, -2), (0, 128)], [(0, 16, 2), (0, 64, 1)],
                                 [(0, 16, 2), (0, 64), (0, 128), (0, 1, 1)], [(0, 16), (0, 64), (0, 129, 4)]])
def test_malformed_slice_is_3(sq, cuda, sel):
    blob = sq.encode_device("bitswap1->lz4", dev(cuda, compressible()))
    out = cuda.empty(16 * 64 * 128, dtype=cuda.int16, device="cuda")
    with pytest.raises(sq.SqeazyError, match=r"decode_slice_device_UI16 returned 3$"):
        sq.decode_roi_device(blob, sel, out)
    with pytest.raises(sq.SqeazyError, match=r"decode_slice_UI16 returned 3$"):
        sq.decode_roi(blob.cpu().numpy(), sel, out=np.empty(2 * 16 * 64 * 128, dtype=np.uint16))


@pytest.mark.parametrize("pipeline", ["bitswap1->lz4", "lz4"])
def test_destination_one_voxel_short_is_1(sq, cuda, pipeline):
    vol = compressible()
    blob = sq.encode_device(pipeline, dev(cuda, vol))
    sel = [(1, 16, 4), (5, 60, 9), (0, 128, 3)]
    n = count(sel)
    out = cuda.full((n - 1 + GUARD,), SENTINEL, dtype=cuda.int16, device="cuda")
    with pytest.raises(sq.SqeazyError, match=r"returned 1$"):
        sq.decode_roi_device(blob, sel, out[: n - 1])
    assert np.all(host16(out) == SENTINEL)
    arr = (ctypes.c_long * 9)(*[v for t in sel for v in t])
    h = np.full(n + GUARD, SENTINEL, dtype=np.uint16)
    b = blob.cpu().numpy()
    assert sq.lib().sqyx_decode_slice_UI16(b.ctypes.data_as(ctypes.c_void_p), ctypes.c_long(b.size), arr, ctypes.c_uint(3),
                                           h.ctypes.data_as(ctypes.c_void_p), ctypes.c_long(2 * n - 2), ctypes.c_int(1)) == 1
    assert np.all(h == SENTINEL)
    got, guard = slice_device(sq, cuda, blob, sel)
    assert guard and np.array_equal(got, cut(vol, sel).ravel())


# ---------------------------------------------------------------------------------------------------------------- other blobs
def test_reference_style_blob_is_decoded_whole_and_cropped(sq, cuda, ref_or_standin):
    vol = numpy_volume((16, 128, 256), "scmos", index=10)
    name = "bitswap1(num_bits_per_plane=1)->lz4(accel=1,blocksize_kb=256,framestep_kb=256,n_chunks_of_input=0)"
    payload, _ = ref_or_standin.pipeline_encode_stages(0, vol, 8)
    h = orc.pack_header(vol.shape, name, payload.size, version="0.5.2", headref="4c45a9b")
    blob = np.concatenate([np.frombuffer(h.encode(), dtype=np.uint8), payload])
    check_all_slices(sq, cuda, blob, vol, 2)
    sel = slices(vol.shape)["all_steps"]
    slice_host(sq, blob, sel)
    assert sq.last_roi_info()["route"] == 2
    slice_device(sq, cuda, dev(cuda, blob), sel)
    assert sq.last_roi_info()["route"] == 2


def test_ragged_stack_is_decoded_whole_and_cropped(sq, cuda):
    shape = (5, 33, 47)
    vol = numpy_volume(shape, "scmos", index=11)
    blob = sq.encode("bitswap1->lz4", vol)
    for sel in slices(shape).values():
        got, guard = slice_host(sq, blob, sel)
        assert guard and np.array_equal(got, cut(vol, sel).ravel())
        assert sq.last_roi_info()["route"] == 2
        got, guard = slice_device(sq, cuda, dev(cuda, blob), sel)
        assert guard and np.array_equal(got, cut(vol, sel).ravel())
        assert sq.last_roi_info()["route"] == 2


def test_uint8_stack_is_decoded_whole_and_cropped(sq, cuda):
    shape = (24, 64, 128)
    vol = vol8(shape, seed=3)
    blob = sq.encode_device_u8("bitswap1->lz4", dev(cuda, vol))
    for sel in slices(shape).values():
        got, guard = slice_device(sq, cuda, blob, sel, 1)
        assert guard and np.array_equal(got, cut(vol, sel).ravel())
        assert sq.last_roi_info()["route"] == 2
        got, guard = slice_host(sq, blob.cpu().numpy(), sel, 1)
        assert guard and np.array_equal(got, cut(vol, sel).ravel())
        assert sq.last_roi_info()["route"] == 2


# ---------------------------------------------------------------------------------------------------------------- CLI
def test_cli_decompress_roi_writes_the_slice(sq, cuda, tmp_path):
    vol = numpy_volume((16, 64, 128), "scmos", index=2)
    f = tmp_path / "stack.sqy"
    sq.encode("bitswap1->lz4", vol).tofile(str(f))
    out = str(tmp_path / "slice.tif")
    r = subprocess.run([SQY, "decompress", "--roi", "0:16:4,0:64:8,0:128:16", str(f), "-o", out], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stderr
    assert np.array_equal(read_tiff(out), vol[0:16:4, 0:64:8, 0:128:16])
    r = subprocess.run([SQY, "decompress", "--roi", "1:16:3,5:64,0:128:7", str(f), "-o", out], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stderr
    assert np.array_equal(read_tiff(out), vol[1:16:3, 5:64, 0:128:7])
    for bad in ("0:4:0,0:64,0:128", "0:4:-2,0:64,0:128", "0:4:,0:64,0:128", "0:4:2:1,0:64,0:128"):
        r = subprocess.run([SQY, "decompress", "--roi", bad, str(f), "-o", out], capture_output=True, text=True, timeout=300)
        assert r.returncode == 1 and "--roi expects" in r.stderr, bad
