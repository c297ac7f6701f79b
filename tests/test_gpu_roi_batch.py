"""Batches of selections (`sqyx_decode_slice_batch_*`): many boxes and strided slices of one stack in one call.

The packed output of a batch must equal the selections of the whole-stack decode, cut with numpy and concatenated in order, and
the single calls' outputs concatenated, through the device and the host entry points, with nothing written behind it. On the
indexed route the batch decodes the union of the selections' blocks once: the test restates that union from the selected voxels
and, from the blob's index words, what the host route sends. A batch of boxes takes the launches of one box call; every further
thread program of the gather adds one launch. Every other blob is decoded whole once (route 2).
"""
import ctypes

import numpy as np
import pytest

from oracle import oracle as orc
from sqeazy_b200.synth import numpy_volume, torch_volume
from test_gpu_device_routes import PIPES16, PIPES8, SHAPES, SHAPES8, compressible, counted_device
from test_gpu_parity import dev, host16
from test_gpu_roi_decode import BIG, GUARD, INDEXED, ROI_LAUNCHES, SENTINEL, boxes, compressed_block, geometry, sub_frame_bytes
from test_gpu_slice_decode import big_slices, count, cut, needed_blocks, slices
from test_gpu_uint8 import vol8

pytestmark = pytest.mark.gpu


def every_selection(shape):
    """every box and every slice of the single-call tests: the whole stack, empty selections, one voxel, every gather program"""
    return list(boxes(shape).values()) + list(slices(shape).values())


def packed(full, sels):
    return np.concatenate([cut(full, s).ravel() for s in sels])


def batch_device(sq, cuda, d_blob, sels, elem=2):
    """the device batch into a buffer with GUARD sentinel elements behind it; returns (packed voxels, guard intact)"""
    n = sum(count(s) for s in sels)
    out = cuda.full((n + GUARD,), SENTINEL, dtype=cuda.int16 if elem == 2 else cuda.uint8, device="cuda")
    (sq.decode_roi_batch_device if elem == 2 else sq.decode_roi_batch_device_u8)(d_blob, sels, out)
    h = out.cpu().numpy().view(np.uint16 if elem == 2 else np.uint8)
    return h[:n], bool(np.all(h[n:] == (np.uint16(SENTINEL) if elem == 2 else np.uint8(SENTINEL))))


def batch_host(sq, blob, sels, elem=2):
    n = sum(count(s) for s in sels)
    out = np.full(n + GUARD, SENTINEL, dtype=np.uint16 if elem == 2 else np.uint8)
    (sq.decode_roi_batch if elem == 2 else sq.decode_roi_batch_u8)(blob, sels, nthreads=4, out=out)
    return out[:n], bool(np.all(out[n:] == SENTINEL))


def check_batch(sq, cuda, blob, full, elem):
    sels = every_selection(full.shape)
    want = packed(full, sels)
    got, guard = batch_device(sq, cuda, dev(cuda, blob), sels, elem)
    assert guard and np.array_equal(got, want), "device"
    assert sq.last_roi_info()["voxels"] == want.size
    got, guard = batch_host(sq, blob, sels, elem)
    assert guard and np.array_equal(got, want), "host"
    assert sq.last_roi_info()["voxels"] == want.size
    single = sq.decode_roi if elem == 2 else sq.decode_roi_u8
    assert np.array_equal(np.concatenate([single(blob, s).ravel() for s in sels]), want)


# ---------------------------------------------------------------------------------------------------------------- every pipeline
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("pipeline", PIPES16)
def test_one_batch_of_every_selection_of_every_u16_pipeline(sq, cuda, pipeline, shape):
    vol = numpy_volume(shape, "scmos", index=8)
    blob = sq.encode_device(pipeline, dev(cuda, vol).reshape(shape))
    full = cuda.empty(shape, dtype=cuda.int16, device="cuda")
    sq.decode_device(blob, full)
    check_batch(sq, cuda, blob.cpu().numpy(), host16(full), 2)


@pytest.mark.parametrize("shape", SHAPES8)
@pytest.mark.parametrize("pipeline", PIPES8)
def test_one_batch_of_every_selection_of_every_u8_pipeline(sq, cuda, pipeline, shape):
    vol = vol8(shape, seed=len(pipeline))
    blob = sq.encode_device_u8(pipeline, dev(cuda, vol))
    full = cuda.empty(shape, dtype=cuda.uint8, device="cuda")
    sq.decode_device_u8(blob, full)
    check_batch(sq, cuda, blob.cpu().numpy(), full.cpu().numpy(), 1)
    assert sq.last_roi_info()["route"] == 2   # (no indexed route for uint8)


# ---------------------------------------------------------------------------------------------------------------- indexed route
@pytest.fixture(scope="module")
def big_vol():
    v = torch_volume(BIG, "scmos", index=46)
    v[: BIG[0] // 4] = 100
    return v.cpu().numpy().view(np.uint16)


def union(sels, pipeline):
    if any(count(s) == int(np.prod(BIG)) for s in sels):   # the whole stack: every block
        sets, vpb = geometry(pipeline)
        return np.arange(sets * int(np.prod(BIG)) // vpb)
    return np.unique(np.concatenate([needed_blocks(BIG, s, pipeline) for s in sels if count(s)]))


def tiles(z):
    """the 4 x 4 tiles of plane z"""
    Z, Y, X = BIG
    return [[(z, z + 1), (ty * Y // 4, (ty + 1) * Y // 4), (tx * X // 4, (tx + 1) * X // 4)] for ty in range(4) for tx in range(4)]


def random_boxes(n, edge, seed):
    rng = np.random.default_rng(seed)
    return [[(int(o), int(o) + e) for o, e in zip((rng.integers(0, s - e + 1) for s, e in zip(BIG, edge)), edge)] for _ in range(n)]


def check_indexed(sq, cuda, blob, d_blob, full, sels, pipeline, launches):
    """device and host batch of `sels`: the packed voxels, the union's blocks once, the sub-frame of the union, the launches"""
    hsz = sq.header_size(blob)
    want = packed(full, sels)
    n = want.size
    out = cuda.full((n + GUARD,), SENTINEL, dtype=cuda.int16, device="cuda")
    assert counted_device(sq, cuda, sq.decode_roi_batch_device, d_blob, sels, out) == launches
    got = host16(out)
    assert np.array_equal(got[:n], want) and np.all(got[n:] == SENTINEL)
    blocks = union(sels, pipeline)
    assert sq.last_roi_info() == {"route": 1, "blocks": blocks.size, "h2d_bytes": 0, "voxels": n}
    k0 = sq.kernel_launches()
    host, guard = batch_host(sq, blob, sels)
    assert sq.kernel_launches() - k0 == launches
    assert guard and np.array_equal(host, want)
    assert sq.last_roi_info() == {"route": 1, "blocks": blocks.size, "h2d_bytes": sub_frame_bytes(blob, hsz, blocks), "voxels": n}
    return blocks.size


@pytest.mark.parametrize("pipeline", INDEXED)
def test_indexed_route_decodes_the_union_of_the_selections_once(sq, cuda, big_vol, pipeline):
    blob = sq.encode(pipeline, big_vol, nthreads=4)
    d_blob = dev(cuda, blob)
    full = sq.decode(blob, nthreads=4)
    # the tiles of one plane share the blocks of their rows: a quarter of what the single calls decode
    t = tiles(BIG[0] // 2)
    blocks = check_indexed(sq, cuda, blob, d_blob, full, t, pipeline, ROI_LAUNCHES)
    assert 4 * blocks == sum(needed_blocks(BIG, s, pipeline).size for s in t)
    # boxes only: the launches of one box call, whatever their number
    for sels in (random_boxes(1, (5, 100, 300), 1), random_boxes(16, (3, 64, 64), 2), random_boxes(1000, (2, 9, 40), 3)):
        check_indexed(sq, cuda, blob, d_blob, full, sels, pipeline, ROI_LAUNCHES)
    # the slices of the single-call tests (every gather program), an empty box and the whole stack: route 1, every block, one
    # extra launch per extra gather program
    mixed = list(big_slices().values()) + [boxes(BIG)["empty"], boxes(BIG)["whole"]] + t
    check_indexed(sq, cuda, blob, d_blob, full, mixed, pipeline, ROI_LAUNCHES + 2)
    # a repeated selection is written twice, its blocks decoded once
    box = [(2, 5), (100, 300), (7, 1500)]
    assert check_indexed(sq, cuda, blob, d_blob, full, [box, box], pipeline, ROI_LAUNCHES) == needed_blocks(BIG, box, pipeline).size


# ---------------------------------------------------------------------------------------------------------------- random access
@pytest.mark.parametrize("pipeline, code", [("bitswap1->lz4", 11), ("quantiser->lz4", 101)])
def test_a_broken_block_matters_only_when_a_selection_needs_it(sq, cuda, big_vol, pipeline, code):
    blob = sq.encode(pipeline, big_vol, nthreads=4).copy()
    good = sq.decode(blob, nthreads=4)
    hsz = sq.header_size(blob)
    k, off, size = compressed_block(blob[hsz:])
    blob[hsz + off : hsz + off + size] = 0xFF
    _, vpb = geometry(pipeline)
    set_blocks = int(np.prod(BIG)) // vpb
    z_broken = (k % set_blocks) * vpb // (BIG[1] * BIG[2])           # the z-plane the broken block holds voxels of
    clean = [tiles(z)[i] for z in range(BIG[0]) if z != z_broken for i in (0, 5, 15)]
    d_blob = dev(cuda, blob)
    want = packed(good, clean)
    got_d, guard_d = batch_device(sq, cuda, d_blob, clean)
    assert sq.last_roi_info()["route"] == 1
    got_h, guard_h = batch_host(sq, blob, clean)
    assert sq.last_roi_info()["route"] == 1
    assert guard_d and guard_h and np.array_equal(got_d, want) and np.array_equal(got_h, want)
    hit = clean[:4] + [[(z_broken, z_broken + 1), (0, BIG[1], 2), (0, BIG[2], 5)]] + clean[4:8]
    n = sum(count(s) for s in hit)
    out = cuda.full((n + GUARD,), SENTINEL, dtype=cuda.int16, device="cuda")
    with pytest.raises(sq.SqeazyError, match=rf"returned {code}$"):
        sq.decode_roi_batch_device(d_blob, hit, out)
    assert np.all(host16(out)[n:] == SENTINEL)
    h = np.full(n + GUARD, SENTINEL, dtype=np.uint16)
    with pytest.raises(sq.SqeazyError, match=rf"returned {code}$"):
        sq.decode_roi_batch(blob, hit, out=h)
    assert np.all(h[n:] == SENTINEL)


# ---------------------------------------------------------------------------------------------------------------- refusals
SMALL = (16, 64, 128)
GOOD = [[(1, 16, 4), (5, 60, 9), (0, 128, 3)], [(0, 2), (0, 64), (0, 128)]]


def c_batch(sq, blob, arr, nsel, ndims, dst, capacity, device):
    """the C batch call itself (device: blob and dst are CUDA tensors)"""
    L = sq.lib()
    if device:
        return L.sqyx_decode_slice_batch_device_UI16(ctypes.c_void_p(blob.data_ptr()), ctypes.c_long(blob.numel()), arr,
                                                     ctypes.c_uint(nsel), ctypes.c_uint(ndims), ctypes.c_void_p(dst.data_ptr()),
                                                     ctypes.c_long(capacity), ctypes.c_void_p(0))
    return L.sqyx_decode_slice_batch_UI16(blob.ctypes.data_as(ctypes.c_void_p), ctypes.c_long(blob.size), arr, ctypes.c_uint(nsel),
                                          ctypes.c_uint(ndims), dst.ctypes.data_as(ctypes.c_void_p), ctypes.c_long(capacity),
                                          ctypes.c_int(1))


@pytest.mark.parametrize("bad", [[(3, 2), (0, 64), (0, 128)], [(0, 16), (0, 65), (0, 128)], [(0, 16, 0), (0, 64), (0, 128)],
                                 [(0, 16), (0, 64, -2), (0, 128)], [(-1, 2), (0, 64), (0, 128)]])
def test_one_malformed_selection_refuses_the_batch_with_3_and_writes_nothing(sq, cuda, bad):
    blob = sq.encode_device("bitswap1->lz4", dev(cuda, compressible()))
    sels = [GOOD[0], bad, GOOD[1]]
    n = 2 * int(np.prod(SMALL))
    out = cuda.full((n,), SENTINEL, dtype=cuda.int16, device="cuda")
    with pytest.raises(sq.SqeazyError, match=r"decode_slice_batch_device_UI16 returned 3$"):
        sq.decode_roi_batch_device(blob, sels, out)
    assert np.all(host16(out) == SENTINEL)
    h = np.full(n, SENTINEL, dtype=np.uint16)
    with pytest.raises(sq.SqeazyError, match=r"decode_slice_batch_UI16 returned 3$"):
        sq.decode_roi_batch(blob.cpu().numpy(), sels, out=h)
    assert np.all(h == SENTINEL)


def test_wrong_ndims_and_nsel_out_of_range_are_3(sq, cuda):
    """The C calls take one ndims for the whole batch, so a wrong ndims refuses every selection at once; Python refuses a batch
    whose selections differ in their number of dimensions before it reaches the library"""
    blob = sq.encode_device("bitswap1->lz4", dev(cuda, compressible()))
    b = blob.cpu().numpy()
    n = int(np.prod(SMALL))
    out = cuda.full((n,), SENTINEL, dtype=cuda.int16, device="cuda")
    h = np.full(n, SENTINEL, dtype=np.uint16)
    one = [0, 1, 1, 0, 1, 1, 0, 1, 1]
    for nsel, ndims in ((2, 2), (0, 3), (65537, 3)):
        arr = (ctypes.c_long * max(len(one) * nsel, 1))(*(one * nsel))
        assert c_batch(sq, blob, arr, nsel, ndims, out, 2 * n, True) == 3, (nsel, ndims)
        assert c_batch(sq, b, arr, nsel, ndims, h, 2 * n, False) == 3, (nsel, ndims)
    assert np.all(host16(out) == SENTINEL) and np.all(h == SENTINEL)
    with pytest.raises(sq.SqeazyError):
        sq.decode_roi_batch(b, [GOOD[0], [(0, 2), (0, 64)]])
    arr = (ctypes.c_long * (9 * 65536))(*(one * 65536))   # the most a batch takes: one voxel 65536 times
    assert c_batch(sq, b, arr, 65536, 3, h, 2 * n, False) == 0
    assert np.all(h[:65536] == compressible()[0, 0, 0]) and sq.last_roi_info()["voxels"] == 65536


def test_destination_one_voxel_short_is_1_and_empty_selections_are_route_minus_1(sq, cuda):
    vol = compressible()
    blob = sq.encode_device("bitswap1->lz4", dev(cuda, vol))
    b = blob.cpu().numpy()
    n = sum(count(s) for s in GOOD)
    out = cuda.full((n + GUARD,), SENTINEL, dtype=cuda.int16, device="cuda")
    with pytest.raises(sq.SqeazyError, match=r"returned 1$"):
        sq.decode_roi_batch_device(blob, GOOD, out[: n - 1])
    assert np.all(host16(out) == SENTINEL)
    arr = (ctypes.c_long * 18)(*[v for s in GOOD for t in s for v in (t if len(t) == 3 else (*t, 1))])
    h = np.full(n + GUARD, SENTINEL, dtype=np.uint16)
    assert c_batch(sq, b, arr, 2, 3, h, 2 * n - 2, False) == 1
    assert np.all(h == SENTINEL)
    empty = [[(2, 2), (0, 64), (0, 128)], [(0, 16), (5, 60, 9), (7, 7, 3)]]
    for got in (sq.decode_roi_batch(b, empty), sq.decode_roi_batch_device(blob, empty, out)):
        assert [tuple(a.shape) for a in got] == [(0, 64, 128), (16, 7, 0)]
        assert sq.last_roi_info() == {"route": -1, "blocks": 0, "h2d_bytes": 0, "voxels": 0}
    assert np.all(host16(out) == SENTINEL)


# ---------------------------------------------------------------------------------------------------------------- other blobs
def check_route_2(sq, cuda, blob, vol, elem):
    """route 2: every selection cropped from one whole decode; the host route sends the payload once, whatever nsel is"""
    hsz = sq.header_size(blob)
    sels = every_selection(vol.shape)
    for batch in (sels[3:4], sels, sels * 3):
        want = packed(vol, batch)
        got, guard = batch_host(sq, blob, batch, elem)
        assert guard and np.array_equal(got, want)
        assert sq.last_roi_info() == {"route": 2, "blocks": 0, "h2d_bytes": blob.size - hsz, "voxels": want.size}
        got, guard = batch_device(sq, cuda, dev(cuda, blob), batch, elem)
        assert guard and np.array_equal(got, want)
        assert sq.last_roi_info() == {"route": 2, "blocks": 0, "h2d_bytes": 0, "voxels": want.size}


def test_other_blobs_are_decoded_whole_once(sq, cuda, ref_or_standin):
    vol = vol8((24, 64, 128), seed=3)
    check_route_2(sq, cuda, sq.encode_device_u8("bitswap1->lz4", dev(cuda, vol)).cpu().numpy(), vol, 1)
    vol = numpy_volume((5, 33, 47), "scmos", index=11)
    check_route_2(sq, cuda, sq.encode("bitswap1->lz4", vol), vol, 2)
    vol = numpy_volume((16, 128, 256), "scmos", index=10)
    name = "bitswap1(num_bits_per_plane=1)->lz4(accel=1,blocksize_kb=256,framestep_kb=256,n_chunks_of_input=0)"
    payload, _ = ref_or_standin.pipeline_encode_stages(0, vol, 8)
    h = orc.pack_header(vol.shape, name, payload.size, version="0.5.2", headref="4c45a9b")
    check_route_2(sq, cuda, np.concatenate([np.frombuffer(h.encode(), dtype=np.uint8), payload]), vol, 2)


# ---------------------------------------------------------------------------------------------------------------- Python
def test_python_returns_views_of_one_buffer_in_the_selections_shapes(sq, cuda, big_vol):
    blob = sq.encode("quantiser->lz4", big_vol, nthreads=4)
    full = sq.decode(blob, nthreads=4)
    patches = random_boxes(8, (4, 32, 32), 7)
    sels = patches + [[(0, 16, 5), (3, 99), (10, 2000, 7)]]
    n = sum(count(s) for s in sels)
    out = np.empty(n + 3, dtype=np.uint16)
    got = sq.decode_roi_batch(blob, sels, out=out)
    assert all(np.shares_memory(a, out) for a in got)
    assert [a.shape for a in got] == [cut(full, s).shape for s in sels]
    assert all(np.array_equal(a, cut(full, s)) for a, s in zip(got, sels))
    own = sq.decode_roi_batch(blob, sels)
    assert own[0].base is not None and all(a.base is own[0].base for a in own) and all(np.array_equal(a, b) for a, b in zip(own, got))
    d_out = cuda.empty(n, dtype=cuda.int16, device="cuda")
    views = sq.decode_roi_batch_device(dev(cuda, blob), sels, d_out)
    assert all(v.untyped_storage().data_ptr() == d_out.untyped_storage().data_ptr() for v in views)
    assert all(np.array_equal(host16(v), a) for v, a in zip(views, got))
    batch = d_out[: 8 * 4 * 32 * 32].view(8, 4, 32, 32)   # K patches of one shape: the training batch, no copy
    assert np.array_equal(host16(batch), np.stack([cut(full, p) for p in patches]))
