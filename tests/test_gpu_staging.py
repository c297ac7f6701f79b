"""Host-pointer entry points with caller buffers of both kinds (SURVEY §8b: every buffer is caller-allocated; the
reference's `nthreads` knob, src/sqeazy.cpp:108-142). Pageable buffers go through the pinned chunk ring with
`nthreads` staging threads (csrc/staging.cu); the bytes must not depend on the route."""
import numpy as np
import pytest

from sqeazy_b200.synth import numpy_volume

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("pipeline", ["bitswap1->lz4", "rmestbkrd->bitswap1->lz4", "quantiser->lz4", "pass_through"])
@pytest.mark.parametrize("shape", [(40, 512, 512), (33, 500, 517)])   # 20 MiB (not a multiple of the 32 MiB chunk), ragged
def test_pageable_staging_matches_single_thread(sq, cuda, pipeline, shape):
    vol = numpy_volume(shape, "scmos", index=3)
    # (the encoder is deterministic: every route and thread count writes the same bytes)
    ref_blob = sq.encode(pipeline, vol, nthreads=1)
    want = sq.decode(sq.encode(pipeline, vol, nthreads=1), nthreads=1)
    if pipeline in ("bitswap1->lz4", "pass_through"):   # the lossless ones
        assert np.array_equal(want.reshape(vol.shape), vol)
    for t in (2, 5, 0, 64):             # <= 0 and > cores: all cores (sqeazy_algorithms.hpp:14-22)
        blob = sq.encode(pipeline, vol, nthreads=t)
        assert np.array_equal(blob, ref_blob), f"blob bytes differ at nthreads={t}"
        assert np.array_equal(sq.decode(blob, nthreads=1), want), f"encode nthreads={t}"
        assert np.array_equal(sq.decode(blob, nthreads=t), want), f"decode nthreads={t}"


def test_staging_many_chunks_and_pinned_buffers(sq, cuda):
    """160 MiB = five full 32 MiB ring chunks (the ring has three slots: slots are reused) from pageable memory, and the
    same volume from page-locked memory (one DMA, no ring)"""
    vol = numpy_volume((80, 1024, 1024), "scmos")
    blob = sq.encode("bitswap1->lz4", vol, nthreads=4)
    back = sq.decode(blob, nthreads=4)
    assert np.array_equal(back.reshape(vol.shape), vol)
    pinned = cuda.empty(vol.shape, dtype=cuda.int16).pin_memory()
    pinned.numpy().view(np.uint16)[...] = vol
    blob_p = sq.encode("bitswap1->lz4", pinned.numpy().view(np.uint16), nthreads=4)
    assert np.array_equal(sq.decode(blob_p, nthreads=1).reshape(vol.shape), vol)
    out_p = cuda.empty(vol.shape, dtype=cuda.int16).pin_memory()
    sq.decode(blob, nthreads=4, out=out_p.numpy().view(np.uint16).reshape(-1))
    assert np.array_equal(out_p.numpy().view(np.uint16), vol)


def test_staging_uint8(sq, cuda):
    rng = np.random.default_rng(5)
    vol = np.clip(np.rint(20 + 2 * rng.standard_normal((24, 1024, 1024))), 0, 255).astype(np.uint8)
    many = sq.encode_u8("bitswap1->lz4", vol, nthreads=6)
    assert np.array_equal(sq.decode_u8(many, nthreads=1).reshape(vol.shape), vol)
    assert np.array_equal(sq.decode_u8(many, nthreads=6).reshape(vol.shape), vol)


@pytest.mark.parametrize("pipeline", ["bitswap1->lz4", "rmestbkrd->bitswap1->lz4", "remove_background(threshold=110)->bitswap4->lz4",
                                      "rmbkrd(threshold=104)->bitswap2->lz4", "quantiser->lz4"])
@pytest.mark.parametrize("kind", ["pageable", "pinned"])
def test_streamed_host_paths_match_the_device_path(sq, cuda, pipeline, kind):
    """stacks of >= 512 MiB take the streamed host paths (api.cu: host_encode_streamed, take_slabs, decode_streamed, ship_slabs):
    z-slabs are transposed and LZ4-compressed while the next slab is still on the PCIe bus; slabs of the decoded stack leave
    as soon as they are transposed back. 80 frames of 2048x2048 = 640 MiB = 2.5 slabs (ragged last slab). The voxels must be
    the ones the all-at-once device path produces."""
    from sqeazy_b200.synth import torch_volume

    shape = (80, 2048, 2048)
    d_vol = torch_volume(shape, "scmos", index=2)
    d_blob = sq.encode_device(pipeline, d_vol)
    d_want = cuda.empty(shape, dtype=cuda.int16, device="cuda")
    sq.decode_device(d_blob, d_want)
    want = d_want.cpu().numpy().view(np.uint16)
    if pipeline == "bitswap1->lz4":
        assert np.array_equal(want, d_vol.cpu().numpy().view(np.uint16))
    if kind == "pinned":
        h_vol = cuda.empty(shape, dtype=cuda.int16).pin_memory()
        h_out = cuda.empty(shape, dtype=cuda.int16).pin_memory()
    else:
        h_vol = cuda.empty(shape, dtype=cuda.int16)
        h_out = cuda.empty(shape, dtype=cuda.int16)
    h_vol.copy_(d_vol)
    del d_vol, d_want
    vol = h_vol.numpy().view(np.uint16)
    out = h_out.numpy().view(np.uint16)
    for t in (1, 6):
        blob = sq.encode(pipeline, vol, nthreads=t)
        assert np.array_equal(blob, d_blob.cpu().numpy()), "the streamed host path and the device path must write the same bytes"
        assert sq.decompressed_shape(blob) == list(shape) or tuple(sq.decompressed_shape(blob)) == shape
        out[...] = 0xABCD
        sq.decode(blob, nthreads=t, out=out.reshape(-1))                      # streamed encode + streamed decode
        assert np.array_equal(out, want), f"nthreads={t}"
    # a streamed blob through the device path, a device-path blob through the streamed host decode
    d_out = cuda.empty(shape, dtype=cuda.int16, device="cuda")
    sq.decode_device(cuda.from_numpy(blob).cuda(), d_out)
    assert np.array_equal(d_out.cpu().numpy().view(np.uint16), want)
    out[...] = 0
    sq.decode(d_blob.cpu().numpy(), nthreads=3, out=out.reshape(-1))
    assert np.array_equal(out, want)
    sq.release_scratch()
