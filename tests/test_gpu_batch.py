"""Batches of independent stacks through sqyx_*_batch_device_UI16 (BASELINE cfg4: decode-only of reference-produced
blobs; cfg5: a time-lapse stream). The reference handles a list of files one after the other
(verbs/compress.hpp:204-338); here up to 8 stacks are in flight, and every one of them must come out exactly as it
does from a call of its own."""
import numpy as np
import pytest

from oracle import oracle as orc
from sqeazy_b200.synth import numpy_volume
from test_gpu_parity import dev, host16

pytestmark = pytest.mark.gpu

CFG5 = "remove_background(threshold=110)->bitswap4->lz4"


@pytest.mark.parametrize("n", [1, 3, 8, 11, 19])
def test_timelapse_batch_matches_single_calls(sq, cuda, port, n):
    shape = (8, 128, 256)
    vols = [numpy_volume(shape, "scmos", index=i) for i in range(n)]
    d_vols = [dev(cuda, v) for v in vols]
    blobs = sq.encode_batch_device(CFG5, d_vols)
    assert len(blobs) == n
    outs = [cuda.empty(shape, dtype=cuda.int16, device="cuda") for _ in range(n)]
    sq.decode_batch_device(blobs, outs)
    for v, blob, out in zip(vols, blobs, outs):
        want = port.remove_background(v.reshape(-1), 110).reshape(shape)
        assert np.array_equal(host16(out), want)                     # batch encode + batch decode
        single = cuda.empty(shape, dtype=cuda.int16, device="cuda")
        sq.decode_device(blob, single)                                # batch-encoded blob through the single-stack call
        assert np.array_equal(host16(single), want)
        assert np.array_equal(sq.decode(blob.cpu().numpy()), want)   # ... and through the host entry point


def test_decode_batch_of_mixed_pipelines(sq, cuda):
    shape = (6, 96, 160)
    pipes = ["bitswap1->lz4", "quantiser->lz4", "pass_through", "rmestbkrd->bitswap1->lz4", "lz4", "bitswap2->lz4", "quantiser",
             "bitswap1", "remove_background(threshold=105)->bitswap1->lz4", "bitswap8->lz4"]
    vols = [numpy_volume(shape, "ref" if i % 3 == 0 else "scmos", index=20 + i) for i in range(len(pipes))]
    blobs = [sq.encode_device(p, dev(cuda, v)).clone() for p, v in zip(pipes, vols)]
    want = []
    for b in blobs:
        o = cuda.empty(shape, dtype=cuda.int16, device="cuda")
        sq.decode_device(b, o)
        want.append(host16(o).copy())
    outs = [cuda.full(shape, -1, dtype=cuda.int16, device="cuda") for _ in blobs]
    sq.decode_batch_device(blobs, outs)
    for o, w in zip(outs, want):
        assert np.array_equal(host16(o), w)


def test_decode_batch_of_reference_blobs(sq, cuda, ref_or_standin):
    """cfg4 in small: blobs made by the reference's own stage chain, both framings (block-linked frame = sqy CLI default,
    one frame per chunk = the multi-threaded mode), decoded as one batch, bit-exact"""
    name = "bitswap1(num_bits_per_plane=1)->lz4(accel=1,blocksize_kb=256,framestep_kb=256,n_chunks_of_input=0)"
    shape = (16, 128, 256)
    vols, blobs = [], []
    for i in range(10):
        vol = numpy_volume(shape, "scmos", index=40 + i)
        payload, _ = ref_or_standin.pipeline_encode_stages(0, vol, 1 if i % 2 else 8)
        h = orc.pack_header(vol.shape, name, payload.size, version="0.5.2", headref="4c45a9b")
        vols.append(vol)
        blobs.append(cuda.from_numpy(np.concatenate([np.frombuffer(h.encode(), dtype=np.uint8), payload])).cuda())
    outs = [cuda.empty(shape, dtype=cuda.int16, device="cuda") for _ in blobs]
    sq.decode_batch_device(blobs, outs)
    for v, o in zip(vols, outs):
        assert np.array_equal(host16(o), v)


def test_decode_batch_of_linked_blobs_on_the_deferred_route(sq, cuda, ref_or_standin):
    """stacks of 12 linked 256 KiB blocks each: every lane of the batch runs the deferred-reference decoder (pass 1 and the
    chain walk side by side on two streams of its own) at the same time as the others"""
    name = "bitswap1(num_bits_per_plane=1)->lz4(accel=1,blocksize_kb=256,framestep_kb=256,n_chunks_of_input=0)"
    shape = (24, 256, 256)
    vols, blobs = [], []
    for i in range(9):
        vol = numpy_volume(shape, "scmos" if i % 2 else "ref", index=70 + i)
        payload, _ = ref_or_standin.pipeline_encode_stages(0, vol, 1)
        h = orc.pack_header(vol.shape, name, payload.size, version="0.5.2", headref="4c45a9b")
        vols.append(vol)
        blobs.append(cuda.from_numpy(np.concatenate([np.frombuffer(h.encode(), dtype=np.uint8), payload])).cuda())
    for _ in range(2):
        outs = [cuda.full(shape, -1, dtype=cuda.int16, device="cuda") for _ in blobs]
        sq.decode_batch_device(blobs, outs)
        for v, o in zip(vols, outs):
            assert np.array_equal(host16(o), v)


def test_batch_reports_the_broken_stack(sq, cuda):
    shape = (4, 64, 128)
    vols = [numpy_volume(shape, "scmos", index=60 + i) for i in range(5)]
    blobs = [b.clone() for b in sq.encode_batch_device("bitswap1->lz4", [dev(cuda, v) for v in vols])]
    blobs[2][: 512] = 0x78                   # header gone (it sits right-aligned in a 256-byte slot)
    outs = [cuda.empty(shape, dtype=cuda.int16, device="cuda") for _ in blobs]
    with pytest.raises(sq.SqeazyError) as e:
        sq.decode_batch_device(blobs, outs)
    assert "[0, 0, 1, 0, 0]" in str(e.value)
    for i in (0, 1, 3, 4):                   # the others were decoded all the same
        assert np.array_equal(host16(outs[i]), vols[i])
    assert sq.decode_batch_device([], []) == []
    assert sq.encode_batch_device("bitswap1->lz4", []) == []
    with pytest.raises(sq.SqeazyError):
        sq.encode_batch_device("no_such_stage->lz4", [dev(cuda, vols[0])])
