"""Block-LINKED LZ4 frames — what the reference writes in its serial mode, i.e. the sqy CLI default and any
`SQY_PipelineEncode_UI16(..., nthreads = 1)` (encoders/lz4_utils.hpp:99-173, SURVEY F6; BASELINE cfg4 decodes such blobs).
Both GPU routes must give the bytes liblz4 was fed: the block-after-block route (every linked block waits for its
predecessor) and the deferred-reference route (lz4_decode.cu: all blocks at once, bytes from in front of a block are
remembered as origins and resolved afterwards)."""
import numpy as np
import pytest

from sqeazy_b200.synth import numpy_volume
from test_gpu_lz4_decoders import _mixed_content
from test_gpu_parity import dev

pytestmark = pytest.mark.gpu


@pytest.fixture(params=[0, 1, 8], ids=["serial", "deferred-always", "default"])
def route(request, sq, cuda):
    prev = sq.set_lz4_defer_min(request.param)
    yield request.param
    sq.set_lz4_defer_min(prev)


def roundtrip(sq, cuda, ref_or_standin, a, config=b"", nthreads=1):
    a = np.ascontiguousarray(a).view(np.uint8).ravel()
    payload = ref_or_standin.lz4_encode(a, nthreads=nthreads, config=config)
    out = cuda.full((a.size + 64,), 0x5A, dtype=cuda.uint8, device="cuda")
    assert sq.lz4_decode_device(dev(cuda, payload), out[: a.size]) == a.size
    h = out.cpu().numpy()
    assert np.array_equal(h[: a.size], a)
    assert np.all(h[a.size:] == 0x5A)
    return payload


CONTENT = {
    # zero runs that run across many block borders: one origin byte feeds whole blocks
    "zeros": lambda rng: np.zeros(3_000_000, np.uint8),
    "thresholded_planes": lambda rng: None,
    # a 200-byte pattern repeated for 2 MB: every block starts with a match into its predecessor, with wrap-around
    "period200": lambda rng: np.tile(rng.integers(0, 256, 200, dtype=np.uint8), 10_000),
    "period7": lambda rng: np.tile(rng.integers(0, 256, 7, dtype=np.uint8), 300_000),
    # repeats at a distance close to the 64 KiB window, across borders
    "period60000": lambda rng: np.tile(rng.integers(0, 256, 60_000, dtype=np.uint8), 40),
    "noise": lambda rng: rng.integers(0, 256, 1_500_000, dtype=np.uint8),              # stored blocks inside a linked frame
    "mixed": lambda rng: _mixed_content(rng, 2_500_000),
    "ragged_small": lambda rng: _mixed_content(rng, 300_001),
}


@pytest.mark.parametrize("name", list(CONTENT))
@pytest.mark.parametrize("config", [b"", b"blocksize_kb=64,framestep_kb=64"], ids=["256k", "64k"])
def test_linked_frames_decode_bit_exact(sq, cuda, port, ref_or_standin, route, name, config):
    rng = np.random.default_rng(len(name) * 101)
    a = CONTENT[name](rng)
    if a is None:
        vol = numpy_volume((12, 512, 512), "scmos", index=4)
        a = port.bitswap_encode(1, port.remove_background(vol.reshape(-1), 107)).view(np.uint8)
    roundtrip(sq, cuda, ref_or_standin, a, config)


def test_several_linked_frames_and_independent_ones_in_one_stream(sq, cuda, ref_or_standin, route):
    """n_chunks_of_input with one thread: a few linked frames one after the other; then frames with independent blocks
    (multi-threaded mode) in front of and behind a linked one"""
    rng = np.random.default_rng(77)
    a = _mixed_content(rng, 4_000_000)
    roundtrip(sq, cuda, ref_or_standin, a, b"n_chunks_of_input=3")
    parts = [a[:1_000_000], a[1_000_000:3_200_000], a[3_200_000:]]
    payload = np.concatenate([ref_or_standin.lz4_encode(parts[0], nthreads=4), ref_or_standin.lz4_encode(parts[1], nthreads=1),
                              ref_or_standin.lz4_encode(parts[2], nthreads=4)])
    out = cuda.zeros(a.size, dtype=cuda.uint8, device="cuda")
    assert sq.lz4_decode_device(dev(cuda, payload), out) == a.size
    assert np.array_equal(out.cpu().numpy(), a)


def test_routes_agree_on_a_reference_blob(sq, cuda, ref_or_standin):
    """whole blob of the reference's serial mode through SQY_Decode_UI16, both routes"""
    from oracle import oracle as orc

    vol = numpy_volume((24, 512, 512), "scmos", index=12)
    name = "bitswap1(num_bits_per_plane=1)->lz4(accel=1,blocksize_kb=256,framestep_kb=256,n_chunks_of_input=0)"
    payload, _ = ref_or_standin.pipeline_encode_stages(0, vol, 1)
    h = orc.pack_header(vol.shape, name, payload.size, version="0.5.2", headref="4c45a9b")
    blob = np.concatenate([np.frombuffer(h.encode(), dtype=np.uint8), payload])
    for n in (0, 8):
        prev = sq.set_lz4_defer_min(n)
        try:
            assert np.array_equal(sq.decode(blob), vol)
        finally:
            sq.set_lz4_defer_min(prev)


def test_corrupt_linked_stream_fails_cleanly(sq, cuda, ref_or_standin, route):
    rng = np.random.default_rng(5)
    a = _mixed_content(rng, 3_000_000)
    payload = ref_or_standin.lz4_encode(a, nthreads=1).copy()
    for pos in (payload.size // 3, payload.size // 2, payload.size - 3000):
        bad = payload.copy()
        bad[pos: pos + 64] ^= 0xA5
        out = cuda.full((a.size + 4096,), 0x11, dtype=cuda.uint8, device="cuda")
        try:
            sq.lz4_decode_device(dev(cuda, bad), out[: a.size])
        except sq.SqeazyError:
            pass
        assert bool((out[a.size:] == 0x11).all())      # whatever happened, nothing was written behind the buffer


def test_linked_frames_into_unaligned_buffers(sq, cuda, ref_or_standin, route):
    """destination at odd addresses: the chain walk takes its element-wise route (no 16-byte vectors), same bytes"""
    rng = np.random.default_rng(9)
    a = _mixed_content(rng, 2_000_003)
    payload = dev(cuda, ref_or_standin.lz4_encode(a, nthreads=1))
    for off in (1, 3, 8):
        out = cuda.full((a.size + 64,), 0x33, dtype=cuda.uint8, device="cuda")
        assert sq.lz4_decode_device(payload, out[off: off + a.size]) == a.size
        h = out.cpu().numpy()
        assert np.array_equal(h[off: off + a.size], a)
        assert np.all(h[:off] == 0x33) and np.all(h[off + a.size:] == 0x33)
