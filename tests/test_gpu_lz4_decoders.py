"""The LZ4 block decoder of the library (one block per warp, sliding window) on this library's frames, on liblz4's frames
(reference encoder, encoders/lz4_utils.hpp:99-274) and on the oracle's frames; corrupt streams must fail cleanly."""
import numpy as np
import pytest

from sqeazy_b200.synth import numpy_volume
from test_gpu_parity import dev, host16, lz4_inputs

pytestmark = pytest.mark.gpu

@pytest.mark.parametrize("name", [k for k in lz4_inputs().keys() if k != "empty"])
def test_own_frames(sq, cuda, port, name):
    a = lz4_inputs()[name]
    if a is None:
        a = port.bitswap_encode(1, numpy_volume((8, 256, 256), "scmos", index=5)).view(np.uint8)
    payload = sq.lz4_encode_device(dev(cuda, a))
    out = cuda.full((a.size + 64,), 0x5A, dtype=cuda.uint8, device="cuda")
    assert sq.lz4_decode_device(payload, out[: a.size]) == a.size
    h = out.cpu().numpy()
    assert np.array_equal(h[: a.size], a)
    assert np.all(h[a.size:] == 0x5A), "decoder wrote past the end of the output"


@pytest.mark.parametrize("period", [1, 2, 3, 4, 5, 6, 7, 8, 9, 15, 16, 17, 31, 32, 33, 39, 40, 41, 48, 63, 64, 65, 1000, 70000])
def test_foreign_frames_with_any_offset(sq, cuda, port, period):
    """256 KiB blocks from the oracle's encoder: single-step, periodic and far copies"""
    rng = np.random.default_rng(period)
    a = np.tile(rng.integers(0, 256, size=period, dtype=np.uint8), (300000 // period) + 2)[:300001]
    a[100000:100040] = rng.integers(0, 256, size=40, dtype=np.uint8)   # break the period once
    payload = port.lz4_frames_encode(a, chunk=1 << 18)
    out = cuda.zeros(a.size, dtype=cuda.uint8, device="cuda")
    assert sq.lz4_decode_device(dev(cuda, payload), out) == a.size
    assert np.array_equal(out.cpu().numpy(), a)


def test_reference_frames(sq, cuda, ref_or_standin):
    """liblz4 frames made by the reference's lz4_scheme: serial (linked: always the warp decoder), parallel, 64 KiB blocks"""
    vol = numpy_volume((10, 256, 512), "ref", index=9)
    planes = ref_or_standin.bitswap_encode(1, vol)
    for nthreads, config in ((1, b""), (8, b""), (3, b"n_chunks_of_input=7"), (4, b"blocksize_kb=64,framestep_kb=64")):
        payload = ref_or_standin.lz4_encode(planes, nthreads=nthreads, config=config)
        out = cuda.zeros(planes.size, dtype=cuda.int16, device="cuda")
        assert sq.lz4_decode_device(dev(cuda, payload), out) == planes.nbytes, (nthreads, config)
        assert np.array_equal(host16(out), planes), (nthreads, config)


def test_corrupt_blocks_fail_cleanly(sq, cuda, port):
    """bit flips inside the compressed blocks: the decode either fails or returns the promised size (LZ4 has no checksum
    here), never crashes or writes out of bounds, and the library keeps working afterwards"""
    rng = np.random.default_rng(99)
    planes = port.bitswap_encode(1, numpy_volume((4, 256, 256), "scmos", index=2)).view(np.uint8)
    payload = sq.lz4_encode_device(dev(cuda, planes)).cpu().numpy()
    nblocks = (planes.size + 16383) // 16384
    first = 8 + 32 + 4 * nblocks + 7     # skippable header + index header + block words + frame header
    failures = 0
    for trial in range(25):
        bad = payload.copy()
        if trial < 24:
            pos = rng.integers(first, bad.size - 4, size=1 + trial % 5)
            bad[pos] ^= rng.integers(1, 256, size=pos.size, dtype=np.uint8)
        else:
            bad[first + 4: first + 4 + 4096] = 0xFF   # length chains that run past every bound: must be refused
        out = cuda.full((planes.size + 4096,), 0x33, dtype=cuda.uint8, device="cuda")
        try:
            sq.lz4_decode_device(dev(cuda, bad), out[: planes.size])
        except sq.SqeazyError:
            failures += 1
        assert np.all(out[planes.size:].cpu().numpy() == 0x33)
    assert failures > 0
    out = cuda.zeros(planes.size, dtype=cuda.uint8, device="cuda")
    assert sq.lz4_decode_device(dev(cuda, payload), out) == planes.size
    assert np.array_equal(out.cpu().numpy(), planes)


def test_large_ragged_frame_uses_the_tiled_table_build(sq, cuda):
    """>= 8192 blocks: the block table comes from lz4_tile_sums_kernel + lz4_expand_kernel (many CTAs) instead of the
    single-CTA directory scan; ragged block count, short last block, mixed constant / general / stored blocks"""
    n = 16384 * 8192 + 16384 * 37 + 12345
    g = cuda.Generator(device="cuda")
    g.manual_seed(5)
    a = cuda.zeros(n, dtype=cuda.uint8, device="cuda")
    # sparse bytes over the first third, noise in the middle of the second third, zeros elsewhere
    third = n // 3
    sparse = cuda.rand(third, generator=g, device="cuda") < 0.03
    a[:third] = sparse.to(cuda.uint8) * cuda.randint(1, 256, (third,), generator=g, device="cuda", dtype=cuda.uint8)
    a[third + 1000: third + 1000 + (1 << 20)] = cuda.randint(0, 256, (1 << 20,), generator=g, device="cuda", dtype=cuda.uint8)
    payload = sq.lz4_encode_device(a)
    st = sq.last_lz4_stats()
    assert st["general_blocks"] > 1000 and st["constant_blocks"] > 1000 and st["stored_blocks"] > 30
    out = cuda.full((n + 64,), 0x77, dtype=cuda.uint8, device="cuda")
    assert sq.lz4_decode_device(payload, out[:n]) == n
    assert cuda.equal(out[:n], a)
    assert bool((out[n:] == 0x77).all())


def _mixed_content(rng, n):
    """runs, short and long periods, text-like low-entropy bytes, noise, long literal stretches — in random order"""
    parts, total = [], 0
    while total < n:
        kind = rng.integers(0, 7)
        m = int(rng.integers(1, 6000))
        if kind == 0:
            p = np.full(m, rng.integers(0, 256), np.uint8)
        elif kind == 1:
            per = int(rng.integers(1, 40))
            p = np.tile(rng.integers(0, 256, per, dtype=np.uint8), m // per + 1)[:m]
        elif kind == 2:
            per = int(rng.integers(40, 5000))
            p = np.tile(rng.integers(0, 256, per, dtype=np.uint8), m // per + 2)[:m]
        elif kind == 3:
            p = rng.integers(0, 4, m, dtype=np.uint8) * 17
        elif kind == 4:
            p = rng.integers(0, 256, m, dtype=np.uint8)
        elif kind == 5 and parts:
            src = parts[int(rng.integers(0, len(parts)))]
            p = np.tile(src, m // max(src.size, 1) + 1)[:m].copy()        # far repeat of something seen earlier
            if p.size > 10:
                p[rng.integers(0, p.size, max(1, p.size // 50))] ^= 1    # with sparse differences
        else:
            p = (rng.random(m) < 0.06).astype(np.uint8) * rng.integers(1, 256, m, dtype=np.uint8)
        parts.append(p)
        total += p.size
    return np.concatenate(parts)[:n]


@pytest.mark.parametrize("seed", range(10))
def test_random_mixed_streams_from_liblz4_and_own_encoder(sq, cuda, ref_or_standin, seed):
    """the batch walk, the single-sequence path, near / far / overlapping copies and the length chains
    on streams with every kind of sequence: liblz4 frames (64 KiB and 256 KiB blocks, linked and independent) and our own"""
    rng = np.random.default_rng(1000 + seed)
    a = _mixed_content(rng, int(rng.integers(200_000, 900_000)))
    configs = ((1, b""), (4, b""), (2, b"blocksize_kb=64,framestep_kb=64"), (3, b"n_chunks_of_input=3"))
    nthreads, config = configs[seed % len(configs)]
    for payload in (ref_or_standin.lz4_encode(a, nthreads=nthreads, config=config), sq.lz4_encode_device(dev(cuda, a)).cpu().numpy()):
        out = cuda.full((a.size + 32,), 0x42, dtype=cuda.uint8, device="cuda")
        assert sq.lz4_decode_device(dev(cuda, payload), out[: a.size]) == a.size
        h = out.cpu().numpy()
        assert np.array_equal(h[: a.size], a)
        assert np.all(h[a.size:] == 0x42)


@pytest.mark.parametrize("nblocks", [40, 9000], ids=["directory-scan", "tiled-table-build"])
def test_corrupt_index_words_are_refused(sq, cuda, nblocks):
    """The block offsets of this library's frames are prefix sums of the index words in the skippable frame — untrusted
    input. Both table builders (directory CTA below 8192 blocks, lz4_tile_sums_kernel + lz4_expand_kernel above) must
    refuse an index whose sizes do not add up to exactly the frame the index header promises, before any block is read."""
    n = 16384 * nblocks - 77
    g = cuda.Generator(device="cuda")
    g.manual_seed(nblocks)
    sparse = cuda.rand(n, generator=g, device="cuda") < 0.02
    a = sparse.to(cuda.uint8) * cuda.randint(1, 256, (n,), generator=g, device="cuda", dtype=cuda.uint8)
    payload = sq.lz4_encode_device(a).cpu().numpy()
    words = payload[40: 40 + 4 * nblocks].view(np.uint32)

    def try_decode(p):
        out = cuda.full((n + 4096,), 0x11, dtype=cuda.uint8, device="cuda")
        try:
            got = sq.lz4_decode_device(dev(cuda, p), out[:n])
        except sq.SqeazyError:
            got = None
        assert bool((out[n:] == 0x11).all()), "decoder wrote past the end of the output"
        return got, out

    for k, (pos, new) in enumerate([(5, int(words[5]) + 1000), (nblocks // 2, 0x7FFFFFFF), (nblocks - 1, 0xFFFFFFFF),
                                    (3, 0), (nblocks - 2, int(words[nblocks - 2]) - 1)]):
        bad = payload.copy()
        bad[40: 40 + 4 * nblocks].view(np.uint32)[pos] = new
        got, _ = try_decode(bad)
        assert got is None, f"corrupt index word {k} was accepted"
    # sizes that still add up but belong to other blocks: no out-of-bounds access; an error or garbage, never a crash
    bad = payload.copy()
    w = bad[40: 40 + 4 * nblocks].view(np.uint32)
    i = int(np.argmax(w[:-1] != w[1:]))
    w[i], w[i + 1] = w[i + 1], w[i]
    try_decode(bad)
    # an index that claims a frame longer than the stream is not trusted at all: the LZ4 frame behind it is still valid and
    # is walked like a foreign one (or the stream is refused)
    bad = payload.copy()
    bad[32:40].view(np.uint64)[0] += 16
    got, out = try_decode(bad)
    assert got is None or (got == n and cuda.equal(out[:n], a))
    got, out = try_decode(payload)
    assert got == n and cuda.equal(out[:n], a)
