"""The LZ4 decoder on hand-built streams (tests/lz4_craft.py; the same streams decode with liblz4 in test_lz4_craft.py):
a grid of offsets, match lengths and literal runs around the decoder's thresholds, frame features liblz4 at level 1 never
writes, and malformed streams. Bytes are compared exactly, and every decode writes into a buffer with a sentinel tail."""
import functools
import struct

import numpy as np
import pytest

import lz4_craft as lc
from test_gpu_linked_frames import route  # noqa: F401  (fixture: serial / deferred-always / default route)
from test_gpu_parity import dev
from test_lz4_craft import (closed_form_streams, feature_streams, grid_frame, malformed_streams, tolerated_streams)

pytestmark = pytest.mark.gpu

SENTINEL = 0x5A
PAD = 256


@functools.lru_cache(maxsize=None)
def _grid(bsid, linked):
    data, want = grid_frame(bsid, linked)
    return np.frombuffer(data, np.uint8), np.frombuffer(want, np.uint8)


def decode(sq, cuda, payload, n, out_off=0, src_off=0):
    """decodes into out[out_off: out_off + n] of a sentinel-filled buffer, the payload starting src_off bytes into a device
    buffer of its own; returns (decoded count or None when refused, the whole output buffer on the host)"""
    p = dev(cuda, payload)
    if src_off:
        big = cuda.full((p.numel() + src_off + 64,), 0xEE, dtype=cuda.uint8, device="cuda")
        big[src_off: src_off + p.numel()] = p
        p = big[src_off: src_off + p.numel()]
    out = cuda.full((out_off + n + PAD,), SENTINEL, dtype=cuda.uint8, device="cuda")
    try:
        got = sq.lz4_decode_device(p, out[out_off: out_off + n])
    except sq.SqeazyError:
        got = None
    h = out.cpu().numpy()
    assert np.all(h[:out_off] == SENTINEL) and np.all(h[out_off + n:] == SENTINEL), "decoder wrote outside its output"
    return got, h[out_off: out_off + n]


def assert_decodes(sq, cuda, payload, want, **kw):
    got, h = decode(sq, cuda, payload, want.size, **kw)
    assert got == want.size, kw
    if not np.array_equal(h, want):
        bad = int(np.argmax(h != want))
        raise AssertionError(f"{kw}: first wrong byte at {bad} of {want.size}")


# ------------------------------------------------------------------------------------------------ path grid
@pytest.mark.parametrize("bsid", [4, 5], ids=["64k", "256k"])
@pytest.mark.parametrize("out_off", [0, 1, 4, 16, 128])
def test_grid_independent_blocks_output_placement(sq, cuda, bsid, out_off):
    payload, want = _grid(bsid, False)
    assert_decodes(sq, cuda, payload, want, out_off=out_off)


@pytest.mark.parametrize("bsid", [4, 5], ids=["64k", "256k"])
def test_grid_independent_blocks_payload_placement(sq, cuda, bsid):
    payload, want = _grid(bsid, False)
    for src_off in range(16):
        assert_decodes(sq, cuda, payload, want, src_off=src_off)


@pytest.mark.parametrize("bsid", [4, 5], ids=["64k", "256k"])
def test_grid_linked_blocks(sq, cuda, route, bsid):
    payload, want = _grid(bsid, True)
    for out_off in (0, 1, 4, 16, 128):
        assert_decodes(sq, cuda, payload, want, out_off=out_off)
    for src_off in (1, 3, 7, 15):
        assert_decodes(sq, cuda, payload, want, src_off=src_off)


@pytest.mark.parametrize("bsid", [6, 7], ids=["1m", "4m"])
@pytest.mark.parametrize("linked", [False, True], ids=["independent", "linked"])
def test_grid_big_blocks(sq, cuda, route, bsid, linked):
    payload, want = _grid(bsid, linked)
    assert_decodes(sq, cuda, payload, want)
    assert_decodes(sq, cuda, payload, want, out_off=1, src_off=5)


@pytest.mark.parametrize("out_off", [0, 1, 4, 16, 128])
def test_closed_form_near_misses_and_stored_sizes(sq, cuda, out_off):
    """only the exact closed form may take the 16-byte fill; stored blocks around the 256-byte vector copy"""
    data, want = closed_form_streams()
    assert_decodes(sq, cuda, np.frombuffer(data, np.uint8), np.frombuffer(want, np.uint8), out_off=out_off)


# ------------------------------------------------------------------------------------------------ frame features
@pytest.mark.parametrize("name", list(feature_streams()))
def test_frame_features(sq, cuda, route, name):
    data, want = feature_streams()[name]
    payload, want = np.frombuffer(data, np.uint8), np.frombuffer(want, np.uint8)
    assert_decodes(sq, cuda, payload, want)
    assert_decodes(sq, cuda, payload, want, out_off=1, src_off=3)


# ------------------------------------------------------------------------------------------------ malformed streams
@pytest.mark.parametrize("name", list(malformed_streams()))
def test_malformed_streams_are_refused(sq, cuda, route, name):
    """refused with SqeazyError, nothing written outside the output, and the next decode works"""
    data, n = malformed_streams()[name]
    got, _ = decode(sq, cuda, np.frombuffer(data, np.uint8), n)
    assert got is None, f"{name}: accepted ({got} bytes)"
    got, _ = decode(sq, cuda, np.frombuffer(data, np.uint8), n, out_off=3)
    assert got is None, f"{name}: accepted ({got} bytes) into an unaligned buffer"
    payload, want = _grid(4, True)
    assert_decodes(sq, cuda, payload, want)


@pytest.mark.parametrize("name", list(tolerated_streams()))
def test_tolerated_rule_breaks_stay_in_bounds(sq, cuda, route, name):
    """end-rule violations and an oversize block: the obvious bytes or a refusal, never a write outside the buffers"""
    data, want = tolerated_streams()[name]
    want = np.frombuffer(want, np.uint8)
    for out_off in (0, 1):
        got, h = decode(sq, cuda, np.frombuffer(data, np.uint8), want.size, out_off=out_off)
        assert got is None or (got == want.size and np.array_equal(h, want)), name


def test_more_blocks_than_the_table_holds_is_refused(sq, cuda):
    """k_lz4_decode_capacity: output bytes / 16 KiB + 1024 blocks; a stream of more small blocks is refused cleanly"""
    rng = np.random.default_rng(3)
    blocks = [lc.Block(stored=rng.integers(0, 256, 90, dtype=np.uint8).tobytes()) for _ in range(1100)]
    data, want = lc.frame(blocks)
    got, _ = decode(sq, cuda, np.frombuffer(data, np.uint8), len(want))
    assert got is None
    payload, want = _grid(4, False)
    assert_decodes(sq, cuda, payload, want)


# ------------------------------------------------------------------------------------------------ the encoder
def check_encoded(sq, ref_or_standin, payload, a):
    """this library's payload for `a` against liblz4 and the strict reader: liblz4 decodes it (the frame decoder on the
    whole payload, LZ4_decompress_safe block by block with room for exactly the block's bytes), no block breaks a rule,
    and the index in the skippable frame agrees with the frame"""
    n, p = a.size, payload.tobytes()
    assert len(p) <= sq.lz4_bound(n)
    rc, back = ref_or_standin.lz4_decode_bytes(payload, n)
    assert rc == 0 and np.array_equal(back, a)
    got, frames = lc.check_stream(p)
    assert got == a.tobytes()
    magic, size = struct.unpack_from("<II", p, 0)
    imagic, version, bb, nblk, raw, fbytes = struct.unpack_from("<IIIIQQ", p, 8)
    assert (magic, imagic, version, bb, nblk, raw) == (0x184D2A5B, 0x42595153, 1, 16384, -(-n // 16384), n)
    assert size == 32 + 4 * nblk and fbytes == len(p) - 8 - size
    words = list(struct.unpack_from(f"<{nblk}I", p, 40))
    assert len(frames) == 1 and frames[0].flg == 0x60 and frames[0].bd == 0x40
    assert frames[0].words == words and frames[0].raw == [min(16384, n - 16384 * i) for i in range(nblk)]
    pos = 8 + size + 7
    for i, w in enumerate(words):
        csize = w & ~lc.STORED
        if not w & lc.STORED:
            assert lc.decompress_block(p[pos + 4: pos + 4 + csize], frames[0].raw[i]) == frames[0].raw[i], i
        pos += 4 + csize


def _encoder_corpus():
    """name -> list of (input, pitch hint)"""
    rng = np.random.default_rng(21)
    noise = lambda k: rng.integers(0, 256, k, dtype=np.uint8)

    def mixed(k):
        a = noise(k)
        a[rng.random(k) < 0.7] = 0
        return a

    C = {}
    C["sizes_1_to_13"] = [(noise(k), 0) for k in range(1, 14)] + [(np.full(k, 7, np.uint8), 0) for k in range(1, 14)]
    C["ragged_block_tails"] = [(mixed(16384 * k + t), 0) for k in (1, 3) for t in (1, 4, 5, 11, 12, 13, 17)]
    runs = []
    for end in [16384] + [1024 * j + d for j in range(1, 16) for d in (-1, 0, 1)]:
        a = noise(16384 * 2)
        a[end - 300: end] = 0                                  # a run that ends right at the border
        a[16384 + end - 40: 16384 + end] = 9
        runs.append((a, 0))
    C["runs_ending_at_borders"] = runs
    C["periodic_across_sub_blocks"] = [(np.tile(noise(p), 2 * 16384 // p + 1)[:2 * 16384 + 5], 0) for p in (1, 2, 3, 7, 64, 100, 1000)]
    rows = []
    for pitch in range(32, 8193, 32):
        r = np.tile(noise(pitch), 32768 // pitch + 1)[:32768]
        r[rng.integers(0, r.size, 200)] ^= 0x10                 # rows that repeat with sparse differences
        rows += [(r, 0), (r, pitch)]
    C["row_repeats_every_pitch"] = rows
    early = []
    for k in range(4):
        a = np.zeros(16384 * 2, np.uint8)
        a[:2048] = noise(2048)
        a[16384: 16384 + 2048 + 64 * k] = noise(2048 + 64 * k)
        early.append((a, 0))
    C["noise_then_compressible"] = early
    lit = []
    for gap in (15, 16, 269, 270, 1000, 5000, 14000):
        parts = []
        while sum(x.size for x in parts) < 40000:
            parts += [noise(gap), np.zeros(40, np.uint8)]
        lit.append((np.concatenate(parts), 0))
    C["long_literal_runs"] = lit
    C["constant_ragged_tails"] = [(np.full(16384 * 2 + t, v, np.uint8), 0) for v in (0, 0xAB)
                                  for t in list(range(0, 20)) + [100, 1000, 16383]]
    return C


@pytest.mark.parametrize("name", list(_encoder_corpus()))
def test_encoder_obeys_liblz4_block_rules(sq, cuda, ref_or_standin, name):
    if lc.liblz4() is None:
        pytest.skip("liblz4 not installed")
    for a, pitch in _encoder_corpus()[name]:
        payload = sq.lz4_encode_device(dev(cuda, a), pitch=pitch).cpu().numpy()
        try:
            check_encoded(sq, ref_or_standin, payload, a)
        except (AssertionError, lc.Broken) as e:
            raise AssertionError(f"{name}: {a.size} bytes, pitch {pitch}: {e}") from e
