"""Hand-built LZ4 streams (tests/lz4_craft.py) against liblz4, the library the reference decodes with: every stream the
GPU conformance tests (test_gpu_lz4_conformance.py) call valid must come out of LZ4F_decompress as exactly the expected
bytes, every stream they call malformed must be refused. The grid those tests decode is built here from the decoder's
thresholds, and a test reads the thresholds back from lz4_decode.cu so that a retuned constant cannot leave it stale."""
import os
import random
import re
import struct

import numpy as np
import pytest

import lz4_craft as lc
from lz4_craft import Block

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# ------------------------------------------------------------------------------------------------ the decoder's thresholds
# (lz4_decode.cu; test_grid_constants_match_the_decoder keeps these in step)
DEC = {"kWin": 2048, "kRing": 1024, "kBatchOut": 512, "kLitOwn": 4, "kFarMax": 24, "kDeferMin": 8, "kChainTail": 65536}
NEAR = DEC["kWin"] - DEC["kBatchOut"] - 64          # kNear: ring copy up to here, far copy from L2 behind it
SIMPLE_LIT, SIMPLE_MATCH = 15 + 254, 4 + 15 + 254   # a sequence with one length byte at most takes the batch path

OFFSETS = list(range(1, 41)) + [NEAR - 1, NEAR, NEAR + 1, DEC["kWin"] - 1, DEC["kWin"], DEC["kWin"] + 1, 65535, "op"]
MATCHES = list(range(4, 41)) + [255, 256, 257, SIMPLE_LIT, SIMPLE_MATCH, SIMPLE_MATCH + 1, SIMPLE_MATCH + 2,
                                1023, 1024, 1025, 5000]
LITS = [0, DEC["kLitOwn"], DEC["kLitOwn"] + 1, 14, 15, 16, SIMPLE_LIT, SIMPLE_LIT + 1, 1023, 1024, 1025]
LONG_LIT = 20000


def _grid_items():
    """(literals, offset, match length) in stream order: every offset x match length with the literal runs cycling, then
    runs aimed at the batch walk"""
    items = []
    for i, (o, m) in enumerate((o, m) for o in OFFSETS for m in MATCHES):
        items.append((LONG_LIT if i % 211 == 100 else LITS[i % len(LITS)], o, m))
    far = DEC["kFarMax"]
    items += [(1, NEAR + 1 + 13 * k, far) for k in range(40)]                 # far group: four at a time
    items += [(1, NEAR + 5 + k, far + 1) for k in range(40)]                  # one byte too long: whole warp
    items += [(k % 3, NEAR + 40 + 7 * k, 4 + k % 22) for k in range(64)]      # mixed far lengths around the limit
    items += [(4, 7, 28)] * 16 + [(0, 100, 300)]                              # a batch of exactly kBatchOut bytes
    items += [(4, 9, 28)] * 15 + [(5, 9, 28), (0, 3, 300)]                   # and of one more
    items += [(2, NEAR + 3, 62)] * 8 + [(0, 1, 300)]                          # kBatchOut bytes of far copies
    items += [(15, 3, 19)] * 80 + [(16, 5, 19)] * 80                          # 20- and 21-byte sequences: headers at every
    items += [(14, 33, 18)] * 80                                              # position of the 512-byte stream chunks
    return items


def grid_frame(bsid, linked, seed=0):
    """one frame of the grid: blocks filled to the frame's maximum (the last one short). A sequence whose offset does not
    reach yet waits until it does (65535 never does in an independent 64 KiB block); "op" copies from the block's first
    byte."""
    rng = random.Random(seed * 10 + bsid)
    bmax = lc.BLOCK_MAX[bsid]
    blocks, seqs, op, window, pending = [], [], 0, 0, []
    todo = _grid_items()

    def fits(item, lit):
        o = op + lit if item[1] == "op" else item[1]
        return 1 <= o <= min(op + lit + window, 65535)

    i = 0
    while i < len(todo) or pending:
        ready = next((k for k, p in enumerate(pending) if fits(p, p[0])), None)
        if ready is not None:
            item = pending.pop(ready)
        elif i < len(todo):
            item = todo[i]
            i += 1
            if not fits(item, item[0]):
                pending.append(item)
                continue
        elif seqs or op:
            item = None        # close the block: what waits may fit in the next one
        else:
            break              # nothing fits in a fresh block either
        if item is None or op + item[0] + item[2] > bmax - 16:
            blocks.append(Block(seqs, rng.randbytes(bmax - op)))
            window = min(window + bmax, 65535) if linked else 0
            seqs, op = [], 0
            if item is None:
                continue
            if not fits(item, item[0]):
                pending.append(item)
                continue
        lit, o, m = item
        o = op + lit if o == "op" else o
        seqs.append((rng.randbytes(lit), o, m))
        op += lit + m
    if seqs or op:
        blocks.append(Block(seqs, rng.randbytes(16)))
    return lc.frame(blocks, linked=linked, bsid=bsid)


# ------------------------------------------------------------------------------------------------ frame features
def _content_block(rng, n, window=0):
    """a block of about n bytes (>= 16) with short and long matches, some reaching `window` bytes in front of it"""
    seqs, op = [], 0
    while op + 60 < n - 16:
        lit = rng.choice([0, 1, 3, 17, 40])
        m = rng.choice([4, 7, 19, 40, 200])
        if op + lit + m > n - 16:
            break
        o = rng.randint(1, min(op + lit + window, 65535)) if op + lit + window else None
        if o is None:
            lit = max(lit, 1)
            o = 1
        seqs.append((rng.randbytes(lit), o, m))
        op += lit + m
    return Block(seqs, rng.randbytes(n - op))


def _linked_blocks(rng, sizes, window=0):
    """content blocks of a linked frame, each reaching into all of the frame in front of it (up to 64 KiB)"""
    out = []
    for n in sizes:
        out.append(_content_block(rng, n, min(window, 65535)))
        window += n
    return out


def feature_streams():
    """name -> (stream, decoded bytes): frame features every decoder of LZ4 frames must take"""
    rng = random.Random(5)
    S = {}
    S["blocks_1m"] = lc.frame([_content_block(rng, 1 << 20), _content_block(rng, 300000)], bsid=6)
    S["blocks_4m_linked"] = lc.frame([_content_block(rng, 4 << 20), _content_block(rng, 70000, 65535)], bsid=7, linked=True)
    blocks = _linked_blocks(rng, (65536, 65536, 1234))
    S["block_checksums"] = lc.frame(blocks, linked=True, block_checksum=True)
    S["content_checksum"] = lc.frame(blocks, linked=True, content_checksum=True)
    S["content_size"] = lc.frame(blocks, linked=True, content_size=True)
    S["dict_id"] = lc.frame(blocks, linked=True, dict_id=0x12345678)
    S["everything"] = lc.frame(blocks, linked=True, block_checksum=True, content_checksum=True, content_size=True,
                               dict_id=7)
    # short blocks in front of the last one (liblz4 writes full ones; any writer may flush early)
    S["short_nonfinal"] = lc.frame([_content_block(rng, n) for n in (1000, 70, 65536, 20, 5000)])
    S["short_nonfinal_linked"] = lc.frame(_linked_blocks(rng, (1000, 70, 65536, 20, 5000)), linked=True)
    # single-block frames that are not full, followed by more frames
    S["short_single_block_frames"] = lc.stream(*[lc.frame([_content_block(rng, n)]) for n in (3000, 65536, 17, 40000)],
                                               lc.frame([_content_block(rng, 65536), _content_block(rng, 100)]))
    S["empty_and_skippable_frames"] = lc.stream(lc.frame([]), lc.skippable(b"x" * 13, 3), lc.frame([_content_block(rng, 9000)]),
                                                lc.frame([], linked=True), lc.skippable(), lc.frame([_content_block(rng, 65536)]),
                                                lc.skippable(b"tail", 15), lc.frame([]))
    # stored blocks of a linked frame that later blocks copy from
    st = [Block(stored=rng.randbytes(n)) for n in (65536, 3000)]
    S["stored_in_linked"] = lc.frame([st[0], _content_block(rng, 65536, 65535), st[1], _content_block(rng, 20000, 65535),
                                      Block([(b"", 65535, 4000), (b"", 60000, 300), (b"a", 3001, 5000)], rng.randbytes(20))],
                                     linked=True)
    # many short linked blocks: an offset of 65535 reaches back across dozens of them (irregular chain steps)
    many = _linked_blocks(rng, [rng.randint(900, 1600) for _ in range(150)])
    many.append(Block([(b"", 65535, 3000), (b"", 40000, 700), (b"q", 65535, 30)], rng.randbytes(16)))
    many += [Block([(rng.randbytes(1), 65535, 1000 + k)], rng.randbytes(12)) for k in range(20)]
    S["linked_many_short_blocks"] = lc.frame(many, linked=True)
    # exactly 64 KiB blocks (regular chain steps) with short ones between them (irregular steps), and two linked frames
    sizes = (65536, 65536, 1000, 65536, 65536, 65536, 30000, 65536, 65536, 65536, 65536, 7)
    S["linked_chain_regular_irregular"] = lc.stream(
        lc.frame(_linked_blocks(rng, sizes), linked=True), lc.frame(_linked_blocks(rng, sizes[:5]), linked=True))
    return S


def closed_form_streams():
    """near misses of the closed-form run block (token 1F, byte, offset 1, length bytes, token 50, five bytes), one
    16 KiB block per frame, the exact form first; and stored blocks at the sizes around the 256-byte vector copy"""
    v = b"\x61"
    n = 16384
    near = [
        Block([(v, 1, n - 6)], v * 5),                               # the closed form itself
        Block([(v, 1, n - 6)], v * 4 + b"w"),                        # last byte differs
        Block([(v, 1, n - 6)], b"w" + v * 4),
        Block([(v + b"b", 2, n - 7)], v * 5),                        # offset 2
        Block([(v, 1, n - 7)], v * 6),                               # six final literals
        Block([(v, 1, n - 6 - 300)], v * 305),                       # a long final run
        Block([(v, 1, 300), (b"", 1, n - 311)], v * 5),              # two matches
        Block([(v * 2, 1, n - 7)], v * 5),                           # two literals in front
        Block([(b"w", 1, n - 6)], v * 5),                            # match byte differs from the final ones
    ]
    parts = [lc.frame([b]) for b in near]
    rng = random.Random(11)
    parts += [lc.frame([Block(stored=rng.randbytes(k))]) for k in (255, 256, 257, 271, 272, 16384, 1, 4097)]
    parts.append(lc.frame([Block(stored=rng.randbytes(k)) for k in (255, 256, 257, 271, 272)]))
    return lc.stream(*parts)


def malformed_streams():
    """name -> (stream, decoded size the caller offers): streams every decoder must refuse"""
    rng = random.Random(9)
    good = lc.frame([_content_block(rng, 4000)])[0]
    S = {}
    S["offset0_batch"] = lc.frame([Block([(b"ab", 1, 8), (b"c", 0, 6), (b"d", 2, 9)], rng.randbytes(16))])
    S["offset0_single"] = lc.frame([Block([(b"ab", 1, 8), (b"c", 0, 600)], rng.randbytes(16))])
    S["independent_in_front"] = lc.stream(lc.frame([Block(stored=rng.randbytes(5000))]),
                                          lc.frame([Block([(b"xyz", 100, 50)], rng.randbytes(16))]))
    S["linked_head_in_front"] = lc.stream(lc.frame([Block(stored=rng.randbytes(5000))], linked=True),
                                          lc.frame([Block([(b"xyz", 100, 50)], rng.randbytes(16)),
                                                    _content_block(rng, 3000, 65535)], linked=True))
    # a linked block behind the head of its frame reaching in front of the frame, into a linked / independent /
    # stored frame; nine stored blocks in front of it keep the stream on the deferred route at the default threshold
    front = {"linked": lc.frame([_content_block(rng, 65536), _content_block(rng, 3000, 65535)], linked=True),
             "independent": lc.frame([_content_block(rng, 65536), _content_block(rng, 3000)]),
             "stored": lc.frame([Block(stored=rng.randbytes(65536))])}
    for k, f in front.items():
        S["linked_crosses_into_" + k] = lc.stream(
            f, lc.frame([Block(stored=rng.randbytes(100)) for _ in range(9)] +
                        [Block([(b"", 2000, 20), (b"", 1, 40)], rng.randbytes(16))], linked=True))
        S["linked_crosses_into_" + k + "_in_batch"] = lc.stream(
            f, lc.frame([Block(stored=rng.randbytes(1000)), _content_block(rng, 2000, 1000),
                         Block([(b"ab", 3, 5), (b"c", 3100, 9), (b"", 1, 8)], rng.randbytes(16))], linked=True))
    S["literal_chain_off_block"] = (good + lc.frame([Block()])[0][:7] + struct.pack("<I", 40) + b"\xf0" + b"\xff" * 39
                                    + b"\0\0\0\0", None)
    S["match_chain_off_block"] = (lc.frame([Block([(b"abcd", 4, 19)], b"")])[0][:-5] + b"\0\0\0\0", None)
    blk = lc.encode_block([(b"abcd", 4, 30)], b"x" * 20)
    S["literals_past_block_end"] = (lc.frame([])[0][:7] + struct.pack("<I", len(blk) - 3) + blk[:-3] + b"\0\0\0\0", None)
    S["block_past_stream_end"] = (good[:-4] + struct.pack("<I", 5000) + b"\0" * 100, None)
    S["truncated_header"] = (good + lc.frame([])[0][:6], None)
    for bsid in (0, 1, 3):
        S[f"bsid{bsid}"] = lc.frame([_content_block(rng, 200)], bsid=bsid)
    for ver in (0, 2, 3):
        S[f"version{ver}"] = lc.frame([_content_block(rng, 200)], version=ver)
    return {k: (s, 70000) for k, (s, _) in S.items()}


def tolerated_streams():
    """name -> (stream, decoded bytes): broken rules a decoder may accept (with the obvious bytes) or refuse"""
    rng = random.Random(13)
    S = {}
    S["ends_with_match"] = lc.frame([Block([(b"abcdefgh", 4, 8)], None), _content_block(rng, 100)])
    S["four_final_literals"] = lc.frame([Block([(b"abcdefgh", 4, 8)], b"1234"), _content_block(rng, 100)])
    S["last_match_11_from_end"] = lc.frame([Block([(b"abcdefgh", 4, 4)], b"xyzuvwa")])
    S["nonfinal_above_block_max"] = lc.frame([Block([(b"z", 1, 70000)], rng.randbytes(16)), _content_block(rng, 100)])
    return S


# ------------------------------------------------------------------------------------------------ the tests
@pytest.fixture(scope="module")
def standin():
    from oracle import oracle

    s = oracle.standin()
    if not s.available:
        pytest.skip("liblz4 not installed")
    return s


def _liblz4_gives(standin, data, want):
    rc, out = standin.lz4_decode_bytes(np.frombuffer(data, np.uint8), len(want))
    return rc == 0 and out.tobytes() == want


def test_xxh32_known_values():
    assert lc.xxh32(b"") == 0x02CC5D05 and lc.xxh32(b"abc") == 0x32D153FF
    assert lc.xxh32(b"", 1) != lc.xxh32(b"")


@pytest.mark.parametrize("bsid", [4, 5, 6, 7])
@pytest.mark.parametrize("linked", [False, True], ids=["independent", "linked"])
def test_grid_frames_decode_with_liblz4(standin, bsid, linked):
    data, want = grid_frame(bsid, linked)
    assert want is not None and len(want) > 1_000_000
    assert _liblz4_gives(standin, data, want)
    got, frames = lc.check_stream(data)
    assert got == want and frames[0].linked == linked


def test_grid_covers_every_offset_and_length():
    """each (offset, match length) pair of the grid is written in the 256 KiB blocks; 64 KiB independent blocks lack only
    the offsets they cannot hold"""
    for bsid, linked in ((5, False), (4, True), (4, False)):
        data, _ = grid_frame(bsid, linked)
        _, frames = lc.check_stream(data)
        p, seen = 7, set()
        for w in frames[0].words:
            size = w & ~lc.STORED
            seqs, _ = lc.parse_block(data[p + 4:p + 4 + size])
            seen |= {(o, m) for _, o, m in seqs}
            p += 4 + size
        missing = {(o, m) for o in OFFSETS if o != "op" for m in MATCHES} - seen
        if bsid == 4 and not linked:
            assert {o for o, _ in missing} == {65535}
        else:
            assert not missing, sorted(missing)[:10]


def test_feature_streams_decode_with_liblz4(standin):
    for name, (data, want) in feature_streams().items():
        assert want is not None, name
        assert _liblz4_gives(standin, data, want), name
        assert lc.check_stream(data, shrink=False)[0] == want, name


def test_closed_form_and_stored_streams_decode_with_liblz4(standin):
    data, want = closed_form_streams()
    assert _liblz4_gives(standin, data, want)


def test_malformed_streams_are_refused_by_liblz4(standin):
    for name, (data, n) in malformed_streams().items():
        for size in (n, 200000):
            rc, _ = standin.lz4_decode_bytes(np.frombuffer(data, np.uint8), size)
            assert rc != 0, (name, size)
        with pytest.raises(lc.Broken):
            lc.check_stream(data)


def test_frame_crossing_match_is_refused_but_in_frame_one_decodes(standin):
    """liblz4 limits a linked block's window to its own frame: the same match decodes when the bytes are in the frame"""
    rng = random.Random(1)
    a = lc.frame([Block(stored=rng.randbytes(65536))], linked=True)
    crossing = lc.stream(a, lc.frame([Block(stored=rng.randbytes(1000)), Block([(b"", 2000, 20)], b"abcde" * 3)], linked=True))
    inside = lc.stream(a, lc.frame([Block(stored=rng.randbytes(3000)), Block([(b"", 2000, 20)], b"abcde" * 3)], linked=True))
    assert crossing[1] is None and inside[1] is not None
    assert _liblz4_gives(standin, *inside)
    rc, _ = standin.lz4_decode_bytes(np.frombuffer(crossing[0], np.uint8), 65536 + 1035)
    assert rc != 0


@pytest.mark.parametrize("name", ["ends_with_match", "four_final_literals", "last_match_11_from_end"])
def test_end_rules_agree_with_liblz4(name):
    """the strict reader and LZ4_decompress_safe (room for exactly the block's bytes, where liblz4 checks the end rules)
    refuse the same end-rule violations; the minimal legal endings pass"""
    if lc.liblz4() is None:
        pytest.skip("liblz4 not installed")
    data, _ = tolerated_streams()[name]
    blk = data[11:11 + (struct.unpack_from("<I", data, 7)[0] & ~lc.STORED)]
    assert lc.check_block(blk) is not None
    assert lc.decompress_block(blk, len(lc.expand(*lc.parse_block(blk)))) < 0
    for seqs, final in (([(b"abcdefgh", 4, 7)], b"12345"), ([(b"abcdefgh", 4, 4)], b"x" * 8), ([], b"1234"), ([], b"")):
        ok = lc.encode_block(seqs, final)
        n = len(lc.expand(seqs, final))
        assert lc.check_block(ok) is None and lc.decompress_block(ok, n) == n, (seqs, final)


def test_long_length_chains_cross_the_32_byte_steps(standin):
    """length chains of 31, 32 and 33 bytes of 255 (read_ext looks at 32 bytes per step), literals and matches"""
    rng = random.Random(2)
    for k in (30, 31, 32, 33, 64, 65):
        lit = rng.randbytes(15 + 255 * k + 7)
        ml = 19 + 255 * k + 11
        blk = Block([(lit, 5, ml), (b"", 1, 15 + 4 + 255 * k)], rng.randbytes(12))
        enc = blk.data()
        assert enc[1:1 + k] == b"\xff" * k
        data, want = lc.frame([blk])
        assert _liblz4_gives(standin, data, want), k


def test_check_stream_reports_broken_rules():
    rng = random.Random(3)
    ok, _ = lc.frame([_content_block(rng, 5000)])
    lc.check_stream(ok)
    big = lc.frame([Block(stored=rng.randbytes(100)), Block([(b"ab", 1, 70000)], b"x" * 12)])[0]
    with pytest.raises(lc.Broken, match="above the block maximum"):
        lc.check_stream(big)
    fat = lc.frame([Block([(b"abcdefghijklmnopqrstuvwxyz", 26, 4)], b"0123456789ab")])[0]
    with pytest.raises(lc.Broken, match="not smaller than raw"):
        lc.check_stream(fat)
    with pytest.raises(lc.Broken, match="bad header checksum"):
        lc.check_stream(ok[:6] + bytes([ok[6] ^ 1]) + ok[7:])


def test_grid_constants_match_the_decoder():
    """the grid is built from the decoder's thresholds: retuning one must fail here, not leave the grid aimed elsewhere"""
    src = open(os.path.join(ROOT, "sqeazy_b200", "csrc", "device", "lz4_decode.cu")).read()
    got = {}
    for name in DEC:
        m = re.search(r"constexpr\s+\w+\s+" + name + r"\s*=\s*(\d+)\s*;", src)
        assert m, name
        got[name] = int(m.group(1))
    assert got == DEC
    assert re.search(r"constexpr\s+\w+\s+kNear\s*=\s*kWin\s*-\s*kBatchOut\s*-\s*64\s*;", src)
    assert NEAR == 1472
