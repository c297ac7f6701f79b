"""Pins the oracle (oracle/sqy_oracle.c + oracle/oracle.py) against the reference's known-answer vectors, the committed
golden vectors (made by the reference's own code, tests/golden/make_golden.py) and, where oracle/_ref exists, the
reference's stage classes run live. CPU only."""
import numpy as np
import pytest

from oracle import oracle as orc


# ---- bitswap: tests/test_bitswap_scheme_impl.cpp:286-329 ----
KAT = {1: [0x00FF, 0x0F0F, 0x3333, 0x5555], 2: [0x0055, 0xAAFF, 0x1B1B, 0x1B1B], 4: [0x0123, 0x4567, 0x89AB, 0xCDEF]}


@pytest.mark.parametrize("w", [1, 2, 4])
def test_bitswap_kat(port, w):
    out = port.bitswap_encode(w, np.arange(16, dtype=np.uint16))
    assert list(out[12:]) == KAT[w]
    assert not out[:12].any()
    assert np.array_equal(port.bitswap_decode(w, out), np.arange(16, dtype=np.uint16))


@pytest.mark.parametrize("w", [1, 2, 4, 8])
@pytest.mark.parametrize("name", ["kat", "ragged", "aligned"])
def test_bitswap_golden(port, golden, w, name):
    a = golden[f"bitswap_{name}_in"]
    enc = port.bitswap_encode(w, a)
    assert np.array_equal(enc, golden[f"bitswap_{name}_w{w}"])
    assert np.array_equal(port.bitswap_decode(w, enc), a)


@pytest.mark.parametrize("w", [1, 2, 4, 8])
def test_bitswap_vs_ref_live(port, ref, w):
    rng = np.random.default_rng(w)
    for n in (0, 1, 15, 16, 127, 128, 4096 + 3, 128 * 33):
        a = rng.integers(0, 65536, size=n, dtype=np.uint16)
        enc = port.bitswap_encode(w, a)
        if n:
            assert np.array_equal(enc, ref.bitswap_encode(w, a, nthreads=1, scalar=(n % 128 != 0)))
            assert np.array_equal(ref.bitswap_decode(w, enc), a)


# ---- background ----
def test_remove_background_golden(port, golden):
    assert np.array_equal(port.remove_background(golden["bg_vol"], 110), golden["bg_rm110"])


def test_rmestbkrd_golden(port, golden):
    vol = golden["bg_vol"]
    l2 = int(golden["bg_l2_bytes"][0])
    sup = port.darkest_face_supports(vol, l2)
    assert np.array_equal(sup.view(np.uint32), golden["bg_supports"].view(np.uint32))  # bit-exact floats
    out, thr = port.rmestbkrd(vol, l2)
    assert np.array_equal(out, golden["bg_rmest"])
    assert thr == int(np.uint16(golden["bg_supports"].min()))


def test_rmestbkrd_l2_portion_golden(port, golden):
    """frame (1536x2048 elements) larger than the build host's L2 (bytes): only 0.75*L2 elements are sampled (SURVEY F9)"""
    from sqeazy_b200.synth import numpy_volume

    big = numpy_volume(tuple(golden["bg_big_seed_shape"]), "ref", index=2)
    sup = port.darkest_face_supports(big, int(golden["bg_l2_bytes"][0]))
    assert np.array_equal(sup.view(np.uint32), golden["bg_big_supports"].view(np.uint32))
    other = port.darkest_face_supports(big, 1 << 30)
    assert other.shape == (4,)


def test_support_constant_cube(port):
    """tests/test_background_scheme_impl.cpp:21-51: constant-1 cube -> all four supports ~ 1"""
    vol = np.ones((8, 8, 8), dtype=np.uint16)
    sup = port.darkest_face_supports(vol, 2 << 20)
    assert np.allclose(sup, 1.0, rtol=1e-4)


def test_histogram_kat(port):
    """tests/test_histogram_fill.cpp:31-53: c % 32 over 1024 values -> 32 per bin"""
    a = (np.arange(1024) % 32).astype(np.uint16)
    h = port.histogram(a)
    assert (h[:32] == 32).all() and not h[32:].any()


# ---- quantiser ----
@pytest.mark.parametrize("name", ["q_small", "q_big", "q_ramp"])
def test_quantiser_golden(port, golden, name):
    a = golden[name + "_in"]
    hist = port.histogram(a)
    expect = np.zeros(65536, dtype=np.uint32)
    expect[golden[name + "_hist_nonzero_idx"]] = golden[name + "_hist_nonzero_val"]
    assert np.array_equal(hist, expect)
    enc, dec = port.quantiser_luts(hist)
    assert np.array_equal(enc, golden[name + "_enc"])
    assert np.array_equal(dec, golden[name + "_dec"])


def test_quantiser_ramp_kat(port):
    """tests/test_quantiser_impl.cpp:862-1020: ramp 0..4095 -> enc[0]=0, enc[16]=enc[0]+1, rec[0..15]=8, rec[last]=4088"""
    a = np.arange(4096, dtype=np.uint16)
    hist = port.histogram(a)
    assert (hist[:4096] == 1).all()
    enc, dec = port.quantiser_luts(hist)
    assert enc[0] == 0 and enc[16] == enc[0] + 1
    rec = port.lut_decode(port.lut_apply(a, enc), dec)
    assert (rec[:16] == 8).all() and rec[16] != 8 and rec[-1] == 4088
    assert len(set(dec.tolist())) == 256  # decode LUT entries unique (:1022-1086)


def test_quantiser_lossless_kat(port):
    """tests/test_quantiser_impl.cpp:992-1020: <= 256 distinct values round-trip exactly"""
    a = (np.arange(1 << 14) % 63).astype(np.uint16) * 7
    enc, dec = port.quantiser_luts(port.histogram(a))
    assert np.array_equal(port.lut_decode(port.lut_apply(a, enc), dec), a)


def test_quantiser_lut_string_golden(golden):
    s = orc.lut_to_verbatim(golden["q_big_dec"])
    assert s.encode() == golden["q_big_lutstring"].tobytes()


def test_quantiser_vs_ref_live(port, ref):
    rng = np.random.default_rng(5)
    for a in (np.clip(rng.exponential(400, 1 << 17) + 100, 0, 65535).astype(np.uint16),
              rng.integers(0, 65536, 1 << 17, dtype=np.uint16), np.zeros(1000, dtype=np.uint16)):
        hist, enc, dec = ref.quantiser_setup(a)
        e2, d2 = port.quantiser_luts(port.histogram(a))
        assert np.array_equal(enc, e2) and np.array_equal(dec, d2)
        codes, _ = ref.quantiser_encode(a)
        assert np.array_equal(codes, port.lut_apply(a, e2))


# ---- lz4 ----
@pytest.mark.parametrize("kb,expect", [(0, 64), (64, 64), (128, 64), (160, 256), (256, 256), (511, 256), (640, 1024),
                                       (2048, 1024), (2560, 4096), (4096, 4096), (8000, 4096)])
def test_closest_blocksize(port, kb, expect):
    """tests/test_lz4_utils_impl.cpp:147-180"""
    assert port.closest_blocksize_kb(kb) == expect


def test_lz4_decode_reference_payloads(port, golden):
    from sqeazy_b200.synth import numpy_volume  # noqa: F401

    planes = port.bitswap_encode(1, golden["lz4_vol"])
    for key in ("lz4_serial", "lz4_parallel"):
        got = port.lz4_frames_decode(golden[key], planes.nbytes)
        assert np.array_equal(got.view(np.uint16), planes), key
    got = port.lz4_frames_decode(golden["lz4_linked"], golden["lz4_linked_in"].nbytes)
    assert np.array_equal(got.view(np.uint16), golden["lz4_linked_in"])


def test_standin_lz4_encoder_writes_the_reference_payloads(port, golden):
    """oracle.Standin restates the reference's lz4_scheme encode over liblz4: the same bytes as the reference made for the
    golden vectors (one linked frame, a frame per 256 KiB chunk, cross-block matches) and the same default config"""
    s = orc.standin()
    if not s.available:
        pytest.skip("liblz4 not present")
    planes = port.bitswap_encode(1, golden["lz4_vol"])
    assert np.array_equal(s.lz4_encode(planes, nthreads=1), golden["lz4_serial"])
    assert np.array_equal(s.lz4_encode(planes, nthreads=4), golden["lz4_parallel"])
    assert np.array_equal(s.lz4_encode(golden["lz4_linked_in"], nthreads=1), golden["lz4_linked"])
    assert s.lz4_config(b"").encode() == golden["lz4_default_config"].tobytes()
    rc, out = s.lz4_decode_u16(golden["lz4_parallel"], planes.size)
    assert rc == 0 and np.array_equal(out, planes)


def test_lz4_port_encoder_is_reference_decodable(port, ref_or_standin):
    rng = np.random.default_rng(9)
    a = np.repeat(rng.integers(0, 50, 40000, dtype=np.uint16), 7)[: 3 * 131072 + 77]
    payload = port.lz4_frames_encode(a, chunk=262144)
    rc, out = ref_or_standin.lz4_decode_u16(payload, a.size)
    assert rc == 0 and np.array_equal(out, a)
    assert np.array_equal(port.lz4_frames_decode(payload, a.nbytes).view(np.uint16), a)


def test_lz4_skippable_frames_pass_the_reference_decoder(port, ref_or_standin):
    """the block index this library prepends is a skippable LZ4 frame; the reference's loop (lz4.hpp:257-339) skips it"""
    import struct

    a = (np.arange(1 << 16) % 251).astype(np.uint16)
    payload = port.lz4_frames_encode(a)
    skip = np.frombuffer(struct.pack("<II", 0x184D2A5B, 12) + b"x" * 12, dtype=np.uint8)
    rc, out = ref_or_standin.lz4_decode_u16(np.concatenate([skip, payload]), a.size)
    assert rc == 0 and np.array_equal(out, a)
    assert np.array_equal(port.lz4_frames_decode(np.concatenate([skip, payload]), a.nbytes).view(np.uint16), a)


# ---- control layer ----
def test_parser_fixtures():
    """tests/test_string_parsers_impl.cpp:13-120 style fixtures"""
    assert orc.to_pairs("a->b(c=d)->e") == [("a", ""), ("b", "c=d"), ("e", "")]
    assert orc.minors("x=1,y=<verbatim>a,b=c-></verbatim>,z=3") == {"x": "1", "y": "<verbatim>a,b=c-></verbatim>", "z": "3"}
    assert orc.to_pairs("q(l=<verbatim>->,=</verbatim>)->lz4")[0] == ("q", "l=<verbatim>->,=</verbatim>")


def test_pipeline_possible_fixtures():
    """tests/test_pipeline_interface.cpp:28-61, tests/test_dynamic_pipeline_impl.cpp:679-709"""
    assert orc.can_be_built_from("bitswap1->lz4")
    assert not orc.can_be_built_from("")
    assert not orc.can_be_built_from("bswap1_lz4")
    assert not orc.can_be_built_from("bitswap1->lz4!!")


def test_header_roundtrip():
    """tests/test_sqeazy_header_impl.cpp:101-188: size % sizeof(T) == 0, pack/unpack, trailing bytes tolerated"""
    name = "quantiser(decode_lut_string=<verbatim>ab/+c=</verbatim>)->lz4(accel=1)"
    h = orc.pack_header([3, 5, 7], name, 42)
    assert len(h) % 2 == 0 and h.endswith(orc.HEADER_DELIM)
    u = orc.unpack_header(h.encode() + b"\x00\xffgarbage|01307#!")
    assert u["pipeline"] == name and u["shape"] == [3, 5, 7] and u["bytes"] == 42 and u["size"] == len(h)


# ------------------------------------------------------------------------------------------------ uint8 volumes
@pytest.mark.parametrize("w", [1, 2, 4])
def test_bitswap8_kat_and_ref_live(port, w):
    """the scalar template of bitplane_reorder_scalar.hpp:27-116 with raw_type = uint8_t: first element of a group in the
    most significant field, most significant plane first; the C port equals the reference's own instantiation"""
    ref = orc.ref()
    a = np.arange(8, dtype=np.uint8)
    e = port.bitswap8_encode(w, a)
    if w == 1:   # planes 7..3 empty; bit 2 of 0..7 = 00001111, bit 1 = 00110011, bit 0 = 01010101
        assert e.tolist() == [0, 0, 0, 0, 0, 0x0F, 0x33, 0x55]
    if w == 4:   # P = 2: high nibbles first, then low nibbles, pairs packed first-element-high
        assert e.tolist() == [0x00, 0x00, 0x00, 0x00, 0x01, 0x23, 0x45, 0x67]
    rng = np.random.default_rng(w)
    for n in (0, 1, 7, 8, 9, 64, 1000, 4099):
        x = rng.integers(0, 256, n, dtype=np.uint8)
        y = port.bitswap8_encode(w, x)
        assert np.array_equal(port.bitswap8_decode(w, y), x)
        if ref.available:
            assert np.array_equal(ref.bitswap8_encode(w, x), y)
            assert np.array_equal(ref.bitswap8_decode(w, y), x)


def test_remove_background8_vs_ref_live(port):
    ref = orc.ref()
    x = np.random.default_rng(5).integers(0, 256, 5000, dtype=np.uint8)
    for t in (0, 1, 100, 255, 300):   # 300 is stored as uint8 (44), remove_background_scheme_impl.hpp:41-44
        y = port.remove_background8(x, t)
        assert np.array_equal(y, np.where(x > (t & 0xFF), x - (t & 0xFF), 0).astype(np.uint8))
        if ref.available:
            assert np.array_equal(ref.remove_background8(x, t), y)
