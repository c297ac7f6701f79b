"""GPU parity tests: every call goes through the C ABI of libsqeazy.so (ctypes), results are compared bit-for-bit with
the oracle on the same seeded inputs, with the committed golden vectors (reference-made), and — where oracle/_ref
travelled to the box — with the reference's own stage code and decoder."""
import numpy as np
import pytest

from oracle import oracle as orc
from sqeazy_b200.synth import numpy_volume

pytestmark = pytest.mark.gpu


def dev(cuda, a):
    a = np.ascontiguousarray(a)
    if a.dtype == np.uint16:
        return cuda.from_numpy(a.view(np.int16)).cuda()
    if a.dtype == np.uint32:
        return cuda.from_numpy(a.view(np.int32)).cuda()
    return cuda.from_numpy(a).cuda()


def host16(t):
    return t.cpu().numpy().view(np.uint16)


# ------------------------------------------------------------------------------------------------ bitswap
@pytest.mark.parametrize("w", [1, 2, 4, 8])
@pytest.mark.parametrize("n", [0, 1, 15, 16, 127, 128, 1000 + 389, 128 * 40, 128 * 4099, 1 << 21])
def test_bitswap_parity(sq, cuda, port, w, n):
    rng = np.random.default_rng(n + w)
    a = rng.integers(0, 65536, size=n, dtype=np.uint16)
    d_in = dev(cuda, a) if n else cuda.empty(0, dtype=cuda.int16, device="cuda")
    d_out = cuda.empty_like(d_in)
    sq.bitswap_encode_device(w, d_in, d_out)
    enc = host16(d_out)
    assert np.array_equal(enc, port.bitswap_encode(w, a))
    d_back = cuda.empty_like(d_in)
    sq.bitswap_decode_device(w, d_out, d_back)
    assert np.array_equal(host16(d_back), a)


@pytest.mark.parametrize("w", [1, 2, 4, 8])
@pytest.mark.parametrize("name", ["kat", "ragged", "aligned"])
def test_bitswap_golden(sq, cuda, golden, w, name):
    a = golden[f"bitswap_{name}_in"]
    d_in = dev(cuda, a)
    d_out = cuda.empty_like(d_in)
    sq.bitswap_encode_device(w, d_in, d_out)
    assert np.array_equal(host16(d_out), golden[f"bitswap_{name}_w{w}"])


def test_bitswap_unaligned_pointers(sq, cuda, port):
    """sub-tensor views start at odd offsets: the generic kernel must take over"""
    a = np.random.default_rng(3).integers(0, 65536, size=128 * 64 + 1, dtype=np.uint16)
    d = dev(cuda, a)
    out = cuda.empty(a.size + 1, dtype=cuda.int16, device="cuda")
    sq.bitswap_encode_device(1, d[1:], out[1 : a.size])
    assert np.array_equal(host16(out[1 : a.size]), port.bitswap_encode(1, a[1:]))


@pytest.mark.parametrize("w", [1, 4])
@pytest.mark.parametrize("thr", [1, 97, 110, 65535])
def test_fused_threshold_bitswap(sq, cuda, port, w, thr):
    vol = numpy_volume((8, 64, 128), "scmos", index=4)
    d_in = dev(cuda, vol)
    d_out = cuda.empty_like(d_in)
    sq.bitswap_encode_device(w, d_in.view(-1), d_out.view(-1), threshold=thr)
    assert np.array_equal(host16(d_out).ravel(), port.bitswap_encode(w, port.remove_background(vol, thr)))


# ------------------------------------------------------------------------------------------------ background
@pytest.mark.parametrize("thr", [0, 1, 110, 40000])
@pytest.mark.parametrize("n", [1, 7, 8, 4096 + 5])
def test_remove_background(sq, cuda, port, thr, n):
    a = np.random.default_rng(n).integers(0, 65536, size=n, dtype=np.uint16)
    d_in = dev(cuda, a)
    d_out = cuda.empty_like(d_in)
    sq.remove_background_device(d_in, d_out, thr)
    assert np.array_equal(host16(d_out), port.remove_background(a, thr))


def test_remove_background_golden(sq, cuda, golden):
    d_in = dev(cuda, golden["bg_vol"])
    d_out = cuda.empty_like(d_in)
    sq.remove_background_device(d_in.view(-1), d_out.view(-1), 110)
    assert np.array_equal(host16(d_out), golden["bg_rm110"])


@pytest.mark.parametrize("shape,preset", [((12, 96, 128), "scmos"), ((5, 40, 64), "ref"), ((3, 16, 16), "random"), ((4, 1536, 2048), "ref")])
@pytest.mark.parametrize("l2", [2 << 20, 1 << 16, 0, 1 << 30])
def test_estimate_background(sq, cuda, port, shape, preset, l2):
    vol = numpy_volume(shape, preset, index=2)
    sup, thr = sq.estimate_background_device(dev(cuda, vol), l2_bytes=l2)
    exp = port.darkest_face_supports(vol, l2)
    assert np.array_equal(sup.view(np.uint32), exp.view(np.uint32))
    assert thr == int(np.uint16(exp.min()))


def test_estimate_background_golden(sq, cuda, golden):
    sup, _ = sq.estimate_background_device(dev(cuda, golden["bg_vol"]), l2_bytes=int(golden["bg_l2_bytes"][0]))
    assert np.array_equal(sup.view(np.uint32), golden["bg_supports"].view(np.uint32))
    big = numpy_volume(tuple(golden["bg_big_seed_shape"]), "ref", index=2)
    sup, _ = sq.estimate_background_device(dev(cuda, big), l2_bytes=int(golden["bg_l2_bytes"][0]))
    assert np.array_equal(sup.view(np.uint32), golden["bg_big_supports"].view(np.uint32))


# ------------------------------------------------------------------------------------------------ quantiser
@pytest.mark.parametrize("n", [1, 1000, (1 << 20) + 3, (1 << 22) + 17])
@pytest.mark.parametrize("kind", ["concentrated", "uniform", "high"])
def test_histogram(sq, cuda, port, n, kind):
    rng = np.random.default_rng(n)
    if kind == "concentrated":
        a = np.clip(rng.normal(100, 3, n), 0, 65535).astype(np.uint16)
    elif kind == "uniform":
        a = rng.integers(0, 65536, size=n, dtype=np.uint16)
    else:
        a = rng.integers(49000, 65536, size=n, dtype=np.uint16)
    hist = cuda.zeros(65536, dtype=cuda.int32, device="cuda")
    sq.histogram_device(dev(cuda, a), hist)
    cuda.cuda.synchronize()
    assert np.array_equal(hist.cpu().numpy().view(np.uint32), port.histogram(a))


HIST_KINDS = {
    # (bins below 49152 are CTA-private shared-memory atomics, the rest global atomics: quantise.cu)
    "camera": lambda rng, n: np.clip(rng.normal(100, 3, n), 0, 65535),
    "one_value": lambda rng, n: np.full(n, 4242),
    "zero_mode": lambda rng, n: np.abs(rng.normal(0, 4, n)),
    "two_modes": lambda rng, n: np.where(rng.random(n) < 0.5, rng.normal(300, 2, n), rng.normal(9000, 2, n)),
    "window_edges": lambda rng, n: 1000 + rng.integers(-40, 40, n),              # wider than the window on both sides
    "private_bin_limit": lambda rng, n: 49152 + rng.integers(-20, 20, n),        # mode at the edge of the CTA-private bins
    "above_private_bins": lambda rng, n: 60000 + rng.integers(-5, 5, n),         # global atomics only
    "drifting": lambda rng, n: np.linspace(50, 3000, n) + rng.normal(0, 2, n),   # the mode of the first voxels is not the stack's
    "wide": lambda rng, n: rng.exponential(400, n) + 100,
}


@pytest.mark.parametrize("kind", list(HIST_KINDS))
def test_histogram_distributions(sq, cuda, port, kind):
    """exact counts whatever the distribution: one value, modes at both ends of the private bins, values above them, drift"""
    n = (1 << 24) + 11
    rng = np.random.default_rng(len(kind))
    a = np.clip(np.rint(HIST_KINDS[kind](rng, n)), 0, 65535).astype(np.uint16)
    hist = cuda.zeros(65536, dtype=cuda.int32, device="cuda")
    d = dev(cuda, a)
    sq.histogram_device(d, hist)
    sq.histogram_device(d[5: n - 3], hist)                                        # unaligned view, accumulating
    cuda.cuda.synchronize()
    want = port.histogram(a).astype(np.uint64) + port.histogram(a[5: n - 3])
    assert np.array_equal(hist.cpu().numpy().view(np.uint32), want.astype(np.uint32))


@pytest.mark.parametrize("kind", ["uniform", "all_high", "bright_tail"])
def test_histogram_bright_stacks(sq, cuda, port, kind):
    """stacks with many voxels above the CTA-private bins (>= 49152): a thread that has sent more than 64 of them to global
    atomics leaves the rest to a second sweep in shared memory (quantise.cu) — enough iterations per thread here to get there"""
    n = (1 << 26) + 5
    rng = np.random.default_rng(7)
    if kind == "uniform":
        a = rng.integers(0, 65536, size=n, dtype=np.uint16)
    elif kind == "all_high":
        a = rng.integers(49152, 65536, size=n, dtype=np.uint16)
    else:                               # camera-like, the second half of the stack saturated here and there
        a = np.clip(rng.normal(100, 3, n), 0, 65535).astype(np.uint16)
        a[n // 2:][rng.random(n - n // 2) < 0.2] = 65535
    hist = cuda.zeros(65536, dtype=cuda.int32, device="cuda")
    d = dev(cuda, a)
    sq.histogram_device(d, hist)
    sq.histogram_device(d[3: n - 1], hist)                                        # unaligned view, accumulating
    cuda.cuda.synchronize()
    want = port.histogram(a).astype(np.uint64) + port.histogram(a[3: n - 1])
    assert np.array_equal(hist.cpu().numpy().view(np.uint32), want.astype(np.uint32))


def test_histogram_unaligned_and_accumulating(sq, cuda, port):
    a = np.random.default_rng(0).integers(0, 3000, size=(1 << 21) + 5, dtype=np.uint16)
    d = dev(cuda, a)
    hist = cuda.zeros(65536, dtype=cuda.int32, device="cuda")
    sq.histogram_device(d[3:], hist)
    sq.histogram_device(d[:3], hist)
    cuda.cuda.synchronize()
    assert np.array_equal(hist.cpu().numpy().view(np.uint32), port.histogram(a))


@pytest.mark.parametrize("name", ["q_small", "q_big", "q_ramp"])
def test_quantiser_stage_golden(sq, cuda, port, golden, name):
    a = golden[name + "_in"]
    d = dev(cuda, a)
    hist = cuda.zeros(65536, dtype=cuda.int32, device="cuda")
    sq.histogram_device(d, hist)
    cuda.cuda.synchronize()
    enc, dec = sq.quantiser_luts(hist.cpu().numpy().view(np.uint32))
    assert np.array_equal(enc, golden[name + "_enc"]) and np.array_equal(dec, golden[name + "_dec"])
    codes = cuda.empty(a.size, dtype=cuda.uint8, device="cuda")
    sq.lut_apply_device(d, codes, enc)
    assert np.array_equal(codes.cpu().numpy(), port.lut_apply(a, enc))
    back = cuda.empty(a.size, dtype=cuda.int16, device="cuda")
    sq.lut_decode_device(codes, back, dec)
    assert np.array_equal(host16(back), port.lut_decode(port.lut_apply(a, enc), dec))


@pytest.mark.parametrize("n", [1, 9, 4099, (1 << 20) + 1])
def test_lut_kernels_ragged(sq, cuda, port, n):
    rng = np.random.default_rng(n)
    a = rng.integers(0, 65536, size=n, dtype=np.uint16)
    enc = rng.integers(0, 256, size=65536, dtype=np.uint8)
    dec = rng.integers(0, 65536, size=256, dtype=np.uint16)
    codes = cuda.empty(n, dtype=cuda.uint8, device="cuda")
    sq.lut_apply_device(dev(cuda, a), codes, enc)
    assert np.array_equal(codes.cpu().numpy(), port.lut_apply(a, enc))
    back = cuda.empty(n, dtype=cuda.int16, device="cuda")
    sq.lut_decode_device(codes, back, dec)
    assert np.array_equal(host16(back), dec[enc[a]])


# ------------------------------------------------------------------------------------------------ lz4
def lz4_inputs():
    rng = np.random.default_rng(11)
    cases = {
        "empty": np.zeros(0, dtype=np.uint8),
        "one": np.array([7], dtype=np.uint8),
        "twelve": np.arange(12, dtype=np.uint8),
        "thirteen_same": np.full(13, 9, dtype=np.uint8),
        "sixteen_same": np.full(16, 9, dtype=np.uint8),
        "block_minus1": np.full(16383, 1, dtype=np.uint8),
        "block_exact_zero": np.zeros(16384, dtype=np.uint8),
        "block_plus1": np.zeros(16385, dtype=np.uint8),
        "random_64k": rng.integers(0, 256, size=65536, dtype=np.uint8),
        "random_ragged": rng.integers(0, 256, size=16384 * 3 + 1234, dtype=np.uint8),
        "text_like": np.frombuffer((b"the quick brown fox jumps over the lazy dog. " * 3000), dtype=np.uint8).copy(),
        "runs": np.repeat(rng.integers(0, 4, size=5000, dtype=np.uint8), rng.integers(1, 60, size=5000)),
        "period3": np.tile(np.array([1, 2, 3], dtype=np.uint8), 30000),
        "period64": np.tile(rng.integers(0, 256, size=64, dtype=np.uint8), 2000),
        "sparse_bits": (rng.random(200000) < 0.05).astype(np.uint8) * rng.integers(1, 256, size=200000, dtype=np.uint8),
        "ramp16": (np.arange(1 << 18) % 32768).astype(np.uint16).view(np.uint8),
        # long periods: match sources lie outside the decoder's 2 KiB shared-memory window (far path), overlapping copies
        "period3000": np.tile(rng.integers(0, 256, size=3000, dtype=np.uint8), 40),
        "period5000_ragged": np.tile(rng.integers(0, 256, size=5000, dtype=np.uint8), 13)[:-77],
        "far_and_near": np.concatenate([np.tile(rng.integers(0, 256, size=2500, dtype=np.uint8), 3), np.zeros(700, np.uint8),
                                        np.tile(np.array([5, 6], np.uint8), 900), np.tile(rng.integers(0, 256, size=2500, dtype=np.uint8), 4)]),
        "planes_scmos": None,
    }
    return cases


@pytest.mark.parametrize("name", list(lz4_inputs().keys()))
def test_lz4_roundtrip(sq, cuda, port, ref_or_standin, name):
    a = lz4_inputs()[name]
    if a is None:
        a = port.bitswap_encode(1, numpy_volume((8, 256, 256), "scmos", index=5)).view(np.uint8)
    d = dev(cuda, a) if a.size else cuda.empty(0, dtype=cuda.uint8, device="cuda")
    payload = sq.lz4_encode_device(d)
    assert payload.numel() <= sq.lz4_bound(a.size)
    hp = payload.cpu().numpy()
    # (1) the oracle's frame decoder reproduces the input from the GPU stream
    assert np.array_equal(port.lz4_frames_decode(hp, a.size), a)
    # (2) the reference's decoder (lz4.hpp:257-339 over liblz4), or liblz4's frame decoder where it is not built, does too
    if a.size:
        rc, out = ref_or_standin.lz4_decode_bytes(hp, a.size)
        assert rc == 0 and np.array_equal(out, a)
    # (3) GPU decode of the GPU stream
    out = cuda.zeros(max(a.size, 1), dtype=cuda.uint8, device="cuda")
    if a.size:
        got = sq.lz4_decode_device(payload, out[: a.size])
        assert got == a.size
        assert np.array_equal(out[: a.size].cpu().numpy(), a)


def test_lz4_constant_blocks_use_closed_form(sq, cuda):
    d = cuda.zeros(16384 * 64, dtype=cuda.uint8, device="cuda")
    payload = sq.lz4_encode_device(d)
    st = sq.last_lz4_stats()
    assert st["constant_blocks"] == 64 and st["general_blocks"] == 0 and st["stored_blocks"] == 0
    assert payload.numel() < 64 * 90 + 400


def test_lz4_random_blocks_are_stored(sq, cuda):
    a = np.random.default_rng(1).integers(0, 256, size=16384 * 8, dtype=np.uint8)
    payload = sq.lz4_encode_device(dev(cuda, a))
    st = sq.last_lz4_stats()
    assert st["stored_blocks"] == 8
    assert payload.numel() == sq.lz4_bound(a.size)


def test_lz4_noise_blocks_are_stored_early(sq, cuda, port, ref_or_standin):
    """blocks with fewer than 128 match candidates — fixed-offset ones of the whole block + hash ones of the first 2 KiB —
    (camera-noise bit planes, 8-bit quantiser codes of a noisy stack) are stored without a parse (lz4_encode.cu: kEarlyBytes /
    kEarlyMin; tools/lz4_model2.c EARLY=2048 DUMP=1: noise blocks count <= 29, every compressible block of the sample sets >= 243). The
    stated price: such blocks shrink by < 3 % under the reference's liblz4, so the payload stays within 3 % of the
    reference's; compressible blocks never take that exit."""
    vol = numpy_volume((16, 512, 512), "scmos", index=8)
    enc, dec = port.quantiser_luts(port.histogram(vol.reshape(-1)))
    codes = port.lut_apply(vol.reshape(-1), enc)                     # noisy 8-bit codes: liblz4 gets ~1.02
    payload = sq.lz4_encode_device(dev(cuda, codes))
    st = sq.last_lz4_stats()
    assert st["stored_blocks"] >= 0.9 * (codes.size // 16384), st
    theirs = ref_or_standin.lz4_encode(codes, nthreads=8).size    # (lz4_scheme<char>, the quantiser's tail)
    assert payload.numel() <= 1.03 * theirs, (payload.numel(), theirs)
    out = cuda.zeros(codes.size, dtype=cuda.uint8, device="cuda")
    assert sq.lz4_decode_device(payload, out) == codes.size
    assert np.array_equal(out.cpu().numpy(), codes)
    rc, back = ref_or_standin.lz4_decode_bytes(payload.cpu().numpy(), codes.size)
    assert rc == 0 and np.array_equal(back, codes)
    # bit planes of the same stack: the noise planes (low bits) are stored, everything else is parsed; a block that is noise
    # in its first 4 KiB only but full of runs elsewhere is parsed too (short-offset candidates count over the whole block)
    planes = port.bitswap_encode(1, vol.reshape(-1)).view(np.uint8)
    sq.lz4_encode_device(dev(cuda, planes))
    st = sq.last_lz4_stats()
    nb = planes.size // 16384
    assert 0.15 * nb <= st["stored_blocks"] <= 0.35 * nb and st["constant_blocks"] >= 0.4 * nb, st
    rng = np.random.default_rng(3)
    mixed = np.concatenate([rng.integers(0, 256, size=4096, dtype=np.uint8), np.zeros(12288, np.uint8)] * 6)
    p2 = sq.lz4_encode_device(dev(cuda, mixed))
    assert sq.last_lz4_stats()["stored_blocks"] == 0 and p2.numel() < 0.3 * mixed.size
    out2 = cuda.zeros(mixed.size, dtype=cuda.uint8, device="cuda")
    sq.lz4_decode_device(p2, out2)
    assert np.array_equal(out2.cpu().numpy(), mixed)


@pytest.mark.parametrize("key,src", [("lz4_serial", "lz4_vol"), ("lz4_parallel", "lz4_vol"), ("lz4_linked", "lz4_linked_in")])
def test_lz4_decodes_reference_payloads(sq, cuda, port, golden, key, src):
    """reference-produced frames (liblz4 1.9.4 through lz4_scheme::encode): block-linked single frame (CLI default,
    SURVEY F6), one frame per chunk (parallel mode), and a linked frame with real cross-block matches"""
    raw = golden[src]
    expect = port.bitswap_encode(1, raw) if src == "lz4_vol" else raw
    out = cuda.zeros(expect.size, dtype=cuda.int16, device="cuda")
    got = sq.lz4_decode_device(dev(cuda, golden[key]), out)
    assert got == expect.nbytes
    assert np.array_equal(host16(out).ravel(), expect.ravel())


def test_lz4_decodes_live_reference_payloads(sq, cuda, ref_or_standin):
    vol = numpy_volume((10, 256, 512), "ref", index=6)
    planes = ref_or_standin.bitswap_encode(1, vol)
    for nthreads, config in ((1, b""), (8, b""), (2, b"n_chunks_of_input=5"), (1, b"blocksize_kb=64,framestep_kb=128")):
        payload = ref_or_standin.lz4_encode(planes, nthreads=nthreads, config=config)
        out = cuda.zeros(planes.size, dtype=cuda.int16, device="cuda")
        got = sq.lz4_decode_device(dev(cuda, payload), out)
        assert got == planes.nbytes, (nthreads, config)
        assert np.array_equal(host16(out), planes), (nthreads, config)


def test_lz4_decodes_port_frames(sq, cuda, port):
    a = np.repeat(np.random.default_rng(2).integers(0, 30, 90000, dtype=np.uint16), 5)
    payload = port.lz4_frames_encode(a, chunk=1 << 18)
    out = cuda.zeros(a.size, dtype=cuda.int16, device="cuda")
    assert sq.lz4_decode_device(dev(cuda, payload), out) == a.nbytes
    assert np.array_equal(host16(out), a)


@pytest.mark.parametrize("period", [1, 2, 3, 4, 5, 7, 8, 16, 31, 32, 33, 40, 1984, 1985, 2048, 3000, 40000, 70000])
def test_lz4_decodes_foreign_frames_with_any_offset(sq, cuda, port, period):
    """256 KiB blocks from the oracle's encoder: offsets from 1 to 64 KiB, near / far / overlapping copies"""
    rng = np.random.default_rng(period)
    a = np.tile(rng.integers(0, 256, size=period, dtype=np.uint8), (700000 // period) + 2)[:700001]
    payload = port.lz4_frames_encode(a, chunk=1 << 19)
    out = cuda.zeros(a.size, dtype=cuda.uint8, device="cuda")
    assert sq.lz4_decode_device(dev(cuda, payload), out) == a.size
    assert np.array_equal(out.cpu().numpy(), a)


def test_lz4_decodes_long_literal_runs_in_big_blocks(sq, cuda, ref_or_standin):
    """a 256 KiB liblz4 block with ~200 KB of literals carries ~800 length bytes: the stream window must follow them"""
    rng = np.random.default_rng(8)
    a = np.concatenate([np.zeros(30000, np.uint8), rng.integers(0, 256, size=200000, dtype=np.uint8), np.zeros(32144, np.uint8)])
    payload = ref_or_standin.lz4_encode(a, nthreads=1)
    out = cuda.zeros(a.size, dtype=cuda.uint8, device="cuda")
    assert sq.lz4_decode_device(dev(cuda, payload), out) == a.size
    assert np.array_equal(out.cpu().numpy(), a)


def test_lz4_rejects_garbage(sq, cuda):
    bad = np.random.default_rng(4).integers(0, 256, size=4096, dtype=np.uint8)
    out = cuda.zeros(1 << 16, dtype=cuda.uint8, device="cuda")
    with pytest.raises(sq.SqeazyError):
        sq.lz4_decode_device(dev(cuda, bad), out)


def test_lz4_ratio_close_to_reference(sq, cuda, ref_or_standin):
    """compression ratio within 5 % of the reference's (lz4_scheme, 8 threads) on bit-plane data of both presets"""
    for preset in ("scmos", "ref"):
        vol = numpy_volume((32, 256, 512), preset, index=7)
        planes = ref_or_standin.bitswap_encode(1, vol)
        ours = sq.lz4_encode_device(dev(cuda, planes)).numel()
        theirs = ref_or_standin.lz4_encode(planes, nthreads=8).size
        assert ours <= theirs * 1.05, (preset, ours, theirs)


# ------------------------------------------------------------------------------------------------ pipelines (C API, host buffers)
PIPES = ["bitswap1->lz4", "rmestbkrd->bitswap1->lz4", "quantiser->lz4", "remove_background(threshold=110)->bitswap4->lz4",
         "rmbkrd(threshold=105)->bitswap1->lz4", "lz4", "bitswap1", "bitswap2->lz4", "bitswap8", "quantiser", "pass_through",
         "remove_background(threshold=100)", "rmestbkrd", "bitswap1->pass_through->lz4", "rmestbkrd->lz4"]


def expected_roundtrip(port, sq, pipeline, vol):
    """what decode(encode(vol)) must return: lossy stages applied by the oracle"""
    cur = vol
    for name, args in orc.to_pairs(pipeline):
        if name in ("remove_background", "rmbkrd"):
            cur = port.remove_background(cur, int(orc.minors(args).get("threshold", 0)))
        elif name == "rmestbkrd":
            cur, _ = port.rmestbkrd(cur, sq.host_l2_bytes())
        elif name == "quantiser":
            enc, dec = port.quantiser_luts(port.histogram(cur))
            cur = port.lut_decode(port.lut_apply(cur, enc), dec).reshape(vol.shape)
    return cur


@pytest.mark.parametrize("pipeline", PIPES)
@pytest.mark.parametrize("shape,preset", [((8, 8, 8), "ramp"), ((16, 64, 128), "scmos"), ((5, 33, 47), "ref")])
def test_pipeline_roundtrip(sq, cuda, port, pipeline, shape, preset):
    vol = numpy_volume(shape, preset, index=8)
    blob = sq.encode(pipeline, vol)
    assert blob.size <= sq.max_compressed_length(pipeline, vol.nbytes)
    assert sq.decompressed_shape(blob) == shape
    assert sq.decompressed_length(blob) == vol.nbytes
    assert sq.decompressed_sizeof(blob) == 2
    hdr = orc.unpack_header(blob.tobytes())
    assert hdr is not None and hdr["size"] == sq.header_size(blob) and hdr["size"] % 2 == 0
    assert hdr["bytes"] == blob.size - hdr["size"]
    assert orc.can_be_built_from(hdr["pipeline"].replace("bitswap2", "bitswap1").replace("bitswap4", "bitswap1").replace("bitswap8", "bitswap1"))
    back = sq.decode(blob)
    assert np.array_equal(back, expected_roundtrip(port, sq, pipeline, vol))


def test_constant_cube_roundtrip(sq, cuda):
    """tests/test_pipeline_interface.cpp:388-416"""
    vol = np.full((8, 8, 8), 42, dtype=np.uint16)
    blob = sq.encode("bitswap1->lz4", vol, nthreads=1)
    assert np.array_equal(sq.decode(blob), vol)


def test_java_boundary_cases(sq, cuda):
    """SqeazyLibraryTests.java:28-84,163-227"""
    data = (np.arange(512) % 256).astype(np.uint16).reshape(1, 1, 512)
    blob = sq.encode("lz4", data)
    assert np.array_equal(sq.decode(blob), data)
    vol = (1 << (np.arange(256 * 128 * 128) % 8)).astype(np.uint16).reshape(256, 128, 128)
    blob = sq.encode("quantiser->lz4", vol)
    assert np.array_equal(sq.decode(blob), vol)  # 8 distinct values: lossless mapping


def test_blob_is_decodable_by_the_reference_chain(sq, cuda, port, ref_or_standin):
    """header parsed by the restated reference reader, payload by the reference's lz4 decoder + bitswap decoder"""
    vol = numpy_volume((16, 128, 256), "scmos", index=9)
    blob = sq.encode("bitswap1->lz4", vol)
    hdr = orc.unpack_header(blob.tobytes())
    assert hdr["pipeline"] == "bitswap1(num_bits_per_plane=1)->lz4(accel=1,blocksize_kb=256,framestep_kb=256,n_chunks_of_input=0)"
    rc, out, _ = ref_or_standin.pipeline_decode_stages(1, blob[hdr["size"]:], vol.size)
    assert rc == 0 and np.array_equal(out.reshape(vol.shape), vol)


def test_reference_blob_decodes_on_gpu(sq, cuda, ref_or_standin):
    """blob = reference-style header (oracle restatement of header::pack) + payload made by the reference's stage chain"""
    vol = numpy_volume((16, 128, 256), "scmos", index=10)
    name = "bitswap1(num_bits_per_plane=1)->lz4(accel=1,blocksize_kb=256,framestep_kb=256,n_chunks_of_input=0)"
    for nthreads in (1, 8):
        payload, _ = ref_or_standin.pipeline_encode_stages(0, vol, nthreads)
        h = orc.pack_header(vol.shape, name, payload.size, version="0.5.2", headref="4c45a9b")
        blob = np.concatenate([np.frombuffer(h.encode(), dtype=np.uint8), payload])
        assert np.array_equal(sq.decode(blob), vol)


def test_quantiser_blob_matches_reference_encode(sq, cuda, port, ref_or_standin):
    vol = numpy_volume((8, 128, 256), "ref", index=11)
    blob = sq.encode("quantiser", vol)
    hdr = orc.unpack_header(blob.tobytes())
    codes_ref, dec_ref = ref_or_standin.quantiser_encode(vol)
    assert np.array_equal(blob[hdr["size"]:], codes_ref.ravel())
    lut = orc.minors(orc.to_pairs(hdr["pipeline"])[0][1])["decode_lut_string"]
    assert lut == ref_or_standin.quantiser_lut_string(dec_ref)


def test_device_api_matches_host_api(sq, cuda, port):
    vol = numpy_volume((16, 64, 128), "scmos", index=12)
    for pipeline in ("bitswap1->lz4", "quantiser->lz4"):
        d_blob = sq.encode_device(pipeline, dev(cuda, vol))
        hb = d_blob.cpu().numpy()
        assert np.array_equal(sq.decode(hb), sq.decode(sq.encode(pipeline, vol)))
        out = cuda.empty(vol.shape, dtype=cuda.int16, device="cuda")
        sq.decode_device(d_blob, out)
        assert np.array_equal(host16(out), sq.decode(hb))


def test_quantiser_with_global_histogram(sq, cuda, port):
    """multi-GPU path on one GPU: two z-slabs encoded with the all-reduced histogram == slabs of the whole-volume result"""
    vol = numpy_volume((16, 64, 128), "ref", index=13)
    d = dev(cuda, vol)
    hist = cuda.zeros(65536, dtype=cuda.int32, device="cuda")
    sq.histogram_device(d[:8], hist)
    sq.histogram_device(d[8:], hist)
    cuda.cuda.synchronize()
    whole = sq.decode(sq.encode("quantiser->lz4", vol))
    for sl in (slice(0, 8), slice(8, 16)):
        blob = sq.encode_device("quantiser->lz4", d[sl].contiguous(), global_hist=hist)
        assert np.array_equal(sq.decode(blob.cpu().numpy()), whole[sl])


def test_distributed_threshold_matches_single_gpu(sq, cuda, port):
    """sqeazy_b200.dist.global_background_threshold (the multi-GPU path, here with one rank) == sqyx_estimate_background"""
    from sqeazy_b200 import dist as sqdist

    vol = numpy_volume((9, 64, 96), "ref", index=14)
    d = dev(cuda, vol)
    sup, thr = sq.estimate_background_device(d, l2_bytes=1 << 12)
    thr2, sup2 = sqdist.global_background_threshold(d, 0, vol.shape, l2_bytes=1 << 12, histogram_fn=lambda sub, row: sq.histogram_device(sub, row),
                                                   support_fn=lambda h: sq.histogram_support(h, 0.99))
    assert thr2 == thr and np.array_equal(sup2.view(np.uint32), sup.view(np.uint32))
    assert np.array_equal(sup.view(np.uint32), port.darkest_face_supports(vol, 1 << 12).view(np.uint32))


def test_large_volume_roundtrip_properties(sq, cuda):
    """config-1 sized volume (512x512x256): encode -> decode identity and idempotence of the lossy filter"""
    from sqeazy_b200.synth import torch_volume

    vol = torch_volume((256, 512, 512), "scmos", index=0)
    blob = sq.encode_device("bitswap1->lz4", vol)
    out = cuda.empty_like(vol)
    sq.decode_device(blob, out)
    assert cuda.equal(out, vol)
    blob2 = sq.encode_device("rmestbkrd->bitswap1->lz4", vol)
    sq.decode_device(blob2, out)
    assert int((out.to(cuda.int32) & 0xFFFF).max()) <= int((vol.to(cuda.int32) & 0xFFFF).max())
    st = sq.last_lz4_stats()
    assert st["constant_blocks"] + st["general_blocks"] + st["stored_blocks"] == 256 * 512 * 512 * 2 // 16384


def test_concurrent_callers(sq, cuda, port):
    """the reference's entry points are re-entrant (SURVEY §8b); here concurrent host threads are serialised inside the
    library: four threads encode and decode different volumes through the host-pointer API at the same time"""
    import threading

    vols = [numpy_volume((8, 64, 96), "scmos", index=40 + i) for i in range(4)]
    results, errors = [None] * 4, []

    def work(i):
        try:
            for _ in range(3):
                blob = sq.encode("rmestbkrd->bitswap1->lz4" if i % 2 else "bitswap1->lz4", vols[i])
                results[i] = sq.decode(blob)
        except Exception as exc:  # pragma: no cover
            errors.append(exc)

    threads = [threading.Thread(target=work, args=(i,)) for i in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors
    for i in range(4):
        expect = port.rmestbkrd(vols[i], sq.host_l2_bytes())[0] if i % 2 else vols[i]
        assert np.array_equal(results[i], expect)
