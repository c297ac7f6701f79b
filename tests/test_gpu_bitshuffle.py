"""bitshuffle head filter on the GPU (SURVEY §8f-4; the reference's own full-pipeline benchmark runs `bitshuffle->lz4` and
`rmestbkrd->bitshuffle->lz4`, bench/benchmark_full_pipeline_impl.cpp:11-12): kernels bit-exact against the oracle's
restatement of the bitshuffle library (parity unpinned, see tests/test_bitshuffle_cpu.py), pipelines through the C ABI."""
import numpy as np
import pytest

from oracle import oracle as orc
from sqeazy_b200.synth import numpy_volume
from test_gpu_parity import dev, host16

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("bs", [0, 8, 24, 64, 1000, 4096, 8192])
@pytest.mark.parametrize("n", [0, 1, 7, 8, 9, 31, 32, 4095, 4096, 4097, 4104, 32003, 32 * 1024, 32 * 1024 + 1, (1 << 21) + 5])
def test_bitshuffle_stage_parity(sq, cuda, port, n, bs):
    a = np.random.default_rng(n * 31 + bs).integers(0, 65536, size=n, dtype=np.uint16)
    d_in = dev(cuda, a) if n else cuda.empty(0, dtype=cuda.int16, device="cuda")
    d_out = cuda.full((n + 16,), 0x7EEE, dtype=cuda.int16, device="cuda")
    sq.bitshuffle_encode_device(d_in, d_out[:n], bs)
    got = host16(d_out)
    assert np.array_equal(got[:n], port.bitshuffle(a, bs))
    assert np.all(got[n:] == 0x7EEE)
    back = cuda.empty(n, dtype=cuda.int16, device="cuda")
    sq.bitshuffle_decode_device(d_out[:n], back, bs)
    assert np.array_equal(host16(back), a)


def test_bitshuffle_unaligned_and_bad_block_size(sq, cuda, port):
    a = np.random.default_rng(4).integers(0, 65536, size=4096 * 9 + 77, dtype=np.uint16)
    d = dev(cuda, a)
    for off in (1, 3, 8):                                  # 2-, 6-, 16-byte offsets: the thread-per-group kernels
        n = a.size - off - 5
        out = cuda.zeros(n + 8, dtype=cuda.int16, device="cuda")
        sq.bitshuffle_encode_device(d[off: off + n], out[1: 1 + n])
        assert np.array_equal(host16(out)[1: 1 + n], port.bitshuffle(a[off: off + n]))
    with pytest.raises(sq.SqeazyError):
        sq.bitshuffle_encode_device(d[:64], cuda.zeros(64, dtype=cuda.int16, device="cuda"), 12)
    with pytest.raises(sq.SqeazyError):
        sq.encode("bitshuffle(block_size=12)->lz4", a[: 4096].reshape(4, 32, 32))


def test_bitshuffle_full_size_many_sweeps(sq, cuda):
    """2^28 voxels = several grid sweeps of the fast kernels, checked against torch arithmetic on the device: row r of
    block b = bit r of its 4096 elements"""
    torch = cuda
    n = 1 << 28
    g = torch.Generator(device="cuda"); g.manual_seed(5)
    x = torch.randint(0, 65536, (n,), generator=g, device="cuda", dtype=torch.int32)
    d_in = x.to(torch.int16)
    d_out = torch.empty_like(d_in)
    sq.bitshuffle_encode_device(d_in, d_out)
    rows = d_out.view(torch.uint8).view(n // 4096, 16, 512)              # [block][row][byte]
    xb = x.view(n // 4096, 512, 8)                                        # [block][byte][bit position in the byte]
    weights = (1 << torch.arange(8, device="cuda", dtype=torch.int32))
    for r in (0, 3, 7, 8, 15):
        want = (((xb >> r) & 1) * weights).sum(dim=2).to(torch.uint8)
        assert torch.equal(rows[:, r, :], want), r
    back = torch.empty_like(d_in)
    sq.bitshuffle_decode_device(d_out, back)
    assert torch.equal(back, d_in)


@pytest.mark.parametrize("pipeline", ["bitshuffle->lz4", "bitshuffle", "bitshuffle(block_size=512)->lz4", "rmestbkrd->bitshuffle->lz4",
                                      "remove_background(threshold=105)->bitshuffle->lz4", "bitshuffle->pass_through->lz4"])
@pytest.mark.parametrize("shape", [(16, 128, 256), (5, 33, 77), (1, 1, 512)])
def test_bitshuffle_pipelines(sq, cuda, port, ref_or_standin, pipeline, shape):
    vol = numpy_volume(shape, "scmos", index=9)
    blob = sq.encode(pipeline, vol)
    assert blob.size <= sq.max_compressed_length(pipeline, vol.nbytes)
    hdr = orc.unpack_header(blob.tobytes())
    assert "bitshuffle(block_size=" in hdr["pipeline"] and tuple(hdr["shape"]) == shape
    want = vol
    if "rmestbkrd" in pipeline:
        want, _ = port.rmestbkrd(vol, sq.host_l2_bytes())
    elif "remove_background" in pipeline:
        want = port.remove_background(vol, 105)
    out = sq.decode(blob)
    assert np.array_equal(out.reshape(shape), np.asarray(want).reshape(shape))
    # what a reader built on the reference would do with the payload: LZ4 frames (liblz4 through the reference's decode
    # loop) -> bshuf_bitunshuffle
    bs = 512 if "block_size=512" in pipeline else 0
    payload = blob[hdr["size"]:]
    if pipeline.endswith("lz4"):
        rc, raw = ref_or_standin.lz4_decode_bytes(payload, vol.nbytes)
        assert rc == 0
        payload = raw
    shuffled = np.frombuffer(payload.tobytes(), dtype=np.uint16)
    assert np.array_equal(port.bitshuffle(shuffled, bs, decode=True).reshape(shape), np.asarray(want).reshape(shape))


def test_bitshuffle_device_pipeline_and_ratio(sq, cuda):
    vol = numpy_volume((32, 512, 512), "scmos", index=3)
    d = dev(cuda, vol)
    sizes = {}
    for p in ("bitshuffle->lz4", "bitswap1->lz4"):
        blob = sq.encode_device(p, d)
        out = cuda.empty(vol.shape, dtype=cuda.int16, device="cuda")
        sq.decode_device(blob, out)
        assert np.array_equal(host16(out), vol)
        sizes[p] = blob.numel()
    # rows of 512 bytes per 4096-voxel block instead of whole-stack planes: the runs are shorter, the ratio a little lower
    assert sizes["bitshuffle->lz4"] < 0.6 * vol.nbytes and sizes["bitshuffle->lz4"] < 1.25 * sizes["bitswap1->lz4"]


@pytest.mark.parametrize("bs", [0, 8, 24, 64, 1000, 8192])
@pytest.mark.parametrize("n", [0, 1, 7, 8, 9, 31, 32, 8191, 8192, 8193, 8200, 32003, (1 << 22) + 5])
def test_bitshuffle_uint8_stage_parity(sq, cuda, port, n, bs):
    a = np.random.default_rng(n * 7 + bs).integers(0, 256, size=n, dtype=np.uint8)
    d_in = dev(cuda, a) if n else cuda.empty(0, dtype=cuda.uint8, device="cuda")
    d_out = cuda.full((n + 16,), 0xEE, dtype=cuda.uint8, device="cuda")
    sq.bitshuffle_encode_device(d_in, d_out[:n], bs)
    got = d_out.cpu().numpy()
    assert np.array_equal(got[:n], port.bitshuffle(a, bs))
    assert np.all(got[n:] == 0xEE)
    back = cuda.empty(n, dtype=cuda.uint8, device="cuda")
    sq.bitshuffle_decode_device(d_out[:n], back, bs)
    assert np.array_equal(back.cpu().numpy(), a)
    if n > 64:                                             # unaligned views: the thread-per-group kernel
        out2 = cuda.zeros(n, dtype=cuda.uint8, device="cuda")
        sq.bitshuffle_encode_device(d_in[3:], out2[1: n - 2], bs)
        assert np.array_equal(out2.cpu().numpy()[1: n - 2], port.bitshuffle(a[3:], bs))


@pytest.mark.parametrize("pipeline", ["bitshuffle->lz4", "bitshuffle", "remove_background(threshold=19)->bitshuffle(block_size=256)->lz4"])
def test_bitshuffle_uint8_pipelines(sq, cuda, port, ref_or_standin, pipeline):
    rng = np.random.default_rng(6)
    vol = np.clip(np.rint(20 + 2 * rng.standard_normal((9, 130, 257))), 0, 255).astype(np.uint8)
    blob = sq.encode_u8(pipeline, vol)
    hdr = orc.unpack_header(blob.tobytes())
    assert hdr["raw_type"] in ("uint8", "unsigned char", "h") or "8" in str(hdr["raw_type"])
    want = port.remove_background8(vol.reshape(-1), 19).reshape(vol.shape) if "remove_background" in pipeline else vol
    assert np.array_equal(sq.decode_u8(blob).reshape(vol.shape), want)
    payload = blob[hdr["size"]:]
    if pipeline.endswith("lz4"):
        rc, payload = ref_or_standin.lz4_decode_bytes(payload, vol.nbytes)
        assert rc == 0
    bs = 256 if "block_size=256" in pipeline else 0
    assert np.array_equal(port.bitshuffle(np.frombuffer(payload.tobytes(), dtype=np.uint8), bs, decode=True).reshape(vol.shape), want)
