"""diff3x3x1 head filter on the GPU (SURVEY §8f-4, reference: encoders/diff_scheme_impl.hpp:78-199): the kernels bit-exact
against the oracle (pinned by golden vectors of the reference and oracle/_ref, tests/test_diff_cpu.py), pipelines through
the C ABI read back the way a reader built on the reference would, the recurrence at size against plain torch arithmetic."""
import numpy as np
import pytest

from oracle import oracle as orc
from sqeazy_b200.synth import numpy_volume
from test_diff_cpu import BIG, GOLDEN, REFUSED, REFUSED_U8, SHAPES, _volume
from test_gpu_parity import dev, host16

pytestmark = pytest.mark.gpu


def _host(t, dtype):
    return t.cpu().numpy().view(dtype)


@pytest.mark.parametrize("dtype", [np.uint16, np.uint8])
@pytest.mark.parametrize("shape", SHAPES + BIG + [(7, 9, 520), (10, 23, 264), (40, 250, 264), (64, 256, 512)])
def test_diff_stage_parity(sq, cuda, port, shape, dtype):
    if not port.diff_supported(shape, np.dtype(dtype).itemsize):
        assert shape in REFUSED_U8 + BIG + [(7, 9, 520), (10, 23, 264), (40, 250, 264), (64, 256, 512)] and dtype == np.uint8
        assert not sq.diff_shape_supported(*shape, sizeof_voxel=1)
        d = cuda.zeros(shape, dtype=cuda.uint8, device="cuda")
        with pytest.raises(sq.SqeazyError):
            sq.diff_device(d, cuda.zeros_like(d))
        return
    tdt = cuda.int16 if dtype == np.uint16 else cuda.uint8
    poison = 0x7EEE if dtype == np.uint16 else 0xEE
    n = int(np.prod(shape))
    for seed in (1, 2):
        a = _volume(shape, dtype, seed)
        want = port.diff(a)
        d_in = dev(cuda, a)
        d_out = cuda.full((n + 16,), poison, dtype=tdt, device="cuda")
        sq.diff_device(d_in, d_out[:n].view(shape))
        got = _host(d_out, dtype)
        assert np.array_equal(got[:n].reshape(shape), want)
        assert np.all(got[n:] == poison)
        back = cuda.full((n,), poison, dtype=tdt, device="cuda").view(shape)
        sq.diff_device(d_out[:n].view(shape), back, decode=True)
        assert np.array_equal(_host(back, dtype), a)


def test_diff_golden_on_gpu(sq, cuda):
    g = np.load(GOLDEN)
    for case in ("u16_cube", "u16_flat", "u16_spill", "u16_vec", "u16_tall", "u8_cube", "u8_spill", "u8_vec"):
        a, enc = g[case + "_in"], g[case + "_enc"]
        dtype = a.dtype.type
        d_out = cuda.zeros(a.shape, dtype=cuda.int16 if dtype == np.uint16 else cuda.uint8, device="cuda")
        sq.diff_device(dev(cuda, a), d_out)
        assert np.array_equal(_host(d_out, dtype), enc), case
        back = cuda.zeros_like(d_out)
        sq.diff_device(d_out, back, decode=True)
        assert np.array_equal(_host(back, dtype), a), case


def test_diff_unaligned_buffers(sq, cuda, port):
    shape = (12, 40, 72)
    n = int(np.prod(shape))
    a = _volume(shape, np.uint16, 5)
    want = port.diff(a)
    for off_in, off_out in ((1, 0), (0, 3), (5, 1), (8, 8)):
        src = cuda.zeros(n + 16, dtype=cuda.int16, device="cuda")
        src[off_in: off_in + n] = dev(cuda, a).reshape(-1)
        out = cuda.zeros(n + 16, dtype=cuda.int16, device="cuda")
        sq.diff_device(src[off_in: off_in + n].view(shape), out[off_out: off_out + n].view(shape))
        assert np.array_equal(host16(out)[off_out: off_out + n].reshape(shape), want)
        back = cuda.zeros(n + 16, dtype=cuda.int16, device="cuda")
        sq.diff_device(out[off_out: off_out + n].view(shape), back[off_in: off_in + n].view(shape), decode=True)
        assert np.array_equal(host16(back)[off_in: off_in + n].reshape(shape), a)


@pytest.mark.parametrize("shape", [s for s in REFUSED if int(np.prod(s)) < 1 << 20])
def test_diff_refused_shapes(sq, cuda, shape):
    assert not sq.diff_shape_supported(*shape)
    d = cuda.zeros(shape, dtype=cuda.int16, device="cuda")
    with pytest.raises(sq.SqeazyError):
        sq.diff_device(d, cuda.zeros_like(d))
    with pytest.raises(sq.SqeazyError):
        sq.encode("diff3x3x1->lz4", np.zeros(shape, dtype=np.uint16))
    with pytest.raises(sq.SqeazyError):
        sq.diff_device(d, d)                               # in place: the decode recurrence needs both buffers


@pytest.mark.parametrize("pipeline", ["diff3x3x1->lz4", "diff3x3x1", "diff3x3x1->bitswap1->lz4", "rmestbkrd->diff3x3x1->bitswap1->lz4",
                                      "remove_background(threshold=105)->diff3x3x1->lz4", "diff3x3x1->pass_through->lz4",
                                      "bitswap1->diff3x3x1->lz4"])
@pytest.mark.parametrize("shape", [(16, 128, 256), (5, 33, 77), (40, 24, 32)])
def test_diff_pipelines(sq, cuda, port, ref_or_standin, pipeline, shape):
    vol = numpy_volume(shape, "scmos", index=11)
    blob = sq.encode(pipeline, vol)
    assert blob.size <= sq.max_compressed_length(pipeline, vol.nbytes)
    hdr = orc.unpack_header(blob.tobytes())
    assert "diff3x3x1" in hdr["pipeline"] and "diff3x3x1(" not in hdr["pipeline"] and tuple(hdr["shape"]) == shape
    want = vol
    if "rmestbkrd" in pipeline:
        want, _ = port.rmestbkrd(vol, sq.host_l2_bytes())
    elif "remove_background" in pipeline:
        want = port.remove_background(vol, 105)
    want = np.asarray(want).reshape(shape)
    assert np.array_equal(sq.decode(blob).reshape(shape), want)
    # a reader built on the reference: LZ4 frames (liblz4 through the reference's decode loop), then the head filters backwards
    payload = blob[hdr["size"]:]
    if pipeline.endswith("lz4"):
        rc, payload = ref_or_standin.lz4_decode_bytes(payload, vol.nbytes)
        assert rc == 0
    stage_out = np.frombuffer(payload.tobytes(), dtype=np.uint16)
    if pipeline.startswith("bitswap1->diff"):
        assert np.array_equal(stage_out.reshape(shape), ref_or_standin.diff(port.bitswap_encode(1, want).reshape(shape)))
        stage_out = port.bitswap_decode(1, ref_or_standin.diff(stage_out.reshape(shape), decode=True))
    else:
        if "bitswap1" in pipeline:
            stage_out = port.bitswap_decode(1, stage_out)
        assert np.array_equal(stage_out.reshape(shape), ref_or_standin.diff(want))
        stage_out = ref_or_standin.diff(stage_out.reshape(shape), decode=True)
    assert np.array_equal(stage_out.reshape(shape), want)


def test_diff_uint8_pipelines(sq, cuda, port, ref_or_standin):
    rng = np.random.default_rng(8)
    vol = np.clip(np.rint(20 + 2 * rng.standard_normal((9, 120, 128))), 0, 255).astype(np.uint8)
    with pytest.raises(sq.SqeazyError):                      # 130 rows: beyond the reference's int8 coordinates
        sq.encode_u8("diff3x3x1->lz4", np.zeros((9, 130, 64), dtype=np.uint8))
    for pipeline in ("diff3x3x1->lz4", "diff3x3x1", "diff3x3x1->bitswap1->lz4"):
        blob = sq.encode_u8(pipeline, vol)
        assert np.array_equal(sq.decode_u8(blob).reshape(vol.shape), vol)
        if pipeline == "diff3x3x1":
            hdr = orc.unpack_header(blob.tobytes())
            assert np.array_equal(np.frombuffer(blob[hdr["size"]:].tobytes(), dtype=np.uint8).reshape(vol.shape), ref_or_standin.diff(vol))


def test_diff_device_pipeline_and_ratio(sq, cuda):
    """a smooth stack is mostly its own neighbourhood mean: the residuals compress better than the voxels"""
    vol = numpy_volume((32, 512, 512), "scmos", index=3)
    d = dev(cuda, vol)
    sizes = {}
    for p in ("diff3x3x1->bitswap1->lz4", "bitswap1->lz4", "diff3x3x1->lz4", "lz4"):
        blob = sq.encode_device(p, d)
        out = cuda.empty(vol.shape, dtype=cuda.int16, device="cuda")
        sq.decode_device(blob, out)
        assert np.array_equal(host16(out), vol)
        sizes[p] = blob.numel()
    assert all(v < vol.nbytes for v in sizes.values())


def test_diff_at_size_against_torch(sq, cuda):
    """256 MiB stack: encode against the formula written with torch slices (int32 arithmetic, wrap of the sum applied by
    hand), decode as the round trip; launches = 1 + (1 + Z - 1) + 0 for Z <= X"""
    z, y, x = 128, 1024, 1024
    g = cuda.Generator(device="cuda")
    g.manual_seed(12)
    a = cuda.randint(0, 65536, (z, y, x), generator=g, device="cuda", dtype=cuda.int32)
    a[: z // 2] = 200 + (a[: z // 2] % 37)                  # half camera-like, half full-range (wrapping sums)
    src = cuda.where(a >= 32768, a - 65536, a).to(cuda.int16)
    out = cuda.empty_like(src)
    before = sq.kernel_launches()
    sq.diff_device(src, out)
    assert sq.kernel_launches() - before == 1
    s = cuda.zeros((z - 1, y - 2, x - 2), dtype=cuda.int32, device="cuda")
    for dy in range(3):
        for dx in range(3):
            s += a[: z - 1, dy: dy + y - 2, dx: dx + x - 2]
    q = (s & 0xFFFF) // 9
    want = a.clone()
    want[1:, 1: y - 1, 1: z - 1] = (a[1:, 1: y - 1, 1: z - 1] - q[:, :, : z - 2]) & 0xFFFF     # x range from the Z extent
    assert cuda.equal(out.to(cuda.int32) & 0xFFFF, want)
    del s, q, want
    back = cuda.empty_like(src)
    before = sq.kernel_launches()
    sq.diff_device(out, back, decode=True)
    assert sq.kernel_launches() - before == z
    assert cuda.equal(back, src)
