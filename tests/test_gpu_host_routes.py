"""Which route a host call (`SQY_PipelineEncode_UI16` / `SQY_Decode_UI16`) takes, told apart by the kernels it launches and by
`last_shard_info()`. The other host-path suites compare voxels only; a call that silently changed route (a slab size, a
threshold, a guard) would pass them. The counts are derived from the slab counts of api.cu and sharded.inl:

- LZ4 encode in one go: begin (prefix) + blocks + end (3) = 5; streamed: begin, 2 per slab (transpose, blocks), end (3);
- LZ4 decode: the block table takes 5 launches; then one block-decoder launch per slab (streamed) or one in all;
- rmestbkrd's estimate: 2 face histograms, 6 row histograms, the support index.
"""
import numpy as np
import pytest

from sqeazy_b200.synth import torch_volume

pytestmark = pytest.mark.gpu

MiB = 1 << 20
SHAPE = (80, 2048, 2048)          # 640 MiB: streamed, 2.5 slabs of 256 MiB
SMALL = (40, 2048, 2048)          # 320 MiB: below the 512 MiB of the streamed routes
GIB = (128, 2048, 2048)           # 1 GiB: the device call fuses the last transpose into the LZ4 decoder

TABLES = 5
LZ4_ENCODE = 5
ENC_BEGIN, ENC_END = 1, 3
ESTIMATE = 9
SLAB_VOXELS = 128 * MiB           # kStreamSlabBytes / 2
SUB_SLAB_VOXELS = 32 * MiB        # kShardSubSlabVoxels: slabs of the sharded calls

FOREIGN_NAME = "bitswap1(num_bits_per_plane=1)->lz4(accel=1,blocksize_kb=256,framestep_kb=256,n_chunks_of_input=0)"


def slabs(n, slab=SLAB_VOXELS):
    return -(-n // slab)


def voxels(shape):
    return int(np.prod(shape))


def host_volume(shape, index, constant_slices=0):
    v = torch_volume(shape, "scmos", index=index)
    if constant_slices:
        v[:constant_slices] = 100
    return v.cpu().numpy().view(np.uint16)


def counted(sq, fn, *args, **kw):
    k0 = sq.kernel_launches()
    out = fn(*args, **kw)
    return out, sq.kernel_launches() - k0


def counted_device(sq, cuda, fn, *args):
    cuda.cuda.synchronize()
    k0 = sq.kernel_launches()
    fn(*args)
    cuda.cuda.synchronize()
    return sq.kernel_launches() - k0


def first_compressed_block(payload):
    """(offset, size) of the data of the first compressed block behind the index frame and the LZ4 frame header"""
    p = 8 + int(payload[4:8].view(np.uint32)[0]) + 7
    while True:
        word = int(payload[p : p + 4].view(np.uint32)[0])
        assert word != 0, "no compressed block in the payload"
        if not word >> 31:
            return p + 4, word & 0x7FFFFFFF
        p += 4 + (word & 0x7FFFFFFF)


@pytest.fixture
def one_gpu(sq, cuda):
    sq.set_devices([0])
    yield
    sq.set_device(0)


@pytest.fixture
def two_gpus(sq, cuda):
    if cuda.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    sq.set_devices([0, 1])
    yield
    sq.set_device(0)


@pytest.fixture(scope="module")
def vol640(cuda):
    return host_volume(SHAPE, 41)


# ---------------------------------------------------------------------------------------------------------------- one GPU
STREAMED = {
    # pipeline: (encode launches, decode launches, shard GPUs of the encode)
    "bitswap1->lz4": (ENC_BEGIN + 2 * slabs(voxels(SHAPE)) + ENC_END, TABLES + 2 * slabs(voxels(SHAPE)), 0),
    "rmestbkrd->bitswap1->lz4": (ESTIMATE + ENC_BEGIN + 2 * slabs(voxels(SHAPE)) + ENC_END, TABLES + 2 * slabs(voxels(SHAPE)), 0),
    # the one-GPU sharded encoder: a histogram per sub-slab, LUT apply, LZ4; the codes decoder: LZ4 + LUT^-1 per slab
    "quantiser->lz4": (slabs(voxels(SHAPE), SUB_SLAB_VOXELS) + 1 + LZ4_ENCODE, TABLES + 2 * slabs(voxels(SHAPE)), 1),
}


@pytest.mark.parametrize("pipeline", list(STREAMED))
def test_streamed_routes_on_one_gpu(sq, cuda, one_gpu, vol640, pipeline):
    enc, dec, gpus = STREAMED[pipeline]
    blob, n = counted(sq, sq.encode, pipeline, vol640, nthreads=4)
    assert n == enc
    assert sq.last_shard_info() == {"gpus": gpus, "nccl": False, "pieces": gpus}
    back, n = counted(sq, sq.decode, blob, nthreads=4)
    assert n == dec
    assert sq.last_shard_info()["gpus"] == 0
    if pipeline == "bitswap1->lz4":
        assert np.array_equal(back, vol640)


def test_foreign_blob_takes_the_last_transpose_per_slab(sq, cuda, one_gpu, ref_or_standin, vol640):
    """a blob that is not one frame of this library: the streamed decoder builds the table, finds it foreign and gives up;
    the general route builds it again, decodes all blocks in one launch, and transposes back slab by slab"""
    from oracle import oracle as orc

    payload, _ = ref_or_standin.pipeline_encode_stages(0, vol640, 8)         # one frame per 256 KiB chunk
    h = orc.pack_header(vol640.shape, FOREIGN_NAME, payload.size, version="0.5.2", headref="4c45a9b")
    blob = np.concatenate([np.frombuffer(h.encode(), dtype=np.uint8), payload])
    back, n = counted(sq, sq.decode, blob, nthreads=4)
    assert n == TABLES + TABLES + 1 + slabs(voxels(SHAPE))
    assert np.array_equal(back, vol640)


@pytest.mark.parametrize("pipeline, enc, dec", [("bitswap1->lz4", 1 + LZ4_ENCODE, TABLES + 1 + 1),
                                                ("quantiser->lz4", 1 + 1 + LZ4_ENCODE, TABLES + 1 + 1)])
def test_general_route_below_512_mib(sq, cuda, one_gpu, pipeline, enc, dec):
    vol = host_volume(SMALL, 42)
    blob, n = counted(sq, sq.encode, pipeline, vol, nthreads=4)
    assert n == enc
    assert sq.last_shard_info()["gpus"] == 0
    back, n = counted(sq, sq.decode, blob, nthreads=4)
    assert n == dec
    if pipeline == "bitswap1->lz4":
        assert np.array_equal(back, vol)


def test_one_gib_stack_streamed_to_the_host_and_fused_on_the_device(sq, cuda, one_gpu):
    vol = host_volume(GIB, 43)
    blob, n = counted(sq, sq.encode, "bitswap1->lz4", vol, nthreads=4)
    assert n == ENC_BEGIN + 2 * slabs(voxels(GIB)) + ENC_END
    back, n = counted(sq, sq.decode, blob, nthreads=4)
    assert n == TABLES + 2 * slabs(voxels(GIB))
    assert np.array_equal(back, vol)
    del back
    d_blob = cuda.from_numpy(blob).cuda()
    out = cuda.empty(GIB, dtype=cuda.int16, device="cuda")
    assert counted_device(sq, cuda, sq.decode_device, d_blob, out) == TABLES + 1
    assert np.array_equal(out.cpu().numpy().view(np.uint16), vol)


@pytest.mark.parametrize("pipeline, code", [("bitswap1->lz4", 11), ("quantiser->lz4", 101)])
def test_streamed_decode_refuses_a_corrupt_block(sq, cuda, one_gpu, pipeline, code):
    """a compressed block turned into one endless literal run: the index and the frame stay intact, so the streamed decoder
    runs every slab and refuses the stream at the end with the code of the general route"""
    vol = host_volume(SHAPE, 44, constant_slices=4)
    blob = sq.encode(pipeline, vol, nthreads=4).copy()
    hsz = sq.header_size(blob)
    off, size = first_compressed_block(blob[hsz:])
    blob[hsz + off : hsz + off + size] = 0xFF
    k0 = sq.kernel_launches()
    with pytest.raises(sq.SqeazyError, match=rf"returned {code}$"):
        sq.decode(blob, nthreads=4)
    assert sq.kernel_launches() - k0 == TABLES + 2 * slabs(voxels(SHAPE))


# ---------------------------------------------------------------------------------------------------------------- two GPUs
def test_sharded_planes_on_two_gpus(sq, cuda, two_gpus, vol640):
    per_gpu = slabs(voxels(SHAPE) // 2, SUB_SLAB_VOXELS)
    blob, n = counted(sq, sq.encode, "bitswap1->lz4", vol640, nthreads=8)
    assert n == 2 * (ENC_BEGIN + 2 * per_gpu + ENC_END)
    assert sq.last_shard_info() == {"gpus": 2, "nccl": False, "pieces": 2 * 16}
    back, n = counted(sq, sq.decode, blob, nthreads=8)
    assert n == 2 * (TABLES + 2 * per_gpu)
    assert sq.last_shard_info() == {"gpus": 2, "nccl": False, "pieces": 2 * 16}
    assert np.array_equal(back, vol640)


def test_sharded_quantiser_on_two_gpus(sq, cuda, two_gpus, vol640):
    per_gpu = slabs(voxels(SHAPE) // 2, SUB_SLAB_VOXELS)
    blob, n = counted(sq, sq.encode, "quantiser->lz4", vol640, nthreads=8)
    assert n == 2 * (per_gpu + 1 + LZ4_ENCODE)
    info = sq.last_shard_info()
    assert info["gpus"] == 2 and info["pieces"] == 2
    _, n = counted(sq, sq.decode, blob, nthreads=8)
    assert n == 2 * (TABLES + 2 * per_gpu)
    assert sq.last_shard_info() == {"gpus": 2, "nccl": False, "pieces": 2}
