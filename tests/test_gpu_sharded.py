"""One stack sharded over several GPUs INSIDE the C ABI (csrc/sharded.inl; SURVEY §8e, north_star: "stacks and z-slabs are
partitioned over the GPUs; the only collective is an allreduce of the quantiser's global histogram"). The reference's
entry points SQY_PipelineEncode_UI16 / SQY_Decode_UI16 (src/cpp/src/sqeazy.cpp:108-142, 281-307) know nothing of devices:
the blob a sharded call writes must be a plain blob — decodable by one GPU, by several, and by the reference's own stage
code — with the voxels of the single-GPU path. Needs >= 2 GPUs (gpurun --gpus 2); skipped on a single-GPU box."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SHAPE = (64, 2048, 2048)          # 512 MiB: 256 MiB per GPU at G = 2
EXACT = True                      # byte equality of blobs (needs the deterministic encoder)


def _same_blob(a, b):
    if EXACT:
        return a.size == b.size and np.array_equal(a, b)
    return abs(int(a.size) - int(b.size)) <= 0.02 * b.size


@pytest.fixture
def two_gpus(sq, cuda):
    if cuda.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    yield [0, 1] if cuda.cuda.device_count() < 4 else [0, 1, 2, 3]
    sq.set_device(0)


def _host_volume(cuda, kind, index):
    from sqeazy_b200.synth import torch_volume

    d_vol = torch_volume(SHAPE, "scmos", index=index)
    h = cuda.empty(SHAPE, dtype=cuda.int16)
    if kind == "pinned":
        h = h.pin_memory()
    h.copy_(d_vol)
    del d_vol
    return h


@pytest.mark.parametrize("kind", ["pinned", "pageable"])
@pytest.mark.parametrize("pipeline", ["bitswap1->lz4", "rmestbkrd->bitswap1->lz4", "remove_background(threshold=110)->bitswap4->lz4"])
def test_sharded_planes_blob_is_the_single_gpu_blob(sq, cuda, ref_or_standin, two_gpus, pipeline, kind):
    h = _host_volume(cuda, kind, 21)
    vol = h.numpy().view(np.uint16)
    sq.set_device(0)
    blob1 = sq.encode(pipeline, vol, nthreads=8).copy()
    assert sq.last_shard_info()["gpus"] == 0
    want = sq.decode(blob1, nthreads=8)
    if pipeline == "bitswap1->lz4":
        assert np.array_equal(want.reshape(SHAPE), vol)
    sq.set_devices(two_gpus)
    blobn = sq.encode(pipeline, vol, nthreads=8).copy()
    info = sq.last_shard_info()
    assert info["gpus"] == len(two_gpus), info
    # same blocks, same header: the sharded blob IS the single-GPU blob (the encoder is deterministic)
    assert _same_blob(blobn, blob1)
    # several GPUs decode what one GPU wrote and the other way round; pageable and pinned destinations
    out = cuda.empty(SHAPE, dtype=cuda.int16)
    if kind == "pinned":
        out = out.pin_memory()
    o = out.numpy().view(np.uint16).reshape(-1)
    o[...] = 0xABCD
    sq.decode(blob1, nthreads=8, out=o)
    assert sq.last_shard_info()["gpus"] == len(two_gpus)
    assert np.array_equal(o, want.reshape(-1))
    sq.set_device(0)
    o[...] = 0
    sq.decode(blobn, nthreads=3, out=o)
    assert sq.last_shard_info()["gpus"] == 0
    assert np.array_equal(o, want.reshape(-1))
    # the reference's own decoder (LZ4F loop + scalar bitswap decode) reads the sharded blob
    if "bitswap1" in pipeline:
        rc, back, _ = ref_or_standin.pipeline_decode_stages(1, blobn[sq.header_size(blobn):], vol.size)
        assert rc == 0 and np.array_equal(back, want.reshape(-1))


@pytest.mark.parametrize("nccl", [True, False])
def test_sharded_quantiser_uses_one_global_histogram(sq, cuda, two_gpus, nccl, monkeypatch):
    """quantiser -> lz4: local histograms, ncclAllReduce (or the host sum when NCCL is switched off), ONE LUT: header text
    (it carries the decode LUT), codes and decoded voxels are those of the single-GPU encode"""
    h = _host_volume(cuda, "pinned", 22)
    vol = h.numpy().view(np.uint16)
    sq.set_device(0)
    blob1 = sq.encode("quantiser->lz4", vol, nthreads=4).copy()
    want = sq.decode(blob1, nthreads=4)
    sq.set_devices(two_gpus)
    before = sq.nccl_allreduces()
    if not nccl:
        pytest.skip("host-sum variant is selected per process (SQY_NO_NCCL=1): covered by tests/test_sharded_env.py")
    blobn = sq.encode("quantiser->lz4", vol, nthreads=4).copy()
    info = sq.last_shard_info()
    # (a GPU takes at least 128 MiB of the LZ4 stream — here the 256 MiB of 8-bit codes: two GPUs, however many there are)
    assert info["gpus"] == min(len(two_gpus), vol.size // (128 << 20))
    assert info["nccl"], "NCCL was not used for the histogram all-reduce"
    assert sq.nccl_allreduces() == before + 1
    assert _same_blob(blobn, blob1)
    assert sq.decompressed_shape(blobn) == sq.decompressed_shape(blob1)
    hs = sq.header_size(blob1)
    assert bytes(blobn[:hs]).strip().split(b'"encoded"')[0] == bytes(blob1[:hs]).strip().split(b'"encoded"')[0]   # same LUT in the header
    back = sq.decode(blobn, nthreads=4)
    assert sq.last_shard_info()["gpus"] == min(len(two_gpus), vol.size // (128 << 20))
    assert np.array_equal(back, want)


def test_sharded_calls_are_reentrant_and_respect_the_device_set(sq, cuda, two_gpus):
    """two host threads encode at the same time (the device locks are taken in ascending order), then the set is narrowed"""
    import threading

    h = _host_volume(cuda, "pinned", 23)
    vol = h.numpy().view(np.uint16)
    sq.set_devices(two_gpus)
    blobs = [None, None]

    def run(i):
        blobs[i] = sq.encode("bitswap1->lz4", vol, nthreads=2).copy()

    th = [threading.Thread(target=run, args=(i,)) for i in range(2)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert _same_blob(blobs[0], blobs[1])
    sq.set_devices([1])
    b = sq.encode("bitswap1->lz4", vol, nthreads=2)
    assert sq.last_shard_info()["gpus"] == 0 and _same_blob(b, blobs[0])
    sq.set_devices(None)         # default: every visible device
    b = sq.encode("bitswap1->lz4", vol, nthreads=2)
    assert sq.last_shard_info()["gpus"] >= 2 and _same_blob(b, blobs[0])
    assert np.array_equal(sq.decode(b).reshape(SHAPE), vol)
