"""The LZ4 block decoder transposes the bit planes of `[filter ->] bitswapW -> lz4` back itself (lz4_decode_kernel with FW != 0)
when the stack has at least 1 GiB (api.cu: kFuseMinBytes), the stream is one frame of this library, N is a multiple of
8192 * 16/W voxels (no 16 KiB block straddles two planes) and the buffers are 32-byte aligned. The voxels must be exactly what the
two-launch route (LZ4 decode, then bitswap decode) gives. The route is told apart by the launch count of a decode call: 5 table
kernels + the block decoder, plus one bitswap launch when it is not fused."""
import numpy as np
import pytest

from oracle import oracle as orc
from sqeazy_b200.synth import numpy_volume, torch_volume
from test_gpu_parity import dev, host16

pytestmark = pytest.mark.gpu

FUSED_LAUNCHES = 6
TWO_LAUNCH = 7
GIB_SHAPE = (128, 2048, 2048)        # 1 GiB: the smallest stack that takes the fused route

FILTERS = ["", "remove_background(threshold=110)->", "rmestbkrd->"]


def decode_counted(sq, cuda, blob, out):
    cuda.cuda.synchronize()
    k0 = sq.kernel_launches()
    sq.decode_device(blob, out)
    cuda.cuda.synchronize()
    return sq.kernel_launches() - k0


def two_launch_reference(sq, cuda, blob, w, n):
    """the standalone entry points: LZ4 decode of the payload, then the bitswap decode"""
    hsz = sq.header_size(blob[:65536].cpu().numpy())
    planes = cuda.empty(n, dtype=cuda.int16, device="cuda")
    assert sq.lz4_decode_device(blob[hsz:], planes) == 2 * n
    out = cuda.empty(n, dtype=cuda.int16, device="cuda")
    sq.bitswap_decode_device(w, planes, out)
    del planes
    return out


def filtered(sq, filt, vol):
    """what a lossy pipeline decodes to, in torch arithmetic on the device (int16 tensors hold the uint16 bit patterns)"""
    import torch

    if not filt:
        return vol
    thr = sq.estimate_background_device(vol)[1] if filt.startswith("rmestbkrd") else 110
    x = ((vol.to(torch.int32) & 0xFFFF) - thr).clamp_min(0)
    return torch.where(x >= 32768, x - 65536, x).to(torch.int16)


@pytest.mark.parametrize("filt", FILTERS)
@pytest.mark.parametrize("w", [1, 2, 4, 8])
def test_fused_decode_matches_the_two_launch_route(sq, cuda, w, filt):
    vol = torch_volume(GIB_SHAPE, "scmos", index=w)
    blob = sq.encode_device(f"{filt}bitswap{w}->lz4", vol).clone()
    out = cuda.empty_like(vol)
    assert decode_counted(sq, cuda, blob, out) == FUSED_LAUNCHES
    assert cuda.equal(out, filtered(sq, filt, vol))
    assert cuda.equal(out.view(-1), two_launch_reference(sq, cuda, blob, w, vol.numel()))


# below 1 GiB, ragged N, and a destination that is not 32-byte aligned: the two launches
@pytest.mark.parametrize("shape", [(127, 2048, 2048), (129, 2048, 2047), (8, 128, 256), (12, 128, 250)])
def test_other_stacks_take_the_two_launch_route(sq, cuda, shape):
    vol = torch_volume(shape, "scmos", index=3)
    blob = sq.encode_device("rmestbkrd->bitswap1->lz4", vol).clone()
    out = cuda.empty_like(vol)
    assert decode_counted(sq, cuda, blob, out) == TWO_LAUNCH
    assert cuda.equal(out, filtered(sq, "rmestbkrd->", vol))


def test_misaligned_destination_takes_the_two_launch_route(sq, cuda):
    vol = torch_volume(GIB_SHAPE, "scmos", index=4)
    blob = sq.encode_device("bitswap1->lz4", vol).clone()
    room = cuda.empty(vol.numel() + 16, dtype=cuda.int16, device="cuda")
    out = room[1 : 1 + vol.numel()]                          # 2 bytes past a 256-byte boundary
    assert decode_counted(sq, cuda, blob, out) == TWO_LAUNCH
    assert cuda.equal(out, vol.view(-1))


def test_fused_decode_behind_another_transform(sq, cuda):
    """the LZ4 decoder does the first of two transforms back; the bitshuffle decode follows as before"""
    vol = torch_volume(GIB_SHAPE, "scmos", index=7)
    blob = sq.encode_device("bitshuffle->bitswap2->lz4", vol).clone()
    out = cuda.empty_like(vol)
    launches = decode_counted(sq, cuda, blob, out)
    assert cuda.equal(out, vol)
    scratch = cuda.empty_like(out)
    k0 = sq.kernel_launches()
    sq.bitshuffle_decode_device(out, scratch)
    assert launches == FUSED_LAUNCHES + sq.kernel_launches() - k0


def test_fused_decode_of_constant_stacks(sq, cuda):
    for value in (0, 0x7FFF, -1):
        vol = cuda.full(GIB_SHAPE, value, dtype=cuda.int16, device="cuda")
        blob = sq.encode_device("bitswap1->lz4", vol).clone()
        out = cuda.empty_like(vol)
        assert decode_counted(sq, cuda, blob, out) == FUSED_LAUNCHES
        assert cuda.equal(out, vol)
        del vol, blob, out


def test_fused_decode_of_a_batch(sq, cuda):
    pipe = "remove_background(threshold=110)->bitswap4->lz4"
    vols = [torch_volume(GIB_SHAPE, "scmos", index=30 + i) for i in range(2)]
    blobs = [b.clone() for b in sq.encode_batch_device(pipe, vols)]
    outs = [cuda.empty_like(v) for v in vols]
    k0 = sq.kernel_launches()
    sq.decode_batch_device(blobs, outs)
    assert sq.kernel_launches() - k0 == FUSED_LAUNCHES * len(vols)
    for v, o in zip(vols, outs):
        assert cuda.equal(o, filtered(sq, pipe, v))


def test_reference_framed_stack_builds_its_block_table_once(sq, cuda, ref_or_standin):
    """a fusable shape whose blob is not a frame of this library: the table built for the fused route serves the block decoder"""
    n = int(np.prod(GIB_SHAPE))
    vol = (np.arange(n, dtype=np.uint32) * 2654435761 >> 27).astype(np.uint16).reshape(GIB_SHAPE)   # 5-bit values
    payload, _ = ref_or_standin.pipeline_encode_stages(0, vol, 8)            # one frame per 256 KiB chunk
    name = "bitswap1(num_bits_per_plane=1)->lz4(accel=1,blocksize_kb=256,framestep_kb=256,n_chunks_of_input=0)"
    h = orc.pack_header(vol.shape, name, payload.size, version="0.5.2", headref="4c45a9b")
    blob = cuda.from_numpy(np.concatenate([np.frombuffer(h.encode(), dtype=np.uint8), payload])).cuda()
    out = cuda.empty(GIB_SHAPE, dtype=cuda.int16, device="cuda")
    assert decode_counted(sq, cuda, blob, out) == TWO_LAUNCH
    assert cuda.equal(out, dev(cuda, vol))


def first_compressed_block(payload):
    """(offset, size) of the data of the first compressed block of the payload's LZ4 frame"""
    p = 8 + int(payload[4:8].view(np.uint32)[0]) + 7      # skippable index frame, LZ4 frame header
    while True:
        word = int(payload[p : p + 4].view(np.uint32)[0])
        assert word != 0
        if not word >> 31:
            return p + 4, word & 0x7FFFFFFF
        p += 4 + (word & 0x7FFFFFFF)


@pytest.mark.parametrize("where", ["block", "index"])
def test_corrupt_blob_is_refused_and_nothing_is_written_past_dst(sq, cuda, where):
    vol = torch_volume(GIB_SHAPE, "scmos", index=5)
    blob = sq.encode_device("rmestbkrd->bitswap1->lz4", vol).clone()
    good = cuda.empty_like(vol)
    assert decode_counted(sq, cuda, blob, good) == FUSED_LAUNCHES
    h = blob.cpu().numpy()
    hsz = sq.header_size(h[:65536])
    bad = h.copy()
    if where == "block":
        # a compressed block turned into one endless literal run: the frame and its index stay intact, the fused decoder runs
        # and finds the block broken
        off, csize = first_compressed_block(h[hsz:])
        bad[hsz + off : hsz + off + csize] = 0xFF
    else:
        # the index promises a block size the frame does not have: refused while the block table is built
        bad[hsz + 8 + 32] ^= 0x01
    n = vol.numel()
    guard = 4096
    full = cuda.full((n + guard,), 0x5A5A, dtype=cuda.int16, device="cuda")
    with pytest.raises(sq.SqeazyError):
        sq.decode_device(cuda.from_numpy(bad).cuda(), full[:n])
    assert bool((full[n:] == 0x5A5A).all())
    del full
    again = cuda.empty_like(vol)
    assert decode_counted(sq, cuda, blob, again) == FUSED_LAUNCHES      # the next decode works
    assert cuda.equal(again, good)


def test_small_stacks_keep_their_results(sq, cuda, port):
    """a sample of the shapes the fused route does not take, through device and host entry points"""
    for w in (1, 4):
        vol = numpy_volume((8, 128, 256), "scmos", index=w)
        blob = sq.encode_device(f"remove_background(threshold=110)->bitswap{w}->lz4", dev(cuda, vol)).clone()
        out = cuda.empty((8, 128, 256), dtype=cuda.int16, device="cuda")
        assert decode_counted(sq, cuda, blob, out) == TWO_LAUNCH
        want = port.remove_background(vol.reshape(-1), 110).reshape(vol.shape)
        assert np.array_equal(host16(out), want)
        assert np.array_equal(sq.decode(blob.cpu().numpy()), want)
