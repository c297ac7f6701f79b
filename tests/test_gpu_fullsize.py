"""BASELINE.json's full sizes, checked through size-independent properties (the oracle cannot run 4-8 GiB in test time):
the pipeline's result must equal what the single-stage kernels — a different code path — produce, lossless pipelines must
return their input, and the 2^31 / 2^32 voxel boundaries (where the reference's 32-bit sizes give up, SURVEY F7) must hold."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture
def roomy(sq, cuda):
    free, _ = cuda.cuda.mem_get_info()
    if free < 60 << 30:
        pytest.skip("needs ~60 GB of free device memory")
    yield
    sq.release_scratch()
    cuda.cuda.empty_cache()


def _oracle_slabs(Z, frames=16):
    """z-ranges the oracle restates at full size: the first frames, a slab in the middle of the shell, the last frames"""
    return [(0, frames), (Z // 2 - frames // 2, Z // 2 + frames // 2), (Z - frames, Z)]


def test_cfg2_full_size(sq, cuda, port, roomy):
    """rmestbkrd->bitswap1->lz4 on 2048x2048x512 uint16 = 2^31 voxels, 4 GiB"""
    from sqeazy_b200.synth import torch_volume

    shape = (512, 2048, 2048)
    vol = torch_volume(shape, "scmos", index=0)
    assert vol.numel() == 1 << 31
    # expected voxels from the stage kernels: threshold estimate + stand-alone remove_background (not the fused transpose)
    _, thr = sq.estimate_background_device(vol)
    assert 90 < thr < 130
    expect = cuda.empty_like(vol)
    sq.remove_background_device(vol.view(-1), expect.view(-1), thr)
    blob = sq.encode_device("rmestbkrd->bitswap1->lz4", vol)
    assert blob.numel() <= sq.max_compressed_length("rmestbkrd->bitswap1->lz4", vol.numel() * 2)
    st = sq.last_lz4_stats()
    assert st["constant_blocks"] + st["general_blocks"] + st["stored_blocks"] == (vol.numel() * 2) // 16384
    assert st["constant_blocks"] > st["general_blocks"] > 0      # the upper planes of a background-removed stack are empty
    out = cuda.empty_like(vol)
    sq.decode_device(blob, out)
    assert cuda.equal(out, expect)
    ratio = vol.numel() * 2 / blob.numel()
    assert 10 < ratio < 40
    # SURVEY F7: the reference cannot index 2^31 voxels (dynamic_pipeline.hpp:514), so the ORACLE pins the full-size result
    # slab by slab: the threshold of the whole stack from the faces / rows it samples (background_scheme_utils.hpp:35-105),
    # then remove_background (remove_background_scheme_impl.hpp:73-95) on three 16-frame slabs of the decoded stack
    h_vol = vol.cpu().numpy().view(np.uint16)
    supports = port.darkest_face_supports(h_vol, sq.host_l2_bytes())
    assert int(np.uint16(supports.min())) == thr
    for z0, z1 in _oracle_slabs(shape[0]):
        want = port.remove_background(h_vol[z0:z1], thr)
        got = out[z0:z1].cpu().numpy().view(np.uint16)
        assert np.array_equal(got, want), (z0, z1)
    del h_vol
    # idempotence of the lossy filter + a lossless pipeline on the result returns it unchanged
    blob2 = sq.encode_device("bitswap1->lz4", out)
    back = cuda.empty_like(vol)
    sq.decode_device(blob2, back)
    assert cuda.equal(back, expect)
    del blob, blob2, back, out, expect, vol


def test_cfg3_full_size(sq, cuda, port, roomy):
    """quantiser->lz4 on 2048x2048x1024 uint16 = 2^32 voxels, 8 GiB raw, 4 GiB of 8-bit codes"""
    from sqeazy_b200.synth import torch_volume

    shape = (1024, 2048, 2048)
    vol = torch_volume(shape, "scmos", index=1)
    assert vol.numel() == 1 << 32
    hist = cuda.zeros(65536, dtype=cuda.int32, device="cuda")
    sq.histogram_device(vol, hist)
    cuda.cuda.synchronize()
    h = hist.cpu().numpy().view(np.uint32)
    assert int(h.astype(np.uint64).sum()) == 1 << 32
    ref_hist = cuda.zeros(65536, dtype=cuda.int64, device="cuda")
    flat = vol.view(-1)
    for lo in range(0, flat.numel(), 1 << 28):      # independent count: torch.bincount, 2^28 voxels at a time
        ref_hist += cuda.bincount(flat[lo: lo + (1 << 28)].to(cuda.int32) & 0xFFFF, minlength=65536)
    assert np.array_equal(ref_hist.cpu().numpy().astype(np.uint64), h.astype(np.uint64))
    enc, dec = sq.quantiser_luts(h)
    codes = cuda.empty(vol.numel(), dtype=cuda.uint8, device="cuda")
    sq.lut_apply_device(vol, codes, enc)
    expect = cuda.empty_like(vol)
    sq.lut_decode_device(codes, expect.view(-1), dec)
    del codes
    blob = sq.encode_device("quantiser->lz4", vol)
    out = cuda.empty_like(vol)
    sq.decode_device(blob, out)
    assert cuda.equal(out, expect)
    assert 1.9 < vol.numel() * 2 / blob.numel() < 4
    # the oracle at full size: LUTs of the WHOLE stack's histogram (quantiser_utils.hpp:227-306), then LUT apply and decode
    # (quantiser_scheme_impl.hpp:206-223, 245-282) on three 16-frame slabs
    o_enc, o_dec = port.quantiser_luts(h)
    assert np.array_equal(o_enc, enc) and np.array_equal(o_dec, dec)
    for z0, z1 in _oracle_slabs(shape[0]):
        slab = vol[z0:z1].cpu().numpy().view(np.uint16)
        want = port.lut_decode(port.lut_apply(slab, o_enc), o_dec)
        got = out[z0:z1].cpu().numpy().view(np.uint16)
        assert np.array_equal(got.reshape(-1), want.reshape(-1)), (z0, z1)
    del blob, out, expect, vol


@pytest.mark.parametrize("bits", [16, 8])
def test_threshold_kernels_over_many_grid_sweeps(sq, cuda, bits):
    """Regression: the packed saturating subtraction must hold in every grid-stride sweep. With __vsubus2, ptxas 12.9
    unrolled the sweep loop by four and rebuilt the packed constant wrongly in the unrolled copies: beyond ~39 M voxels
    every other voxel lost threshold+1 (stand-alone remove_background only; found by test_cfg2_full_size). Sizes here give
    every thread of the capped grid more than eight sweeps; the expected values come from torch arithmetic."""
    n = 120_000_000 if bits == 16 else 200_000_000
    g = cuda.Generator(device="cuda")
    g.manual_seed(bits)
    if bits == 16:
        v = cuda.randint(0, 400, (n,), generator=g, device="cuda", dtype=cuda.int32).to(cuda.int16)
        thr = 106
        ref = (v.to(cuda.int32) - thr).clamp_(min=0).to(cuda.int16)
        out = cuda.empty_like(v)
        sq.remove_background_device(v, out, thr)
        assert cuda.equal(out, ref)
        n128 = n - n % 128
        planes = cuda.empty(n128, dtype=cuda.int16, device="cuda")
        sq.bitswap_encode_device(1, v[:n128], planes, threshold=thr)
        sq.bitswap_decode_device(1, planes, out[:n128])
        assert cuda.equal(out[:n128], ref[:n128])
    else:
        v = cuda.randint(0, 256, (n,), generator=g, device="cuda", dtype=cuda.uint8)
        thr = 19
        ref = (v.to(cuda.int16) - thr).clamp_(min=0).to(cuda.uint8)
        out = cuda.empty_like(v)
        sq.remove_background_device_u8(v, out, thr)
        assert cuda.equal(out, ref)
        n128 = n - n % 128
        planes = cuda.empty(n128, dtype=cuda.uint8, device="cuda")
        for w in (1, 4):
            sq.bitswap_encode_device_u8(w, v[:n128], planes, threshold=thr)
            sq.bitswap_decode_device_u8(w, planes, out[:n128])
            assert cuda.equal(out[:n128], ref[:n128])


def _torch_bitswap(cuda, x, w, bits):
    """independent restatement of bitplane_reorder_scalar.hpp:27-74 with torch integer arithmetic (int64 lanes)"""
    P = bits // w
    n = x.numel()
    S = n // P
    v = x.to(cuda.int64) & ((1 << bits) - 1)
    g = v[: S * P].view(S, P)
    out = cuda.empty(n, dtype=cuda.int64, device=x.device)
    for p in range(P):
        word = cuda.zeros(S, dtype=cuda.int64, device=x.device)
        for j in range(P):
            word |= ((g[:, j] >> (p * w)) & ((1 << w) - 1)) << ((bits - w) - j * w)
        out[(P - 1 - p) * S: (P - p) * S] = word
    out[S * P:] = v[S * P:]
    return out


@pytest.mark.parametrize("bits,w", [(16, 2), (16, 4), (16, 8), (16, 1), (8, 1), (8, 2), (8, 4)])
def test_bitswap_over_many_grid_sweeps(sq, cuda, bits, w):
    """every fast transpose kernel over > 8 sweeps of its capped grid, against torch arithmetic; ragged tail included"""
    n = 40_000_000 * 2 + (0 if w != 4 else 5)      # the +5 takes the generic kernel (n % 128 != 0)
    g = cuda.Generator(device="cuda")
    g.manual_seed(bits * 10 + w)
    if bits == 16:
        x = cuda.randint(0, 65536, (n,), generator=g, device="cuda", dtype=cuda.int32).to(cuda.int16)
        out = cuda.empty_like(x)
        sq.bitswap_encode_device(w, x, out)
        ref = _torch_bitswap(cuda, x, w, 16)
        assert cuda.equal(out.to(cuda.int64) & 0xFFFF, ref)
        back = cuda.empty_like(x)
        sq.bitswap_decode_device(w, out, back)
        assert cuda.equal(back, x)
    else:
        x = cuda.randint(0, 256, (n,), generator=g, device="cuda", dtype=cuda.uint8)
        out = cuda.empty_like(x)
        sq.bitswap_encode_device_u8(w, x, out)
        ref = _torch_bitswap(cuda, x, w, 8)
        assert cuda.equal(out.to(cuda.int64), ref)
        back = cuda.empty_like(x)
        sq.bitswap_decode_device_u8(w, out, back)
        assert cuda.equal(back, x)


def test_lossless_pipeline_on_eight_gib(sq, cuda, roomy):
    """bitswap1->lz4 on 2^32 voxels: 8 GiB of bit planes, 524288 LZ4 blocks, every size beyond 32 bits"""
    from sqeazy_b200.synth import torch_volume

    vol = torch_volume((1024, 2048, 2048), "scmos", index=2)
    blob = sq.encode_device("bitswap1->lz4", vol)
    st = sq.last_lz4_stats()
    assert st["constant_blocks"] + st["general_blocks"] + st["stored_blocks"] == (vol.numel() * 2) // 16384 == 524288
    out = cuda.empty_like(vol)
    sq.decode_device(blob, out)
    assert cuda.equal(out, vol)
    assert 2.0 < vol.numel() * 2 / blob.numel() < 4.0
    del blob, out, vol


def test_cfg2_slab_ratio_against_the_reference_on_the_same_voxels(sq, cuda, ref_or_standin):
    """DESIGN.md 5: on background-removed, very compressible stacks the blob may be at most 10 % larger than the reference's
    (ratio >= 0.90 x): 16 KiB independent blocks against liblz4's 64 KiB window inside 256 KiB blocks. Same 2^26 voxels through
    both encoders (the reference's own stage chain, dynamic_pipeline.hpp:560-690 re-driven by oracle/ref_harness.cpp), and the
    reference's decode chain (lz4.hpp:257-339 + bitplane_reorder_scalar.hpp:81-116) must read the GPU's blob."""
    from sqeazy_b200.synth import numpy_volume

    vol = numpy_volume((16, 2048, 2048), "scmos", index=0)
    theirs, _ = ref_or_standin.pipeline_encode_stages(1, vol, 8)
    blob = sq.encode("rmestbkrd->bitswap1->lz4", vol)
    hs = sq.header_size(blob)
    ours = blob.size - hs
    assert ours <= theirs.size / 0.90, (ours, theirs.size, vol.nbytes / ours, vol.nbytes / theirs.size)
    rc, back_theirs, _ = ref_or_standin.pipeline_decode_stages(1, theirs, vol.size)
    rc2, back_ours, _ = ref_or_standin.pipeline_decode_stages(1, blob[hs:], vol.size)
    assert rc == 0 and rc2 == 0
    assert np.array_equal(back_ours, back_theirs)
    assert np.array_equal(sq.decode(blob).reshape(-1), back_theirs.reshape(-1))
