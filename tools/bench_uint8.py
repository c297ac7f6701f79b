"""uint8 path: device times of the uint8 bitswap / remove_background kernels (1 GiB) and of bitswap1->lz4 through sqyx_*_UI8."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import sqeazy_b200 as sq

torch.cuda.set_device(0); sq.set_device(0)
n = 1 << 30
g = torch.Generator(device="cuda"); g.manual_seed(1)
vol = (20 + 2 * torch.randn(n, generator=g, device="cuda")).round_().clamp_(0, 255).to(torch.uint8)
vol.view(256, 2048, 2048)[80:120, 500:1200] += 90
out = torch.empty_like(vol)


def timed(fn, reps=5):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record(); e1.synchronize()
    return e0.elapsed_time(e1) / reps


for w in (1, 2, 4):
    ms = timed(lambda: sq.bitswap_encode_device_u8(w, vol, out))
    ms_f = timed(lambda: sq.bitswap_encode_device_u8(w, vol, out, threshold=19))
    back = torch.empty_like(vol)
    sq.bitswap_encode_device_u8(w, vol, out)
    ms_d = timed(lambda: sq.bitswap_decode_device_u8(w, out, back))
    print(f"bitswap{w} uint8 1 GiB: encode {ms:.3f} ms = {2 * n / ms / 1e6:.0f} GB/s, fused threshold {ms_f:.3f} ms, decode {ms_d:.3f} ms = {2 * n / ms_d / 1e6:.0f} GB/s, roundtrip ok {torch.equal(back, vol)}")
ms = timed(lambda: sq.remove_background_device_u8(vol, out, 19))
print(f"remove_background uint8 1 GiB: {ms:.3f} ms = {2 * n / ms / 1e6:.0f} GB/s")
v3 = vol.view(256, 2048, 2048)
blob = sq.encode_device_u8("remove_background(threshold=19)->bitswap1->lz4", v3)
buf = torch.empty(sq.max_compressed_length_u8("remove_background(threshold=19)->bitswap1->lz4", n), dtype=torch.uint8, device="cuda")
ms_e = timed(lambda: sq.encode_device_u8("remove_background(threshold=19)->bitswap1->lz4", v3, out=buf), 3)
blob = sq.encode_device_u8("remove_background(threshold=19)->bitswap1->lz4", v3, out=buf)
ms_d = timed(lambda: sq.decode_device_u8(blob, out), 3)
print(f"remove_background(threshold=19)->bitswap1->lz4 uint8 1 GiB: encode {ms_e:.2f} ms = {n / ms_e / 1e6:.0f} voxel-GB/s, decode {ms_d:.2f} ms = {n / ms_d / 1e6:.0f} voxel-GB/s, ratio {n / blob.numel():.2f}, {sq.last_lz4_stats()}")
