"""cfg4 probe: GPU decode of REFERENCE-produced bitswap1->lz4 blobs (oracle/_ref = the reference's stage code + liblz4;
oracle.Standin, the reference's frame encoder restated over liblz4, where oracle/_ref is not built):
serial mode = one block-linked frame (sqy CLI default), parallel mode = one frame per 256 KiB chunk.
usage: bench_cfg4.py [ZxYxX] [serial|parallel] [both-routes]   (both-routes: the linked frame also block after block)"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import sqeazy_b200 as sq
from oracle import oracle as orc
from sqeazy_b200.synth import numpy_volume

shape = (64, 2048, 2048) if len(sys.argv) < 2 else tuple(int(v) for v in sys.argv[1].split("x"))
ref = orc.ref() if orc.ref().available else orc.standin()
assert ref.available
print(f"payloads from {type(ref).__name__}")
torch.cuda.set_device(0); sq.set_device(0)
vol = numpy_volume(shape, "scmos", index=0)
name = "bitswap1(num_bits_per_plane=1)->lz4(accel=1,blocksize_kb=256,framestep_kb=256,n_chunks_of_input=0)"
modes = [("serial/linked", 1, 8), ("parallel/framed", os.cpu_count(), 8)]
if len(sys.argv) > 2 and sys.argv[2] in ("serial", "parallel"):
    modes = [m for m in modes if m[0].startswith(sys.argv[2])]
if len(sys.argv) > 3:
    modes.append(("serial/linked, block after block", 1, 0))
for label, nthreads, defer_min in modes:
    sq.set_lz4_defer_min(defer_min)
    payload, t_enc = ref.pipeline_encode_stages(0, vol, nthreads)
    h = orc.pack_header(vol.shape, name, payload.size, version="0.5.2", headref="4c45a9b")
    blob = torch.from_numpy(np.concatenate([np.frombuffer(h.encode(), dtype=np.uint8), payload])).cuda()
    out = torch.empty(vol.shape, dtype=torch.int16, device="cuda")
    reps = 1 if defer_min == 0 else 3
    for _ in range(1 if defer_min == 0 else 2):
        sq.decode_device(blob, out)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(reps):
        sq.decode_device(blob, out)
    ev1.record(); ev1.synchronize()
    ms = ev0.elapsed_time(ev1) / reps
    ok = np.array_equal(out.cpu().numpy().view(np.uint16), vol)
    rc, _, t_dec = ref.pipeline_decode_stages(1, payload, vol.size)
    print(f"{label}: blob {blob.numel()} B ratio {vol.nbytes / blob.numel():.3f}  GPU decode {ms:.2f} ms = {vol.nbytes / ms / 1e6:.1f} GB/s  bit-exact {ok}  | reference CPU decode {t_dec*1e3:.0f} ms = {vol.nbytes / t_dec / 1e9:.3f} GB/s")
sq.set_lz4_defer_min(8)
