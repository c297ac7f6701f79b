"""A/B of whole SQY_Decode_UI16 calls between library builds on the same GPU in the same process (development tool), for the
host decode of a `bitswap1->lz4` blob that is not one frame of this library: the general decode, whose last inverse transpose
runs slab by slab with every slab leaving for the host as soon as it is done. bench.py has no workload on that route.
usage: ab_host_decode.py libA.so libB.so ...   (env AB_ROUNDS: rounds, default 3; AB_CALLS: calls per timing, default 3;
AB_Z: z-slices of 2048x2048, default 80 = 640 MiB)
The blob is made by oracle.Standin (liblz4, one frame per 256 KiB chunk, as the reference writes with several threads). Builds
run one after the other inside every round; the decoded voxels must be identical across builds and equal to the stack."""
import ctypes, os, statistics, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from ctypes import c_char_p, c_int, c_long
from oracle import oracle as orc
from sqeazy_b200.synth import torch_volume

rounds = int(os.environ.get("AB_ROUNDS", "3"))
calls = int(os.environ.get("AB_CALLS", "3"))
shape = (int(os.environ.get("AB_Z", "80")), 2048, 2048)
libs = [(os.path.basename(p), ctypes.CDLL(os.path.abspath(p))) for p in sys.argv[1:]]
torch.cuda.set_device(0)
for _, L in libs:
    assert L.sqyx_set_device(c_int(0)) == 0
    L.sqyx_kernel_launches.restype = c_long
print("device:", torch.cuda.get_device_name(0), flush=True)

vol = torch_volume(shape, "scmos", index=12).cpu().numpy().view(np.uint16)
name = "bitswap1(num_bits_per_plane=1)->lz4(accel=1,blocksize_kb=256,framestep_kb=256,n_chunks_of_input=0)"
payload, _ = orc.standin().pipeline_encode_stages(0, vol, 8)
h = orc.pack_header(vol.shape, name, payload.size, version="0.5.2", headref="4c45a9b")
blob = np.concatenate([np.frombuffer(h.encode(), dtype=np.uint8), payload])
out = np.empty(vol.size, dtype=np.uint16)
print(f"stack {shape} = {vol.nbytes >> 20} MiB, blob {blob.size >> 20} MiB", flush=True)


def decode(L):
    rc = L.SQY_Decode_UI16(c_char_p(blob.ctypes.data), c_long(blob.size), c_char_p(out.ctypes.data), c_int(8))
    assert rc == 0, rc


def timed(L):
    t0 = time.perf_counter()
    for _ in range(calls):
        decode(L)
    return (time.perf_counter() - t0) * 1e3 / calls


ms = {n: [] for n, _ in libs}
for rnd in range(rounds + 1):                 # round 0 warms up and checks the outputs
    for lname, L in libs:
        if rnd == 0:
            out[...] = 0
            k0 = L.sqyx_kernel_launches()
            decode(L)
            print(f"{lname}: {L.sqyx_kernel_launches() - k0} kernel launches per call", flush=True)
            assert np.array_equal(out, vol.reshape(-1)), f"{lname} decoded other voxels"
            continue
        ms[lname].append(timed(L))
        print(f"round {rnd} {lname:24s} decode {ms[lname][-1]:8.3f} ms", flush=True)
for lname, _ in libs:
    d = ms[lname]
    print(f"median {lname:24s} decode {statistics.median(d):8.3f} ms [{min(d):.3f}..{max(d):.3f}]  "
          f"{vol.nbytes / statistics.median(d) / 1e6:7.1f} voxel-GB/s  (identical outputs)", flush=True)
