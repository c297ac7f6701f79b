"""A/B of whole host calls (SQY_PipelineEncode_UI16, SQY_Decode_UI16) between library builds on the same GPUs in the same process
(development tool). Workloads:
  cfg2     `rmestbkrd->bitswap1->lz4`, 512x2048x2048 (4 GiB), one GPU: the streamed planes encoder and the slab decoder (the
           route of bench.py's cfg2 `e2e`)
  cfg3     `quantiser->lz4`, 1024x2048x2048 (8 GiB), one GPU: the one-GPU case of the sharded encoder and the slab decoder of
           codes (the route of bench.py's cfg3 `e2e`)
  sharded  `rmestbkrd->bitswap1->lz4`, 4 GiB, over GPUs 0 and 1 (skipped on one GPU)
  foreign  decode of an 80x2048x2048 `bitswap1->lz4` blob that is not one frame of this library (oracle.Standin: liblz4, one
           frame per 256 KiB chunk): the general decode, whose last inverse transpose runs slab by slab
usage: ab_host.py libA.so libB.so ...   (env AB_ROUNDS: rounds, default 5; AB_CALLS: calls per timing, default 3;
AB_WORKLOADS: comma-separated subset, default all)
Pinned host buffers and nthreads = 1, like bench.py's `e2e`. The builds take turns inside every round. Round 0 warms up and
checks: every build must write the same blob bytes, the same last_lz4_stats() and last_shard_info(), and decode to the same
voxels (to the stack itself where the pipeline is lossless)."""
import ctypes, os, statistics, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from ctypes import c_char_p, c_int, c_long, c_uint
import sqeazy_b200 as sq
from sqeazy_b200.synth import torch_volume

rounds = int(os.environ.get("AB_ROUNDS", "5"))
calls = int(os.environ.get("AB_CALLS", "3"))
chosen = os.environ.get("AB_WORKLOADS", "cfg2,cfg3,sharded,foreign").split(",")
libs = [(os.path.basename(p), ctypes.CDLL(os.path.abspath(p))) for p in sys.argv[1:]]
for _, L in libs:
    L.sqyx_kernel_launches.restype = c_long
ngpu = torch.cuda.device_count()
try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                          timeout=30).stdout.strip().splitlines()[0]
except Exception as exc:  # the card name still comes from torch
    card = f"{torch.cuda.get_device_name(0)}, power limit unknown ({exc!r})"
print(f"device: {card}; {ngpu} GPU(s)", flush=True)

FOREIGN = "bitswap1(num_bits_per_plane=1)->lz4(accel=1,blocksize_kb=256,framestep_kb=256,n_chunks_of_input=0)"
WORKLOADS = {   # name: (pipeline, shape, devices, lossless)
    "cfg2": ("rmestbkrd->bitswap1->lz4", (512, 2048, 2048), [0], False),
    "cfg3": ("quantiser->lz4", (1024, 2048, 2048), [0], False),
    "sharded": ("rmestbkrd->bitswap1->lz4", (512, 2048, 2048), [0, 1], False),
    "foreign": (None, (80, 2048, 2048), [0], True),
}


def pinned(nbytes):
    return torch.empty(nbytes, dtype=torch.uint8).pin_memory().numpy()


def use_devices(L, devs):
    if len(devs) == 1:
        assert L.sqyx_set_device(c_int(devs[0])) == 0
    else:
        assert L.sqyx_set_devices(c_int(len(devs)), (c_int * len(devs))(*devs)) == 0


def encode(L, pipeline, vol, shape, blob):
    n = c_long(0)
    rc = L.SQY_PipelineEncode_UI16(pipeline.encode(), c_char_p(vol.ctypes.data), (c_long * 3)(*shape), c_uint(3),
                                   c_char_p(blob.ctypes.data), ctypes.byref(n), c_int(1))
    assert rc == 0, rc
    return n.value


def decode(L, blob, nbytes, out):
    rc = L.SQY_Decode_UI16(c_char_p(blob.ctypes.data), c_long(nbytes), c_char_p(out.ctypes.data), c_int(1))
    assert rc == 0, rc


def info(L):
    stats, shard = (c_long * 4)(), (c_long * 3)()
    assert L.sqyx_last_lz4_stats(stats) == 0 and L.sqyx_last_shard_info(shard) == 0
    return list(stats), list(shard)


def timed(fn):
    t0 = time.perf_counter()
    for _ in range(calls):
        fn()
    return (time.perf_counter() - t0) * 1e3 / calls


for wname in chosen:
    pipeline, shape, devs, lossless = WORKLOADS[wname]
    if len(devs) > ngpu:
        print(f"{wname}: skipped, needs {len(devs)} GPUs", flush=True)
        continue
    torch.cuda.set_device(0)
    nvox = int(np.prod(shape))
    vol = pinned(2 * nvox).view(np.uint16)
    vol[:] = torch_volume(shape, "scmos", index=12).cpu().numpy().view(np.uint16).reshape(-1)
    torch.cuda.empty_cache()
    out = pinned(2 * nvox).view(np.uint16)
    if pipeline is None:      # a foreign blob: decode only
        from oracle import oracle as orc
        payload, _ = orc.standin().pipeline_encode_stages(0, vol.reshape(shape), 8)
        h = np.frombuffer(orc.pack_header(shape, FOREIGN, payload.size, version="0.5.2", headref="4c45a9b").encode(), dtype=np.uint8)
        blob = pinned(h.size + payload.size)
        blob[: h.size] = h
        blob[h.size :] = payload
        nblob = blob.size
    else:
        blob = pinned(sq.max_compressed_length_3d(pipeline, shape))
    print(f"{wname}: {pipeline or FOREIGN} {shape} = {2 * nvox >> 20} MiB on GPU(s) {devs}", flush=True)
    ref = None
    ms = {n: {"encode": [], "decode": []} for n, _ in libs}
    for rnd in range(rounds + 1):             # round 0 warms up and checks the outputs
        for lname, L in libs:
            use_devices(L, devs)
            if rnd == 0:
                k0 = L.sqyx_kernel_launches()
                if pipeline is not None:
                    nblob = encode(L, pipeline, vol, shape, blob)
                k1 = L.sqyx_kernel_launches()
                got = (blob[:nblob].copy(), info(L)) if pipeline is not None else None
                out[:] = 0
                decode(L, blob, nblob, out)
                k2 = L.sqyx_kernel_launches()
                print(f"  {lname}: blob {nblob} B, kernel launches: encode {k1 - k0}, decode {k2 - k1}; "
                      f"lz4 stats / shard info {got[1] if got else '-'}", flush=True)
                if lossless:
                    assert np.array_equal(out, vol), f"{lname} decoded other voxels"
                if ref is None:
                    ref = (got, out.copy() if not lossless else None)
                else:
                    if got is not None:
                        assert np.array_equal(got[0], ref[0][0]), f"{lname} wrote other blob bytes"
                        assert got[1] == ref[0][1], f"{lname}: lz4 stats / shard info {got[1]} != {ref[0][1]}"
                    if not lossless:
                        assert np.array_equal(out, ref[1]), f"{lname} decoded other voxels"
                continue
            if pipeline is not None:
                ms[lname]["encode"].append(timed(lambda: encode(L, pipeline, vol, shape, blob)))
            ms[lname]["decode"].append(timed(lambda: decode(L, blob, nblob, out)))
            print(f"  round {rnd} {lname:24s} " + "  ".join(f"{k} {v[-1]:8.3f} ms" for k, v in ms[lname].items() if v), flush=True)
    for lname, _ in libs:
        for k, d in ms[lname].items():
            if d:
                print(f"{wname} median {lname:24s} {k} {statistics.median(d):8.3f} ms [{min(d):.3f}..{max(d):.3f}]  "
                      f"{2 * nvox / statistics.median(d) / 1e6:7.1f} voxel-GB/s", flush=True)
    print(f"{wname}: identical blobs, stats and voxels across builds", flush=True)
    del vol, out, blob, ref
