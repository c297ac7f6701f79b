"""A/B of whole encode_device / decode_device calls between library builds on the same GPU in the same process (development
tool), for the LZ4 decode with the transpose back folded in. The build without it:
    SRC=api tools/build_variant.sh nofuse -DSQYB_FUSE_TRANSPOSE=0      (-> build/ab/lib_nofuse.so)
usage: ab_fused.py libA.so libB.so ...   (env AB_ROUNDS: rounds, default 3; AB_ONLY=cfg2,cfg1,cfg5; AB_CALLS: calls per timing)
Inputs are bench.py's cfg2, cfg1 and cfg5 (a batch of 8 stacks). Builds run one after the other inside every round; every
blob and every decoded voxel must be identical across builds."""
import ctypes, os, statistics, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import sqeazy_b200 as sq
from sqeazy_b200.synth import torch_volume
from ctypes import c_int, c_long, c_uint, c_void_p

WORK = {  # name: shape, pipeline, preset index, stacks
    "cfg2": ((512, 2048, 2048), "rmestbkrd->bitswap1->lz4", 1, 1),
    "cfg1": ((256, 512, 512), "bitswap1->lz4", 0, 1),
    "cfg5": ((128, 1024, 1024), "remove_background(threshold=110)->bitswap4->lz4", 3, 8),
}
rounds = int(os.environ.get("AB_ROUNDS", "3"))
calls = int(os.environ.get("AB_CALLS", "3"))
only = os.environ.get("AB_ONLY")
torch.cuda.set_device(0)
sq.set_device(0)
libs = [(os.path.basename(p), ctypes.CDLL(os.path.abspath(p))) for p in sys.argv[1:]]
st = c_void_p(torch.cuda.current_stream().cuda_stream)
print("device:", torch.cuda.get_device_name(0), flush=True)


def ptrs(ts):
    return (c_void_p * len(ts))(*[t.data_ptr() for t in ts])


for wname, (shape, pipe, index, nstacks) in WORK.items():
    if only and wname not in only.split(","):
        continue
    vols = [torch_volume(shape, "scmos", index=index + i) for i in range(nstacks)]
    cap = sq.max_compressed_length(pipe, vols[0].numel() * 2)
    shp = (c_long * 3)(*shape)
    bufs = [torch.empty(cap, dtype=torch.uint8, device="cuda") for _ in vols]
    outs = [torch.empty_like(v) for v in vols]
    nbytes = [0] * nstacks
    ref_blobs = ref_outs = None

    def encode(L):
        if nstacks == 1:
            n = c_long(0)
            rc = L.sqyx_encode_device_ex_UI16(pipe.encode(), c_void_p(vols[0].data_ptr()), shp, c_uint(3), c_void_p(bufs[0].data_ptr()),
                                              c_long(cap), ctypes.byref(n), c_void_p(0), st)
            nbytes[0] = n.value
        else:
            nb, rcs = (c_long * nstacks)(), (c_int * nstacks)()
            rc = L.sqyx_encode_batch_device_UI16(c_int(nstacks), pipe.encode(), ptrs(vols), shp, c_uint(3), ptrs(bufs),
                                                 (c_long * nstacks)(*[cap] * nstacks), nb, rcs)
            nbytes[:] = list(nb)
        assert rc == 0, rc

    def decode(L):
        if nstacks == 1:
            rc = L.sqyx_decode_device_UI16(c_void_p(bufs[0].data_ptr()), c_long(nbytes[0]), c_void_p(outs[0].data_ptr()),
                                           c_long(outs[0].numel() * 2), st)
        else:
            rcs = (c_int * nstacks)()
            rc = L.sqyx_decode_batch_device_UI16(c_int(nstacks), ptrs(bufs), (c_long * nstacks)(*nbytes), ptrs(outs),
                                                 (c_long * nstacks)(*[o.numel() * 2 for o in outs]), rcs)
        assert rc == 0, rc

    def timed(fn, L):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(calls):
            fn(L)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3 / calls

    enc_ms = {n: [] for n, _ in libs}
    dec_ms = {n: [] for n, _ in libs}
    for rnd in range(rounds + 1):          # round 0 warms up and checks the outputs
        for lname, L in libs:
            if rnd == 0:
                encode(L)
                decode(L)
                torch.cuda.synchronize()
                blobs = [b[:n].clone() for b, n in zip(bufs, nbytes)]
                if ref_blobs is None:
                    ref_blobs, ref_outs = blobs, [o.clone() for o in outs]
                else:
                    assert all(torch.equal(a, b) for a, b in zip(blobs, ref_blobs)), f"{wname}: {lname} wrote other blobs"
                    assert all(torch.equal(a, b) for a, b in zip(outs, ref_outs)), f"{wname}: {lname} decoded other voxels"
                del blobs
                continue
            enc_ms[lname].append(timed(encode, L))
            dec_ms[lname].append(timed(decode, L))
            print(f"{wname} round {rnd} {lname:24s} encode {enc_ms[lname][-1]:8.3f} ms  decode {dec_ms[lname][-1]:8.3f} ms", flush=True)
    raw = sum(v.numel() * 2 for v in vols)
    for lname, _ in libs:
        e, d = statistics.median(enc_ms[lname]), statistics.median(dec_ms[lname])
        print(f"{wname} median {lname:24s} encode {e:8.3f} ms [{min(enc_ms[lname]):.3f}..{max(enc_ms[lname]):.3f}]  decode {d:8.3f} ms "
              f"[{min(dec_ms[lname]):.3f}..{max(dec_ms[lname]):.3f}]  step {raw / (e + d) / 1e6:7.1f} GB/s  (identical outputs)", flush=True)
    del vols, bufs, outs, ref_blobs, ref_outs
    torch.cuda.empty_cache()
