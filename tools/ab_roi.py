"""A/B of the box calls (sqyx_decode_roi_device_UI16, sqyx_decode_roi_UI16) between library builds on the same GPU in the same
process (development tool): the one-plane and the 256^3 tile box of cfg2 (`rmestbkrd->bitswap1->lz4`) and cfg3 (`quantiser->lz4`)
on a seeded synthetic 512x2048x2048 uint16 stack, each encoded once by the first build. The builds take turns inside every
round: device calls timed with CUDA events, host calls (pageable buffers, nthreads = 8) with a wall clock, median over rounds.
One torch.profiler pass per build and box gives the gather kernel's time. Round 0 checks that every build writes the same
voxels and reports the same last_roi_info().
usage: ab_roi.py libA.so libB.so ...   (env AB_ROUNDS: rounds, default 7; AB_CALLS: calls per timing, default 5)"""
import ctypes
import os
import statistics
import subprocess
import sys
import time
from ctypes import c_int, c_long, c_uint, c_void_p

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import sqeazy_b200 as sq  # noqa: E402
from sqeazy_b200.synth import torch_volume  # noqa: E402

rounds = int(os.environ.get("AB_ROUNDS", "7"))
calls = int(os.environ.get("AB_CALLS", "5"))
libs = [(p, ctypes.CDLL(os.path.abspath(p))) for p in sys.argv[1:]]
SHAPE = (512, 2048, 2048)
Z, Y, X = SHAPE
CONFIGS = {"cfg2": "rmestbkrd->bitswap1->lz4", "cfg3": "quantiser->lz4"}
BOXES = {
    "one_plane": [(Z // 2, Z // 2 + 1), (0, Y), (0, X)],
    "box_256": [(Z // 2 - 128, Z // 2 + 128), (Y // 2 - 128, Y // 2 + 128), (X // 2 - 128, X // 2 + 128)],
}
try:
    card = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                          text=True, timeout=30).stdout.strip()
except Exception as exc:  # the card name still comes from torch
    card = f"{torch.cuda.get_device_name(0)}, power limit unknown ({exc!r})"
print(f"device: {card}", flush=True)


def box_arr(box):
    return (c_long * 6)(*[v for p in box for v in p])


def roi_device(L, blob, box, out):
    rc = L.sqyx_decode_roi_device_UI16(c_void_p(blob.data_ptr()), c_long(blob.numel()), box_arr(box), c_uint(3),
                                       c_void_p(out.data_ptr()), c_long(2 * out.numel()), c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, rc


def roi_host(L, h_blob, box, h_out):
    rc = L.sqyx_decode_roi_UI16(c_void_p(h_blob.ctypes.data), c_long(h_blob.size), box_arr(box), c_uint(3), c_void_p(h_out.ctypes.data),
                                c_long(h_out.nbytes), c_int(8))
    assert rc == 0, rc


def info(L):
    o = (c_long * 4)()
    assert L.sqyx_last_roi_info(o) == 0
    return list(o)


def device_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(calls):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / calls


def host_ms(fn):
    t0 = time.perf_counter()
    for _ in range(calls):
        fn()
    return (time.perf_counter() - t0) * 1e3 / calls


def gather_ms(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    return sum(e.self_device_time_total for e in prof.key_averages() if "roi_gather_kernel" in e.key) / 1e3 / calls


torch.cuda.set_device(0)
for _, L in libs:
    assert L.sqyx_set_device(c_int(0)) == 0
sq.set_device(0)
vol = torch_volume(SHAPE, "scmos", index=0)
for cfg, pipeline in CONFIGS.items():
    L0 = libs[0][1]
    blob = sq.encode_device(pipeline, vol).clone()
    h_blob = blob.cpu().numpy()
    for bname, box in BOXES.items():
        n = int(np.prod([hi - lo for lo, hi in box]))
        out = torch.empty(n, dtype=torch.int16, device="cuda")
        h_out = np.empty(n, dtype=np.uint16)
        ms = {name: {"device": [], "host": []} for name, _ in libs}
        ref = None
        for rnd in range(rounds + 1):
            for name, L in libs:
                if rnd == 0:   # warm up and check
                    out.zero_()
                    roi_device(L, blob, box, out)
                    torch.cuda.synchronize()
                    got = (out.cpu().numpy().copy(), info(L))
                    roi_host(L, h_blob, box, h_out)
                    got_h = (h_out.copy(), info(L))
                    if ref is None:
                        ref = (got, got_h)
                    else:
                        assert np.array_equal(got[0], ref[0][0]) and got[1] == ref[0][1], (cfg, bname, name, "device")
                        assert np.array_equal(got_h[0], ref[1][0]) and got_h[1] == ref[1][1], (cfg, bname, name, "host")
                    continue
                ms[name]["device"].append(device_ms(lambda: roi_device(L, blob, box, out)))
                ms[name]["host"].append(host_ms(lambda: roi_host(L, h_blob, box, h_out)))
        for name, L in libs:
            g = gather_ms(lambda: roi_device(L, blob, box, out))
            print(f"{cfg} {bname:10s} {os.path.basename(os.path.dirname(os.path.abspath(name))) + '/' + os.path.basename(name):36s} "
                  + "  ".join(f"{k} {statistics.median(v):8.3f} ms [{min(v):.3f}..{max(v):.3f}]" for k, v in ms[name].items())
                  + f"  gather {g:.4f} ms", flush=True)
    del blob
    torch.cuda.empty_cache()
print("identical voxels and last_roi_info() across builds", flush=True)
