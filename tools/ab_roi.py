"""A/B of the box and slice calls (sqyx_decode_roi_device_UI16 / sqyx_decode_roi_UI16, sqyx_decode_slice_*_UI16 for the strided
cases) between library builds on the same GPU in the same process (development tool): the boxes and slices of bench_roi.py on
cfg2 (`rmestbkrd->bitswap1->lz4`) and cfg3 (`quantiser->lz4`) on a seeded synthetic 512x2048x2048 uint16 stack, each encoded once
by the first build. A build that has the batch calls is also timed with each selection as a batch of one
(sqyx_decode_slice_batch_*_UI16, nsel = 1): the batch gather kernel against the single calls' by-value one. The variants take
turns inside every round: device calls timed with CUDA events, host calls (pageable buffers, nthreads = 8) with a wall clock,
median over rounds. One torch.profiler pass per variant and box gives the gather kernel's time. Round 0 checks that every
variant writes the same voxels and reports the same last_roi_info().
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
from bench_roi import BOXES  # noqa: E402
from sqeazy_b200.synth import torch_volume  # noqa: E402

rounds = int(os.environ.get("AB_ROUNDS", "7"))
calls = int(os.environ.get("AB_CALLS", "5"))
libs = [(p, ctypes.CDLL(os.path.abspath(p))) for p in sys.argv[1:]]
SHAPE = (512, 2048, 2048)
Z, Y, X = SHAPE
CONFIGS = {"cfg2": "rmestbkrd->bitswap1->lz4", "cfg3": "quantiser->lz4"}
try:
    card = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                          text=True, timeout=30).stdout.strip()
except Exception as exc:  # the card name still comes from torch
    card = f"{torch.cuda.get_device_name(0)}, power limit unknown ({exc!r})"
print(f"device: {card}", flush=True)


def box_arr(box):
    """(the C array, whether it holds triples: the slice calls)"""
    strided = any(len(t) == 3 for t in box)
    vals = [v for t in box for v in ((t if len(t) == 3 else (*t, 1)) if strided else t)]
    return (c_long * len(vals))(*vals), strided


def triples(box):
    return (c_long * (3 * len(box)))(*[v for t in box for v in (t if len(t) == 3 else (*t, 1))])


def roi_device(L, batch, blob, box, out):
    args = (c_void_p(out.data_ptr()), c_long(2 * out.numel()), c_void_p(torch.cuda.current_stream().cuda_stream))
    if batch:
        rc = L.sqyx_decode_slice_batch_device_UI16(c_void_p(blob.data_ptr()), c_long(blob.numel()), triples(box), c_uint(1), c_uint(3), *args)
    else:
        arr, strided = box_arr(box)
        fn = L.sqyx_decode_slice_device_UI16 if strided else L.sqyx_decode_roi_device_UI16
        rc = fn(c_void_p(blob.data_ptr()), c_long(blob.numel()), arr, c_uint(3), *args)
    assert rc == 0, rc


def roi_host(L, batch, h_blob, box, h_out):
    args = (c_void_p(h_out.ctypes.data), c_long(h_out.nbytes), c_int(8))
    if batch:
        rc = L.sqyx_decode_slice_batch_UI16(c_void_p(h_blob.ctypes.data), c_long(h_blob.size), triples(box), c_uint(1), c_uint(3), *args)
    else:
        arr, strided = box_arr(box)
        fn = L.sqyx_decode_slice_UI16 if strided else L.sqyx_decode_roi_UI16
        rc = fn(c_void_p(h_blob.ctypes.data), c_long(h_blob.size), arr, c_uint(3), *args)
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
    return sum(e.self_device_time_total for e in prof.key_averages() if "roi_gather" in e.key) / 1e3 / calls


torch.cuda.set_device(0)
for _, L in libs:
    assert L.sqyx_set_device(c_int(0)) == 0
# (label, library, as a batch of one)
variants = [(os.path.basename(os.path.dirname(os.path.abspath(p))) + "/" + os.path.basename(p) + kind, L, batch) for p, L in libs
            for kind, batch in (("", False), (" batch of 1", True)) if not batch or hasattr(L, "sqyx_decode_slice_batch_UI16")]
sq.set_device(0)
vol = torch_volume(SHAPE, "scmos", index=0)
for cfg, pipeline in CONFIGS.items():
    L0 = libs[0][1]
    blob = sq.encode_device(pipeline, vol).clone()
    h_blob = blob.cpu().numpy()
    for bname, box in BOXES.items():
        n = int(np.prod([len(range(*t)) for t in box]))
        out = torch.empty(n, dtype=torch.int16, device="cuda")
        h_out = np.empty(n, dtype=np.uint16)
        ms = {name: {"device": [], "host": []} for name, _, _ in variants}
        ref = None
        for rnd in range(rounds + 1):
            for name, L, batch in variants:
                if rnd == 0:   # warm up and check
                    out.zero_()
                    roi_device(L, batch, blob, box, out)
                    torch.cuda.synchronize()
                    got = (out.cpu().numpy().copy(), info(L))
                    roi_host(L, batch, h_blob, box, h_out)
                    got_h = (h_out.copy(), info(L))
                    if ref is None:
                        ref = (got, got_h)
                    else:
                        assert np.array_equal(got[0], ref[0][0]) and got[1] == ref[0][1], (cfg, bname, name, "device")
                        assert np.array_equal(got_h[0], ref[1][0]) and got_h[1] == ref[1][1], (cfg, bname, name, "host")
                    continue
                ms[name]["device"].append(device_ms(lambda: roi_device(L, batch, blob, box, out)))
                ms[name]["host"].append(host_ms(lambda: roi_host(L, batch, h_blob, box, h_out)))
        for name, L, batch in variants:
            g = gather_ms(lambda: roi_device(L, batch, blob, box, out))
            print(f"{cfg} {bname:18s} {name:48s} "
                  + "  ".join(f"{k} {statistics.median(v):8.3f} ms [{min(v):.3f}..{max(v):.3f}]" for k, v in ms[name].items())
                  + f"  gather {g:.4f} ms", flush=True)
    del blob
    torch.cuda.empty_cache()
print("identical voxels and last_roi_info() across variants", flush=True)
