"""Sub-volume and strided-slice decode against the whole-stack decode of the same blob, in one process.

cfg2 (`rmestbkrd->bitswap1->lz4`) and cfg3 (`quantiser->lz4`) on a seeded synthetic 512x2048x2048 uint16 stack, each encoded once.
Device: sqyx_decode_roi_device_UI16 for one z-plane, 16 z-planes, a 64-row band through all planes and a 256^3 box in the middle,
and the full sqyx_decode_device_UI16 — CUDA events, after warm-up, median of --reps. Host: sqyx_decode_roi_UI16 for the same
boxes against SQY_Decode_UI16 (pageable buffers, wall clock), with the bytes each sends to the device. A torch.profiler pass
over the one-plane device call gives its per-kernel times. Slices (sqyx_decode_slice_*): an overview [::8, ::4, ::4], every
8th plane [::8, :, :] and every 4th column of one plane [Z/2, :, ::4], each with its call times, blocks decoded, bytes sent and
the gather kernel's time (torch.profiler). The card's name and power limit are read in the same run.

usage: python tools/bench_roi.py [--reps 20] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import sqeazy_b200 as sq  # noqa: E402
from sqeazy_b200.synth import torch_volume  # noqa: E402

SHAPE = (512, 2048, 2048)
CONFIGS = {"cfg2": "rmestbkrd->bitswap1->lz4", "cfg3": "quantiser->lz4"}
Z, Y, X = SHAPE
BOXES = {
    "one_plane": [(Z // 2, Z // 2 + 1), (0, Y), (0, X)],
    "16_planes": [(Z // 2, Z // 2 + 16), (0, Y), (0, X)],
    "64_row_band": [(0, Z), (Y // 2 - 32, Y // 2 + 32), (0, X)],
    "box_256": [(Z // 2 - 128, Z // 2 + 128), (Y // 2 - 128, Y // 2 + 128), (X // 2 - 128, X // 2 + 128)],
    "overview": [(0, Z, 8), (0, Y, 4), (0, X, 4)],
    "z_step_8": [(0, Z, 8), (0, Y), (0, X)],
    "x_step_4_one_plane": [(Z // 2, Z // 2 + 1), (0, Y), (0, X, 4)],
}


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    parts = [p.strip() for p in q.stdout.strip().split(",")] if q.returncode == 0 else []
    return {"name": parts[0] if parts else torch.cuda.get_device_name(0), "power_limit": parts[1] if len(parts) > 1 else None,
            "max_sm_clock": parts[2] if len(parts) > 2 else None}


def device_ms(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times))


def host_ms(fn, reps):
    for _ in range(2):
        fn()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        times.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(times))


def kernel_breakdown(fn):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if e.device_type.name == "CUDA" and e.count:
            name = e.key.split("(")[0].split("<")[0].split("::")[-1][:60]
            out[name] = round(out.get(name, 0.0) + e.self_device_time_total / 1e3, 4)
    return out


def gather_ms(fn, reps=5):
    """the gather kernel's device time per call (roi_gather_kernel, or roi_gather_batch_kernel for the batch calls)"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    return sum(e.self_device_time_total for e in prof.key_averages() if "roi_gather" in e.key) / 1e3 / reps


def sel_of(box):
    return tuple(slice(*t) for t in box)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    sq.set_device(0)
    result = {"card": card(), "shape": SHAPE, "configs": {}}
    vol = torch_volume(SHAPE, "scmos", index=0)
    full = torch.empty(SHAPE, dtype=torch.int16, device="cuda")
    for cfg, pipeline in CONFIGS.items():
        blob = sq.encode_device(pipeline, vol).clone()
        h_blob = blob.cpu().numpy()
        r = {"pipeline": pipeline, "blob_bytes": int(blob.numel())}
        r["full_device_ms"] = device_ms(lambda: sq.decode_device(blob, full), args.reps)
        h_full = np.empty(vol.numel(), dtype=np.uint16)
        r["full_host_ms"] = host_ms(lambda: sq.decode(h_blob, nthreads=8, out=h_full), max(3, args.reps // 4))
        r["boxes"] = {}
        for name, box in BOXES.items():
            n = int(np.prod([len(range(*t)) for t in box]))
            out = torch.empty(n, dtype=torch.int16, device="cuda")
            d = {"voxels": n}
            d["device_ms"] = device_ms(lambda: sq.decode_roi_device(blob, box, out), args.reps)
            d["device_route"], d["device_blocks"] = sq.last_roi_info()["route"], sq.last_roi_info()["blocks"]
            d["device_share_of_full"] = d["device_ms"] / r["full_device_ms"]
            want = full.view(SHAPE)[sel_of(box)].reshape(-1)
            assert torch.equal(out, want), (cfg, name, "device")
            h_out = np.empty(n, dtype=np.uint16)
            d["host_ms"] = host_ms(lambda: sq.decode_roi(h_blob, box, nthreads=8, out=h_out), max(3, args.reps // 4))
            info = sq.last_roi_info()
            d["host_route"], d["host_h2d_bytes"], d["blocks"] = info["route"], info["h2d_bytes"], info["blocks"]
            d["host_h2d_share_of_blob"] = info["h2d_bytes"] / r["blob_bytes"]
            assert np.array_equal(h_out, want.cpu().numpy().view(np.uint16)), (cfg, name, "host")
            d["gather_ms"] = gather_ms(lambda: sq.decode_roi_device(blob, box, out))
            r["boxes"][name] = d
        one = BOXES["one_plane"]
        out = torch.empty(Y * X, dtype=torch.int16, device="cuda")
        r["one_plane_device_kernels_ms"] = kernel_breakdown(lambda: sq.decode_roi_device(blob, one, out))
        r["full_device_kernels_ms"] = kernel_breakdown(lambda: sq.decode_device(blob, full))
        result["configs"][cfg] = r
        del blob
        torch.cuda.empty_cache()
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
