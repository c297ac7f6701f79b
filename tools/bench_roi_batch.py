"""Batches of selections (sqyx_decode_slice_batch_*) against the same selections one call at a time and against the whole-stack
decode followed by indexing, in one process.

cfg2 (`rmestbkrd->bitswap1->lz4`) and cfg3 (`quantiser->lz4`) on the seeded synthetic 512x2048x2048 uint16 stack of
bench_roi.py, each encoded once. Cases: the 16 tiles of 512x512 of one z-plane (a viewer's page), 64 random 64^3 patches and
256 random 32^3 patches (a training loader's batch; seeded), and one 256^3 box (nsel = 1, against the single call). For each:
- device: the batch call, the K single calls, and sqyx_decode_device_UI16 followed by torch indexing — CUDA events, medians;
- host: the batch call, the K single calls, and SQY_Decode_UI16 followed by numpy indexing — wall clock around synchronous
  calls (pageable buffers, nthreads = 8), medians;
- LZ4 blocks decoded and host->device bytes of the batch and summed over the single calls;
- the gather kernel's device time of the batch call (torch.profiler, a pass of its own).
Every output is checked against the whole-stack decode. The card's name and power limit are read in the same run.

usage: python tools/bench_roi_batch.py [--reps 10] [--out result.json]
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import sqeazy_b200 as sq  # noqa: E402
from bench_roi import CONFIGS, SHAPE, card, device_ms, gather_ms, host_ms  # noqa: E402
from sqeazy_b200.synth import torch_volume  # noqa: E402

Z, Y, X = SHAPE


def patches(n, edge, seed):
    rng = np.random.default_rng(seed)
    return [[(int(o), int(o) + edge) for o in (rng.integers(0, s - edge + 1) for s in SHAPE)] for _ in range(n)]


CASES = {
    "tiles_16_of_one_plane": [[(Z // 2, Z // 2 + 1), (ty * 512, ty * 512 + 512), (tx * 512, tx * 512 + 512)]
                              for ty in range(Y // 512) for tx in range(X // 512)],
    "patches_64_of_64": patches(64, 64, 1),
    "patches_256_of_32": patches(256, 32, 2),
    "box_256": [[(Z // 2 - 128, Z // 2 + 128), (Y // 2 - 128, Y // 2 + 128), (X // 2 - 128, X // 2 + 128)]],
}


def sl(sel):
    return tuple(slice(lo, hi) for lo, hi in sel)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    sq.set_device(0)
    result = {"card": card(), "shape": SHAPE, "configs": {}}
    vol = torch_volume(SHAPE, "scmos", index=0)
    full = torch.empty(SHAPE, dtype=torch.int16, device="cuda")
    h_full = np.empty(SHAPE, dtype=np.uint16)
    for cfg, pipeline in CONFIGS.items():
        blob = sq.encode_device(pipeline, vol).clone()
        h_blob = blob.cpu().numpy()
        sq.decode_device(blob, full)
        r = {"pipeline": pipeline, "blob_bytes": int(blob.numel()), "cases": {}}
        for name, sels in CASES.items():
            sizes = [int(np.prod([hi - lo for lo, hi in s])) for s in sels]
            n = sum(sizes)
            want = torch.cat([full[sl(s)].reshape(-1) for s in sels])
            h_want = want.cpu().numpy().view(np.uint16)
            out = torch.empty(n, dtype=torch.int16, device="cuda")
            h_out = np.empty(n, dtype=np.uint16)
            offs = np.concatenate([[0], np.cumsum(sizes)]).tolist()
            d = {"nsel": len(sels), "voxels": n}

            def singles_device():
                for s, a, b in zip(sels, offs, offs[1:]):
                    sq.decode_roi_device(blob, s, out[a:b])

            def full_then_index_device():
                sq.decode_device(blob, full)
                for s, a, b in zip(sels, offs, offs[1:]):
                    out[a:b].copy_(full[sl(s)].reshape(-1))

            def singles_host():
                for s, a, b in zip(sels, offs, offs[1:]):
                    sq.decode_roi(h_blob, s, nthreads=8, out=h_out[a:b])

            def full_then_index_host():
                sq.decode(h_blob, nthreads=8, out=h_full.reshape(-1))
                for s, a, b in zip(sels, offs, offs[1:]):
                    h_out[a:b] = h_full[sl(s)].reshape(-1)

            out.zero_()
            d["batch_device_ms"] = device_ms(lambda: sq.decode_roi_batch_device(blob, sels, out), args.reps)
            info = sq.last_roi_info()
            d["route"], d["batch_blocks"] = info["route"], info["blocks"]
            assert torch.equal(out, want), (cfg, name, "batch device")
            d["batch_gather_ms"] = gather_ms(lambda: sq.decode_roi_batch_device(blob, sels, out))
            out.zero_()
            d["singles_device_ms"] = device_ms(singles_device, args.reps)
            assert torch.equal(out, want), (cfg, name, "singles device")
            blocks = 0
            for s, a, b in zip(sels, offs, offs[1:]):
                sq.decode_roi_device(blob, s, out[a:b])
                blocks += sq.last_roi_info()["blocks"]
            d["singles_blocks"] = blocks
            out.zero_()
            d["full_then_index_device_ms"] = device_ms(full_then_index_device, args.reps)
            assert torch.equal(out, want), (cfg, name, "full device")

            h_out[:] = 0
            d["batch_host_ms"] = host_ms(lambda: sq.decode_roi_batch(h_blob, sels, nthreads=8, out=h_out), max(3, args.reps // 2))
            d["batch_h2d_bytes"] = sq.last_roi_info()["h2d_bytes"]
            assert np.array_equal(h_out, h_want), (cfg, name, "batch host")
            h_out[:] = 0
            d["singles_host_ms"] = host_ms(singles_host, max(3, args.reps // 2))
            assert np.array_equal(h_out, h_want), (cfg, name, "singles host")
            h2d = 0
            for s, a, b in zip(sels, offs, offs[1:]):
                sq.decode_roi(h_blob, s, nthreads=8, out=h_out[a:b])
                h2d += sq.last_roi_info()["h2d_bytes"]
            d["singles_h2d_bytes"] = h2d
            h_out[:] = 0
            d["full_then_index_host_ms"] = host_ms(full_then_index_host, 3)
            assert np.array_equal(h_out, h_want), (cfg, name, "full host")
            r["cases"][name] = d
            print(cfg, name, json.dumps(d), flush=True)
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
