#!/usr/bin/env python
"""bench.py — uint16 voxel GB/s of the sqeazy volume pipeline (encode + decode) on B200.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload cfg2|cfg1|cfg3|cfg4|cfg5] [--no-per-config]
                    [--dump-outputs DIR]

A *step* = one encode + one decode of one volume through the pipeline (cfg4: one decode of a batch of reference blobs).
  value    raw volume bytes / (t_encode + t_decode), inputs resident in HBM (sqyx_* device API), summed over ranks
  e2e      the same metric through the reference-facing C API with HOST buffers (SQY_PipelineEncode_UI16 +
           SQY_Decode_UI16, pinned host memory, H2D/D2H inside the timed region); `copy_ceiling` beside it = the same
           bytes moved by bare cudaMemcpyAsync calls on all ranks at once (what the box's PCIe / host memory allows)
  roofline dominant kernel (the LZ4 block encoder): (input bytes + compressed bytes) / its CUDA-event time vs measured HBM peak
  cpu_baseline  the reference's own stage code (oracle/_ref) on this box's host cores on a bounded slab of the same workload
  per_config    the other BASELINE.json configurations (cfg1, cfg3, cfg4, cfg5), a few steps each, same measurements
  e2e_sharded   (N > 1) ONE stack through the same two C calls, sharded over all N GPUs inside libsqeazy.so (rank 0 calls,
                the other ranks' processes wait): strong scaling of the host-buffer path; cfg3 runs its histogram
                all-reduce through NCCL inside the library
N > 1 (torchrun): every rank encodes/decodes its own stack (stacks partitioned over GPUs; weak scaling; no data-path
collective — cfg3's quantiser adds the NCCL histogram all-reduce); time = max over ranks.
`--impl reference` times the reference's CPU implementation (rank 0 only) on bounded slabs of the same workload.
`--dump-outputs DIR` writes what rank 0's timed steps returned in the last step (blobs and decoded stacks of the main
workload) to DIR as .npy files; inputs are seeded, so two builds of the library can be compared output for output. cfg4
times two framings one after the other and dumps the decoded stacks of the last (block-linked) one; without oracle/_ref
it has no reference-made blobs, is skipped and writes nothing (said on stderr).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (shape {Z,Y,X}, pipeline, preset, reference stage-chain id)
    "cfg1": ((256, 512, 512), "bitswap1->lz4", "scmos", 0),
    "cfg2": ((512, 2048, 2048), "rmestbkrd->bitswap1->lz4", "scmos", 1),
    "cfg3": ((1024, 2048, 2048), "quantiser->lz4", "scmos", 2),
    "cfg4": ((256, 2048, 2048), "bitswap1->lz4", "scmos", 0),      # decode-only of reference-made blobs, 8 per GPU
    "cfg5": ((128, 1024, 1024), "remove_background(threshold=110)->bitswap4->lz4", "scmos", 3),   # time-lapse, 32 stacks per GPU
}
CFG4_PER_GPU = 8       # BASELINE cfg4: 64 blobs over 8 GPUs
CFG5_PER_GPU = 32      # BASELINE cfg5: 1000 stacks, stack v -> GPU v mod G; a bounded sample per GPU
METRIC = "uint16 voxel GB/s encode+decode"
DUMP_SAMPLES = 1 << 23   # float32 values over all arrays of one --dump-outputs (32 MiB)
DUMP_CHUNK = 1 << 22     # elements per chunk sum


def dump_outputs(dirname, arrays):
    """Writes each tensor of `arrays` (name -> tensor of uint8 or 16-bit voxels) as DIR/<name>.npy: its elements
    read as unsigned integers in float32 (exact), all of them or, when the array exceeds its share of DUMP_SAMPLES, a
    sorted sample at positions drawn from a generator seeded by the name. DIR/<name>_chunk_sums.npy (float64, exact)
    holds the sums over consecutive DUMP_CHUNK elements, so that every element counts in the comparison."""
    import numpy as np
    import torch

    os.makedirs(dirname, exist_ok=True)
    per_array = DUMP_SAMPLES // len(arrays)
    for name, t in arrays.items():
        flat = t.reshape(-1)
        n = flat.numel()
        mask = (1 << (8 * flat.element_size())) - 1
        sums = [int((flat[s:s + DUMP_CHUNK].to(torch.int64) & mask).sum().item()) for s in range(0, n, DUMP_CHUNK)]
        np.save(os.path.join(dirname, name + "_chunk_sums.npy"), np.array(sums, dtype=np.float64))
        if n > per_array:
            idx = np.sort(np.random.default_rng(zlib.crc32(name.encode())).integers(0, n, size=per_array))
            flat = flat[torch.from_numpy(idx).to(flat.device)]
        np.save(os.path.join(dirname, name + ".npy"), ((flat.to(torch.int64) & mask).cpu().numpy()).astype(np.float32))


def measured_peak_hbm():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc = None
        self.gpu_index = gpu_index
        self.path = os.path.join(tempfile.gettempdir(), f"sqy_clocks_{os.getpid()}.csv")

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, reasons, mx = [], set(), None
        try:
            for line in open(self.path):
                p = [x.strip() for x in line.split(",")]
                if len(p) < 9:
                    continue
                try:
                    sm.append(float(p[1]))
                    mx = float(p[2])
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.remove(self.path)
        except Exception:
            pass
        if not sm:
            # timed region shorter than one sampling period: one immediate reading (GPU still warm), flagged as such
            try:
                line = subprocess.check_output(["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={self.QUERY}",
                                                "--format=csv,noheader,nounits"], timeout=10).decode().strip()
                p = [x.strip() for x in line.split(",")]
                sm.append(float(p[1]))
                mx = float(p[2])
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
                out["note"] = "timed region < sampling period: sampled right after it"
            except Exception:
                pass
        if sm:
            sm.sort()
            # median of the upper half = clocks under load (idle samples between steps drag a plain median down)
            hi = sm[len(sm) // 2:]
            out["sm_mhz"] = hi[len(hi) // 2]
        out["sm_max_mhz"] = mx
        out["reasons"] = sorted(reasons)
        return out


def reference_arm(shape, pipeline, preset, chain_id, steps, warmup, as_baseline=False, decode_only=False):
    """times the reference's CPU implementation (oracle/_ref: the reference's stage headers compiled in the build
    container) on a bounded z-slab of the workload, all host threads"""
    import numpy as np

    from oracle import oracle as orc
    from sqeazy_b200.synth import numpy_volume

    ref = orc.ref()
    cores = os.cpu_count() or 1
    Z, Y, X = shape
    # bounded sample: a z-slab of ~128 MiB (< 2^31 voxels, which the reference cannot index anyway: SURVEY F7)
    slab_z = max(4, min(Z, (128 << 20) // (Y * X * 2)))
    sample_shape = (slab_z, Y, X)
    vol = numpy_volume(sample_shape, preset, index=0)
    if not ref.available:
        # the C port of the oracle stands in (scalar, 1 core)
        port = orc.port()
        cores = 1
        kind = "port"

        def run():
            t0 = time.perf_counter()
            cur = vol
            if chain_id == 1:
                cur, _ = port.rmestbkrd(cur, 2 << 20)
            if chain_id == 3:
                cur = port.remove_background(cur, 110)
            if chain_id == 2:
                enc, dec = port.quantiser_luts(port.histogram(cur))
                data = port.lut_apply(cur, enc)
            else:
                data = port.bitswap_encode(4 if chain_id == 3 else 1, cur)
            payload = port.lz4_frames_encode(data)
            t1 = time.perf_counter()
            raw = port.lz4_frames_decode(payload, data.nbytes)
            if chain_id == 2:
                port.lut_decode(raw, dec)
            else:
                port.bitswap_decode(4 if chain_id == 3 else 1, raw.view(np.uint16))
            t2 = time.perf_counter()
            return t1 - t0, t2 - t1, payload.size
    else:
        kind = "reference"
        w = 4 if chain_id == 3 else 1

        def run():
            payload, t_enc = ref.pipeline_encode_stages(chain_id, vol, cores, w=w, threshold=110)
            if chain_id == 2:
                t0 = time.perf_counter()
                rc, codes = ref.lz4_decode_bytes(payload, vol.size)
                t_dec = time.perf_counter() - t0  # LUT decode (tiny) not timed: the reference's signed index is UB (F11)
            else:
                rc, _, t_dec = ref.pipeline_decode_stages(w, payload, vol.size)
            assert rc == 0
            return t_enc, t_dec, payload.size

    n_warm = min(warmup, 1) if as_baseline else warmup
    n_steps = min(steps, 2) if as_baseline else steps
    for _ in range(n_warm):
        run()
    t_enc = t_dec = 0.0
    payload = 0
    for _ in range(n_steps):
        e, d, payload = run()
        t_enc += e
        t_dec += d
    raw = vol.nbytes
    t_used = t_dec if decode_only else t_enc + t_dec
    value = raw * n_steps / t_used / 1e9
    info = {"value": value, "unit": "GB/s", "cores": cores, "kind": kind,
            "sample": f"z-slab {sample_shape} of {shape}, {n_steps} steps, encode {raw * n_steps / t_enc / 1e9:.3f} GB/s, "
                      f"decode {raw * n_steps / t_dec / 1e9:.3f} GB/s, ratio {raw / payload:.3f}"
                      + (" (decode only counted)" if decode_only else ""),
            "ratio": raw / payload, "sample_shape": list(sample_shape)}
    return info, t_used / n_steps * 1e3


class Ctx:
    """what every measurement needs: rank layout, device, barriers, max over ranks"""

    def __init__(self, torch, sq, dist, cpu_group, rank, local_rank, world):
        self.torch, self.sq, self.dist, self.cpu_group = torch, sq, dist, cpu_group
        self.rank, self.local_rank, self.world = rank, local_rank, world
        self.dev = torch.device("cuda", local_rank)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def host_barrier(self):
        """rendezvous that leaves the GPUs idle (gloo): used around the sharded call of rank 0"""
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier(group=self.cpu_group)

    def max_over_ranks(self, x):
        if self.dist is None:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x):
        if self.dist is None:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def free(self):
        import gc
        gc.collect()
        self.torch.cuda.empty_cache()
        try:
            self.sq.release_scratch()
        except Exception:
            pass


def copy_ceiling(ctx, h_in, h_out, d_buf, reps=2):
    """the same host<->device bytes as one e2e step, moved by bare cudaMemcpyAsync from/to the same pinned buffers on every
    rank at once: what PCIe and the host memory system allow at this number of GPUs (compressed bytes ignored)"""
    torch = ctx.torch
    n = h_in.numel() * h_in.element_size()
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        d_buf.copy_(h_in, non_blocking=True)
        torch.cuda.synchronize()
    t1 = time.perf_counter()
    for _ in range(reps):
        h_out.copy_(d_buf, non_blocking=True)
        torch.cuda.synchronize()
    t2 = time.perf_counter()
    th = ctx.max_over_ranks(t1 - t0) / reps
    td = ctx.max_over_ranks(t2 - t1) / reps
    return {"value": ctx.world * n / (th + td) / 1e9, "unit": "GB/s", "h2d_gbs": ctx.world * n / th / 1e9, "d2h_gbs": ctx.world * n / td / 1e9,
            "what": "raw stack H2D then D2H by cudaMemcpyAsync from the same pinned buffers, all ranks at once"}


def run_pipeline_workload(ctx, wname, steps, warmup, want_e2e=True, detail=True, sampler_cls=None, dump_dir=None):
    """cfg1 / cfg2 / cfg3: one stack per rank through the whole pipeline, device-resident and through the host API"""
    import numpy as np

    torch, sq, dist = ctx.torch, ctx.sq, ctx.dist
    from sqeazy_b200.synth import torch_volume

    shape, pipeline, preset, chain_id = WORKLOADS[wname]
    dev = ctx.dev
    vol = torch_volume(shape, preset, index=ctx.rank, device=dev)
    raw_bytes = vol.numel() * 2
    cap = sq.max_compressed_length(pipeline, raw_bytes)
    blob_buf = torch.empty(cap, dtype=torch.uint8, device=dev)
    out = torch.empty_like(vol)
    use_hist_allreduce = ctx.world > 1 and "quantiser" in pipeline
    hist = torch.zeros(65536, dtype=torch.int32, device=dev) if use_hist_allreduce else None

    def encode_step():
        if use_hist_allreduce:
            hist.zero_()
            sq.histogram_device(vol, hist)
            dist.all_reduce(hist)  # the path's only collective: NCCL sum of the 65536-bin histogram
            return sq.encode_device(pipeline, vol, out=blob_buf, global_hist=hist)
        return sq.encode_device(pipeline, vol, out=blob_buf)

    # ---- warm-up (also sizes the library's scratch arena) ----
    blob = None
    for _ in range(warmup):
        blob = encode_step()
        sq.decode_device(blob, out)
    torch.cuda.synchronize()
    if pipeline == "bitswap1->lz4":
        assert torch.equal(out, vol), "lossless pipeline did not return the input"
    blob_bytes = int(blob.numel())

    # ---- timed region: device-resident ----
    sampler = sampler_cls(ctx.local_rank) if sampler_cls else None
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    launches0 = sq.kernel_launches()
    ctx.barrier()
    if sampler:
        sampler.start()
    t_enc_ms = t_dec_ms = 0.0
    for _ in range(steps):
        ev[0].record()
        blob = encode_step()
        ev[1].record()
        sq.decode_device(blob, out)
        ev[2].record()
        ev[2].synchronize()
        t_enc_ms += ev[0].elapsed_time(ev[1])
        t_dec_ms += ev[1].elapsed_time(ev[2])
    ctx.barrier()
    clocks = sampler.stop() if sampler else None
    launches = sq.kernel_launches() - launches0
    stats = sq.last_lz4_stats()
    if dump_dir and ctx.rank == 0:
        dump_outputs(dump_dir, {"blob": blob, "decoded": out})
    t_enc_ms = ctx.max_over_ranks(t_enc_ms)
    t_dec_ms = ctx.max_over_ranks(t_dec_ms)
    total_s = (t_enc_ms + t_dec_ms) / 1e3
    res = {"workload": wname, "pipeline": pipeline, "shape_zyx": list(shape),
           "value": ctx.world * raw_bytes * steps / total_s / 1e9, "ms_per_step": (t_enc_ms + t_dec_ms) / steps,
           "encode_gbs": ctx.world * raw_bytes * steps / (t_enc_ms / 1e3) / 1e9,
           "decode_gbs": ctx.world * raw_bytes * steps / (t_dec_ms / 1e3) / 1e9,
           "compression_ratio": raw_bytes / blob_bytes, "blob_bytes": blob_bytes, "gpu_launches": int(launches), "clocks": clocks,
           "collective": "NCCL all-reduce of the 65536-bin histogram per step" if use_hist_allreduce else None}

    # ---- per-stage device times (separate pass: the timers add event syncs) ----
    sq.enable_stage_timing(True)
    sq.stage_ms(reset=True)
    n_prof = 2
    for _ in range(n_prof):
        blob = encode_step()
        sq.decode_device(blob, out)
    torch.cuda.synchronize()
    stage = {k: v / n_prof for k, v in sq.stage_ms(reset=True).items()}
    sq.enable_stage_timing(False)
    lz4_in_bytes = raw_bytes // 2 if "quantiser" in pipeline else raw_bytes
    payload_bytes = stats["payload_bytes"]
    peak, peak_kind = measured_peak_hbm()
    achieved = (lz4_in_bytes + payload_bytes) / (stage["lz4_encode"] / 1e3) / 1e9 if stage["lz4_encode"] > 0 else 0.0
    traffic = None
    try:  # dram__bytes_read.sum + dram__bytes_write.sum of lz4_encode_kernel from the committed `ncu --set full` capture
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic = json.load(f).get(wname, {}).get("lz4_encode_kernel_dram_bytes_per_launch")
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": "lz4_encode_kernel", "achieved": achieved, "peak": peak, "peak_source": peak_kind + " copy bandwidth",
                "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "algorithmic_bytes_per_launch": lz4_in_bytes + payload_bytes, "kernel_ms": stage["lz4_encode"],
                # whole device-resident encode call against the fused-ideal byte count of SURVEY 8d (2N + C; quantiser: 4N + C)
                "encode_call_frac": ((2 * raw_bytes if "quantiser" in pipeline else raw_bytes) + payload_bytes) / (t_enc_ms / steps / 1e3) / 1e9 / peak,
                "stage_ms": stage,
                "stage_gbs": {"filter_bitswap_encode(4B/voxel)": (2 * raw_bytes / (stage["filter_bitswap_encode"] / 1e3) / 1e9) if stage["filter_bitswap_encode"] else None,
                              "bitswap_decode(4B/voxel)": (2 * raw_bytes / (stage["bitswap_decode"] / 1e3) / 1e9) if stage["bitswap_decode"] else None,
                              "lz4_decode(C+B)": ((lz4_in_bytes + payload_bytes) / (stage["lz4_decode"] / 1e3) / 1e9) if stage["lz4_decode"] else None},
                "lz4_blocks": stats}
    if detail:
        # SURVEY §8d: split of the dominant kernel into its closed-form path (all-equal blocks: load, compare, 75 bytes out) and
        # the general path. The closed-form rate is measured on an all-zero buffer of the same size; the general rate follows
        # from the block counts: t_general = t_kernel - constant_bytes / constant_rate.
        try:
            zeros = torch.zeros(lz4_in_bytes, dtype=torch.uint8, device=dev)
            zbuf = torch.empty(sq.lz4_bound(lz4_in_bytes), dtype=torch.uint8, device=dev)
            sq.lz4_encode_device(zeros, out=zbuf)
            zev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            zev[0].record()
            for _ in range(3):
                sq.lz4_encode_device(zeros, out=zbuf)
            zev[1].record()
            zev[1].synchronize()
            const_gbs = lz4_in_bytes / (zev[0].elapsed_time(zev[1]) / 3 / 1e3) / 1e9
            nb = stats["general_blocks"] + stats["constant_blocks"] + stats["stored_blocks"]
            const_bytes = lz4_in_bytes * stats["constant_blocks"] / max(nb, 1)
            t_const = const_bytes / (const_gbs * 1e9)
            t_general = max(stage["lz4_encode"] / 1e3 - t_const, 1e-9)
            roofline["path_split"] = {"constant_blocks_share": stats["constant_blocks"] / max(nb, 1), "constant_path_gbs": const_gbs,
                                      "constant_path_frac_of_peak": const_gbs / peak,
                                      "general_path_gbs": (lz4_in_bytes - const_bytes) / t_general / 1e9,
                                      "general_path_frac_of_peak": (lz4_in_bytes - const_bytes) / t_general / 1e9 / peak}
            del zeros, zbuf
        except Exception as exc:
            roofline["path_split"] = {"error": repr(exc)}
    res["roofline"] = roofline

    # ---- e2e: host buffers through SQY_PipelineEncode_UI16 / SQY_Decode_UI16 ----
    e2e = None
    if want_e2e:
        try:
            h_vol = torch.empty(vol.shape, dtype=torch.int16).pin_memory()
            h_vol.copy_(vol)
            h_blob = torch.empty(cap, dtype=torch.uint8).pin_memory()
            h_out = torch.empty(vol.shape, dtype=torch.int16).pin_memory()
            np_vol = h_vol.numpy().view(np.uint16)
            np_blob = h_blob.numpy()
            np_out = h_out.numpy().view(np.uint16).reshape(-1)
            e_steps = max(1, min(steps, 3))
            sq.set_device(ctx.local_rank)
            b = sq.encode(pipeline, np_vol, out=np_blob)  # warm-up (grows the staging arena)
            sq.decode(b, out=np_out)
            ctx.barrier()
            t0 = time.perf_counter()
            for _ in range(e_steps):
                b = sq.encode(pipeline, np_vol, out=np_blob)
                sq.decode(b, out=np_out)
            torch.cuda.synchronize()
            t_e2e = ctx.max_over_ranks(time.perf_counter() - t0)
            # the host-pointer path must deliver the same voxels as the device-resident path (64-bit checksums)
            host_sum = int(sum(int(np_out[i: i + (1 << 27)].astype(np.uint64).sum()) for i in range(0, np_out.size, 1 << 27)))
            flat = out.view(-1)
            dev_sum = sum(int((flat[i: i + (1 << 28)].to(torch.int64) & 0xFFFF).sum().item()) for i in range(0, flat.numel(), 1 << 28))
            e2e = {"value": ctx.world * raw_bytes * e_steps / t_e2e / 1e9, "unit": "GB/s", "steps": e_steps,
                   "h2d_bytes_per_step": raw_bytes + int(b.size), "d2h_bytes_per_step": int(b.size) + raw_bytes,
                   "api": "SQY_PipelineEncode_UI16 + SQY_Decode_UI16, pinned host buffers, one stack per rank",
                   "same_voxels_as_device_path": host_sum == dev_sum}
            if detail:
                ceil = copy_ceiling(ctx, h_vol, h_out, out)
                e2e["copy_ceiling"] = ceil
                e2e["frac_of_copy_ceiling"] = e2e["value"] / ceil["value"]
                e2e["limiter"] = ("host<->device copies: %.0f %% of what bare cudaMemcpyAsync calls reach on this box at %d GPU(s)"
                                  % (100 * e2e["value"] / ceil["value"], ctx.world))
            del h_vol, h_blob, h_out
        except Exception as exc:  # pinned allocation can fail on small hosts; report instead of dying
            e2e = {"value": None, "unit": "GB/s", "error": repr(exc), "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    res["e2e"] = e2e
    del vol, blob_buf, out, blob
    ctx.free()
    return res


def run_cfg5(ctx, steps, warmup, dump_dir=None):
    """time-lapse: stack v -> rank v mod G; the stacks of a rank as one batch (sqyx_*_batch_device_UI16)"""
    torch, sq = ctx.torch, ctx.sq
    from sqeazy_b200.synth import torch_volume

    shape, pipeline, preset, _ = WORKLOADS["cfg5"]
    n = CFG5_PER_GPU
    vols = [torch_volume(shape, preset, index=ctx.rank + ctx.world * i, device=ctx.dev) for i in range(n)]
    raw = vols[0].numel() * 2
    cap = sq.max_compressed_length(pipeline, raw)
    bufs = [torch.empty(cap, dtype=torch.uint8, device=ctx.dev) for _ in range(n)]
    outs = [torch.empty_like(v) for v in vols]
    blobs = None
    for _ in range(warmup):
        blobs = sq.encode_batch_device(pipeline, vols, outs=bufs)
        sq.decode_batch_device(blobs, outs)
    torch.cuda.synchronize()
    want = torch.clamp(vols[1].to(torch.int32) & 0xFFFF, min=110) - 110
    ok = bool(torch.equal(outs[1].to(torch.int32) & 0xFFFF, want))
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    launches0 = sq.kernel_launches()
    ctx.barrier()
    te = td = 0.0
    for _ in range(steps):
        ev[0].record()
        blobs = sq.encode_batch_device(pipeline, vols, outs=bufs)
        ev[1].record()
        sq.decode_batch_device(blobs, outs)
        ev[2].record()
        ev[2].synchronize()
        te += ev[0].elapsed_time(ev[1])
        td += ev[1].elapsed_time(ev[2])
    ctx.barrier()
    launches = sq.kernel_launches() - launches0
    if dump_dir and ctx.rank == 0:
        dump_outputs(dump_dir, {**{f"blob_{i}": b for i, b in enumerate(blobs)}, **{f"decoded_{i}": o for i, o in enumerate(outs)}})
    te, td = ctx.max_over_ranks(te), ctx.max_over_ranks(td)
    tot = ctx.world * n * raw * steps
    res = {"workload": "cfg5", "pipeline": pipeline, "shape_zyx": list(shape), "stacks_per_gpu": n,
           "what": f"{n} stacks per GPU of the 1000-stack time-lapse (stack v -> GPU v mod G), batched encode + batched decode",
           "value": tot / ((te + td) / 1e3) / 1e9, "encode_gbs": tot / (te / 1e3) / 1e9, "decode_gbs": tot / (td / 1e3) / 1e9,
           "ms_per_step": (te + td) / steps, "compression_ratio": n * raw / sum(int(b.numel()) for b in blobs),
           "bit_exact_vs_torch_arithmetic": ok, "gpu_launches": int(launches)}
    del vols, bufs, outs, blobs
    ctx.free()
    return res


def run_cfg4(ctx, steps, warmup, dump_dir=None):
    """decode-only of REFERENCE-made bitswap1->lz4 blobs: CFG4_PER_GPU stacks per GPU (64 over 8 GPUs), both framings the
    reference produces — one frame per 256 KiB chunk (its multi-threaded mode) and one block-linked frame (its one-thread
    mode, the sqy CLI default). The blobs are made by oracle/_ref (the reference's own stage code + liblz4) before the
    timed region; without it the workload is skipped."""
    import numpy as np

    torch, sq = ctx.torch, ctx.sq
    from oracle import oracle as orc
    from sqeazy_b200.synth import torch_volume

    ref = orc.ref()
    if not ref.available:
        if dump_dir:
            print("bench.py: cfg4 skipped without oracle/_ref: nothing dumped to " + dump_dir, file=sys.stderr)
        return {"workload": "cfg4", "skipped": "oracle/_ref (the compiled reference) is not present: no reference-made blobs"}
    shape, pipeline, preset, _ = WORKLOADS["cfg4"]
    name = "bitswap1(num_bits_per_plane=1)->lz4(accel=1,blocksize_kb=256,framestep_kb=256,n_chunks_of_input=0)"
    cores = os.cpu_count() or 1
    B = CFG4_PER_GPU
    res = {"workload": "cfg4", "pipeline": pipeline, "shape_zyx": list(shape), "blobs_per_gpu": B,
           "what": f"decode-only, {B} reference-made blobs per GPU (2 distinct stacks, repeated), sqyx_decode_batch_device_UI16"}
    vols, planes = [], []
    for i in range(2):
        v = torch_volume(shape, preset, index=100 + ctx.rank * 2 + i, device=ctx.dev)
        vols.append(v)
        if ctx.world == 1:
            planes.append(ref.bitswap_encode(1, v.cpu().numpy().view(np.uint16), nthreads=cores))
        else:
            # N ranks share the host cores: the bit planes come from the GPU transpose (bit-exact with the reference's,
            # tests/test_gpu_parity.py); the LZ4 frames below are the reference's own (lz4_scheme code + liblz4)
            t = torch.empty_like(v)
            sq.bitswap_encode_device(1, v.view(-1), t.view(-1))
            planes.append(t.cpu().numpy().view(np.uint16).reshape(-1))
            del t
    outs = [torch.empty(shape, dtype=torch.int16, device=ctx.dev) for _ in range(B)]
    raw = vols[0].numel() * 2
    total_launches = 0
    for framing, nthreads in (("frame_per_chunk", cores), ("linked_single_frame", 1)):
        blobs = []
        for i in range(2):
            payload = ref.lz4_encode(planes[i], nthreads=nthreads)
            h = orc.pack_header(shape, name, payload.size, version="0.5.2", headref="4c45a9b")
            blobs.append(torch.from_numpy(np.concatenate([np.frombuffer(h.encode(), dtype=np.uint8), payload])).to(ctx.dev))
        batch = [blobs[i % 2] if i < 2 else blobs[i % 2].clone() for i in range(B)]
        for _ in range(max(1, min(warmup, 2))):
            sq.decode_batch_device(batch, outs)
        torch.cuda.synchronize()
        ok = all(bool(torch.equal(outs[i], vols[i % 2])) for i in (0, 1, B - 1))
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        launches0 = sq.kernel_launches()
        ctx.barrier()
        ev[0].record()
        for _ in range(steps):
            sq.decode_batch_device(batch, outs)
        ev[1].record()
        ev[1].synchronize()
        ctx.barrier()
        total_launches += sq.kernel_launches() - launches0
        ms = ctx.max_over_ranks(ev[0].elapsed_time(ev[1]))
        res[framing] = {"decode_gbs": ctx.world * B * raw * steps / (ms / 1e3) / 1e9, "ms_per_batch": ms / steps,
                        "blob_ratio": raw / int(blobs[0].numel()), "bit_exact": ok}
        del blobs, batch
    if dump_dir and ctx.rank == 0:
        dump_outputs(dump_dir, {f"decoded_{i}": o for i, o in enumerate(outs)})
    res["value"] = res["frame_per_chunk"]["decode_gbs"]
    res["gpu_launches"] = int(total_launches)
    del vols, planes, outs
    ctx.free()
    return res


def run_sharded(ctx, wname, steps):
    """ONE stack through SQY_PipelineEncode_UI16 + SQY_Decode_UI16 from pinned host buffers, sharded over all GPUs inside
    libsqeazy.so (csrc/sharded.inl). Rank 0 calls; the other ranks wait on a host-side barrier (their GPUs are idle)."""
    import numpy as np

    torch, sq = ctx.torch, ctx.sq
    from sqeazy_b200.synth import torch_volume

    shape, pipeline, preset, _ = WORKLOADS[wname]
    res = None
    ctx.host_barrier()
    if ctx.rank == 0:
        try:
            h_vol = torch.empty(shape, dtype=torch.int16).pin_memory()
            h_out = torch.empty(shape, dtype=torch.int16).pin_memory()
            zs = max(1, (1 << 28) // (shape[1] * shape[2]))
            for z in range(0, shape[0], zs):     # generated slab-wise: the 8 GiB stack needs no second device copy
                part = torch_volume((min(zs, shape[0] - z), shape[1], shape[2]), preset, index=1000 + z, device=ctx.dev)
                h_vol[z:z + part.shape[0]].copy_(part)
                del part
            torch.cuda.empty_cache()
            vol = h_vol.numpy().view(np.uint16)
            out = h_out.numpy().view(np.uint16).reshape(-1)
            cap = sq.max_compressed_length(pipeline, vol.nbytes)
            h_blob = torch.empty(cap, dtype=torch.uint8).pin_memory()
            blob_buf = h_blob.numpy()
            rows = {}
            for devs in ([ctx.local_rank], list(range(ctx.world))):
                if len(devs) > 1:
                    sq.set_devices(devs)
                else:
                    sq.set_device(devs[0])
                b = sq.encode(pipeline, vol, nthreads=16, out=blob_buf)     # warm-up: arenas, NCCL communicators
                sq.decode(b, nthreads=16, out=out)
                te = td = 0.0
                info = None
                for _ in range(steps):
                    t0 = time.perf_counter()
                    b = sq.encode(pipeline, vol, nthreads=16, out=blob_buf)
                    t1 = time.perf_counter()
                    info = sq.last_shard_info()          # of the encode: the decode has no collective
                    t1b = time.perf_counter()
                    sq.decode(b, nthreads=16, out=out)
                    t2 = time.perf_counter()
                    te += t1 - t0
                    td += t2 - t1b
                rows[len(devs)] = {"value": vol.nbytes * steps / (te + td) / 1e9, "encode_ms": te / steps * 1e3, "decode_ms": td / steps * 1e3,
                                   "gpus_used_by_the_call": max(info["gpus"], 1), "nccl_histogram_allreduce": info["nccl"],
                                   "nccl_allreduces_so_far": sq.nccl_allreduces(),
                                   "blob_bytes": int(b.size), "checksum": int(out[::4097].astype(np.uint64).sum())}
            one, many = rows[1], rows[ctx.world]
            res = {"workload": wname, "pipeline": pipeline, "unit": "GB/s", "value": many["value"], "gpus": ctx.world,
                   "one_gpu_value": one["value"], "speedup_over_one_gpu": many["value"] / one["value"],
                   "encode_ms": many["encode_ms"], "decode_ms": many["decode_ms"], "one_gpu_encode_ms": one["encode_ms"],
                   "one_gpu_decode_ms": one["decode_ms"], "gpus_used_by_the_call": many["gpus_used_by_the_call"],
                   "nccl_histogram_allreduce": many["nccl_histogram_allreduce"], "nccl_allreduces_in_library": many["nccl_allreduces_so_far"],
                   "same_blob_size_and_voxels_as_one_gpu": many["blob_bytes"] == one["blob_bytes"] and many["checksum"] == one["checksum"],
                   "api": "SQY_PipelineEncode_UI16 + SQY_Decode_UI16, one pinned host stack, z-slabs over all GPUs inside the library"}
            del h_vol, h_out, h_blob
        except Exception as exc:
            res = {"workload": wname, "error": repr(exc)}
        finally:
            for d in range(ctx.world):
                try:
                    sq.set_device(d)
                    sq.release_scratch()
                except Exception:
                    pass
            sq.set_device(ctx.local_rank)
    ctx.host_barrier()
    return res


def compact(r):
    """what per_config keeps of a workload result"""
    if r is None:
        return None
    keep = {k: r[k] for k in ("pipeline", "shape_zyx", "what", "value", "encode_gbs", "decode_gbs", "ms_per_step", "compression_ratio",
                              "gpu_launches", "collective", "frame_per_chunk", "linked_single_frame", "bit_exact_vs_torch_arithmetic",
                              "stacks_per_gpu", "blobs_per_gpu", "skipped", "error") if k in r and r[k] is not None}
    if "roofline" in r:
        ro = r["roofline"]
        keep["roofline"] = {"kernel": ro["kernel"], "frac": ro["frac"], "achieved": ro["achieved"], "kernel_ms": ro["kernel_ms"],
                            "encode_call_frac": ro["encode_call_frac"], "stage_ms": ro["stage_ms"], "lz4_blocks": ro["lz4_blocks"]}
    if r.get("e2e"):
        keep["e2e"] = {k: r["e2e"].get(k) for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step", "same_voxels_as_device_path", "error")
                       if k in r["e2e"]}
    return keep


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=list(WORKLOADS))
    ap.add_argument("--preset", default=None)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-per-config", action="store_true", help="only the main workload (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the main workload's outputs of the last timed step to DIR/<name>.npy (cfg4: of its last framing, "
                         "and nothing when it is skipped; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")

    shape, pipeline, preset, chain_id = WORKLOADS[args.workload]
    if args.preset:
        preset = args.preset
        WORKLOADS[args.workload] = (shape, pipeline, preset, chain_id)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    config = {"workload": f"{args.workload}: {pipeline} on synthetic {shape[2]}x{shape[1]}x{shape[0]} uint16 light-sheet stack ({preset})",
              "pipeline": pipeline, "shape_zyx": list(shape), "preset": preset,
              "parallelism": f"{world} stack(s), one per GPU" if world > 1 else "1 GPU",
              "cache": "inputs (>= 256 MiB per step) exceed the 126 MB L2; no flush needed"}
    if args.workload == "cfg4":
        config["parallelism"] = f"{CFG4_PER_GPU} reference-made blobs per GPU, decode only"
    if args.workload == "cfg5":
        config["parallelism"] = f"{CFG5_PER_GPU} stacks per GPU (stack v -> GPU v mod G)"

    if args.impl == "reference":
        if rank != 0:
            return
        info, ms = reference_arm(shape, pipeline, preset, chain_id, args.steps, args.warmup, decode_only=args.workload == "cfg4")
        line = {"metric": METRIC, "value": info["value"], "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u16", "data": "synthetic",
                "impl": "reference", "config": config, "cpu_baseline": info,
                "note": "the reference's CPU stage code on ALL host cores of the box; its throughput is a property of the host and does not "
                        "grow with --gpus (at N > 1 compare whole box against whole box, or per stack: value / n_gpus of the other arm)",
                "e2e": {"value": info["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import torch

    import sqeazy_b200 as sq

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback exists)"
    torch.cuda.set_device(local_rank)
    sq.set_device(local_rank)
    dist = cpu_group = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        cpu_group = dist.new_group(backend="gloo")
    ctx = Ctx(torch, sq, dist, cpu_group, rank, local_rank, world)

    t_start = time.perf_counter()
    if args.workload in ("cfg1", "cfg2", "cfg3"):
        main_res = run_pipeline_workload(ctx, args.workload, args.steps, warmup, want_e2e=not args.no_e2e, detail=True, sampler_cls=ClockSampler,
                                         dump_dir=args.dump_outputs)
    elif args.workload == "cfg4":
        main_res = run_cfg4(ctx, args.steps, warmup, dump_dir=args.dump_outputs)
    else:
        main_res = run_cfg5(ctx, args.steps, warmup, dump_dir=args.dump_outputs)

    # ---- the other BASELINE configurations, a few steps each ----
    per_config = None
    if not args.no_per_config:
        per_config = {}
        for w in ("cfg1", "cfg3", "cfg4", "cfg5"):
            if w == args.workload:
                continue
            try:
                if w in ("cfg1", "cfg3"):
                    r = run_pipeline_workload(ctx, w, 3, 3, want_e2e=(not args.no_e2e) and world == 1, detail=False)
                elif w == "cfg4":
                    r = run_cfg4(ctx, 2, 1)
                else:
                    r = run_cfg5(ctx, 2, 3)
                per_config[w] = compact(r)
            except Exception as exc:
                per_config[w] = {"error": repr(exc)}
                ctx.free()

    # ---- one stack sharded over all GPUs inside the C ABI (strong scaling of the host-buffer path) ----
    e2e_sharded = None
    if world > 1 and not args.no_e2e:
        e2e_sharded = {}
        for w in ("cfg2", "cfg3"):
            r = run_sharded(ctx, w, 2)
            if rank == 0:
                e2e_sharded[w] = r

    # ---- CPU baseline beside it (rank 0, N = 1 only) ----
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline, _ = reference_arm(shape, pipeline, preset, chain_id, 2, 1, as_baseline=True, decode_only=args.workload == "cfg4")
        if "compression_ratio" in main_res and cpu_baseline.get("kind") == "reference":
            # the same voxels through both encoders: the GPU library on the reference arm's slab
            try:
                import numpy as np

                from sqeazy_b200.synth import numpy_volume

                slab = numpy_volume(tuple(cpu_baseline["sample_shape"]), preset, index=0)
                d_slab = torch.from_numpy(slab.view(np.int16)).to(ctx.dev)
                ours = int(sq.encode_device(pipeline, d_slab).numel())
                cpu_baseline["ratio_same_voxels"] = {"gpu": slab.nbytes / ours, "reference": cpu_baseline["ratio"],
                                                     "gpu_over_reference": (slab.nbytes / ours) / cpu_baseline["ratio"]}
                del d_slab
            except Exception as exc:
                cpu_baseline["ratio_same_voxels"] = {"error": repr(exc)}

    if rank == 0:
        line = {"metric": METRIC, "value": main_res["value"], "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": warmup,
                "ms_per_step": main_res.get("ms_per_step"), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u16", "data": "synthetic", "config": config}
        for k in ("encode_gbs", "decode_gbs", "compression_ratio", "blob_bytes", "clocks", "frame_per_chunk", "linked_single_frame", "collective"):
            if main_res.get(k) is not None:
                line[k] = main_res[k]
        line["e2e"] = main_res.get("e2e") or {"value": None, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                                              "note": "device-resident workload (batches): no host-buffer entry point in the reference for it"}
        line["gpu_launches"] = main_res.get("gpu_launches")
        if "roofline" in main_res:
            line["roofline"] = main_res["roofline"]
        line["cpu_baseline"] = cpu_baseline
        if per_config is not None:
            line["per_config"] = per_config
        if e2e_sharded is not None:
            line["e2e_sharded"] = e2e_sharded
        line["bench_wall_s"] = time.perf_counter() - t_start
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
