"""bench.py's reference arm runs without a GPU (it times the reference's CPU stage code, oracle/_ref, or the oracle port):
its JSON line must carry the keys the driver reads."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _line(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", *args],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_reference_arm_line():
    d = _line("--workload", "cfg1")
    assert d["impl"] == "reference" and d["metric"] == "uint16 voxel GB/s encode+decode" and d["unit"] == "GB/s"
    assert d["higher_is_better"] is True and d["dtype"] == "u16" and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["steps"] == 1 and d["warmup"] == 0
    assert d["config"]["pipeline"] == "bitswap1->lz4" and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_under_torchrun_env_prints_on_rank_0_only():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_are_exact_seeded_and_bounded(tmp_path):
    """--dump-outputs: values read as unsigned integers in float32, the whole array or a sample fixed by the array's name,
    and float64 sums over every element; two dumps of the same arrays are identical and stay within 64 MiB"""
    import numpy as np
    import torch

    import bench

    u = np.random.default_rng(1).integers(0, 65536, (80, 256, 256), dtype=np.uint16)
    blob = torch.from_numpy(np.random.default_rng(2).integers(0, 256, 1000, dtype=np.uint8))
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"blob": blob, "decoded": torch.from_numpy(u.view(np.int16))})
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["blob.npy", "blob_chunk_sums.npy", "decoded.npy", "decoded_chunk_sums.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 << 20
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f
    assert np.array_equal(np.load(tmp_path / "a" / "blob.npy"), blob.numpy().astype(np.float32))
    sample = np.load(tmp_path / "a" / "decoded.npy")
    assert sample.dtype == np.float32 and sample.size == bench.DUMP_SAMPLES // 2 < u.size
    assert sample.min() >= 0 and sample.max() > 32767
    sums = np.load(tmp_path / "a" / "decoded_chunk_sums.npy")
    assert sums.dtype == np.float64 and sums.size == -(-u.size // bench.DUMP_CHUNK) and sums.sum() == u.astype(np.uint64).sum()
