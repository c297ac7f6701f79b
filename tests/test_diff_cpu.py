"""diff3x3x1 head filter (SURVEY §8f-4, reference: encoders/diff_scheme_impl.hpp:78-199) without a GPU: the oracle's
restatement against golden vectors made by the reference (tests/golden/make_golden_diff.py) and against oracle/_ref live,
the CUDA kernels' thread program (sqeazy_b200/csrc/device/diff_thread.h, the very source the kernel compiles) replayed on
the CPU in several thread orders against the oracle, and the host logic (stage name, header text, refused shapes)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "golden_diff_v1.npz")

SHAPES = [(8, 8, 8), (5, 7, 9), (16, 16, 16), (4, 6, 32), (9, 8, 8), (12, 9, 8), (17, 9, 8), (3, 3, 3), (3, 4, 2), (20, 5, 10), (7, 3, 40),
          (33, 64, 32), (17, 16, 8), (16, 24, 16), (33, 16, 16), (9, 5, 4), (32, 8, 64), (10, 11, 13), (6, 40, 24)]
REFUSED = [(2, 8, 8), (1, 8, 8), (8, 2, 8), (8, 8, 1), (3, 3, 2), (18, 9, 8), (40000, 3, 3), (100, 4, 4)]
REFUSED_U8 = [(129, 64, 64), (9, 130, 64), (9, 16, 136)]       # int8 coordinates in the reference's naive_sum
BIG = [(24, 128, 128), (128, 20, 128), (130, 9, 72), (20, 129, 24), (6, 16, 136)]   # uint8: the first two only


def _ok(port, shape, dtype):
    return port.diff_supported(shape, np.dtype(dtype).itemsize)


@pytest.fixture(scope="module")
def golden():
    return np.load(GOLDEN)


@pytest.fixture(scope="module")
def sim():
    so = os.path.join(ROOT, "oracle", "_build", "libdiff_sim.so")
    src = os.path.join(ROOT, "tests", "helpers", "diff_sim.cpp")
    hdr = os.path.join(ROOT, "sqeazy_b200", "csrc", "device", "diff_thread.h")
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        os.makedirs(os.path.dirname(so), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", os.path.dirname(hdr), src, "-o", so])
    return ctypes.CDLL(so)


def _volume(shape, dtype, seed):
    rng = np.random.default_rng(seed)
    hi = 65536 if dtype == np.uint16 else 256
    if seed % 2:
        return rng.integers(0, hi, size=shape).astype(dtype)          # wraps of the 9-voxel sum all over
    return np.clip(np.rint(100 + 6 * rng.standard_normal(shape)), 0, hi - 1).astype(dtype)


def test_golden_name(golden):
    assert bytes(golden["name"]).decode() == "diff3x3x1"


@pytest.mark.parametrize("case", ["u16_cube", "u16_flat", "u16_spill", "u16_vec", "u16_tall", "u8_cube", "u8_spill", "u8_vec"])
def test_oracle_matches_golden(port, golden, case):
    a, enc = golden[case + "_in"], golden[case + "_enc"]
    assert np.array_equal(port.diff(a), enc)
    assert np.array_equal(port.diff(enc, decode=True), a)
    assert not np.array_equal(enc, a)


@pytest.mark.parametrize("dtype", [np.uint16, np.uint8])
@pytest.mark.parametrize("shape", SHAPES + BIG)
def test_oracle_matches_reference_live(port, ref, shape, dtype):
    if not _ok(port, shape, dtype):
        with pytest.raises(ValueError):
            port.diff(np.zeros(shape, dtype=dtype))
        return
    for seed in (1, 2):
        a = _volume(shape, dtype, seed + 7 * shape[0])
        enc = ref.diff(a)
        assert np.array_equal(port.diff(a), enc)
        assert np.array_equal(ref.diff(a, nthreads=3), enc)           # the encode loop is free of races (reads `raw` only)
        assert np.array_equal(port.diff(enc, decode=True), ref.diff(enc, decode=True))
        assert np.array_equal(port.diff(enc, decode=True), a)


def test_oracle_semantics_by_hand(port):
    """cube: the coded set is z >= 1, 1 <= y < Y-1, 1 <= x < Z-1; the 9-voxel sum wraps in the voxel type before / 9"""
    a = np.full((4, 4, 4), 60000, dtype=np.uint16)
    enc = port.diff(a)
    q = ((9 * 60000) % 65536) // 9
    want = a.copy()
    want[1:, 1:3, 1:3] = 60000 - q
    assert np.array_equal(enc, want)
    b = np.arange(6 * 5 * 12, dtype=np.uint16).reshape(6, 5, 12)      # Z < X: only x in [1, Z-1) is coded
    eb = port.diff(b)
    assert np.array_equal(eb[:, :, 5:], b[:, :, 5:]) and np.array_equal(eb[0], b[0]) and np.array_equal(eb[:, 0], b[:, 0])
    assert np.all(eb[1:, 1:4, 1:5] == 5 * 12 + 0 * b[1:, 1:4, 1:5])   # a linear ramp minus its mean one plane back = Y*X


@pytest.mark.parametrize("shape", REFUSED)
def test_refused_shapes(port, sim, shape):
    assert not port.diff_supported(shape)
    z, y, x = shape
    if z * y * x < 1 << 20:
        with pytest.raises(ValueError):
            port.diff(np.zeros(shape, dtype=np.uint16))
    assert sim.sim_diff(0, None, None, ctypes.c_uint64(z), ctypes.c_uint64(y), ctypes.c_uint64(x), 2, 0) == 1


@pytest.mark.parametrize("shape", REFUSED_U8)
def test_refused_uint8_extents(port, sim, shape):
    """uint8 stacks: naive_sum keeps z, y, x in int8 (diff_scheme_utils.hpp:81-89); from 129 on the reference reads from
    wrapped coordinates - what it returns there no longer follows its own rule on the shapes where it does not crash"""
    z, y, x = shape
    assert port.diff_supported(shape, 2) and not port.diff_supported(shape, 1)
    with pytest.raises(ValueError):
        port.diff(np.zeros(shape, dtype=np.uint8))
    assert sim.sim_diff(0, None, None, ctypes.c_uint64(z), ctypes.c_uint64(y), ctypes.c_uint64(x), 1, 0) == 1


@pytest.mark.parametrize("dtype", [np.uint16, np.uint8])
@pytest.mark.parametrize("shape", SHAPES + BIG + [(7, 9, 520), (10, 23, 264)])
def test_kernel_thread_program_replay(port, sim, shape, dtype):
    """every launch of the schedule, threads forward / backward / odd first, over poisoned output, any buffer alignment"""
    if not _ok(port, shape, dtype):
        pytest.skip("extent beyond the reference's int8 coordinates")
    z, y, x = shape
    n = z * y * x
    u64 = ctypes.c_uint64
    elem = np.dtype(dtype).itemsize
    for k, (off_in, off_out) in enumerate(((0, 0), (1, 0), (0, 3), (8, 8))):
        for order in (0, 1, 2):
            a_buf = np.zeros(n + 16, dtype)
            a = a_buf[off_in: off_in + n]
            a[:] = _volume(shape, dtype, 3 * k + order).ravel()
            want = port.diff(a.reshape(shape)).ravel()
            e_buf = np.zeros(n + 16, dtype)
            enc = e_buf[off_out: off_out + n]
            assert sim.sim_diff(0, ctypes.c_void_p(a.ctypes.data), ctypes.c_void_p(enc.ctypes.data), u64(z), u64(y), u64(x), elem, order) == 0
            assert np.array_equal(enc, want)
            assert e_buf[:off_out].sum() == 0 and e_buf[off_out + n:].sum() == 0
            w_buf = np.zeros(n + 16, dtype)
            w = w_buf[off_in: off_in + n]
            w[:] = want
            d_buf = np.zeros(n + 16, dtype)
            dec = d_buf[off_out: off_out + n]
            assert sim.sim_diff(1, ctypes.c_void_p(w.ctypes.data), ctypes.c_void_p(dec.ctypes.data), u64(z), u64(y), u64(x), elem, order) == 0
            assert np.array_equal(dec, a)


def test_host_logic_names_and_bounds(sq):
    assert sq.pipeline_possible("diff3x3x1->lz4") and sq.pipeline_possible("diff3x3x1->bitswap1->lz4")
    assert sq.pipeline_possible("rmestbkrd->diff3x3x1->bitswap1->lz4") and sq.pipeline_possible("diff3x3x1")
    assert sq.pipeline_possible("diff3x3x1->lz4", 1)
    assert not sq.pipeline_possible("diff3x3x3->lz4") and not sq.pipeline_possible("lz4->diff3x3x1")
    assert orc.can_be_built_from("diff3x3x1->lz4")
    raw = 64 * 64 * 64 * 2
    assert sq.max_compressed_length("diff3x3x1->lz4", raw) >= sq.max_compressed_length("lz4", raw)
    assert sq.max_compressed_length("diff3x3x1", raw) > raw


def test_reference_offset_kats_on_cube_of_8(port):
    """tests/test_diff_scheme_impl.cpp:50-87 (offset_exact_last_plane) and :91-97 (9 traversed voxels), read off the coded set:
    a constant stack codes to 0 wherever the filter is applied; the first voxel of every run is one of the reference's offsets"""
    n = 8
    enc = port.diff(np.full((n, n, n), 900, dtype=np.uint16)).ravel()      # 9 * 900 / 9 = 900 -> 0
    coded = enc == 0
    starts = np.flatnonzero(coded & ~np.roll(coded, 1))
    assert starts.size == (n - 1) * (n - 2)
    assert starts[0] == n * n + n + 1 and starts[1] == n * n + 2 * n + 1
    assert starts[-1] == (n - 1) * n * n + (n - 2) * n + 1
    runs = np.flatnonzero(coded & ~np.roll(coded, -1)) - starts + 1
    assert np.all(runs == n - 2)                                              # non_halo_end(0) - non_halo_begin(0)
    one = np.zeros((n, n, n), dtype=np.uint16)
    one[3, 4, 4] = 9                                                          # seen by the 9 voxels below it, each gets 9 / 9
    e1 = port.diff(one).astype(np.int32)
    assert np.all(e1[4, 3:6, 3:6] == 65535) and (e1 != one).sum() == 9
