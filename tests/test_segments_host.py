"""removeSmallSegments: the device code's replay logic (csrc/segments_core.cuh) compiled for the HOST.

The CUDA implementation labels connected components in parallel and replays the reference's scan at component
granularity (see segments_core.cuh for why that is exact).  The replay functions are plain C++ shared by the kernel
and by tests/seg_host_emul.cpp; here they are checked on the CPU against the golden fixtures (the reference's own
function) and against the C oracle on random fields.  The kernels themselves are covered by tests/test_z_gpu_segments.py.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from helpers import SEGMENT_KINDS, load_npz, segment_test_field
from oracle import cport

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("seg") / "libseg_emul.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-Wall", "-ffp-contract=off", "-o", so,
                    os.path.join(HERE, "seg_host_emul.cpp")], check=True)
    lib = C.CDLL(so)

    def run(flow, tresh, ms, prefilter=0):
        f = np.array(flow, dtype=np.float32, copy=True)
        assert lib.seg_emul(f.ctypes.data_as(C.c_void_p), f.shape[0], f.shape[1], C.c_float(tresh), int(ms),
                            int(prefilter)) == 0
        return f
    return run


@pytest.mark.parametrize("prefilter", [0, 1])
def test_replay_logic_golden(emul, prefilter):
    z = load_npz("segments")
    for i in range(int(z["n"])):
        f, (tresh, ms) = z[f"c{i}_in"], z[f"c{i}_par"]
        out = emul(f, float(tresh), int(ms), prefilter)
        assert np.array_equal(out[..., :2], f[..., :2])
        assert np.array_equal(out[..., 2], z[f"c{i}_valid_out"].astype(np.float32)), i


@pytest.mark.parametrize("prefilter", [0, 1])
def test_replay_logic_vs_oracle_random(emul, prefilter):
    rng = np.random.default_rng(77)
    removed = 0
    for it in range(120):
        kind = SEGMENT_KINDS[it % 4]
        A, B = int(rng.integers(2, 90)), int(rng.integers(2, 90))
        f = segment_test_field(rng, A, B, kind)
        tresh = [10, 3, 1.5, 0][int(rng.integers(0, 4))]
        ms = [100, 10, 4, 2, 1000, 1 << 30][int(rng.integers(0, 6))]
        want, n = cport.remove_small_segments(f, tresh, ms, want_count=True)
        removed += n
        assert np.array_equal(emul(f, tresh, ms, prefilter), want), (it, kind, A, B, tresh, ms)
    assert removed > 1000


def planted_cases():
    from helpers import (SEG_INVALID_MIN, seg_invalid_seed_cases, seg_prefilter_cases, seg_rebind_cases)
    for name, (f, _) in seg_rebind_cases().items():
        yield name, f, 1.0, 100
    for name, (f, _, _) in seg_invalid_seed_cases().items():
        yield name, f, 1.0, SEG_INVALID_MIN
    for name, (f, _, _) in seg_prefilter_cases().items():
        yield name, f, 1.0, 10


@pytest.mark.parametrize("prefilter", [0, 1])
def test_replay_logic_planted_cases(emul, prefilter):
    """The planted scan rebinds, invalid seeds and prefilter boundaries of test_zz_gpu_postprocess_edges.py through
    the host build of the replay; the Python restatement is pinned to the C oracle on each of them."""
    from helpers import bitwise_equal, seg_restated
    events = 0
    for name, f, tresh, ms in planted_cases():
        want = cport.remove_small_segments(f, tresh, ms)
        ref, ev = seg_restated(f, tresh, ms)
        assert bitwise_equal(ref, want), name
        assert bitwise_equal(emul(f, tresh, ms, prefilter), want), name
        events += len(ev)
    assert events > 60


@pytest.mark.parametrize("prefilter", [0, 1])
def test_replay_logic_special_values(emul, prefilter):
    """NaN / +-inf / +-0 flows, valid flags around 0.5, NaN, -1, 2, 1e30 and tresh 0, negative, NaN, +inf: bytewise,
    NaN payloads included."""
    from helpers import bitwise_equal, seg_restated, seg_value_fields
    rng = np.random.default_rng(12)
    removed = 0
    for it in range(80):
        f = seg_value_fields(rng, int(rng.integers(1, 10)), int(rng.integers(1, 10)))
        for tresh in (0.0, 0.5, -1.0, float("nan"), float("inf")):
            want = cport.remove_small_segments(f, tresh, 4)
            ref, ev = seg_restated(f, tresh, 4)
            assert bitwise_equal(ref, want)
            assert bitwise_equal(emul(f, tresh, 4, prefilter), want), (it, tresh)
            removed += len(ev)
    assert removed > 50


def test_restatement_min_size_rule():
    """The drop-in's bound rule matches the reference's float comparison: NaN and -inf remove nothing, +inf removes
    every segment of two or more pixels, a fractional bound acts like its ceiling."""
    from helpers import bitwise_equal, seg_restated
    rng = np.random.default_rng(13)
    f = segment_test_field(rng, 23, 19, "stale")
    for ms, bound in ((float("nan"), 0), (float("-inf"), 0), (float("inf"), 2**31 - 1), (2.5, 3), (3.0000001, 4),
                      (1e12, 2**31 - 1)):
        assert bitwise_equal(seg_restated(f, 3.0, ms)[0], cport.remove_small_segments(f, 3.0, bound)), ms
