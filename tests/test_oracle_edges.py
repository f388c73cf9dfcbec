"""edge.canny_ivice (edge.py:19-35): the numpy oracle is pinned against the reference's own outputs
(tests/golden/edges.npz) and, step by step, against cv2 itself (imgproc is installed, unlike opencv-contrib); the device
code's per-pixel arithmetic (csrc/edges_core.cuh) is compiled for the host and compared with both.  CPU only."""
import ctypes as C
import os
import subprocess

import cv2
import numpy as np
import pytest

from helpers import load_npz, pkg
from oracle import edges as oe

HERE = os.path.dirname(os.path.abspath(__file__))
CASES = ("texture", "noise", "boxes", "ramp", "row", "column")


def random_image(rng, it):
    H, W = int(rng.integers(1, 150)), int(rng.integers(1, 200))
    if it % 3 == 0:
        return rng.integers(0, 256, size=(H, W, 3), dtype=np.uint8)
    if it % 3 == 1 and H > 20 and W > 20:
        return pkg("synth").texture(H, W, it)
    img = np.zeros((H, W, 3), np.uint8)
    for _ in range(6):
        a, b = int(rng.integers(0, H)), int(rng.integers(0, W))
        img[a:a + int(rng.integers(1, 30)), b:b + int(rng.integers(1, 30))] = rng.integers(0, 256, size=3)
    return img


@pytest.mark.parametrize("case", CASES)
def test_oracle_canny_ivice_golden(case):
    z = load_npz("edges")
    out = oe.canny_ivice(z[case + "_img"])
    assert out.dtype == np.float32 and np.array_equal(out == 0, z[case + "_edges"] == 1)


def test_oracle_steps_equal_cv2():
    rng = np.random.default_rng(1)
    for it in range(30):
        img = random_image(rng, it)
        gray = cv2.cvtColor(img, cv2.COLOR_BGR2GRAY)
        bl = cv2.GaussianBlur(gray, (3, 3), 0)
        assert np.array_equal(oe.blur3(gray), bl)
        dx, dy = oe.sobel3(bl)
        assert np.array_equal(dx, cv2.Sobel(bl, cv2.CV_16S, 1, 0, ksize=3, borderType=cv2.BORDER_REPLICATE))
        assert np.array_equal(dy, cv2.Sobel(bl, cv2.CV_16S, 0, 1, ksize=3, borderType=cv2.BORDER_REPLICATE))
        for lo, hi in ((100, 200), (30, 90), (5, 10)):
            assert np.array_equal(oe.canny(bl, lo, hi), cv2.Canny(image=bl, threshold1=lo, threshold2=hi)), (it, lo, hi)


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("edge") / "libedge_emul.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-Wall", "-o", so,
                    os.path.join(HERE, "edge_host_emul.cpp")], check=True)
    lib = C.CDLL(so)

    def run(img, lo=100, hi=200):
        img = np.ascontiguousarray(img, dtype=np.uint8)
        out = np.empty(img.shape[:2], np.float32)
        assert lib.edge_emul(img.ctypes.data_as(C.c_void_p), img.shape[0], img.shape[1], lo, hi,
                             out.ctypes.data_as(C.c_void_p), None) == 0
        return out
    return run


def test_device_arithmetic_on_host_golden(emul):
    z = load_npz("edges")
    for case in CASES:
        assert np.array_equal(emul(z[case + "_img"]) == 0, z[case + "_edges"] == 1), case


def test_device_arithmetic_on_host_vs_oracle_random(emul):
    rng = np.random.default_rng(2)
    edges = 0
    for it in range(40):
        img = random_image(rng, it)
        lo, hi = [(100, 200), (30, 90), (5, 10)][it % 3 if it % 2 else 0]
        want = oe.canny_ivice(img, lo, hi)
        assert np.array_equal(emul(img, lo, hi), want), (it, img.shape, lo, hi)
        edges += int((want == 0).sum())
    assert edges > 20000


@pytest.mark.parametrize("shape", [(60, 70), (8, 8), (150, 199)])
def test_oracle_descending_thresholds_equal_cv2(shape):
    """cv2.Canny takes its thresholds in either order; so does the oracle.  On blurred noise most survivors are weak,
    so the order matters: the unswapped pair gives another edge map at (200, 100) or (90, 30)."""
    from helpers import canny_blurred_noise, canny_pmap
    rng = np.random.default_rng(shape[0] * 31 + shape[1])
    differs = 0
    for it in range(4):
        bl = cv2.GaussianBlur(cv2.cvtColor(canny_blurred_noise(rng, *shape), cv2.COLOR_BGR2GRAY), (3, 3), 0)
        for lo, hi in ((200, 100), (90, 30), (60, 20), (40.5, -3.5), (-0.5, -2.5)):
            want = cv2.Canny(image=bl, threshold1=lo, threshold2=hi)
            assert np.array_equal(oe.canny(bl, lo, hi), want), (it, lo, hi)
            differs += not np.array_equal(oe.hysteresis(canny_pmap(bl, lo, hi)), want > 0)
    assert differs >= 4


def test_device_arithmetic_on_host_descending_thresholds(emul):
    """The host build of the per-pixel functions with the library's swap, at descending pairs, against cv2."""
    from helpers import canny_blurred_noise
    rng = np.random.default_rng(5)
    for H, W in ((60, 70), (33, 17)):
        img = canny_blurred_noise(rng, H, W)
        for lo, hi in ((200, 100), (90, 30)):
            bl = cv2.GaussianBlur(cv2.cvtColor(img, cv2.COLOR_BGR2GRAY), (3, 3), 0)
            want = np.array((255 - cv2.Canny(image=bl, threshold1=lo, threshold2=hi)) / 255, dtype="float32")
            assert np.array_equal(emul(img, min(lo, hi), max(lo, hi)), want)
