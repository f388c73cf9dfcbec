"""removeSmallSegments (segments.cu, DESIGN 4.6) and edge.canny_ivice (edges.cu, DESIGN 4.7) at their edges.

Both are exact reproductions of a sequential reference on top of the lock-free union-find of csrc/unionfind.cuh.
Segments: whole fields bytewise (float32 viewed as uint32, so dx/dy, NaN payloads and -0.0 must come back untouched)
against the C oracle and the plain-Python restatement in helpers.seg_restated, whose removal events show that every
planted scan rebind, invalid seed and prefilter boundary is reached.  Canny: bytewise against cv2.Canny on the
blurred grey image and against oracle/edges, with threshold pairs in either order and chains only hysteresis links.
(Named to run after the hot-path GPU modules.)"""
import importlib
import math
import os
import sys

import cv2
import numpy as np
import pytest

from helpers import (SEG_INVALID_MIN, SEGMENT_KINDS, bitwise_equal, canny_blurred_noise, canny_chain_points,
                     canny_pmap, canny_polyline_image, canny_sparse_strong_pair, pkg, seg_invalid_seed_cases,
                     seg_paint, seg_prefilter_cases, seg_rebind_cases, seg_restated, seg_singletons,
                     seg_value_fields, segment_test_field)
from oracle import cport
from oracle import edges as oe

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INT_MAX = 2**31 - 1


def dev_segments(f, tresh, ms, workspace=None):
    return pkg("ops").remove_small_segments(torch.from_numpy(f.copy()).cuda(), tresh, ms, workspace).cpu().numpy()


def check_segments(f, tresh, ms, restated=True):
    """Device == C oracle bytewise (and == the Python restatement, pinned to the oracle); returns the events."""
    want = cport.remove_small_segments(f, tresh, ms)
    got = dev_segments(f, tresh, ms)
    assert bitwise_equal(got, want), (tresh, ms, int((got.view(np.uint32) != want.view(np.uint32)).sum()))
    if not restated:
        return None
    ref, events = seg_restated(f, tresh, ms)
    assert bitwise_equal(ref, want)
    return events


# ------------------------------------------------------------------ segments

@pytest.mark.parametrize("shape", [(a, b) for a in (1, 2, 31, 32, 33, 63, 64, 65, 97, 436) for b in (1, 2, 3, 33, 130)]
                         + [(4099, 3), (3, 4099)])
def test_segments_column_length_sweep(shape):
    """Every column length around the replay's 32-row steps, every field kind, tresh and min size."""
    rng = np.random.default_rng(shape[0] * 7919 + shape[1])
    removed = 0
    for kind in SEGMENT_KINDS:
        f = segment_test_field(rng, *shape, kind)
        for tresh in (0, 1.5, 3, 10):
            for ms in (3, 4, 10, 100):
                want, n = cport.remove_small_segments(f, tresh, ms, want_count=True)
                got = dev_segments(f, tresh, ms)
                assert bitwise_equal(got, want), (kind, tresh, ms)
                removed += n
    if shape[0] * shape[1] >= 60:
        assert removed > 0


@pytest.mark.parametrize("name", list(seg_rebind_cases()))
def test_segments_planted_rebinds(name):
    f, want = seg_rebind_cases()[name]
    events = check_segments(f, 1.0, 100)
    got = {(seed, after) for seed, last, before, after in events}
    for w in want:
        assert w in got, (w, events)
    for seed, last, before, after in events:
        assert last[1] == after


@pytest.mark.parametrize("name", list(seg_invalid_seed_cases()))
def test_segments_invalid_seeds(name):
    f, seed, total = seg_invalid_seed_cases()[name]
    events = check_segments(f, 1.0, SEG_INVALID_MIN)
    seeds = [e[0] for e in events]
    assert (seed in seeds) == (1 < total < SEG_INVALID_MIN), events


@pytest.mark.parametrize("name", list(seg_prefilter_cases()))
def test_segments_prefilter_boundaries(name):
    f, pix, removed = seg_prefilter_cases()[name]
    check_segments(f, 1.0, 10)
    out = dev_segments(f, 1.0, 10)
    flags = np.array([out[a, b, 2] for a, b in pix])
    assert np.all(flags == 0) if removed else np.array_equal(flags, np.array([f[a, b, 2] for a, b in pix]))


def serpentine(A, B, rows):
    """One-pixel-wide serpentine over `rows` rows of the scan (every other row, joined alternately at either end)."""
    pix = []
    for k, a in enumerate(range(1, rows, 2)):
        cols = range(1, B - 1) if k % 2 == 0 else range(B - 2, 0, -1)
        pix += [(a, b) for b in cols]
        if a + 2 < rows:
            pix.append((a + 1, cols[-1]))
    return pix


def spiral(A, B, size):
    """Square spiral of one-pixel width inside a size x size box at (1, 1): rings two rows apart, each joined to the
    next by one pixel."""
    pix, seen = [], set()
    a0, b0, a1, b1 = 1, 1, size, size
    while a0 <= a1 and b0 <= b1:
        ring = [(a0, b) for b in range(b0, b1 + 1)] + [(a, b1) for a in range(a0 + 1, a1 + 1)] + \
               [(a1, b) for b in range(b1 - 1, b0 - 1, -1)] + [(a, b0) for a in range(a1 - 1, a0 + 1, -1)]
        if a0 + 2 <= a1 - 2 and b0 + 2 <= b1 - 2:
            ring.append((a0 + 2, b0 + 1))
        for p in ring:
            if p not in seen:
                seen.add(p)
                pix.append(p)
        a0, b0, a1, b1 = a0 + 2, b0 + 2, a1 - 2, b1 - 2
    return pix


def comb(A, B, teeth):
    """Teeth along the scan's second index at every other row, joined only in column B-2."""
    pix = [(a, b) for a in range(1, 2 * teeth, 2) for b in range(1, B - 2)]
    return pix + [(a, B - 2) for a in range(1, 2 * teeth)]


def separated_field(A, B, pix, by):
    """The component `pix` (flow -7) in a background it may not join: flow jumps above tresh or invalid pixels."""
    f = np.zeros((A, B, 3), np.float32)
    f[..., 0] = 50.0
    f[..., 2] = 1 if by == "jump" else 0
    return seg_paint(f, pix, -7)


def uf_cases(A, B):
    big = A * B > 10**6
    ser = serpentine(A, B, 40 if big else A - 1)
    spi = spiral(A, B, 257 if big else min(A, B) - 3)
    com = comb(A, B, 16 if big else (A - 2) // 2)
    return {"serpentine-jump": (ser, "jump"), "serpentine-invalid": (ser, "invalid"),
            "spiral-jump": (spi, "jump"), "spiral-invalid": (spi, "invalid"), "comb-jump": (com, "jump")}


@pytest.mark.parametrize("shape", [(436, 1024), (2160, 3840)])
def test_segments_union_find_under_load(shape):
    """Long one-pixel components whose root is far along the path: kept whole at min_size = size (so labelled as
    one component), removed whole at size + 1 with the scan rebound to the last breadth-first pixel's column.
    At 4K each call runs three times and must give the same bytes."""
    A, B = shape
    reps = 3 if A * B > 10**6 else 1
    for name, (pix, by) in uf_cases(A, B).items():
        f = separated_field(A, B, pix, by)
        n = len(pix)
        assert n > 2000
        for ms in (n, n + 1):
            want, nrem = cport.remove_small_segments(f, 1.0, ms, want_count=True)
            flags = np.array([want[a, b, 2] for a, b in pix])
            assert np.all(flags == 0) if ms == n + 1 else np.all(flags == 1), (name, ms)
            outs = [dev_segments(f, 1.0, ms) for _ in range(reps)]
            for got in outs:
                assert bitwise_equal(got, want), (name, ms)
    # one component of every pixel, and a checkerboard of two flows where every pixel is a singleton
    const = np.zeros((A, B, 3), np.float32)
    const[..., :2] = (1.25, -3.5)
    const[..., 2] = 1
    cb = const.copy()
    cb[(np.arange(A)[:, None] + np.arange(B)[None, :]) % 2 == 1, :2] = (9.0, 9.0)
    for f, ms in ((const, A * B), (const, A * B + 1), (cb, 3)):
        want = cport.remove_small_segments(f, 1.0, ms)
        for _ in range(reps):
            assert bitwise_equal(dev_segments(f, 1.0, ms), want)
    assert np.all(cport.remove_small_segments(const, 1.0, A * B + 1)[..., 2] == 0)


def test_segments_tresh_at_a_float32_difference():
    """tresh exactly at a float32 L1 difference joins the pair; one ulp below does not; one above does."""
    for p, q in (((0.1, 0.7), (0.35, -0.2)), ((1e-3, 3.0), (-2e-3, 3.1)), ((1e6, 0.5), (1e6 + 0.5, 0.25))):
        p32, q32 = np.float32(p), np.float32(q)
        d = np.float32(abs(p32[0] - q32[0]) + abs(p32[1] - q32[1]))
        for t, joined in ((d, True), (np.nextafter(d, np.float32(-1)), False), (np.nextafter(d, np.float32(np.inf)), True)):
            f = seg_singletons(9, 5)
            seg_paint(f, [(4, 2)], *p32)
            seg_paint(f, [(5, 2)], *q32)
            events = check_segments(f, float(t), 3)
            assert (((4, 2), (5, 2), 2, 2) in events) == joined, (p, q, t)


def test_segments_special_values():
    """+-0 flows at tresh 0; negative, NaN and +inf tresh; NaN and +-inf flows; valid flags around 0.5, NaN, -1, 2,
    1e30; NaN payloads and -0.0 must survive bit for bit."""
    f = seg_singletons(8, 6)
    seg_paint(f, [(2, 1)], 0.0, -0.0)
    seg_paint(f, [(3, 1)], -0.0, 0.0)
    assert ((2, 1), (3, 1), 1, 1) in check_segments(f, 0.0, 3)
    for t in (-1.0, float("nan")):
        assert check_segments(f, t, 3) == []
    assert check_segments(f, float("inf"), 48) == []   # all one segment of 48 pixels
    assert len(check_segments(f, float("inf"), 49)) == 1
    rng = np.random.default_rng(11)
    removed = 0
    for it in range(60):
        f = seg_value_fields(rng, int(rng.integers(1, 12)), int(rng.integers(1, 12)))
        for tresh in (0.0, 0.5, 1.0, -1.0, float("nan"), float("inf")):
            removed += len(check_segments(f, tresh, 4))
    assert removed > 50


def test_segments_min_size_through_ops():
    rng = np.random.default_rng(3)
    f = segment_test_field(rng, 37, 29, "stale")
    for ms in (-5, 0, 1, 2):
        assert bitwise_equal(dev_segments(f, 3.0, ms), f)
    for ms in (3, 4, 37 * 29, 37 * 29 + 1, INT_MAX):
        check_segments(f, 3.0, ms, restated=False)
    assert not bitwise_equal(cport.remove_small_segments(f, 3.0, 3), f)


def test_segments_min_size_through_the_drop_in():
    """A fractional bound acts like its ceiling; NaN and -inf remove nothing, +inf every segment of two or more."""
    sys.path.insert(0, ROOT)
    pp = importlib.import_module("postprocessing")
    rng = np.random.default_rng(4)
    f = segment_test_field(rng, 23, 19, "stale")
    for ms in (2.5, 3.0000001, 1e12, float("inf"), float("-inf"), float("nan")):
        g = f.copy()
        assert pp.removeSmallSegments(g, 3.0, ms) is None
        want, events = seg_restated(f, 3.0, ms)
        assert bitwise_equal(g, want), ms
        if not math.isnan(ms) and ms > 0:
            assert len(events) > 0
    assert bitwise_equal(seg_restated(f, 3.0, 2.5)[0], cport.remove_small_segments(f, 3.0, 3))


def test_segments_workspace_and_stream():
    """A workspace prefilled with 0xFF, one left over from another shape, and a side stream."""
    ops, lib = pkg("ops"), pkg("_lib").load()
    rng = np.random.default_rng(8)
    big = segment_test_field(rng, 97, 65, "stale")
    small = segment_test_field(rng, 40, 33, "blocks")
    ws = torch.full((int(lib.flowb200_segments_workspace_bytes(97, 65)),), 0xFF, dtype=torch.uint8, device="cuda")
    for f in (small, big, small):
        want = cport.remove_small_segments(f, 3.0, 10)
        assert bitwise_equal(dev_segments(f, 3.0, 10, workspace=ws), want)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        t = torch.from_numpy(big.copy()).cuda()
        ops.remove_small_segments(t, 3.0, 10)
    s.synchronize()
    assert bitwise_equal(t.cpu().numpy(), cport.remove_small_segments(big, 3.0, 10))


def seg_call(ov):
    L = pkg("_lib")
    lib = L.load()
    A, B = ov.get("A", 8), ov.get("B", 8)
    buf = torch.zeros(8 * 8 * 3, dtype=torch.float32, device="cuda")
    need = lib.flowb200_segments_workspace_bytes(8, 8)
    ws = torch.zeros(need, dtype=torch.uint8, device="cuda")
    wsb = {None: need, "total-1": need - 1}[ov.get("ws_bytes")]
    flow = None if ov.get("null") == "flow" else buf.data_ptr()
    wsp = None if ov.get("null") == "workspace" else ws.data_ptr()
    rc = lib.flowb200_remove_small_segments(flow, A, B, 1.0, 10, wsp, wsb, None)
    torch.cuda.synchronize()
    return rc


SEG_ROWS = [({"null": "flow"}, "EINVAL"), ({"null": "workspace"}, "EINVAL"), ({"A": 0}, "EINVAL"),
            ({"A": -1}, "EINVAL"), ({"B": 0}, "EINVAL"), ({"B": -3}, "EINVAL"),
            ({"A": 65536, "B": 32768}, "EINVAL"), ({"ws_bytes": "total-1"}, "EWORKSPACE"), ({}, "OK")]


@pytest.mark.parametrize("ov,rc", SEG_ROWS, ids=["-".join(f"{k}={v}" for k, v in r[0].items()) or "defaults"
                                                 for r in SEG_ROWS])
def test_segments_return_code(ov, rc):
    assert seg_call(ov) == getattr(pkg("_lib"), rc)


def test_segments_workspace_bytes_of_non_positive_sizes():
    lib = pkg("_lib").load()
    for A, B in ((0, 5), (5, 0), (-1, 5), (5, -1), (0, 0), (-(2**31), 1)):
        assert lib.flowb200_segments_workspace_bytes(A, B) == 0


# ------------------------------------------------------------------ Canny

def cv2_inverted(img, t1, t2):
    bl = cv2.GaussianBlur(cv2.cvtColor(img, cv2.COLOR_BGR2GRAY), (3, 3), 0)
    return np.array((255 - cv2.Canny(image=bl, threshold1=t1, threshold2=t2)) / 255, dtype="float32")


def dev_canny(img, t1, t2, workspace=None):
    return pkg("ops").canny_edges(torch.from_numpy(img).cuda(), t1, t2, workspace).cpu().numpy()


def check_canny(img, t1, t2, oracle=True):
    want = cv2_inverted(img, t1, t2)
    got = dev_canny(img, t1, t2)
    assert bitwise_equal(got, want), (img.shape, t1, t2, int((got != want).sum()))
    assert bitwise_equal(pkg("edges").canny_edges(img, t1, t2), want)
    if oracle:
        assert bitwise_equal(oe.canny_ivice(img, t1, t2), want)
    return want


def unswapped_edges(img, t1, t2):
    """Edge pixels with the thresholds used in the order given (what cv2 does NOT do when t1 > t2)."""
    from scipy import ndimage
    bl = cv2.GaussianBlur(cv2.cvtColor(img, cv2.COLOR_BGR2GRAY), (3, 3), 0)
    pm = canny_pmap(bl, t1, t2)
    lab, _ = ndimage.label(pm != 1, structure=np.ones((3, 3)))
    return np.isin(lab, np.unique(lab[pm == 2])) & (pm != 1)


@pytest.mark.parametrize("shape", [(60, 70), (436, 1024)])
def test_canny_threshold_sweep(shape):
    rng = np.random.default_rng(shape[0])
    img = canny_blurred_noise(rng, *shape)
    bl = cv2.GaussianBlur(cv2.cvtColor(img, cv2.COLOR_BGR2GRAY), (3, 3), 0)
    dx, dy = oe.sobel3(bl)
    M = int((np.abs(dx) + np.abs(dy)).max())
    differs = 0
    for t1, t2 in ((100, 200), (30, 90), (150, 150), (0, 0), (200, 100), (90, 30), (60, 20), (40, 39),
                   (-5, 50), (50, -5), (-2.5, -0.5), (-0.5, 30.7), (30.7, -0.5), (12.5, 40.25), (40.25, 12.5),
                   (0, 40), (40, 0), (M - 1, M), (M, M + 1), (M + 1, M - 1), (10, M), (M, 10), (10, M + 1)):
        want = check_canny(img, t1, t2, oracle=shape[0] < 100)
        if t1 > t2:
            differs += not np.array_equal(want == 0, unswapped_edges(img, t1, t2))
    assert differs >= 4
    for t1, t2 in ((200, 100), (90, 30)):   # the two pairs the swap was found with
        assert not np.array_equal(cv2_inverted(img, t1, t2) == 0, unswapped_edges(img, t1, t2))
    lo, hi, pm = canny_sparse_strong_pair(bl)
    assert 1 <= int((pm == 2).sum()) <= 5 and int((pm == 0).sum()) > 1000
    check_canny(img, lo, hi, oracle=shape[0] < 100)
    check_canny(img, hi, lo, oracle=shape[0] < 100)


@pytest.mark.parametrize("shape", [(436, 1024), (2160, 3840)])
def test_canny_long_chains(shape):
    """Polylines whose contrast falls along their length, so that only one end is strong: spirals, serpentines,
    diagonal and anti-diagonal staircases (joined only through the SE / SW links) and a path along every border."""
    H, W = shape
    big = H * W > 10**6
    for kind in ("spiral", "serpentine", "diagonal", "anti-diagonal", "border"):
        img = canny_polyline_image(H, W, canny_chain_points(H, W, kind, step=6 if not big else 12))
        bl = cv2.GaussianBlur(cv2.cvtColor(img, cv2.COLOR_BGR2GRAY), (3, 3), 0)
        lo, hi, pm = canny_sparse_strong_pair(bl)
        strong = int((pm == 2).sum())
        outs = [check_canny(img, lo, hi, oracle=not big)] + [dev_canny(img, lo, hi) for _ in range(2 if big else 0)]
        for o in outs[1:]:
            assert bitwise_equal(o, outs[0])
        edges = outs[0] == 0
        check_canny(img, hi, lo, oracle=False)
        if kind == "border":
            assert edges[0].any() and edges[-1].any() and edges[:, 0].any() and edges[:, -1].any()
        assert int(edges.sum()) >= 100 * strong, (kind, strong, int(edges.sum()))
        if kind in ("diagonal", "anti-diagonal"):
            from scipy import ndimage
            lab, _ = ndimage.label(pm != 1)          # 4-connected survivors only
            four = np.isin(lab, np.unique(lab[pm == 2]))
            assert int(edges.sum()) >= 50 * int(four.sum()), (kind, int(four.sum()))


def canny_shapes():
    s = [(h, w) for h in range(1, 7) for w in range(1, 7)]
    for n in (255, 256, 257):
        s += [(1, n), (n, 1), (2, n), (n, 2)]
    return s + [(16, 16), (15, 17), (17, 15), (16, 17), (1, 511), (3, 85), (3, 86), (7, 37), (256, 3), (97, 257)]


@pytest.mark.parametrize("shape", canny_shapes())
def test_canny_shapes(shape):
    rng = np.random.default_rng(shape[0] * 1000 + shape[1])
    for it, (t1, t2) in enumerate(((100, 200), (200, 100), (5, 10), (30, 5))):
        img = rng.integers(0, 256, size=shape + (3,), dtype=np.uint8)
        if it % 2:
            img = canny_blurred_noise(rng, *shape)
        check_canny(img, t1, t2)


def test_canny_workspace_and_stream():
    ops, lib = pkg("ops"), pkg("_lib").load()
    rng = np.random.default_rng(9)
    img = canny_blurred_noise(rng, 300, 257)
    ws = torch.full((int(lib.flowb200_edges_workspace_bytes(300, 257)),), 0xFF, dtype=torch.uint8, device="cuda")
    for t1, t2 in ((20, 60), (60, 20)):
        assert bitwise_equal(dev_canny(img, t1, t2, workspace=ws), cv2_inverted(img, t1, t2))
    small = canny_blurred_noise(rng, 61, 45)   # a workspace left over from the larger call
    assert bitwise_equal(dev_canny(small, 20, 60, workspace=ws), cv2_inverted(small, 20, 60))
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        out = ops.canny_edges(torch.from_numpy(img).cuda(), 20, 60)
    s.synchronize()
    assert bitwise_equal(out.cpu().numpy(), cv2_inverted(img, 20, 60))


def canny_call(ov):
    L = pkg("_lib")
    lib = L.load()
    H, W = ov.get("H", 8), ov.get("W", 8)
    img = torch.zeros(8 * 8 * 3, dtype=torch.uint8, device="cuda")
    out = torch.zeros(8 * 8, dtype=torch.float32, device="cuda")
    need = lib.flowb200_edges_workspace_bytes(8, 8)
    ws = torch.zeros(need, dtype=torch.uint8, device="cuda")
    wsb = {None: need, "total-1": need - 1}[ov.get("ws_bytes")]
    p = {k: (None if ov.get("null") == k else t.data_ptr()) for k, t in (("bgr", img), ("out", out), ("ws", ws))}
    rc = lib.flowb200_canny_edges(p["bgr"], H, W, 100, 200, p["out"], p["ws"], wsb, None)
    torch.cuda.synchronize()
    return rc


CANNY_ROWS = [({"null": "bgr"}, "EINVAL"), ({"null": "out"}, "EINVAL"), ({"null": "ws"}, "EINVAL"),
              ({"H": 0}, "EINVAL"), ({"H": -2}, "EINVAL"), ({"W": 0}, "EINVAL"), ({"W": -1}, "EINVAL"),
              ({"H": 65536, "W": 32768}, "EINVAL"), ({"ws_bytes": "total-1"}, "EWORKSPACE"), ({}, "OK")]


@pytest.mark.parametrize("ov,rc", CANNY_ROWS, ids=["-".join(f"{k}={v}" for k, v in r[0].items()) or "defaults"
                                                   for r in CANNY_ROWS])
def test_canny_return_code(ov, rc):
    assert canny_call(ov) == getattr(pkg("_lib"), rc)


def test_canny_workspace_bytes_of_non_positive_sizes():
    lib = pkg("_lib").load()
    for H, W in ((0, 5), (5, 0), (-1, 5), (5, -1), (0, 0)):
        assert lib.flowb200_edges_workspace_bytes(H, W) == 0
