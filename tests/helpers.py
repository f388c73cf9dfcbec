"""Shared test helpers: golden fixture loading and the importable product package."""
import functools
import hashlib
import importlib
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
PKG_NAME = "lk-s-2022-estimacija-pokreta_b200"


def pkg(sub=None):
    return importlib.import_module(PKG_NAME + ("." + sub if sub else ""))


def load_npz(name):
    return dict(np.load(os.path.join(GOLDEN, name + ".npz")))


def digest(a):
    """SHA-256 of an array's dtype, shape and bytes, as uint8 (32,)."""
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str} {a.shape}".encode())
    h.update(a.tobytes())
    return np.frombuffer(h.digest(), dtype=np.uint8)


def ksets_digest(packed, nprop, K):
    """digest of the meaningful K-set bits of a packedksets array (H,W,2,K*K//8+1): pixel p and its down (slot 0) /
    right (slot 1) neighbour q, bits [:nprop[p], :nprop[q]] (oracle.proposals.ksets_masked_equal compares the same)."""
    H, W = nprop.shape
    nq = np.zeros((H, W, 2), np.int64)
    nq[:-1, :, 0] = nprop[1:, :]
    nq[:, :-1, 1] = nprop[:, 1:]
    k = np.arange(K)
    mask = (k[:, None] < nprop[:, :, None, None, None]) & (k[None, :] < nq[..., None, None])
    bits = np.unpackbits(packed, axis=-1)[..., :K * K].reshape(H, W, 2, K, K)
    return digest(np.packbits(bits[mask]))


@functools.lru_cache(maxsize=None)
def _case(name):
    z = load_npz(name)
    out = {}
    for k, v in z.items():
        base = k.split("_", 1)[1] if k[:1] == "b" and k[1:2].isdigit() else k
        if base.endswith("_sha256"):
            continue
        if base in ("proposals", "nprop", "labels00", "draws") or base.startswith("labels"):
            out[k] = v.astype(np.int64)
        elif base == "lcosts" or base.startswith("flow"):
            out[k] = v.astype(np.float64)
        else:
            out[k] = v
    # The reference's stage-1 proposals, costs and K-set bits are stored as digests (the arrays would exceed the
    # fixture size): the oracle recomputes them from the stored descriptors and Gaussian draws, and they must be the
    # reference's bit for bit.
    from oracle import proposals as oprop
    p = oracle_params(out["meta"])
    for b in (0, 1):
        if f"b{b}_proposals_sha256" not in z:
            continue
        d1, d2 = (out["desc1"], out["desc2"]) if b == 0 else (out["desc2"], out["desc1"])
        P, L, N, B = oprop.generisi(d1, d2, p)
        oprop.nasumicni(d1, d2, P, L, N, B, p, out[f"b{b}_draws"])
        pk = oprop.pakovanje(P, N, p)
        for key, ok in (("proposals", np.array_equal(digest(P), z[f"b{b}_proposals_sha256"])),
                        ("lcosts", np.array_equal(digest(L), z[f"b{b}_lcosts_sha256"])),
                        ("nprop", np.array_equal(N, out[f"b{b}_nprop"])),
                        ("packedksets", np.array_equal(ksets_digest(pk, N, p.maxnprop), z[f"b{b}_packedksets_sha256"]))):
            assert ok, f"{name} b{b}_{key}: the oracle's stage 1 differs from the reference's output"
        out.update({f"b{b}_proposals": P, f"b{b}_lcosts": L, f"b{b}_packedksets": pk})
    return out


def load_case(name):
    """Restore the reference dtypes (int64 proposals / nprop / labels, float64 lcosts / flows).  The stage-1 proposals,
    costs and K-set bits are recomputed and checked against the reference's digests once per process (_case)."""
    return {k: v.copy() for k, v in _case(name).items()}


def oracle_params(meta, **kw):
    from oracle.proposals import Params
    H, W, cw, ch = (int(v) for v in meta[:4])
    return Params(H, W, cw, ch, **kw)


def segment_test_field(rng, A, B, kind):
    """float32 (A,B,3) = (dx, dy, valid) fields that exercise removeSmallSegments (postprocessing.py:29-76):
    small islands on piecewise constant / smooth flow, invalid pixels with zeroed or with stale flow, pure noise."""
    f = np.zeros((A, B, 3), np.float32)
    if kind == "blocks":
        ba, bb = int(rng.integers(3, 9)), int(rng.integers(3, 9))
        base = rng.integers(-20, 21, size=((A + ba - 1) // ba, (B + bb - 1) // bb, 2)) * 3
        f[..., :2] = np.repeat(np.repeat(base, ba, 0), bb, 1)[:A, :B] + rng.integers(-1, 2, size=(A, B, 2))
        f[..., 2] = 1
        f[rng.random((A, B)) < 0.08] = 0
    elif kind == "noise":
        f[..., :2] = rng.normal(0, 6, size=(A, B, 2))
        f[..., 2] = rng.random((A, B)) < 0.9
    elif kind == "smooth":
        a = np.arange(A)[:, None]
        b = np.arange(B)[None, :]
        f[..., 0] = 5 * np.sin(a / 7.0) + 0.3 * b
        f[..., 1] = 4 * np.cos(b / 5.0)
        f[..., 2] = 1
        for _ in range(int(rng.integers(3, 12)) * max(1, A * B // 2000)):
            a0, b0 = int(rng.integers(0, max(1, A - 3))), int(rng.integers(0, max(1, B - 3)))
            h, w = int(rng.integers(1, 6)), int(rng.integers(1, 6))
            f[a0:a0 + h, b0:b0 + w, :2] += rng.integers(15, 40)
        f[rng.random((A, B)) < 0.03] = 0
    elif kind == "stale":
        f[..., :2] = rng.integers(-4, 5, size=(A, B, 2)) * 2
        f[..., 2] = rng.random((A, B)) < 0.7      # invalid pixels keep their flow values
    else:
        raise ValueError(kind)
    return f


SEGMENT_KINDS = ("blocks", "noise", "smooth", "stale")


def seg_restated(flow, tresh, min_segment_size):
    """removeSmallSegments (postprocessing.py:29-76) restated in plain Python on a copy of flow, plus its removal
    events.  float32 flow differences compared with tresh in float32, `count > 1 and count < min_segment_size` with
    the bound as given (int or float).  Returns (flow, events); an event is (seed, last, column_before, column_after)
    with seed and last as (row, column): the removal loop (:74) leaves the scan's column at the last pixel's."""
    f = np.array(flow, dtype=np.float32, copy=True)
    A, B = f.shape[:2]
    t = np.float32(tresh)
    check = np.zeros((A, B), dtype=bool)
    events = []
    with np.errstate(invalid="ignore", over="ignore"):
        for bo in range(B):
            b = bo
            for a in range(A):
                if check[a, b]:
                    continue
                q, curr = [(a, b)], 0
                while curr < len(q):
                    ca, cb = q[curr]
                    fc = f[ca, cb]
                    for na, nb in ((ca - 1, cb), (ca + 1, cb), (ca, cb - 1), (ca, cb + 1)):
                        if na < 0 or nb < 0 or na >= A or nb >= B or check[na, nb] or not f[na, nb, 2] > 0.5:
                            continue
                        fm = f[na, nb]
                        if abs(fc[0] - fm[0]) + abs(fc[1] - fm[1]) <= t:
                            q.append((na, nb))
                            check[na, nb] = True
                    curr += 1
                    check[ca, cb] = True
                count = len(q)
                if count > 1 and count < min_segment_size:
                    for u, v in q:
                        f[u, v, 2] = 0
                    events.append(((a, b), q[-1], b, q[-1][1]))
                    b = q[-1][1]
    return f, events


def seg_singletons(A, B):
    """All valid, every pixel its own segment at tresh < 100: a background on which planted segments act alone."""
    f = np.zeros((A, B, 3), np.float32)
    f[..., 0] = 100.0 * np.arange(A * B, dtype=np.float32).reshape(A, B)
    f[..., 2] = 1
    return f


def seg_paint(f, pixels, dx, dy=0.0, valid=1.0):
    for a, b in pixels:
        f[a, b] = (dx, dy, valid)
    return f


def seg_rebind_cases():
    """Fields on the singleton background (tresh 1, min size 100) with planted removals whose last breadth-first
    pixel moves the scan: name -> (field, [(seed, column_after), ...]) with every listed event expected."""
    A, B = 70, 12
    cases = {}
    for r in (0, 31, 32, A - 1):
        if r < A - 1:   # a column segment ends in its own column; below the last row there is nothing
            cases[f"same-r{r}"] = (seg_paint(seg_singletons(A, B), [(r, 4), (r + 1, 4)], -7), [((r, 4), 4)])
        cases[f"later-r{r}"] = (seg_paint(seg_singletons(A, B), [(r, 4), (r, 5), (r, 6)], -7), [((r, 4), 6)])
        cases[f"last-column-r{r}"] = (seg_paint(seg_singletons(A, B), [(r, b) for b in range(3, B)], -7),
                                      [((r, 3), B - 1)])
    for r1, r2 in ((0, 31), (0, 32), (31, 32), (32, A - 1), (0, 1)):
        for c in (0, 5):
            # column c is left at row r1 for column c+2; column c+1's seed at r2 reaches back into column c
            f = seg_singletons(A, B)
            seg_paint(f, [(r1, c), (r1, c + 1), (r1, c + 2)], -7)
            seg_paint(f, [(r2, c + 1), (r2, c)], -9)
            name = "column-0" if c == 0 else "earlier"
            cases[f"{name}-r{r1}-r{r2}"] = (f, [((r1, c), c + 2), ((r2, c + 1), c)])
    for rows in ((0, 1), (30, 31), (31, 32), (5, 69), (0, 1, 2), (31, 32, 63), (2, 40, 64)):
        # a chain: every removal lands in a column whose next seed (below the row the scan resumes at) removes again
        f = seg_singletons(A, B)
        want = []
        for k, r in enumerate(rows):
            c = 1 + 3 * k
            seg_paint(f, [(r, c), (r, c + 1), (r, c + 2), (r, c + 3)], -7 - 2 * k)
            want.append(((r, c), c + 3))
        cases["chain-" + "-".join(map(str, rows))] = (f, want)
    return cases


SEG_INVALID_MIN = 12


def seg_invalid_seed_cases():
    """An invalid seed with stale flow -7 absorbing near neighbouring segments (tresh 1, min size SEG_INVALID_MIN):
    name -> (field, seed, number of pixels the seed's fill takes)."""
    A, B = 40, 9
    cases = {}

    def land(f, r, c):
        # a removal in column 1 whose last pixel lies in column c, so the scan resumes at (r, c) with all four
        # neighbours of (r, c) not yet visited (rows 0..r-1 of column c and column c-1 are still unscanned)
        path = [(r - 1, 1)] + [(a, 1) for a in range(r, r + 3)] + [(r + 2, b) for b in range(2, c + 1)]
        return seg_paint(f, path, -50, 0, 1)

    r, c = 20, 5
    nb = {"up": (r - 1, c), "down": (r + 1, c), "left": (r, c - 1), "right": (r, c + 1)}
    for k in range(5):
        f = land(seg_singletons(A, B), r, c)
        seg_paint(f, [(r, c)], -7, 0, 0)
        for d in list(nb)[:k]:
            seg_paint(f, [nb[d]], -7.5)
        cases[f"absorbs-{k}"] = (f, (r, c), 1 + k)
    f = land(seg_singletons(A, B), r, c)   # one segment reached through up and right
    seg_paint(f, [(r, c)], -7, 0, 0)
    seg_paint(f, [(r - 1, c), (r - 1, c + 1), (r, c + 1)], -7.5)
    cases["one-segment-two-ways"] = (f, (r, c), 4)
    f = land(seg_singletons(A, B), r, c)   # ... through up, right and down
    seg_paint(f, [(r, c)], -7, 0, 0)
    seg_paint(f, [(r - 1, c), (r - 1, c + 1), (r, c + 1), (r + 1, c + 1), (r + 1, c)], -7.5)
    cases["one-segment-three-ways"] = (f, (r, c), 6)
    f = seg_singletons(A, B)               # the up neighbour's segment was taken by its own seed
    seg_paint(f, [(r, c)], -7, 0, 0)
    seg_paint(f, [(r - 1, c), (r - 2, c)], -7.5)
    seg_paint(f, [(r + 1, c), (r + 2, c)], -7.5)
    seg_paint(f, [(r + 2, c + 1)], -30)
    cases["up-already-taken"] = (f, (r, c), 3)
    for name, (sr, sc) in {"corner-00": (0, 0), "corner-0B": (0, B - 1), "corner-A0": (A - 1, 0),
                           "corner-AB": (A - 1, B - 1), "edge-top": (0, 4), "edge-bottom": (A - 1, 4),
                           "edge-left": (17, 0), "edge-right": (17, B - 1)}.items():
        f = seg_singletons(A, B)
        seg_paint(f, [(sr, sc)], -7, 0, 0)
        taken = 1
        for a, b in ((sr + 1, sc), (sr, sc + 1)):   # the neighbours the scan has not passed yet
            if a < A and b < B:
                seg_paint(f, [(a, b)], -7.5)
                taken += 1
        cases[name] = (f, (sr, sc), taken)
    # an absorbed total of exactly min_size - 1 (removed) and exactly min_size (kept)
    for total in (SEG_INVALID_MIN - 1, SEG_INVALID_MIN):
        f = seg_singletons(A, B)
        seg_paint(f, [(r, c)], -7, 0, 0)
        seg_paint(f, [(r + 1 + i, c) for i in range(total - 1 - 2)], -7.5)
        seg_paint(f, [(r, c + 1), (r, c + 2)], -6.5)
        cases[f"total-{total}"] = (f, (r, c), total)
    return cases


def seg_prefilter_cases(min_size=10):
    """Segments of 1, 2, min-1, min, min+1 pixels (flow -7, tresh 1) with and without a near invalid 4-neighbour
    scanned before them, and an invalid pixel near in one direction only: name -> (field, segment pixels, removed)."""
    A, B = 30, 40
    cases = {}
    for n in (1, 2, min_size - 1, min_size, min_size + 1):
        pix = [(10, 3 + i) for i in range(n)]
        for near in (False, True):
            f = seg_singletons(A, B)
            seg_paint(f, pix, -7)
            total = n
            if near:
                seg_paint(f, [(9, 3)], -7.25, 0, 0)   # invalid, scanned first in column 3, absorbs the segment
                total += 1
            cases[f"size-{n}-{'near' if near else 'alone'}"] = (f, pix, 1 < total < min_size)
    # an invalid pixel near its down neighbour's segment (absorbed: 1 + min-1 pixels, kept) and not near its right
    # neighbour's (flow -20, removed by its own seed)
    f = seg_singletons(A, B)
    below = [(11, 1 + i) for i in range(min_size - 1)]
    right = [(10, 2 + i) for i in range(min_size - 1)]
    seg_paint(f, below, -7)
    seg_paint(f, right, -20)
    seg_paint(f, [(10, 1)], -7.5, 0, 0)
    cases["near-one-direction-absorbed"] = (f, below, False)
    cases["near-one-direction-other"] = (f, right, True)
    return cases


def seg_value_fields(rng, A, B):
    """Small fields made of special values: +-0, NaN, +-inf, 1e30 flows and the valid flags around 0.5."""
    flows = np.array([0.0, -0.0, 1.0, -1.0, 0.5, np.nan, np.inf, -np.inf, 1e30, 3.0, 2.999999], np.float32)
    flags = np.array([1.0, 0.0, 0.5, np.nextafter(np.float32(0.5), np.float32(1)), np.nan, -1.0, 2.0, 1e30],
                     np.float32)
    f = np.empty((A, B, 3), np.float32)
    f[..., 0] = rng.choice(flows[:5], size=(A, B)) if rng.random() < 0.5 else rng.choice(flows, size=(A, B))
    f[..., 1] = np.where(rng.random((A, B)) < 0.8, np.float32(0), rng.choice(flows, size=(A, B)))
    f[..., 2] = np.where(rng.random((A, B)) < 0.6, np.float32(1), rng.choice(flags, size=(A, B)))
    # a NaN with a payload and a negative NaN must come back bit for bit wherever they are not removed
    bits = f.view(np.uint32)
    nan = np.isnan(f)
    bits[nan] = np.where(rng.random(int(nan.sum())) < 0.5, np.uint32(0x7fc0beef), np.uint32(0xffc00001))
    return f


def bitwise_equal(x, y):
    x, y = np.ascontiguousarray(x), np.ascontiguousarray(y)
    return x.shape == y.shape and x.dtype == y.dtype and np.array_equal(x.view(np.uint8), y.view(np.uint8))


def canny_blurred_noise(rng, H, W):
    """uint8 BGR noise blurred so that most survivors are weak: the threshold order changes the edge map here."""
    img = rng.integers(0, 256, size=(H, W, 3), dtype=np.uint8)
    return __import__("cv2").GaussianBlur(img, (3, 3), 1.0) if min(H, W) > 1 else img


def canny_polyline_image(H, W, pts, v0=250, v1=40):
    """One 8-connected polyline on black whose grey level falls from v0 to v1 along its length: with a high threshold
    only near its bright end, every other edge pixel of it is reached by hysteresis alone."""
    import cv2
    img = np.zeros((H, W, 3), np.uint8)
    n = len(pts) - 1
    for i in range(n):
        v = int(round(v0 + (v1 - v0) * i / max(n - 1, 1)))
        cv2.line(img, tuple(map(int, pts[i])), tuple(map(int, pts[i + 1])), (v, v, v), 1, cv2.LINE_8)
    return img


def canny_chain_points(H, W, kind, step=6, margin=3):
    """(x, y) vertices of a spiral, a serpentine, a diagonal / anti-diagonal staircase or a path along every border."""
    if kind == "spiral":
        pts, x0, y0, x1, y1 = [], 0, 0, W - 1, H - 1
        while x1 - x0 > 2 * step and y1 - y0 > 2 * step:
            pts += [(x0, y0), (x1, y0), (x1, y1), (x0, y1)]
            x0, y0, x1, y1 = x0 + step, y0 + step, x1 - step, y1 - step
            pts.append((x0 - step, y0))
        return pts
    if kind == "serpentine":
        pts, y, right = [], margin, True
        while y < H - margin:
            pts += [(margin, y), (W - 1 - margin, y)] if right else [(W - 1 - margin, y), (margin, y)]
            right, y = not right, y + step
        return pts
    n = min(H, W) - 1
    if kind == "diagonal":
        return [(0, 0), (n, n)]
    if kind == "anti-diagonal":
        return [(W - 1, 0), (W - 1 - n, n)]
    if kind == "border":
        return [(1, 1), (W - 2, 1), (W - 2, H - 2), (1, H - 2), (1, 3), (W // 2, H // 2)]
    raise ValueError(kind)


def canny_pmap(bl, low, high):
    """The oracle's survivor map {1 none, 0 weak, 2 strong} with low and high used exactly as given."""
    from oracle import edges as oe
    dx, dy = oe.sobel3(bl)
    return oe.nms_map(dx, dy, int(np.floor(low)), int(np.floor(high)))


def canny_sparse_strong_pair(bl, nstrong=5, low=5):
    """A (low, high) pair from the image's magnitude histogram, at most `nstrong` survivors above high, and the
    survivor map at that pair."""
    from oracle import edges as oe
    dx, dy = oe.sobel3(bl)
    mag = (np.abs(dx) + np.abs(dy))[oe.nms_map(dx, dy, 0, 1 << 30) != 1]
    m = np.sort(mag)[::-1]
    high = int(m[nstrong]) if len(m) > nstrong else 0
    return low, high, oe.nms_map(dx, dy, low, high)
