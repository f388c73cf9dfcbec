"""The per-pixel kernels before and after the search and BCD, at the edges where such kernels go wrong.  GPU only.

  DAISY (`daisy.cu`)            bit for bit against oracle/daisy.py at every tile geometry of the 32 x 16 gray / blur
                                tiles and the 32 x 8 sampler tiles (halo 6), on images aimed at its arithmetic, with an
                                unwritten workspace, at its argument limits and on another stream;
  label -> flow (`post.cu`)     the extremes of the 16-bit vector packing, the first and the last slot, one output only;
  consistency (`post.cu`)       planted values (truncation toward zero, float32 sums that round to the next integer,
                                the threshold, the valid flags, non-finite flows) and sub-rectangles, against
                                oracle/consistency.py;
  EPE (`post.cu`)               counts exact and the sum against an exactly rounded sum, around the grid stride;
  energy (`bcd_ksets.cu`)       every mode against exact integer sums / an exactly rounded float64 sum, sums above 2^32.
"""
import ctypes as C
import math

import numpy as np
import pytest

from helpers import pkg

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

F32 = np.float32


def dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda()


def ptr(t):
    return C.c_void_p(t.data_ptr())


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def bits(a):
    """float32 array -> its bit patterns, so that equality is bit for bit (NaN == NaN, -0.0 != 0.0)."""
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


# ---------------------------------------------------------------- DAISY (A2), bit for bit
DAISY_H = (3, 4, 5, 6, 7, 8, 9, 15, 16, 17, 23, 24, 25, 31, 32, 33, 47, 48, 49)
DAISY_W = (3, 4, 5, 6, 7, 11, 12, 13, 31, 32, 33, 63, 64, 65, 95, 96, 97)


def assert_daisy_exact(img, what, got=None):
    from oracle import daisy as od
    want = od.daisy(img)
    if got is None:
        got = pkg("ops").daisy(dev(img)).cpu().numpy()
    if not np.array_equal(got, want):        # NaN (an unwritten output) never compares equal
        diff = np.argwhere(~(got == want))
        y, x, d = diff[0]
        raise AssertionError(f"{what}: {len(diff)} descriptor entries differ, the first at y={y} x={x} entry {d}: "
                             f"{got[y, x, d]!r} instead of {want[y, x, d]!r}")


def noise(H, W):
    return np.random.default_rng(1000 * H + W).integers(0, 256, (H, W, 3), dtype=np.uint8)


@pytest.mark.parametrize("H", DAISY_H)
def test_daisy_bit_identical_at_every_tile_geometry(H):
    """Frames smaller than a tile and than the sampler's halo, one pixel either side of every tile seam."""
    for W in DAISY_W:
        assert_daisy_exact(noise(H, W), f"{H}x{W}")


@pytest.mark.parametrize("H,W", [(3, 4099), (4099, 3)])
def test_daisy_bit_identical_on_long_grids(H, W):
    assert_daisy_exact(noise(H, W), f"{H}x{W}")


def test_daisy_constant_images_give_zero_descriptors():
    for v in (0, 128, 255):
        img = np.full((37, 70, 3), v, np.uint8)
        got = pkg("ops").daisy(dev(img)).cpu().numpy()
        assert not got.any(), v
        assert_daisy_exact(img, f"constant {v}", got)


def test_daisy_checkerboard_and_steps_on_tile_seams():
    """A 0/255 checkerboard, and steps through the point (row 16, column 32), where the seams of every kernel's tiles
    meet: vertical, horizontal (also at the sampler's row seam 8) and both diagonals, each in both polarities, so that
    every orientation layer goes through its rectification on both sides."""
    H, W = 48, 72
    y, x = np.mgrid[0:H, 0:W]
    masks = {"checkerboard": (y + x) % 2 == 1,
             "vertical": x >= 32, "horizontal16": y >= 16, "horizontal8": y >= 8,
             "diagonal": (y - 16) >= (x - 32), "antidiagonal": (y - 16) + (x - 32) >= 0}
    for name, m in masks.items():
        for hi, lo in ((255, 0), (0, 255)):
            img = np.where(m[..., None], hi, lo).astype(np.uint8).repeat(3, axis=2)
            assert_daisy_exact(img, f"{name} {hi}/{lo}")


def test_daisy_impulses_around_seams_and_corners_per_channel():
    """One bright pixel in B, G or R only (the 3735 / 19235 / 9798 gray weights and the channel order) at every offset
    -6..+6 around the column seam 32 and the row seams 8, 16 and 32, and at the four corners."""
    H, W = 48, 72
    spots = [(20, 32 + d) for d in range(-6, 7)]
    spots += [(r + d, 20) for r in (8, 16, 32) for d in range(-6, 7)]
    spots += [(0, 0), (0, W - 1), (H - 1, 0), (H - 1, W - 1)]
    for y, x in spots:
        for ch in range(3):
            img = np.zeros((H, W, 3), np.uint8)
            img[y, x, ch] = 255
            assert_daisy_exact(img, f"impulse at ({y}, {x}) channel {ch}")


def test_daisy_unwritten_workspace_and_every_output_written():
    """Through the C ABI with a workspace of exactly flowb200_daisy_workspace_bytes filled with 0xFF (NaN as float) and
    the descriptors filled with NaN: nothing unwritten is read, every descriptor entry is written."""
    lib = pkg("_lib")
    L = lib.load()
    for H, W in ((3, 3), (17, 33), (49, 97)):
        img = noise(H, W)
        nb = L.flowb200_daisy_workspace_bytes(H, W)
        ws = torch.full((nb,), 0xFF, dtype=torch.uint8, device="cuda")
        desc = torch.full((H, W, 68), float("nan"), dtype=torch.float32, device="cuda")
        g = dev(img)
        assert L.flowb200_daisy(ptr(g), H, W, ptr(desc), ptr(ws), nb, stream()) == lib.OK
        assert_daisy_exact(img, f"{H}x{W} in a 0xFF workspace", desc.cpu().numpy())


def test_daisy_argument_limits():
    lib = pkg("_lib")
    L = lib.load()
    H, W = 8, 8
    g = dev(noise(H, W))
    nb = L.flowb200_daisy_workspace_bytes(H, W)
    ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
    desc = torch.full((H, W, 68), float("nan"), dtype=torch.float32, device="cuda")
    for h, w in [(v, W) for v in (-1, 0, 1, 2)] + [(H, v) for v in (-1, 0, 1, 2)]:
        assert L.flowb200_daisy(ptr(g), h, w, ptr(desc), ptr(ws), nb, stream()) == lib.EINVAL, (h, w)
    assert L.flowb200_daisy(ptr(g), H, W, ptr(desc), ptr(ws), nb - 1, stream()) == lib.EWORKSPACE
    torch.cuda.synchronize()
    assert torch.isnan(desc).all()                     # the refused calls launched nothing
    assert L.flowb200_daisy(ptr(g), H, W, ptr(desc), ptr(ws), nb, stream()) == lib.OK
    assert_daisy_exact(noise(H, W), "8x8 in a workspace of exactly the size asked for", desc.cpu().numpy())


def test_daisy_on_a_side_stream():
    ops = pkg("ops")
    img = noise(49, 97)
    want = ops.daisy(dev(img)).cpu().numpy()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        got = ops.daisy(dev(img))
    s.synchronize()
    assert np.array_equal(got.cpu().numpy(), want)
    assert_daisy_exact(img, "side stream", got.cpu().numpy())


# ---------------------------------------------------------------- label -> flow (A5)
@pytest.mark.parametrize("K", [1, 7, 512])
def test_flow_from_labels_packing_extremes(K):
    """Every (dy, dx) pair of {-32768, -1, 0, 1, 32767} at slot 0 and at slot K-1; 273 pixels (not a multiple of 256).
    flow_yx = float64 (dy, dx), uvv = float32 (dx, dy, 1) exactly; with one output pointer null the other buffer is
    written in full."""
    lib = pkg("_lib")
    L = lib.load()
    H, W = 13, 21
    n = H * W
    ext = np.array([-32768, -1, 0, 1, 32767])
    rng = np.random.default_rng(K)
    dy = rng.choice(ext, (n, K))
    dx = rng.choice(ext, (n, K))
    labels = rng.integers(0, K, n)
    for i, (a, b) in enumerate((a, b) for a in ext for b in ext):
        dy[i, 0], dx[i, 0], labels[i] = a, b, 0
        dy[n - 1 - i, K - 1], dx[n - 1 - i, K - 1], labels[n - 1 - i] = a, b, K - 1
    pvec = ((dy & 0xFFFF) | ((dx & 0xFFFF) << 16)).astype(np.uint32).view(np.int32).reshape(H, W, K)
    sy, sx = dy[np.arange(n), labels].reshape(H, W), dx[np.arange(n), labels].reshape(H, W)
    want_yx = np.stack([sy, sx], -1).astype(np.float64)
    want_uvv = np.stack([sx, sy, np.ones_like(sx)], -1).astype(np.float32)
    gp, gl = dev(pvec), dev(labels.reshape(H, W), torch.int32)
    yx, uvv = pkg("ops").flow_from_labels(gp, gl)
    assert np.array_equal(yx.cpu().numpy(), want_yx)
    assert np.array_equal(bits(uvv.cpu().numpy()), bits(want_uvv))
    for keep in ("yx", "uvv"):
        yx = torch.full((H, W, 2), -7.5, dtype=torch.float64, device="cuda")
        uvv = torch.full((H, W, 3), -7.5, dtype=torch.float32, device="cuda")
        rc = L.flowb200_flow_from_labels(ptr(gp), ptr(gl), H, W, K, ptr(yx) if keep == "yx" else None,
                                         ptr(uvv) if keep == "uvv" else None, stream())
        assert rc == lib.OK
        if keep == "yx":
            assert np.array_equal(yx.cpu().numpy(), want_yx)
            assert (uvv == -7.5).all()
        else:
            assert np.array_equal(bits(uvv.cpu().numpy()), bits(want_uvv))
            assert (yx == -7.5).all()


# ---------------------------------------------------------------- consistency (A12-A14)
CONS_SHAPES = [(7, 300), (300, 7), (1, 300), (300, 1), (40, 53)]


def cons_oracle(f1, f2, tresh):
    from oracle import consistency as ocons
    with np.errstate(invalid="ignore", over="ignore"):      # NaN / inf -> int64: out of range, as intended
        return ocons.forward_backward_consistency(f1, f2, tresh)


def cons_device(f1, f2, tresh, region=None):
    g1 = dev(f1)
    pkg("ops").consistency(g1, dev(f2), tresh, region)
    return g1.cpu().numpy()


def cons_host(f1, f2, tresh, region):
    lib = pkg("_lib")
    h1 = np.array(f1, np.float32, copy=True)
    h2 = np.ascontiguousarray(f2, np.float32)
    A, B, _ = h1.shape
    lib.check(lib.load().flowb200_consistency_host(h1.ctypes.data, h2.ctypes.data, A, B, float(tresh), *region),
              "flowb200_consistency_host")
    return h1


def random_fields(rng, A, B, spread=3.0):
    f1 = np.zeros((A, B, 3), np.float32)
    f2 = np.zeros((A, B, 3), np.float32)
    f1[..., :2] = rng.normal(0, spread, (A, B, 2))
    f2[..., :2] = rng.normal(0, spread, (A, B, 2))
    f1[..., 2] = rng.random((A, B)) > 0.1
    f2[..., 2] = rng.random((A, B)) > 0.1
    return f1, f2


def assert_cons_equal(got, want, what):
    if not np.array_equal(bits(got), bits(want)):
        a, b = np.argwhere((bits(got) != bits(want)).any(-1))[0]
        raise AssertionError(f"{what}: pixel ({a}, {b}) is {got[a, b]} instead of {want[a, b]}")


@pytest.mark.parametrize("A,B", CONS_SHAPES)
def test_consistency_truncation_and_rounding_at_the_borders(A, B):
    """u in {-1, -0.99999994, -0.0, 0.99999994} along rows 0, 3 and A-1 (dx goes to the row index, quirk Q5), v likewise
    along columns 0, 3 and B-1: int() truncates (-0.99999994 stays in row 0), and 3 + 0.99999994f = 4.0f, A-1 +
    0.99999994f = A (out of range) in float32."""
    rng = np.random.default_rng(A * 7 + B)
    f1, f2 = random_fields(rng, A, B)
    U = np.array([-1.0, np.nextafter(F32(-1), F32(0)), -0.0, np.nextafter(F32(1), F32(0))], np.float32)
    for r in sorted({0, 3, A - 1} & set(range(A))):
        f1[r, :, 0] = U[np.arange(B) % 4]
        f1[r, :, 1] = 0
        f1[r, :, 2] = 1
    for c in sorted({0, 3, B - 1} & set(range(B))):
        f1[:, c, 1] = U[np.arange(A) % 4]
        f1[:, c, 0] = 0
        f1[:, c, 2] = 1
    f2[..., 2] = 1
    f2[..., :2] = 0.25                    # every in-range target passes at tresh 5: only the range decides
    want = cons_oracle(f1, f2, 5.0)
    assert_cons_equal(cons_device(f1, f2, 5.0), want, f"{A}x{B}")
    # what the planted rows mean, on columns no column planting overwrote
    cols = np.array([j for j in range(B) if j not in (0, 3, B - 1)], dtype=np.int64)
    if len(cols):
        k = cols % 4
        assert (want[0, cols[k == 0], 2] == 0).all()             # 0 + -1: row -1
        assert (want[0, cols[k == 1], 2] == 1).all()             # 0 + -0.99999994 truncates to row 0
        if A > 4:
            assert (want[3, cols[k == 3], 2] == 1).all()         # 3 + 0.99999994f = 4.0f: row 4
        if A > 1:
            assert (want[A - 1, cols[k == 3], 2] == 0).all()     # A-1 + 0.99999994f = A: out of range


def test_consistency_error_exactly_at_the_threshold():
    """(du, dv) = (+-3, +-4): err = 5 exactly.  Not bad at tresh 5.0, bad at the float32 below it."""
    rng = np.random.default_rng(1)
    A, B = 7, 300
    f1 = np.zeros((A, B, 3), np.float32)
    f1[..., 2] = 1                                       # u = v = 0: every pixel checks itself
    f2 = np.ones((A, B, 3), np.float32)
    f2[..., 0] = rng.choice([-3.0, 3.0], (A, B))
    f2[..., 1] = rng.choice([-4.0, 4.0], (A, B))
    for tresh, kept in ((5.0, True), (float(np.nextafter(F32(5), F32(0))), False)):
        got = cons_device(f1, f2, tresh)
        assert_cons_equal(got, cons_oracle(f1, f2, tresh), f"tresh {tresh!r}")
        assert (got[..., 2] == (1.0 if kept else 0.0)).all(), tresh


@pytest.mark.parametrize("A,B", CONS_SHAPES)
def test_consistency_valid_flags(A, B):
    """flow1 valid flags and flow2 target flags of 0.5 (not valid: the test is > 0.5), nextafter(0.5, 1), -1 and NaN."""
    rng = np.random.default_rng(A + 3 * B)
    f1, f2 = random_fields(rng, A, B, spread=0.8)
    flags = np.array([0.5, np.nextafter(F32(0.5), F32(1)), -1.0, np.nan], np.float32)
    f1[..., 2] = np.where(rng.random((A, B)) < 0.5, flags[rng.integers(0, 4, (A, B))], 1.0)
    f2[..., 2] = np.where(rng.random((A, B)) < 0.5, flags[rng.integers(0, 4, (A, B))], 1.0)
    assert_cons_equal(cons_device(f1, f2, 1.5), cons_oracle(f1, f2, 1.5), f"{A}x{B}")


@pytest.mark.parametrize("A,B", CONS_SHAPES)
def test_consistency_non_finite_flows(A, B):
    """u or v in {NaN, +inf, -inf, +-1e10} at valid pixels: the target is out of range and the pixel is zeroed.  For
    NaN that is a deliberate difference (the reference's int() raises): a float-to-int conversion on the device turns NaN
    into 0, which used to keep such a pixel valid with a NaN flow.  A NaN flow in flow2 at a valid target leaves err NaN,
    `err > tresh` false and the pixel kept, on both sides."""
    rng = np.random.default_rng(11 * A + B)
    f1, f2 = random_fields(rng, A, B)
    vals = np.array([np.nan, np.inf, -np.inf, 1e10, -1e10], np.float32)
    n = A * B
    which = rng.permutation(n)
    pu, pv, p2 = which[:n // 5], which[n // 5:2 * n // 5], which[2 * n // 5:3 * n // 5]
    f1.reshape(n, 3)[pu, 0] = vals[np.arange(len(pu)) % 5]
    f1.reshape(n, 3)[pv, 1] = vals[np.arange(len(pv)) % 5]
    f1.reshape(n, 3)[np.concatenate([pu, pv]), 2] = 1
    # a NaN in flow2 at a valid target: f1 points at itself, f2 there is (NaN, 0, 1) or (0, NaN, 1)
    f1.reshape(n, 3)[p2] = (0, 0, 1)
    f2.reshape(n, 3)[p2] = (0, 0, 1)
    f2.reshape(n, 3)[p2[::2], 0] = np.nan
    f2.reshape(n, 3)[p2[1::2], 1] = np.nan
    want = cons_oracle(f1, f2, 4.0)
    assert (want.reshape(n, 3)[np.concatenate([pu, pv])] == 0).all()
    assert_cons_equal(want.reshape(n, 3)[p2], f1.reshape(n, 3)[p2], "oracle: NaN in flow2 keeps the pixel")
    assert_cons_equal(cons_device(f1, f2, 4.0), want, f"{A}x{B} device")
    assert_cons_equal(cons_host(f1, f2, 4.0, (0, A, 0, B)), want, f"{A}x{B} host")
    h1 = f1.copy()
    pkg("postprocessing").fowardBackwardConsistency(h1, f2, 4.0)
    assert_cons_equal(h1, want, f"{A}x{B} postprocessing.fowardBackwardConsistency")


def test_consistency_sub_rectangles():
    """flowb200_consistency on a region: pixels outside keep their bits, pixels inside equal the full-frame oracle
    (pixels are independent: only flow1 is written, only flow2 is read); the host entry point agrees, and so does
    postprocessing.consistencyCheck, which checks one pixel through the region path."""
    rng = np.random.default_rng(5)
    A, B = 37, 211
    f1, f2 = random_fields(rng, A, B, spread=2.0)
    f2[..., :2] = -f1[..., :2] + rng.normal(0, 1.5, (A, B, 2)).astype(np.float32)
    tresh = 2.5
    full = cons_oracle(f1, f2, tresh)
    assert 0 < (full[..., 2] != f1[..., 2]).sum() < (f1[..., 2] > 0.5).sum()     # some zeroed, some kept
    regions = [(0, A, 0, B), (5, 6, 0, B), (0, A, 17, 18), (A - 1, A, B - 1, B), (0, 1, 0, 1), (12, 13, 100, 101)]
    while len(regions) < 22:
        a0, a1 = sorted(rng.integers(0, A + 1, 2))
        b0, b1 = sorted(rng.integers(0, B + 1, 2))
        if a1 > a0 and b1 > b0:
            regions.append((int(a0), int(a1), int(b0), int(b1)))
    for a0, a1, b0, b1 in regions:
        want = f1.copy()
        want[a0:a1, b0:b1] = full[a0:a1, b0:b1]
        assert_cons_equal(cons_device(f1, f2, tresh, (a0, a1, b0, b1)), want, f"device region {(a0, a1, b0, b1)}")
        assert_cons_equal(cons_host(f1, f2, tresh, (a0, a1, b0, b1)), want, f"host region {(a0, a1, b0, b1)}")
    post = pkg("postprocessing")
    for a, b in ((0, 0), (A - 1, B - 1), (12, 100), (30, 3)):
        h1 = f1.copy()
        post.consistencyCheck(h1, f2, a, b, tresh)
        want = f1.copy()
        want[a, b] = full[a, b]
        assert_cons_equal(h1, want, f"consistencyCheck at {(a, b)}")


# ---------------------------------------------------------------- EPE metric (visualization.errorImage)
def epe_device(t, g, thresh):
    """flowb200_epe's raw accumulators (sum of errors, outliers, valid) through the C ABI."""
    lib = pkg("_lib")
    H, W, _ = t.shape
    out = torch.full((3,), float("nan"), dtype=torch.float64, device="cuda")
    gt_, gg = dev(t), dev(g)
    assert lib.load().flowb200_epe(ptr(gt_), ptr(gg), H, W, float(thresh), ptr(out), stream()) == lib.OK
    s, no, nv = out.tolist()
    return s, no, nv


def epe_reference(t, g, thresh):
    """float32 per-pixel errors, separately rounded products (numpy never contracts them into an FMA), compared with
    the threshold in float32 as the kernel does (the C ABI takes a float)."""
    m = (t[..., 2] > 0.5) & (g[..., 2] > 0.5)
    dfu = t[..., 0][m] - g[..., 0][m]
    dfv = t[..., 1][m] - g[..., 1][m]
    e = np.sqrt(dfu * dfu + dfv * dfv)
    assert e.dtype == np.float32
    return e, int((e > F32(thresh)).sum()), int(m.sum())


@pytest.mark.parametrize("H,W", [(1, 1), (3, 50517), (148, 1024), (1, 151553), (2160, 3840)])
def test_epe_counts_exact_and_sum_exactly_rounded(H, W):
    """Sizes around the grid stride (148 SMs x 4 blocks x 256 threads = 151552 pixels) and a 4K frame.  Errors of
    exactly 5 (3, 4), 3 and 0.1f are planted: an error equal to the threshold is not an outlier, also at 0.1, which
    float32 cannot represent (the comparison is in float32 on both sides)."""
    rng = np.random.default_rng(H + W)
    n = H * W
    g = np.concatenate([rng.normal(0, 5, (H, W, 2)), rng.random((H, W, 1)) > 0.1], -1).astype(np.float32)
    t = np.concatenate([g[..., :2] + rng.normal(0, 2, (H, W, 2)), rng.random((H, W, 1)) > 0.2], -1).astype(np.float32)
    near = rng.random((H, W)) < 0.3                     # errors around 0.1
    t[..., 0] = np.where(near, g[..., 0] + rng.normal(0, 0.07, (H, W)).astype(np.float32), t[..., 0])
    t[..., 1] = np.where(near, g[..., 1], t[..., 1])
    tf, gf = t.reshape(n, 3), g.reshape(n, 3)
    pick = rng.permutation(n)[:max(1, n // 20)]
    for k, (du, dv) in enumerate([(3.0, 4.0), (3.0, 0.0), (0.1, 0.0), (-4.0, 3.0)]):
        p = pick[k::4]
        gf[p] = (0.0, 0.0, 1.0)
        tf[p] = (du, dv, 1.0)
    exact = None
    for thresh in (3.0, 5.0, 0.1):
        e, outliers, nvalid = epe_reference(t, g, thresh)
        s, no, nv = epe_device(t, g, thresh)
        assert nv == nvalid and no == outliers, (thresh, nv, nvalid, no, outliers)
        if thresh == 0.1 and n > 1:       # the planted 0.1f errors lie above the double 0.1 and are not counted
            assert outliers < int((e.astype(np.float64) > 0.1).sum())
        if exact is None:
            exact = math.fsum(e.astype(np.float64).tolist())
        assert abs(s - exact) <= nvalid * 2.0 ** -52 * exact, (thresh, s, exact)


def test_epe_nothing_valid_and_nan_flows():
    from oracle import epe as oepe
    ops = pkg("ops")
    rng = np.random.default_rng(4)
    H, W = 33, 65
    t = np.concatenate([rng.normal(0, 5, (H, W, 2)), rng.random((H, W, 1)) > 0.5], -1).astype(np.float32)
    g = t.copy()
    g[..., 2] = 1 - t[..., 2]                          # no pixel valid in both
    got = ops.epe(dev(t), dev(g))
    assert math.isnan(got[0]) and math.isnan(got[1]) and got[2] == 0
    g = np.concatenate([rng.normal(0, 5, (H, W, 2)), np.ones((H, W, 1))], -1).astype(np.float32)
    t[..., 2] = 1
    t[3, 4, 0] = np.nan                                 # a NaN flow in a valid pixel
    want = oepe.error_image(t, g)
    got = ops.epe(dev(t), dev(g))
    assert math.isnan(want[0]) and math.isnan(got[0])
    assert got[1] == want[1] and got[2] == want[2] == H * W


# ---------------------------------------------------------------- MRF energy (flowb200_energy)
MODES = ("FP64_F32COST", "FP64_F64COST", "INT32", "INT32_F32COST")


def energy_case(rng, H, W, K, mode, spread=12):
    dy = rng.integers(-spread, spread + 1, (H, W, K))
    dx = rng.integers(-spread, spread + 1, (H, W, K))
    pvec = ((dy & 0xFFFF) | ((dx & 0xFFFF) << 16)).astype(np.uint32).view(np.int32)
    nprop = rng.integers(0, K + 1, (H, W))
    labels = rng.integers(-1, K + 1, (H, W))
    if mode == "INT32":
        cost = rng.integers(0, 65536, (H, W, K)).astype(np.int32)
    elif mode == "FP64_F64COST":
        cost = rng.uniform(0, 2.5, (H, W, K))
    else:
        cost = rng.uniform(0, 2.5, (H, W, K)).astype(np.float32)
        cost[np.arange(K)[None, None, :] >= nprop[..., None]] = 1000.0      # unused slots, as the search leaves them
    return dy, dx, pvec, cost, nprop, labels


def energy_reference(dy, dx, cost, nprop, labels, mode, lamda, tpsi, shift):
    """(data terms, pairwise sum as a Python int, number of invalid labels).  Data terms: Python ints m (int32 modes,
    INT32_F32COST m = rint((lamda * c) * 2^S)) or the float64 products lamda * c."""
    H, W = labels.shape
    valid = (labels >= 0) & (labels < nprop)
    lab = np.where(valid, labels, 0)
    ys, xs = np.mgrid[0:H, 0:W]
    vy, vx, c = dy[ys, xs, lab], dx[ys, xs, lab], cost[ys, xs, lab][valid]
    pair = 0
    for sl_a, sl_b in (((slice(None), slice(0, -1)), (slice(None), slice(1, None))),
                       ((slice(0, -1), slice(None)), (slice(1, None), slice(None)))):
        both = valid[sl_a] & valid[sl_b]
        l1 = np.abs(vy[sl_a] - vy[sl_b]) + np.abs(vx[sl_a] - vx[sl_b])
        pair += sum(np.minimum(l1, tpsi)[both].tolist())
    if mode == "INT32":
        terms = [int(v) for v in c.tolist()]
    elif mode == "INT32_F32COST":
        terms = [int(v) for v in np.rint((lamda * c.astype(np.float64)) * float(1 << shift)).tolist()]
    else:
        terms = (lamda * c.astype(np.float64)).tolist()
    return terms, pair, int((~valid).sum())


def check_energy(dy, dx, pvec, cost, nprop, labels, mode, lamda, tpsi, shift, what):
    ops, lib = pkg("ops"), pkg("_lib")
    got = ops.energy(dev(pvec), dev(cost), dev(nprop, torch.int32), dev(labels, torch.int32),
                     mode=getattr(lib, "BCD_" + mode), lamda=lamda, tpsi=tpsi, cost_shift=shift)
    terms, pair, bad = energy_reference(dy, dx, cost, nprop, labels, mode, lamda, tpsi, shift)
    assert got[1] == pair and got[3] == bad, (what, got, pair, bad)
    if mode.startswith("INT32"):
        data = sum(terms)
        assert got[0] == data / 2 ** shift and got[2] == (data + (pair << shift)) / 2 ** shift, (what, got, data, pair)
        if mode == "INT32_F32COST":         # what the chains quantise is what flowb200_quantise_costs computes
            m = ops.quantise_costs(dev(cost), lamda, shift).cpu().numpy()
            valid = (labels >= 0) & (labels < nprop)
            sel = np.take_along_axis(m, np.where(valid, labels, 0)[..., None], -1)[..., 0][valid]
            assert sum(sel.tolist()) == data, what
        return data, pair
    exact, mag = math.fsum(terms), math.fsum(abs(v) for v in terms)
    tol = max(1, len(terms)) * 2.0 ** -52 * (mag + pair)
    assert abs(got[0] - exact) <= tol and abs(got[2] - (exact + pair)) <= tol, (what, got, exact, pair)
    return exact, pair


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("H,W", [(1, 1), (1, 2000), (2000, 1), (33, 64)])
def test_energy_every_mode_against_exact_sums(mode, H, W):
    for K in (1, 2, 512):
        rng = np.random.default_rng(H * 10007 + W * 31 + K)
        case = energy_case(rng, H, W, K, mode)
        for tpsi in (0, 1, 8, 9, 32):
            for shift in ((0, 7, 14) if mode.startswith("INT32") else (12,)):
                check_energy(*case, mode, 0.05, tpsi, shift, (H, W, K, tpsi, shift))


def test_energy_sums_above_2_32():
    """300 x 300, m = 65535 at every chosen label, tpsi 32, shift 14: the data sum (~5.9e9) and the pairwise sum in units
    of 2^-14 (~9e10) pass 2^32, the total stays below 2^53 (the accumulators are 64-bit)."""
    rng = np.random.default_rng(9)
    H, W, K = 300, 300, 2
    dy = rng.integers(-200, 201, (H, W, K))
    dx = rng.integers(-200, 201, (H, W, K))
    pvec = ((dy & 0xFFFF) | ((dx & 0xFFFF) << 16)).astype(np.uint32).view(np.int32)
    nprop = np.full((H, W), K)
    labels = rng.integers(0, K, (H, W))
    for mode, cost, lamda in (("INT32", np.full((H, W, K), 65535, np.int32), 0.05),
                              ("INT32_F32COST", np.full((H, W, K), 65535 / 16384, np.float32), 1.0)):
        data, pair = check_energy(dy, dx, pvec, cost, nprop, labels, mode, lamda, 32, 14, mode)
        assert data == 65535 * H * W and data > 2 ** 32 and (pair << 14) > 2 ** 32 and data + (pair << 14) < 2 ** 53


def test_energy_every_label_invalid():
    ops, lib = pkg("ops"), pkg("_lib")
    rng = np.random.default_rng(2)
    H, W, K = 19, 23, 5
    for mode in MODES:
        dy, dx, pvec, cost, nprop, labels = energy_case(rng, H, W, K, mode)
        labels = np.where(rng.random((H, W)) < 0.5, -1, nprop)          # -1 or exactly nprop
        got = ops.energy(dev(pvec), dev(cost), dev(nprop, torch.int32), dev(labels, torch.int32),
                         mode=getattr(lib, "BCD_" + mode), tpsi=8, cost_shift=12)
        assert got == (0.0, 0.0, 0.0, H * W), (mode, got)
