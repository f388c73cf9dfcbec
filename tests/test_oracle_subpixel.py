"""The sub-pixel refinement's numpy restatement (tests/subpixel_oracle.py, DESIGN section 4.8) on the CPU: its centre
cost is the search's data cost, every branch of the per-axis offset, and the vertex of a quadratic cost surface."""
import numpy as np

import subpixel_oracle as so
from helpers import pkg

F32 = np.float32


def test_centre_cost_equals_the_search_data_cost():
    """At random pixels and NN slots, c(0, 0) of the slot's vector equals cport.generisi's float32 data cost bit for bit
    wherever that cost is below tphi (where it is not, generisi stores tphi)."""
    from oracle import cport, daisy as od, proposals as oprop
    synth = pkg("synth")
    H, W, cw, ch = 75, 146, 29, 15
    img1, img2, _, _ = synth.make_pair(H, W, 3, max_dx=10, max_dy=6, n_rect=2)
    d1, d2 = od.daisy(img1), od.daisy(img2)
    # a tphi low enough that some NN costs are truncated (at 2.5 none of these are; 0.24 is about their median)
    op = oprop.Params(H, W, cw, ch, k_cell=5, n_gauss=0, maxnprop=125, tphi=0.24)
    P, L, N, _ = cport.generisi(d1, d2, op)
    rng = np.random.default_rng(11)
    ys, xs = rng.integers(0, H, 4000), rng.integers(0, W, 4000)
    s = (rng.random(4000) * N[ys, xs]).astype(np.int64)
    keep = N[ys, xs] > 0
    ys, xs, s = ys[keep], xs[keep], s[keep]
    ty, tx = ys + P[ys, xs, s, 0], xs + P[ys, xs, s, 1]
    c = so.costs(d1, d2, ys, xs, ty, tx)
    below = L[ys, xs, s] < op.tphi
    assert below.sum() > 500 and (~below).sum() > 500, below.mean()
    assert np.array_equal(c[below].astype(np.float64), L[ys, xs, s][below])
    assert (c[~below].astype(np.float64) >= op.tphi).all()


def test_axis_offset_branches():
    f = lambda *v: so.axis_offset(*(np.array([x], F32) for x in v))[0]
    # strict minimum: (c- - c+) / (2 (c- - 2 c0 + c+)) = 1 / 6, rounded once
    assert f(3, 1, 2) == F32(1) / F32(6)
    assert f(2, 1, 3) == -(F32(1) / F32(6))
    assert f(2, 1, 2) == 0 and not np.signbit(f(2, 1, 2))
    # a tie on either side is no strict minimum
    assert f(1, 1, 2) == 0 and f(2, 1, 1) == 0
    # the centre is not a minimum: a maximum, a slope, the minimum on one side
    assert f(1, 2, 1) == 0 and f(1, 2, 3) == 0 and f(3, 2, 1) == 0
    # flat: the denominator is 0, the offset 0
    assert f(1.5, 1.5, 1.5) == 0 and f(0, 0, 0) == 0
    # a strict minimum whose float32 quotient rounds past 0.5 is clamped to +-0.5
    cm, c0, cp = F32(270.7888), F32(0.066110544), F32(0.06611055)
    assert c0 < cp < cm
    raw = (cm - cp) / (F32(2) * ((cm - F32(2) * c0) + cp))
    assert raw > F32(0.5)
    assert f(cm, c0, cp) == F32(0.5) and f(cp, c0, cm) == F32(-0.5)


def test_quadratic_cost_surface_gives_its_vertex():
    """Zero source descriptors and target descriptors whose first entry is a*((x - xv)^2 + (y - yv)^2) + b: the cost is
    that entry exactly, the fitted parabola is the surface itself, and the refined vector points at its vertex."""
    rng = np.random.default_rng(5)
    H, W = 21, 23
    for _ in range(50):
        yv, xv = rng.uniform(3, H - 4), rng.uniform(3, W - 4)
        a, b = F32(rng.uniform(0.01, 2)), F32(rng.uniform(0, 3))
        y, x = np.mgrid[0:H, 0:W].astype(np.float64)
        d2 = np.zeros((H, W, 68), F32)
        d2[..., 0] = (a * ((x - xv) ** 2 + (y - yv) ** 2) + b).astype(F32)
        d1 = np.zeros((H, W, 68), F32)
        sy, sx = int(rng.integers(0, H)), int(rng.integers(0, W))
        ty, tx = int(round(yv)), int(round(xv))
        pvec = np.full((H, W, 2), -1, np.int32)
        pvec[sy, sx, 0] = so.pack(ty - sy, tx - sx)
        nprop = np.ones((H, W), np.int32)
        labels = np.zeros((H, W), np.int32)
        out = so.subpixel(d1, d2, pvec, nprop, labels)
        u, v, val = out[sy, sx]
        assert val == 1
        # the three costs are float32 roundings of the surface: the vertex within a few float32 ulps of the costs
        tol = 1e-5 * (1 + float(b) / float(a))
        assert abs(sx + float(u) - xv) <= tol and abs(sy + float(v) - yv) <= tol, (sx + u, xv, sy + v, yv)


def test_unrefined_pixels():
    """Labels in [nprop, K), fill vectors and targets off the frame keep their integer vector; a label outside [0, K)
    gives (0, 0, 0)."""
    rng = np.random.default_rng(2)
    H, W, K = 6, 7, 3
    d1, d2 = rng.random((H, W, 68), dtype=F32), rng.random((H, W, 68), dtype=F32)
    pvec = np.zeros((H, W, K), np.int32)
    nprop = np.full((H, W), 2, np.int32)
    labels = np.zeros((H, W), np.int32)
    pvec[0, 0, 2], labels[0, 0] = so.pack(1, 1), 2               # label >= nprop
    pvec[0, 1, 0] = -1                                            # (-1, -1) fill
    pvec[0, 2, 0] = so.pack(-1, 0)                                # target above the frame
    labels[0, 3] = -1                                             # outside [0, K)
    labels[0, 4] = K
    out = so.subpixel(d1, d2, pvec, nprop, labels)
    assert tuple(out[0, 0]) == (1, 1, 1) and tuple(out[0, 1]) == (-1, -1, 1) and tuple(out[0, 2]) == (0, -1, 1)
    assert tuple(out[0, 3]) == (0, 0, 0) and tuple(out[0, 4]) == (0, 0, 0)
