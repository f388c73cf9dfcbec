"""flowb200_flow_subpixel (`post.cu`, DESIGN section 4.8) bit for bit against tests/subpixel_oracle.py over whole arrays,
and flowb200_flow_pair with flow_refine = 1 against the stages composed by hand.  GPU only.

  kernel     small and odd frames, every frame edge and corner as a target or a target's neighbour, labels at slots 0
             and K-1, labels outside [0, nprop) and outside [0, K), fill vectors, constant descriptors, planted costs for
             every branch of the offset, an output pre-filled with NaN, a side stream, the return codes, and the real
             proposals and labels of the search at 1024x436, K = 300;
  flow_pair  at 1024x436, K = 300, both directions, a float64 and an int32 BCD mode: raw fields = flow_subpixel of the
             stage-by-stage labels, checked field = flowb200_consistency of them; flow_refine = 0 unchanged; the EPE of
             the refined raw forward field below the integer one on the two synthetic pairs of the CPU accuracy check (DESIGN 4.8).
"""
import ctypes as C
import dataclasses

import numpy as np
import pytest

import subpixel_oracle as so
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
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def run(d1, d2, pvec, nprop, labels):
    """Kernel (through ops) and oracle on the same arrays; asserts bit equality and returns the field."""
    got = pkg("ops").flow_subpixel(dev(d1), dev(d2), dev(pvec), dev(nprop, torch.int32), dev(labels, torch.int32))
    got = got.cpu().numpy()
    want = so.subpixel(d1, d2, pvec, nprop, labels)
    if not np.array_equal(bits(got), bits(want)):
        y, x, c = np.argwhere(bits(got) != bits(want))[0]
        raise AssertionError(f"{int((bits(got) != bits(want)).any(-1).sum())} pixels differ, the first ({y}, {x}) "
                             f"channel {c}: {got[y, x]} instead of {want[y, x]}")
    return got


def random_case(H, W, K, seed, reach=None):
    """Random descriptors; vectors whose targets fall inside the frame, on its edges and just outside; nprop over
    [0, K]; unused slots filled (-1, -1), some used slots too; labels mostly in [0, nprop), some at nprop..K-1, -1, K;
    the first pixels take slot 0 and the last slot K-1."""
    rng = np.random.default_rng(seed)
    d1 = rng.random((H, W, 68), dtype=F32)
    d2 = rng.random((H, W, 68), dtype=F32)
    ry, rx = (H + 1, W + 1) if reach is None else reach
    dy = rng.integers(-ry, ry + 1, (H, W, K))
    dx = rng.integers(-rx, rx + 1, (H, W, K))
    pvec = so.pack(dy, dx).reshape(H, W, K)
    nprop = rng.integers(0, K + 1, (H, W)).astype(np.int32)
    nprop[rng.random((H, W)) < 0.7] = K
    slot = np.arange(K)[None, None, :]
    pvec = np.where(slot < nprop[..., None], pvec, np.int32(-1))
    pvec[rng.random((H, W, K)) < 0.02] = -1
    labels = (rng.random((H, W)) * np.maximum(nprop, 1)).astype(np.int32)
    r = rng.random((H, W))
    labels[r < 0.03] = -1
    labels[(r >= 0.03) & (r < 0.06)] = K
    labels[(r >= 0.06) & (r < 0.1)] = K - 1
    flat = labels.reshape(-1)
    n = flat.size
    flat[: max(1, n // 8)] = 0
    flat[n - max(1, n // 8):] = K - 1
    return d1, d2, pvec, nprop, labels


@pytest.mark.parametrize("H,W", [(1, 1), (1, 300), (300, 1), (3, 3), (40, 53)])
@pytest.mark.parametrize("K", [1, 7, 300, 512])
def test_random_fields(H, W, K):
    run(*random_case(H, W, K, 1000 * H + W + K))
    run(*random_case(H, W, K, 7 + K, reach=(2, 2)))        # mostly in the frame: most pixels are refined


def test_targets_on_every_edge_and_corner():
    """Every target in the two outermost rings of the frame and the ring just outside it, from every source pixel in
    turn: targets on an edge (one neighbour off the frame: that axis is not refined), next to an edge (all in), off it."""
    H, W, K = 9, 11, 4
    ring = [(y, x) for y in range(-1, H + 1) for x in range(-1, W + 1)
            if min(y + 1, x + 1, H - y, W - x) <= 2]
    rng = np.random.default_rng(4)
    d1 = rng.random((H, W, 68), dtype=F32)
    d2 = rng.random((H, W, 68), dtype=F32)
    ys, xs = np.mgrid[0:H, 0:W]
    for shift in range(0, len(ring), H * W // 2):
        pvec = np.full((H, W, K), -1, np.int32)
        for i, (y, x) in enumerate(zip(ys.reshape(-1), xs.reshape(-1))):
            ty, tx = ring[(i + shift) % len(ring)]
            s = i % K
            pvec[y, x, s] = so.pack(ty - y, tx - x)
        labels = (np.arange(H * W) % K).reshape(H, W).astype(np.int32)
        run(d1, d2, pvec, np.full((H, W), K, np.int32), labels)


def test_constant_descriptors_tie_everywhere():
    """Every cost is 0: no strict minimum anywhere, every vector stays integer."""
    H, W, K = 23, 31, 5
    _, _, pvec, nprop, labels = random_case(H, W, K, 3, reach=(3, 3))
    for v in (0.0, 0.25, 1.0):
        d = np.full((H, W, 68), v, F32)
        got = run(d, d, pvec, nprop, labels)
        assert np.array_equal(got[..., :2], np.round(got[..., :2]))


def planted(triples_x, triples_y):
    """Source pixel (1, 3j+1) points at (1, 3j+1) + (0, 0) in a 3 x 3m frame with zero source descriptors; entry 0 of
    the target descriptors carries the planted costs (c-, c0, c+) along x and along y (the cost is that entry exactly)."""
    m = len(triples_x)
    H, W, K = 3, 3 * m, 2
    d1 = np.zeros((H, W, 68), F32)
    d2 = np.zeros((H, W, 68), F32)
    for j, ((xm, c0, xp), (ym, c0y, yp)) in enumerate(zip(triples_x, triples_y)):
        assert c0 == c0y
        x = 3 * j + 1
        d2[1, x - 1, 0], d2[1, x, 0], d2[1, x + 1, 0] = xm, c0, xp
        d2[0, x, 0], d2[2, x, 0] = ym, yp
    pvec = np.full((H, W, K), -1, np.int32)
    pvec[..., 0] = 0                                          # (0, 0)
    nprop = np.ones((H, W), np.int32)
    labels = np.zeros((H, W), np.int32)
    return d1, d2, pvec, nprop, labels


def test_planted_costs_every_branch():
    F = F32
    clamp = (F(270.7888), F(0.066110544), F(0.06611055))     # quotient rounds to 0.50000006: clamped
    tx = [(3, 1, 2), (2, 1, 3), (2, 1, 2), (1, 1, 2), (2, 1, 1), (1, 2, 1), (1, 2, 3), (1.5, 1.5, 1.5), (0, 0, 0),
          clamp, clamp[::-1]]
    ty = [t[::-1] for t in tx]
    d1, d2, pvec, nprop, labels = planted(tx, ty)
    got = run(d1, d2, pvec, nprop, labels)
    u = got[1, 1::3, 0]
    v = got[1, 1::3, 1]
    sixth = F(1) / F(6)
    want = [sixth, -sixth, 0, 0, 0, 0, 0, 0, 0, 0.5, -0.5]
    assert np.array_equal(u, np.array(want, F)), u
    assert np.array_equal(v, -np.array(want, F) + F(0)), v


def test_output_prefilled_with_nan_and_side_stream():
    """Every output entry is written (also for refused labels), and the kernel runs on the caller's stream."""
    lib = pkg("_lib")
    L = lib.load()
    H, W, K = 40, 53, 7
    d1, d2, pvec, nprop, labels = random_case(H, W, K, 9, reach=(4, 4))
    want = so.subpixel(d1, d2, pvec, nprop, labels)
    g = [dev(d1), dev(d2), dev(pvec), dev(nprop), dev(labels)]
    s = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        out = torch.full((H, W, 3), float("nan"), dtype=torch.float32, device="cuda")
        rc = L.flowb200_flow_subpixel(*[ptr(t) for t in g], H, W, K, ptr(out), C.c_void_p(s.cuda_stream))
        assert rc == lib.OK
        got = pkg("ops").flow_subpixel(*g)
    s.synchronize()
    assert np.array_equal(bits(out.cpu().numpy()), bits(want))
    assert np.array_equal(bits(got.cpu().numpy()), bits(want))


def test_return_codes():
    lib = pkg("_lib")
    L = lib.load()
    H, W, K = 5, 6, 3
    d1, d2, pvec, nprop, labels = random_case(H, W, K, 2)
    g = [dev(d1), dev(d2), dev(pvec), dev(nprop), dev(labels)]
    out = torch.full((H, W, 3), float("nan"), dtype=torch.float32, device="cuda")
    ok = [ptr(t) for t in g]
    for i in range(6):                                        # each pointer null in turn
        args = ok + [ptr(out)]
        args[i] = C.c_void_p(0)
        assert L.flowb200_flow_subpixel(*args[:5], H, W, K, args[5], stream()) == lib.EINVAL, i
    for h, w, k in ((0, W, K), (-1, W, K), (H, 0, K), (H, -3, K), (H, W, 0), (H, W, -1), (H, W, 513)):
        assert L.flowb200_flow_subpixel(*ok, h, w, k, ptr(out), stream()) == lib.EINVAL, (h, w, k)
    flat = torch.zeros(H * W * 68 + 1, dtype=torch.float32, device="cuda")   # a descriptor base 4 bytes off alignment
    mis = C.c_void_p(flat.data_ptr() + 4)
    assert L.flowb200_flow_subpixel(mis, ok[1], *ok[2:], H, W, K, ptr(out), stream()) == lib.EINVAL
    assert L.flowb200_flow_subpixel(ok[0], mis, *ok[2:], H, W, K, ptr(out), stream()) == lib.EINVAL
    torch.cuda.synchronize()
    assert torch.isnan(out).all()                             # the refused calls launched nothing
    assert L.flowb200_flow_subpixel(*ok, H, W, K, ptr(out), stream()) == lib.OK
    assert np.array_equal(bits(out.cpu().numpy()), bits(so.subpixel(d1, d2, pvec, nprop, labels)))
    p = dataclasses.replace(pkg("params").FlowParams(H=50, W=146), flow_refine=2)
    with pytest.raises(ValueError):
        p.validate()


# ---------------------------------------------------------------- search-sweep geometry and flow_pair at 1024x436
H, W, K, SWEEPS = 436, 1024, 300, 4
ACCURACY_PAIRS = (5, 6)


@pytest.fixture(scope="module")
def bench_pair():
    ops, params, synth = pkg("ops"), pkg("params"), pkg("synth")
    p = params.for_k(K, H=H, W=W, knn_mode=1)
    img = synth.make_pair(H, W, ACCURACY_PAIRS[0])
    g = [dev(img[0]), dev(img[1])]
    return p, img, g, [ops.daisy(g[0]), ops.daisy(g[1])]


def stages(p, desc, bcd_mode, seed, refine):
    ops = pkg("ops")
    flows = []
    for d in (0, 1):
        s, t = desc[d], desc[1 - d]
        pvec, lcost, nprop, labels = ops.knn_proposals(s, t, p)
        ops.random_proposals(s, t, p, pvec, lcost, nprop, labels, seed=seed + d)
        ops.bcd(pvec, lcost, nprop, labels, SWEEPS, mode=bcd_mode, cost_shift=p.cost_shift)
        flows.append(ops.flow_subpixel(s, t, pvec, nprop, labels) if refine else
                     ops.flow_from_labels(pvec, labels, want_yx=False)[1])
        if d == 0:
            keep = (s, t, pvec, nprop, labels)
    return flows, keep


def test_search_sweep_geometry_real_proposals(bench_pair):
    """The kernel on the search's proposals and the BCD's labels of a 1024x436 frame, K = 300."""
    lib = pkg("_lib")
    p, _, _, desc = bench_pair
    _, (s, t, pvec, nprop, labels) = stages(p, desc, lib.BCD_INT32_F32COST, 9, True)
    got = run(s.cpu().numpy(), t.cpu().numpy(), pvec.cpu().numpy(), nprop.cpu().numpy(), labels.cpu().numpy())
    moved = float((got[..., :2] != np.round(got[..., :2])).any(-1).mean())
    print(f"\n1024x436 K=300: {moved:.3f} of the pixels refined")
    assert moved > 0.5


@pytest.mark.parametrize("mode", ["BCD_FP64_F32COST", "BCD_INT32_F32COST"])
def test_flow_pair_refined_equals_the_stages(bench_pair, mode):
    ops, lib = pkg("ops"), pkg("_lib")
    p, _, g, desc = bench_pair
    bcd_mode = getattr(lib, mode)
    pr = dataclasses.replace(p, flow_refine=1)
    out, raw_f, raw_b = ops.flow_pair(g[0], g[1], pr, sweeps=SWEEPS, directions=2, seed=9, bcd_mode=bcd_mode,
                                      want_raw=True)
    flows, _ = stages(p, desc, bcd_mode, 9, True)
    assert torch.equal(raw_f, flows[0]) and torch.equal(raw_b, flows[1])
    assert torch.equal(out, ops.consistency(flows[0].clone(), flows[1], p.con_tresh))
    # forward only: no check, the field is the raw forward one
    fwd = ops.flow_pair(g[0], g[1], pr, sweeps=SWEEPS, directions=1, seed=9, bcd_mode=bcd_mode)
    assert torch.equal(fwd, flows[0])
    # flow_refine = 0 written explicitly: the same bytes as a call that leaves the field at its default, and integers
    a = ops.flow_pair(g[0], g[1], dataclasses.replace(p, flow_refine=0), sweeps=SWEEPS, directions=2, seed=9,
                      bcd_mode=bcd_mode, want_raw=True)
    b = ops.flow_pair(g[0], g[1], p, sweeps=SWEEPS, directions=2, seed=9, bcd_mode=bcd_mode, want_raw=True)
    for x, y in zip(a, b):
        assert torch.equal(x.view(torch.int32), y.view(torch.int32))
    assert torch.equal(a[1], torch.round(a[1])) and not torch.equal(raw_f, a[1])


def test_refined_epe_below_integer_epe():
    """The two synthetic pairs of the CPU accuracy check (DESIGN section 4.8): the refined raw forward EPE is below the integer
    one; raw and checked EPE are logged both ways."""
    ops, lib, params, synth = pkg("ops"), pkg("_lib"), pkg("params"), pkg("synth")
    from oracle import epe as oepe
    p = params.for_k(K, H=H, W=W, knn_mode=1)
    for pair in ACCURACY_PAIRS:
        img1, img2, fwd, _ = synth.make_pair(H, W, pair)
        gt = synth.gt_uvv(fwd)
        e = {}
        for refine in (0, 1):
            out, raw, _ = ops.flow_pair(dev(img1), dev(img2), dataclasses.replace(p, flow_refine=refine),
                                        sweeps=SWEEPS, directions=2, seed=0, bcd_mode=lib.BCD_INT32_F32COST,
                                        want_raw=True)
            e[refine] = (oepe.error_image(raw.cpu().numpy(), gt)[0], oepe.error_image(out.cpu().numpy(), gt)[0])
        print(f"\npair {pair}: EPE raw forward {e[0][0]:.4f} -> {e[1][0]:.4f} px, checked {e[0][1]:.4f} -> "
              f"{e[1][1]:.4f} px (integer -> sub-pixel)")
        assert e[1][0] < e[0][0], e


def test_sharded_pair_on_one_rank_honours_flow_refine():
    """huge.flow_pair_sharded returns what ops.flow_pair returns, sub-pixel fields included (one rank, no exchange)."""
    ops, lib, params, synth, huge = pkg("ops"), pkg("_lib"), pkg("params"), pkg("synth"), pkg("huge")
    h, w = 61, 90
    img1, img2, _, _ = synth.make_pair(h, w, 2, max_dx=6, max_dy=4, n_rect=2)
    p = params.FlowParams(H=h, W=w, cellw=16, cellh=12, n_gauss=10, maxnprop=135, knn_mode=1, flow_refine=1)
    g0, g1 = dev(img1), dev(img2)
    want = ops.flow_pair(g0, g1, p, sweeps=2, directions=2, seed=7, bcd_mode=lib.BCD_INT32, want_raw=True)
    got = huge.flow_pair_sharded(g0, g1, p, 2, 2, 7, lib.BCD_INT32, 0, 1, None, want_raw=True)
    for a, b in zip(got, want):
        assert torch.equal(a, b)
    assert not torch.equal(want[1], torch.round(want[1]))
