"""The random-neighbour proposals (nasumicni, random_proposals_kernel) and the K-set export at their edges.  GPU only.

  a. Replayed draws at every cell geometry of the search sweep and at small cells (4x4, 1xN, Nx1, 2x3) on ragged
     frames, radius 1 / 2 / 3, every k_cell the search compiles, maxnprop exact and with slack, n_gauss 1 / 25 / the
     most K leaves; Gaussian draws at sigma 8 and 30 and planted ones (self-draws, repeats, corners, the remainder
     strips, targets far right / far up-left); the search's argmin and planted labels; NN vectors with a -1 component;
     descriptors that give cost 0, costs above tphi and signed differences that cancel (quirk Q6).  A host restatement
     counts the draws whose slice start is negative, whose slice runs past K, that a wrapped slice rejects, that a
     fill row rejects and that the slice of the random slots rejects, and each case asserts it reaches its targets.
  b. The seeded path against tests/philox_draws.py: identifying proposal sets (every accepted vector names its target
     pixel) at seeds 0, 1, 7, 2^32-1, 2^32, 2^64-1, and the search's proposals at 1024x436, K = 300, both directions.
  c. flowb200_ksets_pack over whole arrays, trailing byte included, against oracle.proposals.pakovanje.
  d. The argument checks of flowb200_knn_proposals, flowb200_random_proposals and flowb200_ksets_pack.
  e. Radius 0: refused on ragged frames with random proposals (the reference's scan order decides the result there),
     working on whole-cell frames and with n_gauss = 0.
Every comparison is over whole arrays, bit for bit: pvec, lcost as float64, nprop.
"""
import ctypes as C
import zlib

import numpy as np
import pytest

import philox_draws as pd
from helpers import pkg

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

OK, EINVAL, EWORKSPACE, EUNSUPPORTED = 0, -1, -2, -4
FILL = 1 << 20          # a component no int16 vector has


def dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda()


def params(H, W, cw, ch, R, k, n_gauss, slack=0, sigma=8.0):
    return pkg("params").FlowParams(H=H, W=W, cellw=cw, cellh=ch, cell_radius=R, k_cell=k, n_gauss=n_gauss,
                                    sigma=sigma, maxnprop=(2 * R + 1) ** 2 * k + n_gauss + slack)


def oracle_params(p):
    from oracle import proposals as oprop
    return oprop.Params(p.H, p.W, p.cellw, p.cellh, cell_radius=p.cell_radius, k_cell=p.k_cell, n_gauss=p.n_gauss,
                        sigma=p.sigma, maxnprop=p.maxnprop, tphi=p.tphi)


def gpu_random(d1, d2, p, P, L, N, B, draws=None, seed=0):
    """flowb200_random_proposals on uploaded copies of (P int64 (H,W,K,2), L, N, B): host (pvec, lcost f64, nprop)."""
    ops, ioc = pkg("ops"), pkg("io_contract")
    pvec, lcost = dev(ioc.pack_proposals(P)), dev(L.astype(np.float32))
    nprop, labels = dev(N.astype(np.int32)), dev(B.astype(np.int32))
    ops.random_proposals(dev(d1), dev(d2), p, pvec, lcost, nprop, labels,
                         draws=None if draws is None else dev(draws.astype(np.int16)), seed=seed)
    return pvec.cpu().numpy(), lcost.cpu().numpy().astype(np.float64), nprop.cpu().numpy()


def assert_equal_arrays(got, P2, L2, N2):
    ioc = pkg("io_contract")
    for name, g, w in zip(("pvec", "lcost", "nprop"), got, (ioc.pack_proposals(P2), L2, N2)):
        assert np.array_equal(g, w), (name, float((g != w).mean()))


# ---------------------------------------------------------------- host restatement with counts
def restate(d1, d2, P, L, N, B, p, draws):
    """nasumicni vectorised over pixels (sequential over draws), with the counts of what the draws reach:
    neg (slice start < 0), over (start + k > K), wrap (rejected by a slice with a negative start), fill (rejected by
    an unused (-1, -1) row of the first slice), second (passed the first slice, rejected by the random slots)."""
    from oracle.proposals import sum_f32_numpy_order
    H, W, K, k, n_g = p.H, p.W, p.maxnprop, p.k_cell, p.n_gauss
    n_pix = H * W
    rows = P.reshape(n_pix, K, 2).copy()
    lc = L.reshape(n_pix, K).copy()
    n = N.reshape(n_pix).astype(np.int64).copy()
    n0 = n.copy()
    ng = np.zeros(n_pix, np.int64)
    acc_store = np.full((n_pix, max(n_g, 1), 2), FILL, np.int64)
    ys, xs = np.divmod(np.arange(n_pix), W)
    mincy = np.maximum(0, ys // p.cellh - 2)
    ncy = np.minimum(p.ncelly, ys // p.cellh + 2) - mincy
    mincx = np.maximum(0, xs // p.cellw - 2)
    best = P.reshape(n_pix, K, 2)[np.arange(n_pix), B.reshape(n_pix)]
    f1, f2 = d1.reshape(n_pix, -1), d2.reshape(n_pix, -1)
    cnt = dict(neg=0, over=0, wrap=0, fill=0, second=0, accepted=0)
    kk = np.arange(k)
    for i in range(n_g):
        tgy, tgx = draws[..., i, 0].reshape(-1).astype(np.int64), draws[..., i, 1].reshape(-1).astype(np.int64)
        broj = k * ((tgy // p.cellh - mincy) + (tgx // p.cellw - mincx) * ncy)
        tpix = tgy * W + tgx
        tv = best[tpix]
        a = np.where(broj < 0, np.maximum(broj + K, 0), np.minimum(broj, K))
        e = broj + k
        b = np.where(e < 0, np.maximum(e + K, 0), np.minimum(e, K))
        idx = a[:, None] + kk[None, :]
        valid = idx < b[:, None]
        sl = rows[np.arange(n_pix)[:, None], np.minimum(idx, K - 1)]
        eq = valid & ((sl[..., 0] == tv[:, None, 0]) | (sl[..., 1] == tv[:, None, 1]))
        hit1 = eq.any(1)
        fill_hit = (eq & (idx >= n[:, None])).any(1)
        hit2 = ((acc_store[..., 0] == tv[:, None, 0]) | (acc_store[..., 1] == tv[:, None, 1])).any(1)
        acc = ~hit1 & ~hit2
        cnt["neg"] += int((broj < 0).sum())
        cnt["over"] += int((broj + k > K).sum())
        cnt["wrap"] += int((hit1 & (broj < 0)).sum())
        cnt["fill"] += int((hit1 & fill_hit).sum())
        cnt["second"] += int((~hit1 & hit2).sum())
        cnt["accepted"] += int(acc.sum())
        q = np.nonzero(acc)[0]
        s = sum_f32_numpy_order(f1[q] - f2[tpix[q]]).astype(np.float64)
        rows[q, n[q]] = tv[q]
        lc[q, n[q]] = np.minimum(np.float64(p.tphi), np.abs(s))
        acc_store[q, ng[q]] = tv[q]
        n[q] += 1
        ng[q] += 1
    assert (n - n0 == ng).all()
    return rows.reshape(P.shape), lc.reshape(L.shape), n.reshape(N.shape), cnt


# ---------------------------------------------------------------- case construction
def nn_inputs(rng, p, labels="argmin", minus_one=0.0):
    """What the search hands to the random proposals, without running it: nprop = k x the cells in range, NN vectors
    that point into the cell of their slot (ci-major, cj-minor), float32 costs in [0, tphi], unused slots (-1, -1) /
    1000; labels = the first strict argmin of the NN costs, or a planted NN slot per pixel; a fraction `minus_one` of
    the NN vectors get dy = -1 or dx = -1."""
    H, W, K, k, R = p.H, p.W, p.maxnprop, p.k_cell, p.cell_radius
    ys, xs = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    cimin, cimax = np.maximum(0, xs // p.cellw - R), np.minimum(p.ncellx - 1, xs // p.cellw + R)
    cjmin, cjmax = np.maximum(0, ys // p.cellh - R), np.minimum(p.ncelly - 1, ys // p.cellh + R)
    nci, ncj = np.maximum(0, cimax - cimin + 1), np.maximum(0, cjmax - cjmin + 1)
    N = (k * nci * ncj).astype(np.int64)
    P = np.full((H, W, K, 2), -1, np.int64)
    L = np.full((H, W, K), 1000.0)
    s = np.arange(K)[None, None, :]
    used = s < N[..., None]
    blk = s // k
    ci = cimin[..., None] + blk // np.maximum(ncj, 1)[..., None]
    cj = cjmin[..., None] + blk % np.maximum(ncj, 1)[..., None]
    t = rng.integers(0, p.cellw * p.cellh, (H, W, K))
    dy = cj * p.cellh + t // p.cellw - ys[..., None]
    dx = ci * p.cellw + t % p.cellw - xs[..., None]
    P[..., 0] = np.where(used, dy, -1)
    P[..., 1] = np.where(used, dx, -1)
    plant = used & (rng.random((H, W, K)) < minus_one)
    comp = rng.integers(0, 2, (H, W, K))
    P[..., 0] = np.where(plant & (comp == 0), -1, P[..., 0])
    P[..., 1] = np.where(plant & (comp == 1), -1, P[..., 1])
    cost = (rng.random((H, W, K), dtype=np.float32) * np.float32(p.tphi)).astype(np.float32)
    cost[rng.random((H, W, K)) < 0.1] = np.float32(p.tphi)
    L = np.where(used, cost.astype(np.float64), 1000.0)
    if labels == "argmin":
        B = np.argmin(np.where(used, L, np.inf), axis=-1)       # first minimum, as finish_nn_kernel
    else:
        B = (rng.integers(0, 1 << 30, (H, W)) % np.maximum(N, 1))
    return P, L, N, B.astype(np.int64)


def descriptors(rng, H, W, kind):
    def rand(scale=0.5):
        return (rng.random((H, W, 68), dtype=np.float32) ** 3 * np.float32(scale)).astype(np.float32)
    if kind == "random":
        return rand(), rand()
    if kind == "identical":                     # one descriptor everywhere: every random proposal costs 0
        d = np.broadcast_to(rand()[0, 0], (H, W, 68)).copy()
        return d, d.copy()
    if kind == "far":                           # |sum| of 68 differences of 0.4-0.6: every cost is tphi
        return (0.5 + rand(0.1)).astype(np.float32), rand(0.1)
    # "cancel": dimensions 2j, 2j+1 hold 0.25 + a_j, 0.25 - a_j: the signed differences cancel in pairs, so Q6's
    # |signed sum| is a few roundings while the L1 distance is large
    out = []
    for _ in range(2):
        a = (0.2 * rng.random((H, W, 34), dtype=np.float32)).astype(np.float32)
        d = np.empty((H, W, 68), np.float32)
        d[..., 0::2], d[..., 1::2] = np.float32(0.25) + a, np.float32(0.25) - a
        out.append(d)
    return tuple(out)


def planted_draws(rng, p, sigma):
    """Per draw i: i % 6 == 0 self, 1 a repeat of draw i-1, 2 a corner, 3 a remainder row / column (a corner when the
    frame has none), 4 the last column, 5 the first row and column; Gaussian otherwise (every 7th)."""
    from test_gpu_baseline_configs import make_draws
    H, W, ng = p.H, p.W, p.n_gauss
    d = make_draws(H, W, ng, sigma, int(rng.integers(1 << 30))).astype(np.int64)
    ys, xs = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    corners = np.array([(0, 0), (0, W - 1), (H - 1, 0), (H - 1, W - 1)])
    ry0, rx0 = p.ncelly * p.cellh, p.ncellx * p.cellw
    for i in range(ng):
        kind = i % 7
        if kind == 0:
            d[:, :, i] = np.stack([ys, xs], -1)
        elif kind == 1 and i > 0:
            d[:, :, i] = d[:, :, i - 1]
        elif kind == 2 or (kind == 3 and ry0 == H and rx0 == W):
            d[:, :, i] = corners[rng.integers(0, 4, (H, W))]
        elif kind == 3:
            ty = np.where(rng.random((H, W)) < 0.5, rng.integers(min(ry0, H - 1), H, (H, W)), rng.integers(0, H, (H, W)))
            tx = np.where(ty >= ry0, rng.integers(0, W, (H, W)), rng.integers(min(rx0, W - 1), W, (H, W)))
            d[:, :, i] = np.stack([ty, tx], -1)
        elif kind == 4:
            d[:, :, i] = np.stack([rng.integers(0, H, (H, W)), np.full((H, W), W - 1)], -1)
        elif kind == 5:
            d[:, :, i] = np.stack([np.zeros((H, W), np.int64), rng.integers(0, 2, (H, W))], -1)
    return d


def K_max(R, k):
    return 512 - (2 * R + 1) ** 2 * k


# (H, W, cellw, cellh, R, k, n_gauss, slack, draws, labels, descriptors, minus_one, counts the case must reach)
G = "gauss8", "gauss30", "planted8", "planted30"
CASES = [
    # the search sweep's geometries (tests/test_gpu_knn_edges.py GEOMETRIES)
    (43, 61, 8, 4, 2, 5, 25, 0, "gauss8", "argmin", "random", 0.1, ("neg", "wrap", "fill", "second")),
    (50, 71, 16, 8, 2, 10, 25, 7, "planted8", "planted", "identical", 0.0, ("neg", "fill", "second")),
    (61, 83, 13, 11, 2, 12, 1, 0, "gauss30", "argmin", "far", 0.0, ("neg", "over")),
    (110, 300, 73, 25, 2, 5, 25, 0, "planted30", "planted", "cancel", 0.1, ("neg", "wrap", "second")),
    (100, 200, 64, 32, 1, 12, 25, 0, "gauss8", "argmin", "random", 0.0, ("over", "second")),
    (37, 390, 128, 16, 2, 10, 25, 512, "planted8", "argmin", "random", 0.0, ("second",)),
    (101, 9, 1, 40, 2, 5, 25, 0, "gauss30", "planted", "far", 0.1, ("neg", "wrap", "fill")),
    (7, 130, 48, 1, 2, 10, 25, 0, "planted8", "argmin", "cancel", 0.0, ("neg", "wrap", "fill", "second")),
    (60, 90, 12, 10, 3, 10, 22, 0, "gauss8", "planted", "random", 0.1, ("second",)),
    (25, 73, 73, 25, 2, 5, 25, 0, "planted30", "argmin", "identical", 0.0, ("second",)),
    (30, 80, 73, 25, 1, 12, 25, 3, "gauss30", "argmin", "random", 0.0, ("second",)),
    # small cells on ragged frames: slice starts negative, wrapped into the tail, past K
    (19, 23, 4, 4, 1, 1, 25, 0, "gauss8", "argmin", "random", 0.2, ("neg", "wrap", "fill", "second")),
    (19, 63, 4, 4, 2, 2, 25, 0, "planted30", "planted", "cancel", 0.2, ("neg", "over", "wrap", "fill", "second")),
    (21, 17, 2, 3, 3, 3, 25, 0, "gauss30", "argmin", "random", 0.2, ("neg", "wrap", "fill", "second")),
    (21, 17, 2, 3, 1, 4, K_max(1, 4), 0, "gauss8", "argmin", "identical", 0.2, ("neg", "wrap", "fill", "second")),
    (15, 37, 1, 7, 2, 5, 25, 0, "planted8", "argmin", "random", 0.2, ("neg", "over", "wrap", "fill", "second")),
    (37, 15, 7, 1, 2, 5, 25, 0, "gauss30", "planted", "far", 0.2, ("neg", "over", "wrap", "fill", "second")),
    (13, 18, 4, 4, 1, 8, 1, 0, "gauss8", "argmin", "random", 0.2, ("neg",)),
    (13, 18, 4, 4, 1, 16, K_max(1, 16), 0, "planted30", "argmin", "random", 0.2, ("neg", "wrap", "fill", "second")),
    (33, 35, 8, 4, 2, 16, 25, 0, "gauss30", "planted", "cancel", 0.2, ("neg", "wrap", "fill", "second")),
    (9, 11, 2, 2, 1, 1, K_max(1, 1), 0, "gauss8", "argmin", "random", 0.2, ("neg", "wrap", "fill", "second")),
    (11, 13, 4, 4, 2, 2, 25, 512, "planted8", "planted", "random", 0.2, ("neg", "fill", "second")),
]


def case_id(c):
    return f"{c[0]}x{c[1]}-c{c[2]}x{c[3]}-R{c[4]}-k{c[5]}-g{c[6]}-s{c[7]}-{c[8]}-{c[9]}-{c[10]}"


def build_case(c):
    H, W, cw, ch, R, k, ng, slack, dk, lk, desc, m1, _ = c
    p = params(H, W, cw, ch, R, k, ng, slack=min(slack, 512 - (2 * R + 1) ** 2 * k - ng))
    rng = np.random.default_rng(zlib.crc32(case_id(c).encode()))
    d1, d2 = descriptors(rng, H, W, desc)
    P, L, N, B = nn_inputs(rng, p, lk, m1)
    sigma = 30.0 if dk.endswith("30") else 8.0
    if dk.startswith("gauss"):
        from test_gpu_baseline_configs import make_draws
        draws = make_draws(H, W, ng, sigma, int(rng.integers(1 << 30))).astype(np.int64)
    else:
        draws = planted_draws(rng, p, sigma)
    return p, d1, d2, P, L, N, B, draws


@pytest.mark.parametrize("c", CASES, ids=[case_id(c) for c in CASES])
def test_replayed_draws_every_geometry(c):
    from oracle import cport
    p, d1, d2, P, L, N, B, draws = build_case(c)
    assert p.maxnprop <= 512 and (N <= p.max_nn).all()
    P2, L2, N2 = cport.nasumicni(d1, d2, P, L, N, B, oracle_params(p), draws=draws)
    R2, RL2, RN2, cnt = restate(d1, d2, P, L, N, B, p, draws)
    assert np.array_equal(R2, P2) and np.array_equal(RL2, L2) and np.array_equal(RN2, N2)   # the restatement = cport
    assert_equal_arrays(gpu_random(d1, d2, p, P, L, N, B, draws=draws), P2, L2, N2)
    for name in c[-1]:
        assert cnt[name] > 0, (name, cnt)               # the case reaches what it targets
    assert 0 < cnt["accepted"] < draws[..., 0].size or p.n_gauss == 1
    rnd = (np.arange(L2.shape[-1]) >= N[..., None]) & (np.arange(L2.shape[-1]) < N2[..., None])
    if c[10] == "identical":
        assert rnd.any() and (L2[rnd] == 0).all()
    if c[10] == "far":
        assert (L2[rnd] == np.float64(np.float32(p.tphi))).all()
    if c[10] == "cancel":
        assert rnd.any() and (L2[rnd] < 1e-5).mean() > 0.9


@pytest.mark.parametrize("R", [0, 1])
def test_radius_0_on_whole_cell_frames(R):
    """Radius 0 on a frame that is a whole multiple of the cell: every pixel has NN proposals, pixels are
    independent, and the kernel equals cport.nasumicni (the same frame at radius 1 for comparison)."""
    from oracle import cport
    from test_gpu_baseline_configs import make_draws
    p = params(24, 36, 4, 6, R, 3, 25)
    rng = np.random.default_rng(8 + R)
    d1, d2 = descriptors(rng, p.H, p.W, "random")
    P, L, N, B = nn_inputs(rng, p, "argmin", 0.1)
    draws = make_draws(p.H, p.W, p.n_gauss, p.sigma, 3)
    P2, L2, N2 = cport.nasumicni(d1, d2, P, L, N, B, oracle_params(p), draws=draws)
    assert_equal_arrays(gpu_random(d1, d2, p, P, L, N, B, draws=draws), P2, L2, N2)
    assert_equal_arrays(gpu_random(d1, d2, p, P, L, N, B, seed=5), *cport.nasumicni(
        d1, d2, P, L, N, B, oracle_params(p), draws=pd.seeded_draws(p.H, p.W, p.n_gauss, p.sigma, 5)[0]))


def test_radius_0_on_a_ragged_frame_is_refused():
    """n_gauss > 0 with radius 0 on a frame with remainder strips: FLOWB200_EUNSUPPORTED before any launch (outputs
    untouched), also through flow_pair; n_gauss = 0 there is a no-op that succeeds."""
    ops, lib = pkg("ops"), pkg("_lib")
    for H, W in ((26, 36), (24, 37), (27, 39)):
        p = params(H, W, 4, 6, 0, 3, 25)
        rng = np.random.default_rng(H + W)
        d1, d2 = descriptors(rng, H, W, "random")
        P, L, N, B = nn_inputs(rng, p)
        assert (N == 0).any()
        pvec, lcost, nprop, labels = (dev(pkg("io_contract").pack_proposals(P)), dev(L.astype(np.float32)),
                                      dev(N.astype(np.int32)), dev(B.astype(np.int32)))
        with pytest.raises(lib.FlowB200Error, match="unsupported|not supported|UNSUPPORTED"):
            ops.random_proposals(dev(d1), dev(d2), p, pvec, lcost, nprop, labels, seed=1)
        assert np.array_equal(nprop.cpu().numpy(), N)
        p0 = params(H, W, 4, 6, 0, 3, 0)
        ops.random_proposals(dev(d1), dev(d2), p0, pvec, lcost, nprop, labels, seed=1)
        assert np.array_equal(nprop.cpu().numpy(), N)
    img = np.zeros((26, 36, 3), np.uint8)
    with pytest.raises(lib.FlowB200Error):
        ops.flow_pair(dev(img), dev(img), params(26, 36, 4, 6, 0, 3, 25), sweeps=1)


# ---------------------------------------------------------------- b. the seeded path equals the restatement
SEEDS = [0, 1, 7, 2 ** 32 - 1, 2 ** 32, 2 ** 64 - 1]
# (H, W, cellw, cellh, n_gauss, seeds)
ID_FRAMES = [(128, 255, 16, 16, 25, SEEDS), (64, 96, 8, 8, 200, [0, 2 ** 64 - 1, 2 ** 32]),
             (2, 4093, 16, 1, 25, [1, 2 ** 32]), (4093, 2, 1, 16, 25, [7, 2 ** 32 - 1])]
ID_CASES = [(f[:5], s) for f in ID_FRAMES for s in f[5]]


@pytest.mark.parametrize("frame,seed", ID_CASES, ids=[f"{f[0]}x{f[1]}-g{f[4]}-seed{s}" for f, s in ID_CASES])
def test_seeded_draws_identifying_sets(frame, seed):
    """nprop 1, labels 0, slot 0 of pixel t = (t+1, t+1), the rest (-1, -1) / 1000: distinct targets differ in both
    components, so only self-hits and genuine repeats are rejected and every accepted vector names its target.  The
    device's seeded output equals cport.nasumicni on the restated draws."""
    from oracle import cport
    H, W, cw, ch, ng = frame
    assert H * W <= 32766
    p = params(H, W, cw, ch, 1, 1, ng)
    K = p.maxnprop
    P = np.full((H, W, K, 2), -1, np.int64)
    t = np.arange(H * W).reshape(H, W) + 1
    P[:, :, 0, 0], P[:, :, 0, 1] = t, t
    L = np.full((H, W, K), 1000.0)
    L[:, :, 0] = 0.5
    N, B = np.ones((H, W), np.int64), np.zeros((H, W), np.int64)
    rng = np.random.default_rng(seed % 1000)
    d1, d2 = descriptors(rng, H, W, "random")
    draws, margin = pd.seeded_draws(H, W, ng, p.sigma, seed)
    assert int((margin < pd.AMBIGUOUS).sum()) == 0          # no pixel the restatement cannot decide
    P2, L2, N2 = cport.nasumicni(d1, d2, P, L, N, B, oracle_params(p), draws=draws)
    got = gpu_random(d1, d2, p, P, L, N, B, seed=seed)
    assert (N2 - 1).sum() > 0.5 * H * W * ng * (0.3 if min(H, W) <= 2 else 1.0)   # most draws observable
    ioc = pkg("io_contract")
    bad = np.nonzero((got[0] != ioc.pack_proposals(P2)).any(-1) | (got[2] != N2))
    if bad[0].size:
        y, x = int(bad[0][0]), int(bad[1][0])
        g = ioc.unpack_proposals(got[0][y, x])[1:got[2][y, x], 0] - 1
        w = P2[y, x, 1:N2[y, x], 0] - 1
        j = next((j for j in range(min(len(g), len(w))) if g[j] != w[j]), min(len(g), len(w)))
        pytest.fail(f"pixel ({y}, {x}): accepted draw {j} targets pixel "
                    f"{divmod(int(g[j]), W) if j < len(g) else None} on the device, "
                    f"{divmod(int(w[j]), W) if j < len(w) else None} restated; restated draws {draws[y, x, :8].tolist()}")
    assert_equal_arrays(got, P2, L2, N2)


def test_seeded_draws_real_sets_1024x436_k300():
    """The search's proposals of a texture pair at 1024x436, K = 300 (for_k), then the seeded random proposals of both
    directions with seeds s and s + 1 as the pipeline runs them, against cport.nasumicni on the restated draws."""
    from oracle import cport
    ops, synth = pkg("ops"), pkg("synth")
    H, W, s = 436, 1024, 9
    p = pkg("params").for_k(300, H=H, W=W)
    a, b, _, _ = synth.make_pair(H, W, 4)
    desc = [ops.daisy(dev(a)), ops.daisy(dev(b))]
    ioc = pkg("io_contract")
    for d in (0, 1):
        pvec, lcost, nprop, labels = ops.knn_proposals(desc[d], desc[1 - d], p)
        P, L = ioc.unpack_proposals(pvec.cpu().numpy()), lcost.cpu().numpy().astype(np.float64)
        N, B = nprop.cpu().numpy().astype(np.int64), labels.cpu().numpy().astype(np.int64)
        ops.random_proposals(desc[d], desc[1 - d], p, pvec, lcost, nprop, labels, seed=s + d)
        draws, margin = pd.seeded_draws(H, W, p.n_gauss, p.sigma, s + d)
        assert int((margin < pd.AMBIGUOUS).sum()) == 0
        h1, h2 = desc[d].cpu().numpy(), desc[1 - d].cpu().numpy()
        P2, L2, N2 = cport.nasumicni(h1, h2, P, L, N, B, oracle_params(p), draws=draws)
        assert_equal_arrays((pvec.cpu().numpy(), lcost.cpu().numpy().astype(np.float64), nprop.cpu().numpy()),
                            P2, L2, N2)
        assert (N2 > N).mean() > 0.5


# ---------------------------------------------------------------- c. the K-set export over whole arrays
def pack_on_device(pvec, nprop, tpsi):
    """flowb200_ksets_pack into a buffer pre-filled with 0xA5, so that every byte must be written."""
    ops, lib = pkg("ops"), pkg("_lib")
    H, W, K = pvec.shape
    out = torch.full((H, W, 2, K * K // 8 + 1), 0xA5, dtype=torch.uint8, device="cuda")
    rc = lib.load().flowb200_ksets_pack(ops._ptr(pvec), ops._ptr(nprop), H, W, K, int(tpsi), ops._ptr(out),
                                        ops._stream())
    lib.check(rc, "flowb200_ksets_pack")
    return out.cpu().numpy()


EXTREMES = np.array([-32768, -32767, -1, 0, 1, 7, 8, 32766, 32767])


@pytest.mark.parametrize("K", [1, 2, 3, 7, 8, 9, 15, 16, 17, 64, 150])
def test_ksets_pack_whole_arrays(K):
    from oracle import proposals as oprop
    ioc = pkg("io_contract")
    rng = np.random.default_rng(K)
    for H, W in ((3, 4), (1, 6), (5, 1)):
        P = rng.integers(-6, 7, (H, W, K, 2))
        ext = rng.random((H, W, K)) < 0.3
        P[ext] = EXTREMES[rng.integers(0, len(EXTREMES), (int(ext.sum()), 2))]
        N = rng.integers(0, K + 1, (H, W))
        N.flat[0], N.flat[-1] = 0, K
        if H * W > 2:
            N.flat[1] = K
        P[np.arange(K)[None, None, :] >= N[..., None]] = -1          # unused rows: the (-1, -1) fill
        pvec, nprop = dev(ioc.pack_proposals(P)), dev(N.astype(np.int32))
        for tpsi in (-1, 0, 1, 8, 33, 2 ** 31 - 1):
            want = oprop.pakovanje(P, N, oprop.Params(H, W, maxnprop=K, tpsi=tpsi, n_gauss=0, k_cell=1,
                                                      cell_radius=0, cellw=1, cellh=1))
            got = pack_on_device(pvec, nprop, tpsi)
            assert np.array_equal(got, want), (H, W, tpsi, int((got != want).sum()))
            bits = np.unpackbits(got, axis=-1)
            assert not bits[..., K * K:].any()                   # the trailing bits (the whole last byte when 8 | K*K)
            if tpsi <= 0:
                assert not bits.any()
            if tpsi == 2 ** 31 - 1:                              # every pair inside the mask is near
                assert bits.sum() == sum(int(N[y, x]) * int(N[y + dy, x + dx]) for y in range(H) for x in range(W)
                                         for dy, dx in ((1, 0), (0, 1)) if y + dy < H and x + dx < W)


# ---------------------------------------------------------------- d. argument checks
def entry_rows():
    """(entry, overrides, expected code).  Defaults: a 12 x 16 frame of 4 x 4 cells, radius 1, k 2, n_gauss 3."""
    R = []
    for e in ("knn0", "knn1", "random"):
        R.append((e, {}, OK))
        ptrs = ("src", "tgt", "pvec", "lcost", "nprop", "labels") + (("ws",) if e == "knn1" else ())
        R += [(e, {"null": q}, EINVAL) for q in ptrs + ("params",)]
        R += [(e, {"H": 0}, EINVAL), (e, {"W": 0}, EINVAL), (e, {"H": 16385, "W": 4}, EINVAL),
              (e, {"H": 4, "W": 16385}, EINVAL), (e, {"W": 3}, EINVAL), (e, {"H": 3}, EINVAL),
              (e, {"k": 0}, EINVAL), (e, {"k": 17}, EINVAL), (e, {"R": -1}, EINVAL), (e, {"ng": -1}, EINVAL),
              (e, {"K": "min-1"}, EINVAL), (e, {"K": 513}, EINVAL), (e, {"K": 512}, OK)]
    R += [("knn0", {"null": "idx"}, OK), ("knn1", {"null": "idx"}, OK), ("random", {"draws": True}, OK)]
    R += [("knn0", {"mode": 2}, EINVAL), ("knn0", {"mode": -1}, EINVAL), ("random", {"mode": 7}, OK)]
    R += [("knn0", {"k": k}, EUNSUPPORTED) for k in (6, 7, 9, 11, 13)]
    R += [("knn1", {"k": k, "cw": 8}, EUNSUPPORTED) for k in (1, 2, 4, 6, 8, 16)]
    R += [("knn0", {"k": k}, OK) for k in (1, 3, 4, 5, 8, 10, 12, 16)]
    R += [("knn1", {"cw": 4, "ch": 7, "k": 5}, EUNSUPPORTED), ("knn1", {"ws": "1"}, EWORKSPACE), ("knn0", {"ws": "1"}, OK)]
    R += [("knn0", {"H": 16384, "W": 4, "cw": 4, "ch": 16, "R": 0, "k": 1, "ng": 0}, OK),
          ("knn1", {"H": 4, "W": 16384, "cw": 16, "ch": 4, "R": 0, "k": 5, "ng": 0}, OK),
          ("random", {"H": 16384, "W": 4, "cw": 4, "ch": 16, "R": 0, "k": 1, "ng": 1}, OK)]
    # radius 0: refused with random proposals on a ragged frame only
    R += [("random", {"R": 0, "H": 13}, EUNSUPPORTED), ("random", {"R": 0, "W": 17}, EUNSUPPORTED),
          ("random", {"R": 0}, OK), ("random", {"R": 0, "H": 13, "ng": 0}, OK),
          ("random", {"R": 0, "H": 13, "null": "pvec"}, EINVAL), ("random", {"R": 0, "H": 13, "K": 513}, EINVAL),
          ("knn0", {"R": 0, "H": 13}, OK), ("knn1", {"R": 0, "H": 13, "cw": 8, "k": 5}, OK),
          ("random", {"ng": 0, "null": "pvec"}, EINVAL)]
    R += [("pack", {}, OK)] + [("pack", {"null": q}, EINVAL) for q in ("pvec", "nprop", "out")]
    R += [("pack", {"H": 0}, EINVAL), ("pack", {"W": 0}, EINVAL), ("pack", {"H": -1}, EINVAL),
          ("pack", {"K": 0}, EINVAL), ("pack", {"K": 513}, EINVAL), ("pack", {"K": 512, "H": 1, "W": 2}, OK),
          ("pack", {"H": 16385, "W": 1, "K": 1}, OK), ("pack", {"tpsi": -5}, OK),
          ("pack", {"H": 4096, "W": 1024, "K": 512, "dummy": True}, EINVAL)]      # 2^38 + 2^23 bytes
    return R


ROWS = entry_rows()


def row_id(r):
    e, ov, rc = r
    return f"{e}-" + ("-".join(f"{k}={v}" for k, v in ov.items()) or "defaults") + f"-rc{rc}"


def call_entry(e, ov):
    ops, L = pkg("ops"), pkg("_lib")
    lib = L.load()
    a = dict(H=12, W=16, cw=4, ch=4, R=1, k=2, ng=3, K=None, mode=0 if e != "knn1" else 1, tpsi=8, ws=None)
    a.update({k: v for k, v in ov.items() if k not in ("null", "dummy", "draws")})
    if e == "knn1" and "k" not in ov and "cw" not in ov:
        a.update(cw=8, k=5)                       # a geometry the tensor-core search takes (T = 32, k = 5)
    nmin = (2 * a["R"] + 1) ** 2 * a["k"] + a["ng"] if a["R"] >= 0 else 1
    K = {None: nmin, "min-1": nmin - 1}.get(a["K"], a["K"])
    H, W = max(a["H"], 1), max(a["W"], 1)
    if ov.get("dummy"):
        H = W = 1
    Kb = max(K, 1)
    null = ov.get("null")
    buf = dict(src=torch.zeros((H, W, 68), device="cuda"), tgt=torch.zeros((H, W, 68), device="cuda"),
               pvec=torch.zeros((H, W, Kb), dtype=torch.int32, device="cuda"),
               lcost=torch.zeros((H, W, Kb), device="cuda"),
               nprop=torch.zeros((H, W), dtype=torch.int32, device="cuda"),
               labels=torch.zeros((H, W), dtype=torch.int32, device="cuda"),
               idx=torch.zeros((H, W, 9 * max(a["k"], 1) * max(1, (2 * max(a["R"], 0) + 1) ** 2)), dtype=torch.int32,
                               device="cuda"),
               draws=torch.zeros((H, W, max(a["ng"], 1), 2), dtype=torch.int16, device="cuda"),
               out=torch.zeros((H, W, 2, Kb * Kb // 8 + 1), dtype=torch.uint8, device="cuda"))
    P = {k: C.c_void_p(0 if null == k else t.data_ptr()) for k, t in buf.items()}
    s = ops._stream()
    if e == "pack":
        rc = lib.flowb200_ksets_pack(P["pvec"], P["nprop"], a["H"], a["W"], K if a["K"] is not None else 8,
                                     a["tpsi"], P["out"], s)
        torch.cuda.synchronize()
        return rc
    cp = L.CParams(H=a["H"], W=a["W"], cellw=a["cw"], cellh=a["ch"], cell_radius=a["R"], k_cell=a["k"],
                   n_gauss=a["ng"], sigma=8.0, maxnprop=K, tphi=2.5, tpsi=8, lamda=0.05, cost_shift=12,
                   bcd_mode=0, knn_mode=a["mode"], con_tresh=10.0, cell_x0=0, cell_x1=0)
    pp = None if null == "params" else C.byref(cp)
    if e == "random":
        rc = lib.flowb200_random_proposals(P["src"], P["tgt"], pp, P["pvec"], P["lcost"], P["nprop"], P["labels"],
                                           P["draws"] if ov.get("draws") else C.c_void_p(0), C.c_uint64(3), s)
    else:
        need = int(lib.flowb200_knn_workspace_bytes(C.byref(cp)))
        nb = 1 if a["ws"] == "1" else max(need, 256)
        ws = torch.zeros(nb, dtype=torch.uint8, device="cuda")
        rc = lib.flowb200_knn_proposals(P["src"], P["tgt"], pp, P["pvec"], P["lcost"], P["nprop"], P["labels"],
                                        P["idx"] if null != "idx" else C.c_void_p(0), C.c_void_p(0),
                                        C.c_void_p(0) if null == "ws" else C.c_void_p(ws.data_ptr()), nb, s)
    torch.cuda.synchronize()
    return rc


@pytest.mark.parametrize("entry,ov,rc", ROWS, ids=[row_id(r) for r in ROWS])
def test_entry_return_code(entry, ov, rc):
    assert call_entry(entry, ov) == rc
