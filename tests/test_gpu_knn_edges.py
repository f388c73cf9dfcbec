"""The proposal search at its edges, both search modes, against the oracle's exact search.  GPU only.

The other search tests feed DAISY of noise textures: no flat regions, no ties below fp16 resolution, two cell
geometries.  Real frames have saturated sky, black borders and uniform walls; DAISY has no normalisation here, so a
flat region gives descriptors that are exactly zero, and its rim gives squared distances that are float32 subnormals.
This module covers
  - every cell geometry knn_tc_supported admits, at and around its limits, ragged frames and one-cell frames;
  - exact ties and near-ties: zero cells, duplicates that straddle rank k / k+1, near-duplicate groups that route a
    task through the one-round re-rank, the two-round re-rank and the brute-force fallback, screening distances
    whose relative gap is 1e-7 / 1e-5 / 3e-5 (exact screening distances, and ones that carry 68 roundings),
    subnormal screening distances, descriptors at the top of DAISY's range;
  - a frame with real flat regions through DAISY, search, random proposals and BCD (mass cost ties);
  - more overflowed (query, cell) tasks than the fallback list holds (1024x436, K = 300, flat top third), and the
    same with radius 0 on a ragged frame, whose remainder pixels have no task, in a workspace full of 0xFF.
Every comparison is over whole arrays, bit for bit: proposals, float32 data costs, nprop, labels and kNN indices.
"""
import math

import numpy as np
import pytest

from helpers import pkg

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

KNN_MODES = [0, 1]     # 0 = float64 CUDA cores, 1 = tcgen05 prefilter + exact re-rank


def dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda()


def flow_params(H, W, cw, ch, R=2, k=5, **kw):
    kw.setdefault("n_gauss", 0)
    kw.setdefault("maxnprop", (2 * R + 1) ** 2 * k + kw["n_gauss"])
    return pkg("params").FlowParams(H=H, W=W, cellw=cw, cellh=ch, cell_radius=R, k_cell=k, **kw)


def oracle_params(p):
    from oracle import proposals as oprop
    return oprop.Params(p.H, p.W, p.cellw, p.cellh, cell_radius=p.cell_radius, k_cell=p.k_cell, n_gauss=p.n_gauss,
                        sigma=p.sigma, maxnprop=p.maxnprop, tphi=p.tphi)


def gpu_search(d1, d2, p, mode):
    ops = pkg("ops")
    pvec, lcost, nprop, labels, idx, stats = ops.knn_proposals(dev(d1), dev(d2), p, want_idx=True, knn_mode=mode)
    return dict(pvec=pvec.cpu().numpy(), lcost=lcost.cpu().numpy().astype(np.float64), nprop=nprop.cpu().numpy(),
                labels=labels.cpu().numpy(), idx=idx.cpu().numpy(), stats=stats.cpu().numpy())


def oracle_search(d1, d2, p):
    from oracle import cport
    P, L, N, B, idx = cport.generisi(d1, d2, oracle_params(p), want_idx=True)
    return dict(pvec=pkg("io_contract").pack_proposals(P), lcost=L, nprop=N, labels=B, idx=idx)


def assert_search_equal(got, want):
    for key in ("nprop", "idx", "pvec", "lcost", "labels"):
        assert np.array_equal(got[key], want[key]), (key, float((got[key] != want[key]).mean()))


def random_desc(rng, H, W):
    """float32 (H, W, 68) in DAISY's range [0, 0.5], skewed towards 0 like DAISY's histograms, 5 % exact zeros."""
    d = (rng.random((H, W, 68), dtype=np.float32) ** 3 * np.float32(0.5)).astype(np.float32)
    d[rng.random((H, W, 68)) < 0.05] = 0
    return d


def stride_s(T):
    """The decimating permutation of a cell's targets in knn_tc.cu (make_tc_geom): position pos holds pos*s mod T."""
    s = max(1, int(0.41421356 * T))
    while math.gcd(s, T) != 1:
        s += 1
    return s


def set_target(d2, p, ci, cj, i, v):
    d2[cj * p.cellh + i // p.cellw, ci * p.cellw + i % p.cellw] = v


def spread_indices(rng, T, n):
    """n target indices of a cell whose permuted positions are evenly spread (randomly offset): with n >= 6 every
    32-column group of a 192-target cell holds one, so the prefilter's bound is the score they share."""
    pos = (int(rng.integers(T)) + np.arange(n) * (T // n)) % T
    return (pos * stride_s(T)) % T


# ---------------------------------------------------------------- geometry sweep
# (H, W, cellw, cellh, cell_radius, k_cell): T = cellw * cellh at and around knn_tc_supported's limits, 1-pixel-wide
# and 1-pixel-high cells (divisions by 1 via the 0xffffffff reciprocal), k 5 / 10 / 12, radius 1 / 2 / 3, frames whose
# size is no multiple of the cell, of 16 or of 8, frames narrower than 2R+1 cells and frames of exactly one cell
GEOMETRIES = [
    (43, 61, 8, 4, 2, 5),          # T = 32: one chunk, 96 padding rows
    (50, 71, 16, 8, 2, 10),        # T = 128: one full chunk
    (61, 83, 13, 11, 2, 12),       # T = 143
    (110, 300, 73, 25, 2, 5),      # the reference's cells, ragged right and bottom
    (100, 200, 64, 32, 1, 12),     # T = 2048, radius 1
    (37, 390, 128, 16, 2, 10),     # T = 2048, 3 x 2 cells: narrower than 2R+1 cells both ways
    (101, 9, 1, 40, 2, 5),         # cellw = 1, T = 40
    (7, 130, 48, 1, 2, 10),        # cellh = 1, T = 48
    (60, 90, 12, 10, 3, 10),       # radius 3: 49 cells x 10 = 490 proposals
    (25, 73, 73, 25, 2, 5),        # exactly one cell
    (30, 80, 73, 25, 1, 12),       # one cell and a ragged rim
]


# the float64 search's other compiled widths (knn_exact_dispatch: k = 1, 2, 3, 4, 8, 16; the tensor-core search has
# only 5 / 10 / 12) on ragged frames: topk_insert<1> has no shift loop, <16> the longest
FP64_GEOMETRIES = [
    (43, 61, 8, 4, 2, 1),
    (50, 71, 16, 8, 1, 2),
    (61, 83, 13, 11, 2, 3),
    (37, 53, 4, 4, 3, 4),          # k = T / 4
    (101, 9, 1, 40, 2, 8),
    (45, 70, 8, 2, 2, 16),         # k = T: every target of a cell is a neighbour
    (60, 90, 12, 10, 1, 16),
]
SWEEP = [(g, m) for g in GEOMETRIES for m in KNN_MODES] + [(g, 0) for g in FP64_GEOMETRIES]


@pytest.mark.parametrize("geom,knn_mode", SWEEP, ids=["x".join(map(str, g)) + f"-{m}" for g, m in SWEEP])
def test_geometry_sweep(geom, knn_mode):
    H, W, cw, ch, R, k = geom
    rng = np.random.default_rng(H * 7 + W)
    d1, d2 = random_desc(rng, H, W), random_desc(rng, H, W)
    d2[H // 2, : W // 2] = d2[H // 3, : W // 2]            # some exact duplicate targets as well
    p = flow_params(H, W, cw, ch, R, k)
    assert_search_equal(gpu_search(d1, d2, p, knn_mode), oracle_search(d1, d2, p))


@pytest.mark.parametrize("geom", [(40, 62, 31, 1, 2, 5),      # T = 31
                                  (9, 700, 683, 3, 2, 5),     # T = 2049
                                  (48, 80, 16, 12, 2, 7)],    # k = 7
                         ids=["T31", "T2049", "k7"])
def test_unsupported_geometry_raises_in_tcgen05_mode(geom):
    """Outside knn_tc_supported the tensor-core search refuses (no silent fall-back); the float64 search takes the
    cell sizes (it has no kernel for k = 7 and refuses that too)."""
    lib = pkg("_lib")
    H, W, cw, ch, R, k = geom
    rng = np.random.default_rng(1)
    d1, d2 = random_desc(rng, H, W), random_desc(rng, H, W)
    p = flow_params(H, W, cw, ch, R, k)
    with pytest.raises(lib.FlowB200Error):
        gpu_search(d1, d2, p, 1)
    if k == 7:
        with pytest.raises(lib.FlowB200Error):
            gpu_search(d1, d2, p, 0)
    else:
        assert_search_equal(gpu_search(d1, d2, p, 0), oracle_search(d1, d2, p))


@pytest.mark.parametrize("k", [6, 7, 9])
def test_float64_search_refuses_widths_it_does_not_compile(k):
    """k = 6, 7, 9 fit the cell but have no knn_exact_kernel instance: FLOWB200_EUNSUPPORTED in mode 0."""
    lib = pkg("_lib")
    rng = np.random.default_rng(k)
    p = flow_params(24, 36, 4, 6, 1, k)
    d1, d2 = random_desc(rng, p.H, p.W), random_desc(rng, p.H, p.W)
    with pytest.raises(lib.FlowB200Error, match="unsupported"):
        gpu_search(d1, d2, p, 0)


# ---------------------------------------------------------------- ties and near-ties
# 5 x 4 cells of 16 x 12 (T = 192, Tpad = 256), radius 2, k = 5
TH, TW, TCW, TCH = 48, 80, 16, 12


def tie_params():
    return flow_params(TH, TW, TCW, TCH, 2, 5)


def far_targets(rng, n):
    """Targets far from every query the constructions below use."""
    return (0.05 + 0.45 * rng.random((n, 68))).astype(np.float32)


def on_grid(rng, shape):
    """Values j / 1024 in [0.125, 0.375]: 64 x value is an fp16 number, so perturbations below 2^-12 leave the fp16
    operands of the tensor-core scores unchanged."""
    return (rng.integers(128, 385, shape) / 1024.0).astype(np.float32)


def case_all_zero(rng, p):
    return np.zeros((p.H, p.W, 68), np.float32), np.zeros((p.H, p.W, 68), np.float32)


def case_zero_cells(rng, p):
    d1, d2 = random_desc(rng, p.H, p.W), random_desc(rng, p.H, p.W)
    d2[0:2 * TCH, 0:2 * TCW] = 0                   # four whole target cells
    d2[3 * TCH:, 4 * TCW:] = 0                     # the corner cell
    d1[TCH:3 * TCH, TCW:3 * TCW + 5] = 0           # zero queries, partly over nonzero targets
    return d1, d2


def case_straddling_duplicates(rng, p):
    """Queries = v.  In every cell: k-1 distinct near targets, then 2-4 exact copies of u at ranks k, k+1, ...; the
    copy with the lowest index is never the one with the lowest permuted position."""
    T, k = p.cellw * p.cellh, p.k_cell
    s = stride_s(T)
    pos = (np.arange(T) * pow(s, -1, T)) % T          # position of target index i in the permuted order
    v = on_grid(rng, 68)
    d1 = np.broadcast_to(v, (p.H, p.W, 68)).copy()
    d2 = random_desc(rng, p.H, p.W)
    for ci in range(p.ncellx):
        for cj in range(p.ncelly):
            for i in range(T):
                set_target(d2, p, ci, cj, i, far_targets(rng, 1)[0])
            m = int(rng.integers(2, 5))
            while True:
                sel = rng.choice(T, k - 1 + m, replace=False)
                dup = np.sort(sel[k - 1:])
                if pos[dup[0]] != pos[dup].min():
                    break
            for r, i in enumerate(sel[:k - 1]):
                set_target(d2, p, ci, cj, i, v + np.float32(0.002 * (r + 1)))
            u = v + np.float32(0.002 * k)
            u[int(rng.integers(68))] += np.float32(0.001)    # (distinct from the near ones' direction)
            for i in dup:
                set_target(d2, p, ci, cj, i, u)
    return d1, d2


def near_duplicate_groups(size):
    """Every cell holds `size` targets u + (perturbations below 2^-12) and queries are u + the same kind of
    perturbation: all of them have the same fp16 operands, so a task has exactly `size` candidates (<= 16: one
    re-rank round, 17-32: two rounds, >= 33: brute-force fallback) while the exact distances all differ."""
    def build(rng, p):
        T = p.cellw * p.cellh
        u = on_grid(rng, 68)

        def jitter(n):
            e = np.zeros((n, 68), np.float32)
            dims = rng.integers(0, 68, (n, 3))
            for j in range(3):
                e[np.arange(n), dims[:, j]] = rng.integers(-200, 201, n) * np.float32(2.0 ** -32)
            return u + e
        d1 = jitter(p.H * p.W).reshape(p.H, p.W, 68)
        d2 = np.zeros((p.H, p.W, 68), np.float32)
        for ci in range(p.ncellx):
            for cj in range(p.ncelly):
                grp = set(spread_indices(rng, T, size).tolist())
                near, far = jitter(T), far_targets(rng, T)
                for i in range(T):
                    set_target(d2, p, ci, cj, i, near[i] if i in grp else far[i])
        return d1, d2
    return build


def gap_pairs(gap):
    """Queries = v.  In every cell the two nearest targets are A = v + a e0 and B = v + a e0 + c e1 with c^2 = gap a^2,
    so the screening distances differ by about `gap` relative (and are exact); B has the lower index in half of the
    cells."""
    def build(rng, p):
        T = p.cellw * p.cellh
        v = on_grid(rng, 68)
        d1 = np.broadcast_to(v, (p.H, p.W, 68)).copy()
        d2 = np.zeros((p.H, p.W, 68), np.float32)
        a = np.float32(2.0 ** -4)
        A = v.copy()
        A[0] += a
        B = A.copy()
        B[1] = np.float32(v[1] + np.float32(a * math.sqrt(gap)))
        got = float((np.float64(B[1]) - np.float64(v[1])) ** 2 / (np.float64(A[0]) - np.float64(v[0])) ** 2)
        assert 0.8 * gap < got < 1.25 * gap, got
        for n, (ci, cj) in enumerate((ci, cj) for ci in range(p.ncellx) for cj in range(p.ncelly)):
            far = far_targets(rng, T)
            for i in range(T):
                set_target(d2, p, ci, cj, i, far[i])
            lo, hi = np.sort(rng.choice(T, 2, replace=False))
            set_target(d2, p, ci, cj, lo, B if n % 2 else A)
            set_target(d2, p, ci, cj, hi, A if n % 2 else B)
        return d1, d2
    return build


def dense_gap_pairs(gap):
    """Queries = v.  In every cell two pairs (A, B) at different distances whose differences from v are of the same order
    in all 68 dimensions, so each float32 screening distance accumulates 68 roundings (up to ~4e-7 relative here, more
    than a 1e-7 gap: about one pair in ten is screened in the wrong order); B's exact distance is A's times 1 + gap to
    within 1 % of the gap, set through dimension 67, where v is 0 and the difference small."""
    def build(rng, p):
        T = p.cellw * p.cellh
        v = (0.1 + 0.3 * rng.random(68)).astype(np.float32)
        v[67] = 0
        v64 = v.astype(np.float64)
        d1 = np.broadcast_to(v, (p.H, p.W, 68)).copy()
        d2 = np.zeros((p.H, p.W, 68), np.float32)

        def pair(scale):
            e = scale * rng.uniform(0.005, 0.02, 68) * rng.choice([-1.0, 1.0], 68)
            e[67] = 0.002 * scale        # small: B's float32 steps there are ~1e-10 of the distance
            A = (v + e).astype(np.float32)
            dA = ((A.astype(np.float64) - v64) ** 2).sum()
            B = (v + e * math.sqrt(1 + gap)).astype(np.float32)
            B[67] = np.float32(math.sqrt(dA * (1 + gap) - ((B[:67].astype(np.float64) - v64[:67]) ** 2).sum()))
            dB = ((B.astype(np.float64) - v64) ** 2).sum()
            assert abs(dB / dA - 1 - gap) < 0.01 * gap, (dB / dA - 1, gap)
            return A, B
        for n, (ci, cj) in enumerate((ci, cj) for ci in range(p.ncellx) for cj in range(p.ncelly)):
            far = far_targets(rng, T)
            for i in range(T):
                set_target(d2, p, ci, cj, i, far[i])
            sel = rng.choice(T, 4, replace=False)
            for m, scale in enumerate((1.0, 1.6)):
                A, B = pair(scale)
                lo, hi = np.sort(sel[2 * m:2 * m + 2])
                set_target(d2, p, ci, cj, lo, B if n % 2 else A)
                set_target(d2, p, ci, cj, hi, A if n % 2 else B)
        return d1, d2
    return build


def tiny_targets(n):
    """Queries = 0.  In every cell n targets whose distances to 0 are below the float32 normal range (their float32
    screening distances are subnormal or 0) and T - n far ones.  The first two are A = 2^-75 in all 68 dimensions and
    B = 2^-74 in dimension 0: fmaf rounds every 2^-150 term of A to 0, so A screens at 0 and B at 2^-148, while the
    exact distances are 17 * 2^-148 for A and 2^-148 for B."""
    def build(rng, p):
        T = p.cellw * p.cellh
        d1 = np.zeros((p.H, p.W, 68), np.float32)
        d2 = np.zeros((p.H, p.W, 68), np.float32)
        A = np.full(68, 2.0 ** -75, np.float32)
        B = np.zeros(68, np.float32)
        B[0] = 2.0 ** -74
        for n_cell, (ci, cj) in enumerate((ci, cj) for ci in range(p.ncellx) for cj in range(p.ncelly)):
            far = far_targets(rng, T)
            tiny = np.zeros((n, 68), np.float32)
            tiny[0], tiny[1] = (A, B) if n_cell % 2 else (B, A)
            for j in range(2, n):
                dims = rng.choice(68, int(rng.integers(1, 69)), replace=False)
                tiny[j, dims] = np.ldexp(1 + rng.random(len(dims)), -rng.integers(70, 80, len(dims))).astype(np.float32)
            sel = spread_indices(rng, T, n)
            for i in range(T):
                set_target(d2, p, ci, cj, i, far[i])
            for j, i in enumerate(sel):
                set_target(d2, p, ci, cj, i, tiny[j])
        return d1, d2
    return build


def case_half_max(rng, p):
    """Descriptors at 0.5 in every dimension (the largest scores, next to the padding rows' 60000 norm): half of the
    targets, a third of the queries; another third of the queries are 0 (the largest distances)."""
    d1, d2 = random_desc(rng, p.H, p.W), random_desc(rng, p.H, p.W)
    d2[rng.random((p.H, p.W)) < 0.5] = 0.5
    r = rng.random((p.H, p.W))
    d1[r < 1 / 3] = 0.5
    d1[r > 2 / 3] = 0
    return d1, d2


TIE_CASES = {
    "all_zero": case_all_zero,
    "zero_cells": case_zero_cells,
    "straddling_duplicates": case_straddling_duplicates,
    "near_dup_12": near_duplicate_groups(12),
    "near_dup_24": near_duplicate_groups(24),
    "near_dup_40": near_duplicate_groups(40),
    "gap_1e-7": gap_pairs(1e-7),
    "gap_1e-5": gap_pairs(1e-5),
    "gap_3e-5": gap_pairs(3e-5),
    "dense_gap_1e-7": dense_gap_pairs(1e-7),
    "dense_gap_1e-5": dense_gap_pairs(1e-5),
    "dense_gap_3e-5": dense_gap_pairs(3e-5),
    "subnormal_pair": tiny_targets(2),
    "subnormal_12": tiny_targets(12),
    "subnormal_24": tiny_targets(24),
    "half_max": case_half_max,
}


@pytest.mark.parametrize("knn_mode", KNN_MODES)
@pytest.mark.parametrize("case", list(TIE_CASES))
def test_ties_and_near_ties(case, knn_mode):
    p = tie_params()
    d1, d2 = TIE_CASES[case](np.random.default_rng(sorted(TIE_CASES).index(case)), p)
    assert d1.dtype == d2.dtype == np.float32 and d1.min() >= 0 and d2.max() <= 0.5
    got = gpu_search(d1, d2, p, knn_mode)
    assert_search_equal(got, oracle_search(d1, d2, p))
    if knn_mode == 1:
        st = got["stats"]
        if case.startswith("subnormal") or case in ("near_dup_12", "near_dup_24"):
            assert st[0] == 0, st       # no brute force: the re-rank alone ordered these tasks
        if case == "near_dup_40":
            assert st[0] == int(got["nprop"].sum()) // p.k_cell, st     # every task overflowed


# ---------------------------------------------------------------- flat regions end to end
FH, FW = 160, 200


def flat_pair():
    """A texture pair with a flat sky band, a black left border and a uniform square that moves between the frames."""
    a, b, _, _ = pkg("synth").make_pair(FH, FW, 3, max_dx=6, max_dy=4, n_rect=2)
    for img, (y, x) in ((a, (95, 120)), (b, (98, 125))):
        img[:80] = (200, 210, 220)
        img[:, :30] = 0
        img[y:y + 40, x:x + 50] = (60, 90, 70)
    return a, b


@pytest.fixture(scope="module")
def flat():
    from oracle import daisy as od
    a, b = flat_pair()
    return a, b, [od.daisy(a), od.daisy(b)]


def test_flat_frame_daisy(flat):
    ops = pkg("ops")
    a, b, want = flat
    for img, w in zip((a, b), want):
        got = ops.daisy(dev(img)).cpu().numpy()
        assert ((w == 0).all(-1)).mean() > 0.25         # the case keeps its point: large exactly-zero areas
        assert ((got == 0) == (w == 0)).all()
        scale = np.abs(w).max(axis=-1, keepdims=True) + 1e-12
        assert (np.abs(got - w) / scale).max() <= 1e-4


@pytest.mark.parametrize("knn_mode", KNN_MODES)
def test_flat_frame_search_random_bcd(flat, knn_mode):
    """Search, random proposals on replayed draws and BCD in every mode after every sweep against the C oracle, on the
    oracle's descriptors of the flat pair (so each stage sees identical inputs): flat regions make exact cost ties."""
    from oracle import cport
    from test_gpu_baseline_configs import make_draws
    ops, lib, ioc = pkg("ops"), pkg("_lib"), pkg("io_contract")
    _, _, (d1, d2) = flat
    p = pkg("params").FlowParams(H=FH, W=FW, knn_mode=knn_mode)          # the reference's 73 x 25 cells, K = 150
    op = oracle_params(p)
    got = gpu_search(d1, d2, p, knn_mode)
    want = oracle_search(d1, d2, p)
    assert_search_equal(got, want)
    P, L, N, B = cport.generisi(d1, d2, op)
    draws = make_draws(FH, FW, p.n_gauss, p.sigma, 5)
    P2, L2, N2 = cport.nasumicni(d1, d2, P, L, N, B, op, draws=draws)
    g1, g2 = dev(d1), dev(d2)
    pvec, lcost, nprop, labels = ops.knn_proposals(g1, g2, p)
    ops.random_proposals(g1, g2, p, pvec, lcost, nprop, labels, draws=dev(draws))
    assert np.array_equal(nprop.cpu().numpy(), N2)
    assert np.array_equal(pvec.cpu().numpy(), ioc.pack_proposals(P2))
    assert np.array_equal(lcost.cpu().numpy().astype(np.float64), L2)
    sweeps, shift = 4, 12
    used = L2 != 1000.0
    m = np.where(used, np.rint(0.05 * L2 * float(1 << shift)), 0.0)
    lq = np.where(used, 20.0 * m / float(1 << shift), 1000.0)
    want_f = cport.ceo_bcd(P2, L2, N2, B, sweeps)
    want_q = cport.ceo_bcd(P2, lq, N2, B, sweeps)
    assert (L2[used] == 0).mean() > 0.2            # mass cost ties: zero queries on zero targets
    for mode, cost, kw, w in ((lib.BCD_FP64_F32COST, lcost, {}, want_f),
                              (lib.BCD_FP64_F64COST, dev(L2, torch.float64), {}, want_f),
                              (lib.BCD_INT32, dev(m.astype(np.int32)), dict(cost_shift=shift), want_q),
                              (lib.BCD_INT32_F32COST, lcost, dict(cost_shift=shift), want_q)):
        lab = labels.clone()
        snaps = ops.bcd(pvec, cost, nprop, lab, sweeps, mode=mode, per_sweep=True, **kw).cpu().numpy()
        for s in range(sweeps):
            assert np.array_equal(snaps[s], w[s]), (mode, s, float((snaps[s] != w[s]).mean()))


# ---------------------------------------------------------------- more overflowed tasks than the fallback list holds
def test_overflow_beyond_the_fallback_list():
    """1024x436, K = 300, top third flat: every query that searches a flat cell ties with all its 1825 targets, which
    is over 2^20 tasks for the brute-force fallback.  The tensor-core search must equal the float64 search over the
    whole arrays (none of those tasks dropped), and sampled tasks must equal the host's exact search."""
    from oracle import proposals as oprop
    ops, params, synth = pkg("ops"), pkg("params"), pkg("synth")
    H, W = 436, 1024
    a, b, _, _ = synth.make_pair(H, W, 0)
    a[:H // 3] = 128
    b[:H // 3] = 128
    d1, d2 = ops.daisy(dev(a)), ops.daisy(dev(b))
    p = params.for_k(300, H=H, W=W)
    ref = ops.knn_proposals(d1, d2, p, want_idx=True, knn_mode=0)
    got = ops.knn_proposals(d1, d2, p, want_idx=True, knn_mode=1)          # (both alive: no reuse of ref's memory)
    stats = got[5].cpu().numpy()
    assert stats[0] > 2 ** 20, stats
    for name, g, w in zip(("pvec", "lcost", "nprop", "labels", "idx"), got[:5], ref[:5]):
        assert torch.equal(g, w), (name, float((g != w).float().mean()))
    rng = np.random.default_rng(4)
    h1, h2 = d1.cpu().numpy(), d2.cpu().numpy()
    cd2 = oprop.cell_descriptors(h2, oracle_params(p))
    idx = got[4]
    R, ncx, ncy = p.cell_radius, p.ncellx, p.ncelly
    in_flat_cells = 0
    for n in range(300):
        y = int(rng.integers(0, H // 3 + 2 * p.cellh)) if n % 2 else int(rng.integers(0, H))
        x = int(rng.integers(0, W))
        cis = [c for c in range(ncx) if p.cellw * (c - R) <= x < p.cellw * (c + R + 1)]
        cjs = [c for c in range(ncy) if p.cellh * (c - R) <= y < p.cellh * (c + R + 1)]
        blk = int(rng.integers(0, len(cis) * len(cjs)))
        ci, cj = cis[blk // len(cjs)], cjs[blk % len(cjs)]
        want = oprop.knn_exact(h1[y, x][None], cd2[ci + cj * ncx], p.k_cell)[0]
        assert np.array_equal(idx[y, x, blk].cpu().numpy(), want), (y, x, ci, cj)
        in_flat_cells += not cd2[ci + cj * ncx].any()
    assert in_flat_cells > 50, in_flat_cells          # the sample reaches the brute-forced ties


def search_in_filled_workspace(d1, d2, p, mode, fill):
    """ops.knn_proposals with a workspace whose bytes are all `fill` instead of whatever the allocator last held there."""
    import ctypes as C
    ops, lib = pkg("ops"), pkg("_lib")
    L = lib.load()
    cp = ops.cparams(p, knn_mode=mode)
    H, W, K = p.H, p.W, p.maxnprop
    out = [torch.empty((H, W, K), dtype=torch.int32, device="cuda"), torch.empty((H, W, K), dtype=torch.float32, device="cuda"),
           torch.empty((H, W), dtype=torch.int32, device="cuda"), torch.empty((H, W), dtype=torch.int32, device="cuda"),
           torch.empty((H, W, (2 * p.cell_radius + 1) ** 2, p.k_cell), dtype=torch.int32, device="cuda"),
           torch.zeros(8, dtype=torch.int32, device="cuda")]
    ws = torch.full((max(int(L.flowb200_knn_workspace_bytes(C.byref(cp))), 256),), fill, dtype=torch.uint8, device="cuda")
    lib.check(L.flowb200_knn_proposals(ops._ptr(d1), ops._ptr(d2), C.byref(cp), *[ops._ptr(t) for t in out],
                                       ops._ptr(ws), ws.numel(), ops._stream()), "flowb200_knn_proposals")
    return out


def test_overflow_scan_skips_pixels_without_cells():
    """Radius 0 on a ragged frame: pixels of the bottom and right remainder strips search no cell, so nothing writes the
    candidate count at their task slot.  A zero target frame makes every other pixel's task overflow (all 64 targets of
    a cell tie), over 2^20 of them, so the fallback scans the counts; with a workspace full of 0xFF (an overflow mark)
    the unwritten counts must not become tasks: those pixels keep nprop 0 and unused slots."""
    ops = pkg("ops")
    H, W = 1203, 1030                    # 16 x 4 cells: 3 remainder rows, 6 remainder columns
    p = flow_params(H, W, 16, 4, R=0, k=5)
    g = torch.Generator(device="cuda").manual_seed(3)
    d1 = torch.rand((H, W, 68), generator=g, device="cuda") ** 3 * 0.5
    d2 = torch.zeros_like(d1)
    got = search_in_filled_workspace(d1, d2, p, 1, 0xFF)
    ref = ops.knn_proposals(d1, d2, p, want_idx=True, knn_mode=0)
    h, w = H // 4 * 4, W // 16 * 16      # the pixels inside the cell grid: one task each
    assert int(got[5][0]) == h * w > 2 ** 20
    for name, a, b in zip(("pvec", "lcost", "nprop", "labels", "idx"), got[:5], ref[:5]):
        assert torch.equal(a, b), (name, float((a != b).float().mean()))
    nprop, idx = got[2], got[4]
    assert (nprop[h:] == 0).all() and (nprop[:, w:] == 0).all() and (nprop[:h, :w] == 5).all()
    assert (idx[h:] == -1).all() and (idx[:, w:] == -1).all()
    assert (idx[:h, :w, 0] == torch.arange(5, dtype=torch.int32, device="cuda")).all()   # equal distances: lowest indices
