"""The restatement of the seeded random-proposal draws (tests/philox_draws.py) on the CPU, and why radius 0 on a ragged
frame is refused: the Random123 known answers of Philox4x32-10, the distribution of the accepted draws against the
exact probabilities of trunc(N(y, sigma)) conditioned on the frame, the two halves of the 64-bit seed, and the
reference's scan order deciding the result when pixels without NN proposals publish their first random proposal."""
import numpy as np
import pytest
from scipy import stats

import philox_draws as pd

P_FLOOR = 1e-6


@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
], ids=["zero", "ones", "pi"])
def test_philox_known_answers(ctr, key, want):
    got = pd.philox4x32_10(np.array(ctr, np.uint64), np.array(key, np.uint64))
    assert got.dtype == np.uint32 and tuple(int(v) for v in got) == want


def trunc_normal_probs(pos, size, sigma):
    """P(trunc(pos + sigma Z) = pos + d | in [0, size)) for d = -pos .. size-1-pos (exact, scipy.stats.norm)."""
    t = np.arange(size, dtype=np.float64)
    lo = np.where(t > 0, t, -1.0)           # trunc maps (-1, 1) to 0 and [t, t+1) to t > 0
    cdf = stats.norm.cdf
    p = cdf((t + 1 - pos) / sigma) - cdf((lo - pos) / sigma)
    return p / p.sum()


def chi2_pvalue(counts, probs):
    """Chi-square of observed counts against probabilities, bins with an expectation below 5 merged into one."""
    n = counts.sum()
    exp = probs * n
    keep = exp >= 5
    obs = np.append(counts[keep], counts[~keep].sum())
    e = np.append(exp[keep], exp[~keep].sum())
    if e[-1] < 5:
        obs[-2] += obs[-1]
        e[-2] += e[-1]
        obs, e = obs[:-1], e[:-1]
    return stats.chisquare(obs, e * (obs.sum() / e.sum())).pvalue


# (frame size along the tested axis, position, sigma): an interior row, the first row (where (-1, 0) truncates to 0
# as well, so it holds twice its share), the last row, a one-row frame
AXIS_CASES = [(436, 200, 8.0), (436, 0, 8.0), (436, 435, 8.0), (1, 0, 8.0), (90, 3, 30.0)]


@pytest.mark.parametrize("axis", ["y", "x"])
@pytest.mark.parametrize("size,pos,sigma", AXIS_CASES, ids=[f"{s}-{p}-{g:g}" for s, p, g in AXIS_CASES])
def test_draw_distribution(size, pos, sigma, axis):
    """About 10^6 accepted draws of one position: their offsets follow trunc(N(pos, sigma)) conditioned on the frame.
    The other coordinate sits in the middle of a wide frame."""
    npix, ng = (20000, 50) if size > 1 else (2000, 50)
    other, wide = 8192, 16384
    y, x, H, W = (pos, other, size, wide) if axis == "y" else (other, pos, wide, size)
    d, margin, used = pd.draws_at(np.arange(npix), np.full(npix, y), np.full(npix, x), H, W, ng, sigma, seed=12345)
    v = d[..., 0 if axis == "y" else 1].ravel()
    assert v.min() >= 0 and v.max() < size
    if size > 1:
        counts = np.bincount(v, minlength=size).astype(np.float64)
        p = chi2_pvalue(counts, trunc_normal_probs(pos, size, sigma))
        assert p > P_FLOOR, p
    assert (margin < pd.AMBIGUOUS).sum() == 0
    if size == 1:       # the acceptance rate is P(|sigma Z| < 1)
        rate = npix * ng / used.sum()
        assert abs(rate - (2 * stats.norm.cdf(1 / sigma) - 1)) < 0.005, rate


def test_seed_halves_are_independent():
    """Seed 1 keys (1, 0) and seed 2^32 keys (0, 1): different streams; both differ from seed 0."""
    a, _ = pd.seeded_draws(16, 24, 25, 8.0, 1)
    b, _ = pd.seeded_draws(16, 24, 25, 8.0, 2 ** 32)
    c, _ = pd.seeded_draws(16, 24, 25, 8.0, 0)
    assert list(pd.seed_key(2 ** 64 - 1)) == [0xFFFFFFFF, 0xFFFFFFFF] and list(pd.seed_key(2 ** 32)) == [0, 1]
    assert (a != b).any(axis=-1).mean() > 0.9 and (a != c).any(axis=-1).mean() > 0.9
    assert (b != c).any(axis=-1).mean() > 0.9


def test_counter_is_per_pixel_and_attempt():
    """The first attempt of pixel p is Philox((p, 0, 0, 0)); a pixel's draws do not depend on the frame around it
    except through the bounds."""
    H, W = 40, 50
    d, _ = pd.seeded_draws(H, W, 5, 8.0, 99)
    one, _, _ = pd.draws_at([17 * W + 23], [17], [23], H, W, 5, 8.0, 99)
    assert np.array_equal(d[17, 23], one[0])
    r = pd.philox4x32_10(np.array([17 * W + 23, 0, 0, 0], np.uint64), pd.seed_key(99)).astype(np.float64)
    u = (r + 0.5) * 2.0 ** -32
    ty = int(np.trunc(17 + 8.0 * np.sqrt(-2 * np.log(u[0])) * np.cos(2 * np.pi * u[1])))
    tx = int(np.trunc(23 + 8.0 * np.sqrt(-2 * np.log(u[2])) * np.cos(2 * np.pi * u[3])))
    if 0 <= ty < H and 0 <= tx < W:
        assert (ty, tx) == tuple(d[17, 23, 0])


# ---------------------------------------------------------------- the scan order at radius 0 on a ragged frame
def scan_order_case(R):
    """10 x 13 frame, 4 x 4 cells (2 remainder rows, 1 remainder column: 34 pixels outside the cell grid), k = 1,
    3 draws; the first draw of every remainder pixel aims at a pixel inside the grid, the other two at another
    remainder pixel."""
    from oracle import proposals as oprop
    H, W = 10, 13
    p = oprop.Params(H, W, 4, 4, cell_radius=R, k_cell=1, n_gauss=3, maxnprop=(2 * R + 1) ** 2 + 3)
    rng = np.random.default_rng(5)
    d1 = rng.random((H, W, 68), dtype=np.float32)
    d2 = rng.random((H, W, 68), dtype=np.float32)
    P, L, N, B = oprop.generisi(d1, d2, p)
    rem = np.zeros((H, W), bool)
    rem[p.ncelly * p.cellh:] = True
    rem[:, p.ncellx * p.cellw:] = True
    ry, rx = np.nonzero(rem)
    draws = np.stack([np.clip(np.trunc(rng.normal(np.arange(H)[:, None, None], 3.0, (H, W, 3))), 0, H - 1),
                      np.clip(np.trunc(rng.normal(np.arange(W)[None, :, None], 3.0, (H, W, 3))), 0, W - 1)], -1)
    draws = draws.astype(np.int64)
    for y, x in zip(ry, rx):
        draws[y, x, 0] = (rng.integers(p.ncelly * p.cellh), rng.integers(p.ncellx * p.cellw))
        for i in (1, 2):
            j = int(rng.integers(len(ry)))
            draws[y, x, i] = (ry[j], rx[j])
    runs = []
    for snap in (False, True):
        P2, L2, N2 = oprop.nasumicni(d1, d2, P.copy(), L.copy(), N.copy(), B, p, draws, snapshot=snap)
        runs.append((P2, L2, N2))
    return rem, N, runs


def test_scan_order_decides_radius_0_on_a_ragged_frame():
    """At radius 0 the remainder pixels have no NN proposal: their first accepted random proposal lands in slot 0,
    which other pixels read as their best vector.  The reference's x-major scan then shows it to the pixels scanned
    later and not to the earlier ones, so no order-free (parallel) evaluation reproduces it:
    flowb200_random_proposals refuses this configuration."""
    rem, N, ((Px, Lx, Nx), (Ps, Ls, Ns)) = scan_order_case(0)
    assert rem.sum() == 34 and (N[rem] == 0).all() and (N[~rem] == 1).all()
    differ = (Px != Ps).any(axis=(-1, -2)) | (Nx != Ns)
    assert differ[rem].sum() >= 17, differ[rem].sum()


def test_scan_order_is_moot_when_every_pixel_has_nn_proposals():
    """At radius 1 on the same frame every pixel searches a cell, neighbours' best vectors are NN slots that the pass
    never rewrites, and the two orders agree exactly."""
    rem, N, ((Px, Lx, Nx), (Ps, Ls, Ns)) = scan_order_case(1)
    assert (N > 0).all()
    assert np.array_equal(Px, Ps) and np.array_equal(Lx, Ls) and np.array_equal(Nx, Ns)
    assert (Nx > N).any()
