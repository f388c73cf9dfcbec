"""The MRF oracles (FLOWB200_BCD_MRF) of tests/mrf_oracle.py: the numpy restatement and the C one (mrf_oracle.c).

- every chain a phase runs reaches the minimum of the energy over all labellings of that chain, the rest fixed, found
  by enumeration (independent of the recurrence; compared as energies, because ties may pick other labels);
- the numpy and C oracles give the same labels after every sweep;
- the energy in integer units never rises from one phase to the next.
Costs are integers or multiples of 2^-S with lamda 1, so that every float64 sum of the oracles is exact.
"""
import itertools

import numpy as np
import pytest

import mrf_oracle as mo
from oracle import bcd as obcd


def case(rng, H, W, K, costs="random", ragged=True, spread=4):
    prop = rng.integers(-spread, spread + 1, (H, W, K, 2)).astype(np.int64)
    nprop = rng.integers(1, K + 1, (H, W)) if ragged else np.full((H, W), K)
    if ragged:
        nprop.flat[0] = 1
    prop[np.arange(K)[None, None, :] >= nprop[..., None]] = -1
    hi = 3 if costs == "ties" else 40
    lc = rng.integers(0, hi, (H, W, K)).astype(np.float64)
    lc[np.arange(K)[None, None, :] >= nprop[..., None]] = 1000.0
    lab0 = rng.integers(0, 1 << 30, (H, W)) % nprop
    return prop, lc, nprop.astype(np.int64), lab0.astype(np.int64)


def energy_int(prop, lc, labels, lamda, tpsi):
    """lamda * sum lcost + sum over 4-connected pairs of min(L1, tpsi), exact for integer costs and lamda 1"""
    H, W = labels.shape
    ys, xs = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    v = prop[ys, xs, labels]
    e = lamda * lc[ys, xs, labels].sum()
    e += np.minimum(tpsi, np.abs(v[1:] - v[:-1]).sum(-1)).sum()
    e += np.minimum(tpsi, np.abs(v[:, 1:] - v[:, :-1]).sum(-1)).sum()
    return e


def chain_pixels(phase, H, W, start):
    ystep, xstep = mo.PHASES[phase]
    L = H if ystep else W
    return [(start[0] + i * ystep, start[1] + i * xstep) for i in range(L)]


def chain_minimum(prop, lc, nprop, labels, pix, lamda, tpsi):
    """min over every labelling of the chain `pix` of the energy terms that involve it, the rest of labels fixed;
    and the same terms at labels"""
    H, W = labels.shape
    combos = np.array(list(itertools.product(*[range(int(nprop[y, x])) for y, x in pix])), dtype=np.int64)
    onchain = set(pix)

    def terms(lab):   # lab: (n, len) -> (n,)
        e = np.zeros(len(lab))
        for i, (y, x) in enumerate(pix):
            v = prop[y, x, lab[:, i]]
            e += lamda * lc[y, x, lab[:, i]]
            for dy, dx in ((0, 1), (0, -1), (1, 0), (-1, 0)):
                yy, xx = y + dy, x + dx
                if not (0 <= yy < H and 0 <= xx < W):
                    continue
                if (yy, xx) in onchain:
                    if (dy, dx) in ((0, 1), (1, 0)):   # each pair inside the chain once
                        u = prop[yy, xx, lab[:, pix.index((yy, xx))]]
                        e += np.minimum(tpsi, np.abs(v - u).sum(-1))
                else:
                    u = prop[yy, xx, labels[yy, xx]]
                    e += np.minimum(tpsi, np.abs(v - u[None]).sum(-1))
        return e
    cur = np.array([[labels[y, x] for y, x in pix]])
    return terms(combos).min(), terms(cur)[0]


def assert_chains_minimal(prop, lc, nprop, labels, phase, tpsi, lamda, what):
    H, W = labels.shape
    for start in mo.phase_starts(phase, H, W):
        pix = chain_pixels(phase, H, W, start)
        best, got = chain_minimum(prop, lc, nprop, labels, pix, lamda, tpsi)
        assert got == best, (what, phase, start, got, best)


BRUTE_CASES = [(0, 3, "random"), (1, 3, "ties"), (2, 2, "ties"), (3, 1, "random")]   # seed, K, costs


@pytest.mark.parametrize("H,W", [(6, 5), (5, 6), (1, 7), (7, 1)])
@pytest.mark.parametrize("tpsi", [1, 3, 8])
def test_every_chain_reaches_its_minimum(H, W, tpsi):
    """both oracles, after every phase: every chain of the phase"""
    lamda = 1.0
    for seed, K, costs in BRUTE_CASES:
        rng = np.random.default_rng(seed * 1000 + H * 10 + W + tpsi)
        prop, lc, nprop, lab0 = case(rng, H, W, K, costs, spread=2 if costs == "ties" else 4)
        labels = lab0.copy()
        for sweep in range(2):
            for phase in range(4):
                mo.run_phase(prop, lc, nprop, labels, phase, tpsi, lamda)
                assert_chains_minimal(prop, lc, nprop, labels, phase, tpsi, lamda, ("numpy", seed, sweep))
                lab = mo.ceo_bcd_c(prop, lc, nprop, lab0, sweep + 1, tpsi=tpsi, lamda=lamda, phases=phase + 1)[-1]
                assert np.array_equal(lab, labels), ("C", seed, sweep, phase)
                assert_chains_minimal(prop, lc, nprop, lab, phase, tpsi, lamda, ("C", seed, sweep))


@pytest.mark.parametrize("tpsi", [0, 3, 8, 12, 32])
def test_numpy_and_c_oracles_agree(tpsi):
    """equal labels after every sweep, float64 costs (lamda 0.05, the reference's arithmetic), K up to 64"""
    for H, W, K, seed in ((9, 11, 5, 0), (12, 7, 17, 1), (5, 13, 64, 2), (1, 9, 8, 3), (10, 1, 33, 4)):
        rng = np.random.default_rng(seed * 100 + tpsi)
        prop, _, nprop, lab0 = case(rng, H, W, K, spread=3 + tpsi)
        lc = rng.random((H, W, K)) * 2.5
        want = mo.ceo_bcd(prop, lc, nprop, lab0, 3, tpsi=tpsi)
        got = mo.ceo_bcd_c(prop, lc, nprop, lab0, 3, tpsi=tpsi)
        for w in range(3):
            assert np.array_equal(got[w], want[w]), (H, W, K, w)


@pytest.mark.parametrize("shift", [4, 12])
def test_energy_never_rises(shift):
    """int32-mode inputs (data costs m, 0 <= m < 65536, in units of 2^-S: lcost = m / 2^S with lamda 1): the energy
    in integer units after every phase is at most the energy before it.  The reference programme is run alongside and
    its phase-to-phase increases are counted (reported, not asserted: it minimises a different objective)."""
    rises = 0
    for H, W, K, tpsi, seed in ((16, 20, 12, 8, 0), (21, 13, 24, 3, 1), (8, 30, 6, 1, 2)):
        rng = np.random.default_rng(seed + shift)
        prop, _, nprop, lab0 = case(rng, H, W, K, spread=6)
        m = rng.integers(0, 65536 if seed % 2 else 4 << shift, (H, W, K))
        lc = m / float(1 << shift)
        scale = float(1 << shift)
        for mrf in (True, False):
            labels = lab0.copy()
            e = energy_int(prop, lc, labels, 1.0, tpsi) * scale
            for _ in range(3):
                for phase in range(4):
                    if mrf:
                        mo.run_phase(prop, lc, nprop, labels, phase, tpsi, 1.0)
                    else:
                        obcd._phase(prop, lc, nprop, labels, tpsi, 1.0, *mo.PHASES[phase], mo.phase_starts(phase, H, W))
                    e2 = energy_int(prop, lc, labels, 1.0, tpsi) * scale
                    assert e2 == int(e2)
                    if mrf:
                        assert e2 <= e, (H, W, K, tpsi, phase, e, e2)
                    else:
                        rises += e2 > e
                    e = e2
    print(f"reference programme: {rises} phase-to-phase energy increases")
