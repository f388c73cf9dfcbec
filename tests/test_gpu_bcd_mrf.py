"""FLOWB200_BCD_MRF on the device: block coordinate descent on the MRF energy, against the C restatement of
tests/mrf_oracle.py (mrf_oracle.ceo_bcd_c) after every sweep, and flowb200_energy against oracle.bcd.energy.

Oracle inputs: the int32 modes run the exact integer programme on m (units of 2^-S), which the oracle reproduces
exactly with lamda 1 on costs m / 2^S; the float64 modes get costs 20 m / 2^S (exact in float32 and float64) and
lamda 0.05, the oracle the same, and both evaluate the same float64 operations in the same order.
"""
import os

import numpy as np
import pytest

import mrf_oracle
from helpers import pkg
from test_gpu_bcd_records import Workspace, device_case, fitting_set, kset_layout, slot_bytes

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

MODES = ("BCD_INT32", "BCD_INT32_F32COST", "BCD_FP64_F64COST", "BCD_FP64_F32COST")


def lib():
    return pkg("_lib")


def dev(a, dtype):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dtype).cuda()


def is_int(mode):
    return mode.startswith("BCD_INT32")


def mode_cost(mode, m, shift):
    if mode == "BCD_INT32":
        return dev(m, torch.int32)
    return dev(20.0 * m / float(1 << shift), torch.float64 if mode == "BCD_FP64_F64COST" else torch.float32)


def oracle_costs(mode, m, shift):
    """(lcost, lamda) that the oracle needs to evaluate what the mode evaluates"""
    if is_int(mode):
        return m / float(1 << shift), 1.0
    return 20.0 * m / float(1 << shift), 0.05


def oracle(prop, nprop, m, lab0, mode, shift, sweeps, tpsi):
    lc, lamda = oracle_costs(mode, m, shift)
    return np.stack(mrf_oracle.ceo_bcd_c(prop, lc, nprop, lab0, sweeps, tpsi=tpsi, lamda=lamda))


def flag(mode):
    return getattr(lib(), mode) | lib().BCD_MRF


def run(pvec, cost, npr, lab0, sweeps, mode, tpsi, shift, nbytes=None):
    ops = pkg("ops")
    lab = dev(lab0, torch.int32)
    return ops.bcd(pvec, cost, npr, lab, sweeps, mode=flag(mode), tpsi=tpsi, cost_shift=shift, per_sweep=True,
                   workspace_bytes=nbytes).cpu().numpy()


def run_parts(pvec, cost, npr, lab0, sweeps, mode, tpsi, shift, nparts):
    """bcd_prepare / bcd_phase with every phase's chains in `nparts` parts, run one after the other on one label
    image (the chains of a phase are independent: what the all-reduce of the single-huge-image mode assembles)"""
    ops = pkg("ops")
    kw = dict(mode=flag(mode), lamda=0.05, tpsi=tpsi, cost_shift=shift)
    wss = []
    for part in range(nparts):
        wss.append(ops.bcd_workspace(pvec))
        ops.bcd_prepare(pvec, cost, npr, wss[-1], part, nparts, **kw)
    lab = dev(lab0, torch.int32)
    out = []
    for _ in range(sweeps):
        for phase in range(4):
            for part in range(nparts):
                ops.bcd_phase(pvec, cost, npr, lab, wss[part], phase, part, nparts, **kw)
        out.append(lab.cpu().numpy())
    return np.stack(out)


def random_case(rng, H, W, K, spread, ragged=True, costs="wide"):
    prop = rng.integers(-spread, spread + 1, (H, W, K, 2)).astype(np.int64)
    nprop = rng.integers(1, K + 1, (H, W)) if ragged else np.full((H, W), K)
    if ragged:
        nprop.flat[0] = 1
    prop[np.arange(K)[None, None, :] >= nprop[..., None]] = -1
    m = rng.integers(0, 65536 if costs == "wide" else 4, (H, W, K)).astype(np.int64)
    lab0 = rng.integers(0, 1 << 30, (H, W)) % nprop
    return prop, nprop.astype(np.int64), m, lab0.astype(np.int64)


# H, W, K, tpsi, shift: ragged nprop (1 included), degenerate shapes, every chain width, K 511 / 512, tpsi without
# records (0, 12, 32) and cost shifts without records (2)
CASES = [
    (7, 9, 5, 3, 12), (1, 13, 40, 8, 4), (13, 1, 33, 0, 12), (9, 11, 100, 12, 2), (6, 7, 500, 8, 14),
    (4, 5, 511, 8, 12), (4, 5, 512, 3, 12), (11, 6, 64, 32, 4), (2, 2, 129, 8, 14), (1, 1, 7, 8, 12),
    (10, 8, 200, 3, 2), (5, 12, 300, 12, 14), (8, 5, 384, 32, 4), (3, 17, 250, 0, 2),
]


def test_cases_cover_the_issue():
    assert {c[3] for c in CASES} >= {0, 3, 8, 12, 32} and {c[4] for c in CASES} >= {2, 4, 12, 14}
    assert {511, 512} <= {c[2] for c in CASES} and max(c[2] for c in CASES if c[2] < 511) >= 500


@pytest.mark.parametrize("H,W,K,tpsi,shift", CASES, ids=[f"{c[0]}x{c[1]}-K{c[2]}-t{c[3]}-s{c[4]}" for c in CASES])
def test_modes_against_the_oracle(H, W, K, tpsi, shift):
    """all four modes with the flag, the oracle's labels after every sweep"""
    sweeps = 2
    rng = np.random.default_rng(H * 1000 + W * 10 + K + tpsi + shift)
    prop, nprop, m, lab0 = random_case(rng, H, W, K, spread=max(2, tpsi), costs="ties" if K % 2 else "wide")
    pvec, npr = device_case(prop, nprop, m)
    for mode in MODES:
        want = oracle(prop, nprop, m, lab0, mode, shift, sweeps, tpsi)
        got = run(pvec, mode_cost(mode, m, shift), npr, lab0, sweeps, mode, tpsi, shift)
        assert np.array_equal(got, want), (mode, float((got != want).mean()))


@pytest.mark.parametrize("K,tpsi,shift", [(100, 8, 12), (300, 5, 7), (33, 1, 14)])
def test_workspace_paths(K, tpsi, shift):
    """record path with every record stored (the fitting sets of test_gpu_bcd_records) and no chain left to the
    fallback in the int32 modes; minimum and partial workspaces and FLOWB200_KSET_FORCE_GENERIC give the same labels"""
    H, W, sweeps = 9, 12, 2
    rng = np.random.default_rng(K + tpsi)
    prop, nprop, m, lab0 = fitting_set(rng, H, W, K, tpsi, costs="ties" if tpsi % 2 else "wide", ragged=True)
    m = m.astype(np.int64)
    pvec, npr = device_case(prop, nprop, m)
    L = lib().load()
    lo, full = L.flowb200_bcd_min_workspace_bytes(H, W, K), L.flowb200_bcd_workspace_bytes(H, W, K)
    ops = pkg("ops")
    for mode in MODES:
        want = oracle(prop, nprop, m, lab0, mode, shift, sweeps, tpsi)
        cost = mode_cost(mode, m, shift)
        # full workspace: every record stored
        ws = torch.zeros(full, dtype=torch.uint8, device="cuda")
        kw = dict(mode=flag(mode), lamda=0.05, tpsi=tpsi, cost_shift=shift)
        lab = dev(lab0, torch.int32)
        if is_int(mode):
            ops.bcd_prepare(pvec, cost, npr, ws, **kw)
            Lw = kset_layout(H, W, K, ws.numel())
            snaps = []
            for _ in range(sweeps):
                for phase in range(4):
                    ops.bcd_phase(pvec, cost, npr, lab, ws, phase, **kw)
                    nch = ((W + 1) // 2, (H + 1) // 2, W // 2, H // 2)[phase]
                    assert not ws[Lw["flags"]:Lw["flags"] + 4 * nch].cpu().numpy().view(np.int32).any(), mode
                snaps.append(lab.cpu().numpy())
            got = np.stack(snaps)
            assert np.all(Workspace(ws, H, W, K).desc != 0), mode
        else:
            got = run(pvec, cost, npr, lab0, sweeps, mode, tpsi, shift, full)
        assert np.array_equal(got, want), (mode, "full")
        for nb in (lo, (lo + full) // 2):
            assert np.array_equal(run(pvec, cost, npr, lab0, sweeps, mode, tpsi, shift, nb), want), (mode, nb)
        os.environ["FLOWB200_KSET_FORCE_GENERIC"] = "1"
        try:
            assert np.array_equal(run(pvec, cost, npr, lab0, sweeps, mode, tpsi, shift), want), (mode, "generic")
        finally:
            del os.environ["FLOWB200_KSET_FORCE_GENERIC"]


@pytest.mark.parametrize("mode", ["BCD_INT32", "BCD_INT32_F32COST"])
def test_parts_equal_the_whole(mode):
    H, W, K, tpsi, shift, sweeps = 13, 10, 60, 8, 12, 2
    prop, nprop, m, lab0 = random_case(np.random.default_rng(5), H, W, K, spread=8)
    pvec, npr = device_case(prop, nprop, m)
    cost = mode_cost(mode, m, shift)
    whole = run(pvec, cost, npr, lab0, sweeps, mode, tpsi, shift)
    assert np.array_equal(whole, oracle(prop, nprop, m, lab0, mode, shift, sweeps, tpsi))
    for nparts in (2, 3):
        assert np.array_equal(run_parts(pvec, cost, npr, lab0, sweeps, mode, tpsi, shift, nparts), whole), nparts


def test_flag_values():
    """the flag with the float64 modes: bcd_prepare / bcd_phase refuse it as they refuse the modes; other unknown
    bits stay invalid; ops.bcd(energy_per_phase) refuses the float64 modes"""
    H, W, K = 4, 5, 8
    prop, nprop, m, lab0 = random_case(np.random.default_rng(1), H, W, K, spread=3)
    pvec, npr = device_case(prop, nprop, m)
    ops, L = pkg("ops"), lib()
    ws = ops.bcd_workspace(pvec)
    lab = dev(lab0, torch.int32)
    c64 = mode_cost("BCD_FP64_F64COST", m, 12)
    with pytest.raises(L.FlowB200Error, match="unsupported"):
        ops.bcd_prepare(pvec, c64, npr, ws, mode=L.BCD_FP64_F64COST | L.BCD_MRF)
    for bad in (32, L.BCD_INT32 | 32, L.BCD_INT32 | L.BCD_MRF | 64):
        rc = L.load().flowb200_bcd(ops._ptr(pvec), ops._ptr(mode_cost("BCD_INT32", m, 12)), ops._ptr(npr),
                                   ops._ptr(lab), H, W, K, bad, 0.05, 8, 12, 1, None, ops._ptr(ws), ws.numel(),
                                   ops._stream())
        assert rc == L.EINVAL, bad
    with pytest.raises(ValueError):
        ops.bcd(pvec, c64, npr, lab, 1, mode=L.BCD_FP64_F64COST | L.BCD_MRF, energy_per_phase=True)


def mrf_len_limit(K, short):
    """largest chain length make_plan admits for the MRF kernels (float64 kernel's check: it is the stricter one), with
    the shorter side `short` (which sets the ring of record slots)"""
    Kpad = (K + 31) // 32 * 32
    mb = next(mb for T, mb in ((64, 8), (128, 6), (192, 5), (256, 4), (320, 4), (384, 3), (512, 2)) if K <= T)
    budget = 227 * 1024 // mb - 1024 - 512
    fixed32 = (4096 + 384 + 8 * short + 2 * short + 127) & ~127
    shift = 1 if 4096 + fixed32 + 4 * slot_bytes(Kpad) > budget else 2
    slots = slot_bytes(Kpad) << shift
    n = 1
    while ((10 * (n + 1) + 4 * Kpad + 127) & ~127) + slots + 1024 + 9216 <= 227 * 1024:
        n += 1
    return n


def test_longest_mrf_chain():
    """K = 512 on 2 x n frames: make_plan admits n = 15001 in the MRF modes and refuses n + 1 (the reference mode
    admits it: its side vectors take half the shared memory); at the limit the chains run and the energy does not
    rise"""
    K, H = 512, 2
    n = mrf_len_limit(K, H)
    assert n == 15001
    ops, L = pkg("ops"), lib()
    for Wc, ok in ((n, True), (n + 1, False)):
        rng = np.random.default_rng(Wc)
        prop = rng.integers(-4, 5, (H, Wc, K, 2)).astype(np.int64)
        nprop = np.full((H, Wc), K, np.int64)
        m = rng.integers(0, 65536, (H, Wc, K)).astype(np.int64)
        lab0 = rng.integers(0, K, (H, Wc)).astype(np.int64)
        pvec, npr = device_case(prop, nprop, m)
        cost = mode_cost("BCD_INT32", m, 12)
        lab = dev(lab0, torch.int32)
        if not ok:
            for mode in ("BCD_INT32", "BCD_FP64_F64COST"):
                with pytest.raises(L.FlowB200Error, match="unsupported"):
                    ops.bcd(pvec, mode_cost(mode, m, 12), npr, lab, 1, mode=flag(mode))
            ops.bcd(pvec, cost, npr, lab, 0, mode=L.BCD_INT32)   # plan only
            continue
        _, energies = ops.bcd(pvec, cost, npr, lab, 1, mode=flag("BCD_INT32"), energy_per_phase=True)
        assert all(b <= a for a, b in zip(energies, energies[1:])), energies


@pytest.mark.parametrize("mode", MODES)
def test_energy(mode):
    """flowb200_energy == oracle.bcd.energy: exactly in the int32 modes, to 1e-12 relative in the float64 ones; the same
    bits on every call; n_bad counts the planted bad labels, which leave their data term and pairs out"""
    from oracle import bcd as obcd
    H, W, K, tpsi, shift = 37, 53, 40, 8, 12
    prop, nprop, m, lab0 = random_case(np.random.default_rng(3), H, W, K, spread=9)
    pvec, npr = device_case(prop, nprop, m)
    ops = pkg("ops")
    cost = mode_cost(mode, m, shift)
    kw = dict(mode=flag(mode), lamda=0.05, tpsi=tpsi, cost_shift=shift)
    lab = dev(lab0, torch.int32)
    got = ops.energy(pvec, cost, npr, lab, **kw)
    lc, lamda = oracle_costs(mode, m, shift)
    want = obcd.energy(prop, lc, lab0, lamda, tpsi)
    assert got[3] == 0
    if is_int(mode):
        assert got[2] == want and got[0] + got[1] == got[2]
    else:
        assert abs(got[2] - want) <= 1e-12 * abs(want)
    for _ in range(3):
        assert ops.energy(pvec, cost, npr, lab, **kw) == got
    bad = lab0.copy()
    planted = [(0, 0, -1), (5, 7, int(nprop[5, 7])), (36, 52, 1000), (20, 0, -7)]
    for y, x, v in planted:
        bad[y, x] = v
    d, p, t, nb = ops.energy(pvec, cost, npr, dev(bad, torch.int32), **kw)
    assert nb == len(planted)
    ok = np.ones((H, W), bool)
    for y, x, _ in planted:
        ok[y, x] = False
    lab_ok = np.where(ok, bad, 0)
    ys, xs = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    v = prop[ys, xs, lab_ok]
    pw = (np.minimum(tpsi, np.abs(v[1:] - v[:-1]).sum(-1)) * (ok[1:] & ok[:-1])).sum() + \
         (np.minimum(tpsi, np.abs(v[:, 1:] - v[:, :-1]).sum(-1)) * (ok[:, 1:] & ok[:, :-1])).sum()
    assert p == pw
    if is_int(mode):
        assert d == (m[ys, xs, lab_ok] * ok).sum() / float(1 << shift)


def test_full_size_config1():
    """BASELINE.json configs[1] (1024x436, K = 300): the device's proposal sets, INT32_F32COST | MRF, 4 sweeps: the C
    oracle's labels after every sweep, and the device energy never rises from one phase to the next"""
    ops, params, synth, ioc, L = pkg("ops"), pkg("params"), pkg("synth"), pkg("io_contract"), lib()
    H, W, K, sweeps = 436, 1024, 300, 4
    p = params.for_k(K, H=H, W=W, knn_mode=1)
    img = synth.make_pair(H, W, 5)[:2]
    d0, d1 = ops.daisy(dev(img[0], torch.uint8)), ops.daisy(dev(img[1], torch.uint8))
    pvec, lcost, nprop, labels = ops.knn_proposals(d0, d1, p)
    ops.random_proposals(d0, d1, p, pvec, lcost, nprop, labels, seed=3)
    m = ops.quantise_costs(lcost, p.lamda, p.cost_shift).cpu().numpy().astype(np.int64)
    prop = ioc.unpack_proposals(pvec.cpu().numpy())
    N, B = nprop.cpu().numpy().astype(np.int64), labels.cpu().numpy().astype(np.int64)
    want = mrf_oracle.ceo_bcd_c(prop, m / float(1 << p.cost_shift), N, B, sweeps, tpsi=p.tpsi, lamda=1.0)
    mode = L.BCD_INT32_F32COST | L.BCD_MRF
    snaps, energies = ops.bcd(pvec, lcost, nprop, labels, sweeps, mode=mode, lamda=p.lamda, tpsi=p.tpsi,
                              cost_shift=p.cost_shift, per_sweep=True, energy_per_phase=True)
    for w in range(sweeps):
        got = snaps[w].cpu().numpy()
        assert np.array_equal(got, want[w]), (w, float((got != want[w]).mean()))
    assert all(b <= a for a, b in zip(energies, energies[1:])), energies
    print(f"\n[1024x436 K300] INT32_F32COST|MRF energy per phase: {energies}")


def test_flow_pair_with_the_flag_equals_its_stages():
    ops, params, synth, L = pkg("ops"), pkg("params"), pkg("synth"), lib()
    H, W = 96, 128
    p = params.FlowParams(H=H, W=W, cellw=16, cellh=12, knn_mode=1)
    img = synth.make_pair(H, W, 4)[:2]
    g0, g1 = dev(img[0], torch.uint8), dev(img[1], torch.uint8)
    for base in (L.BCD_INT32, L.BCD_FP64_F32COST):
        mode = base | L.BCD_MRF
        out, raw_f, raw_b = ops.flow_pair(g0, g1, p, sweeps=2, directions=2, seed=9, bcd_mode=mode, want_raw=True)
        ref = ops.flow_pair(g0, g1, p, sweeps=2, directions=2, seed=9, bcd_mode=base)
        desc = [ops.daisy(g0), ops.daisy(g1)]
        flows = []
        for d in (0, 1):
            pvec, lcost, nprop, labels = ops.knn_proposals(desc[d], desc[1 - d], p)
            ops.random_proposals(desc[d], desc[1 - d], p, pvec, lcost, nprop, labels, seed=9 + d)
            stage_mode = (L.BCD_INT32_F32COST if base == L.BCD_INT32 else base) | L.BCD_MRF
            ops.bcd(pvec, lcost, nprop, labels, 2, mode=stage_mode, lamda=p.lamda, tpsi=p.tpsi,
                    cost_shift=p.cost_shift)
            flows.append(ops.flow_from_labels(pvec, labels, want_yx=False)[1])
        assert torch.equal(raw_f, flows[0]) and torch.equal(raw_b, flows[1]), base
        assert torch.equal(out, ops.consistency(flows[0].clone(), flows[1], p.con_tresh)), base
        assert not torch.equal(out, ref), base   # the flag changes the labels (by design)
