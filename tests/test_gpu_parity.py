"""CUDA path vs the oracle and the golden fixtures (outputs of the reference's own source).  GPU only.

Everything goes through the C ABI (libflowb200.so) via the package's ctypes layer.  Bars:
bit-exact for labels, proposals, nprop, K-set bits, kNN indices, the consistency field and the
float32 data costs; DAISY within 1e-4 relative to the per-descriptor maximum (north star).
"""
import ctypes as C
import os

import numpy as np
import pytest

from helpers import load_case, load_npz, oracle_params, pkg

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

KNN_MODES = [0, 1]    # 0 = float64 CUDA cores, 1 = tcgen05 prefilter + exact re-rank
DAISY_RTOL = 1e-4      # BASELINE.json north_star: "DAISY must agree within 1e-4 relative"
F32 = np.float32


def dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda()


def flow_params(meta, **kw):
    H, W, cw, ch = (int(v) for v in meta[:4])
    return pkg("params").FlowParams(H=H, W=W, cellw=cw, cellh=ch, **kw)


# ---------------------------------------------------------------- consistency (A12-A14)
@pytest.mark.parametrize("case", ["const", "randint", "real"])
def test_consistency_golden(case):
    from oracle import consistency as ocons
    ops = pkg("ops")
    z = load_npz("consistency")
    f1 = dev(ocons.ucitaj_flow(z[case + "_fwd"]))
    f2 = dev(ocons.ucitaj_flow(z[case + "_bwd"]))
    ops.consistency(f1, f2, float(z[case + "_thr"]))
    assert np.array_equal(f1.cpu().numpy(), z[case + "_out"])


def test_consistency_random_float_flows():
    from oracle import consistency as ocons
    ops = pkg("ops")
    rng = np.random.default_rng(3)
    A, B = 97, 131
    f1 = np.concatenate([rng.normal(0, 9, (A, B, 2)), (rng.random((A, B, 1)) > 0.1)], -1).astype(np.float32)
    f2 = np.concatenate([-f1[..., :2] + rng.normal(0, 4, (A, B, 2)), (rng.random((A, B, 1)) > 0.1)], -1).astype(np.float32)
    want = ocons.forward_backward_consistency(f1, f2, 7.5)
    g1 = dev(f1)
    ops.consistency(g1, dev(f2), 7.5)
    assert np.array_equal(g1.cpu().numpy(), want)


def test_consistency_empty_region_and_alias():
    ops, lib = pkg("ops"), pkg("_lib")
    f = torch.zeros((4, 5, 3), dtype=torch.float32, device="cuda")
    ops.consistency(f, torch.zeros_like(f), 1.0, region=(2, 2, 0, 5))      # empty: no-op
    with pytest.raises(lib.FlowB200Error):
        ops.consistency(f, f, 1.0)


# ---------------------------------------------------------------- DAISY (A2)
@pytest.mark.parametrize("shape,seed", [((57, 83), 4), ((40, 48), 1), ((131, 200), 9)])
def test_daisy_vs_oracle(shape, seed):
    from oracle import daisy as od
    ops = pkg("ops")
    img = pkg("synth").texture(shape[0], shape[1], seed)
    want = od.daisy(img)
    got = ops.daisy(dev(img)).cpu().numpy()
    scale = np.abs(want).max(axis=-1, keepdims=True) + 1e-12
    rel = np.abs(got - want) / scale
    assert rel.max() <= DAISY_RTOL, rel.max()
    assert ((want == 0) == (got == 0)).all()          # zeroed border petals are exactly zero


def test_daisy_golden_descriptors():
    ops = pkg("ops")
    z = load_npz("pair_a")
    for img, want in ((z["img1"], z["desc1"]), (z["img2"], z["desc2"])):
        got = ops.daisy(dev(img)).cpu().numpy()
        scale = np.abs(want).max(axis=-1, keepdims=True) + 1e-12
        assert (np.abs(got - want) / scale).max() <= DAISY_RTOL


# ---------------------------------------------------------------- proposals (A3-A8)
def _stage1_gpu(z, b, p, knn_mode=0):
    ops, ioc = pkg("ops"), pkg("io_contract")
    d1, d2 = (z["desc1"], z["desc2"]) if b == 0 else (z["desc2"], z["desc1"])
    g1, g2 = dev(d1), dev(d2)
    pvec, lcost, nprop, labels, idx, stats = ops.knn_proposals(g1, g2, p, want_idx=True, knn_mode=knn_mode)
    out = {"labels00": labels.cpu().numpy().astype(np.int64),
           "flow00": ops.flow_from_labels(pvec, labels)[0].cpu().numpy(),
           "idx": idx.cpu().numpy(), "stats": stats.cpu().numpy()}
    ops.random_proposals(g1, g2, p, pvec, lcost, nprop, labels, draws=dev(z[f"b{b}_draws"], torch.int16))
    out.update(proposals=ioc.unpack_proposals(pvec.cpu().numpy()), lcosts=lcost.cpu().numpy().astype(np.float64),
               nprop=nprop.cpu().numpy().astype(np.int64), pvec=pvec, nprop_dev=nprop)
    return out


@pytest.mark.parametrize("knn_mode", KNN_MODES)
@pytest.mark.parametrize("name,dirs", [("pair_a", (0, 1)), ("pair_b", (0,))])
def test_stage1_golden(name, dirs, knn_mode):
    """generisi + nasumicni (replayed draws) + pakovanje against the reference's own outputs."""
    from oracle import proposals as oprop
    ops = pkg("ops")
    z = load_case(name)
    p = flow_params(z["meta"])
    op = oracle_params(z["meta"])
    for b in dirs:
        r = _stage1_gpu(z, b, p, knn_mode)
        assert np.array_equal(r["labels00"], z[f"b{b}_labels00"])
        assert np.array_equal(r["flow00"], z[f"b{b}_flow00"])
        assert np.array_equal(r["nprop"], z[f"b{b}_nprop"])
        assert np.array_equal(r["proposals"], z[f"b{b}_proposals"])
        assert np.array_equal(r["lcosts"], z[f"b{b}_lcosts"])
        pk = ops.ksets_pack(r["pvec"], r["nprop_dev"]).cpu().numpy()
        assert oprop.ksets_masked_equal(pk, z[f"b{b}_packedksets"], r["nprop"], op)


@pytest.mark.parametrize("knn_mode", KNN_MODES)
@pytest.mark.parametrize("k_cell", [5, 10])
def test_knn_indices_bit_exact(knn_mode, k_cell):
    """kNN indices against exact float64 brute force on the CPU (lowest-index ties), incl. duplicates."""
    from oracle import proposals as oprop
    ops = pkg("ops")
    rng = np.random.default_rng(11)
    H, W, cw, ch = 61, 90, 16, 12
    img1, img2, _, _ = pkg("synth").make_pair(H, W, 5, max_dx=5, max_dy=3, n_rect=2)
    from oracle import daisy as od
    d1, d2 = od.daisy(img1), od.daisy(img2)
    d2[10:14, 20:30] = d2[30:34, 40:50]          # exact duplicate targets -> ties inside / across cells
    d2[5, 5:9] = d2[5, 4]
    p = pkg("params").FlowParams(H=H, W=W, cellw=cw, cellh=ch, k_cell=k_cell, n_gauss=0,
                                 maxnprop=25 * k_cell)
    op = oprop.Params(H, W, cw, ch, k_cell=k_cell, n_gauss=0, maxnprop=25 * k_cell)
    pvec, lcost, nprop, labels, idx, stats = ops.knn_proposals(dev(d1), dev(d2), p, want_idx=True, knn_mode=knn_mode)
    idx = idx.cpu().numpy()
    cd2 = oprop.cell_descriptors(d2, op)
    R = p.cell_radius
    ys = rng.integers(0, H, 40)
    xs = rng.integers(0, W, 40)
    for y, x in list(zip(ys, xs)) + [(0, 0), (H - 1, W - 1), (H - 1, 0), (0, W - 1)]:
        cis = [c for c in range(op.ncellx) if cw * (c - R) <= x < cw * (c + R + 1)]
        cjs = [c for c in range(op.ncelly) if ch * (c - R) <= y < ch * (c + R + 1)]
        blk = 0
        for ci in cis:
            for cj in cjs:
                want = oprop.knn_exact(d1[y, x][None], cd2[ci + cj * op.ncellx], k_cell)[0]
                assert np.array_equal(idx[y, x, blk], want), (y, x, ci, cj)
                blk += 1
        assert (idx[y, x, blk:] == -1).all()
        assert int(nprop[y, x]) == blk * k_cell
    P, L, N, B = oprop.generisi(d1, d2, op)
    ioc = pkg("io_contract")
    assert np.array_equal(ioc.unpack_proposals(pvec.cpu().numpy()), P)
    assert np.array_equal(lcost.cpu().numpy().astype(np.float64), L)
    assert np.array_equal(labels.cpu().numpy(), B)


def test_tcgen05_scores_match_fp16_operands():
    """Raw tensor-core ranking scores (TMA + UMMA descriptors + TMEM read-back) against numpy on the same fp16
    operands: a(q,t) = |q~|^2/2 + |t~|^2/2 - q~.t~ with q~, t~ = fp16(64*d), targets in the pos -> pos*s mod T order."""
    from oracle import daisy as od
    ops = pkg("ops")
    H, W, cw, ch = 40, 48, 12, 10
    img1, img2, _, _ = pkg("synth").make_pair(H, W, 7, max_dx=4, max_dy=3, n_rect=1)
    d1, d2 = od.daisy(img1), od.daisy(img2)
    p = pkg("params").FlowParams(H=H, W=W, cellw=cw, cellh=ch, knn_mode=1)
    scores, g = ops.knn_debug_scores(dev(d1), dev(d2), p)
    scores = scores.cpu().numpy()
    T, Tpad, s = cw * ch, g["Tpad"], g["stride_s"]
    ncx, ncy, R = W // cw, H // ch, p.cell_radius
    q16 = (d1 * np.float32(64)).astype(np.float16).astype(np.float64)
    checked = 0
    for cell in range(ncx * ncy):
        ci, cj = cell % ncx, cell // ncx
        idx = (np.arange(T) * s) % T
        tg = d2[cj * ch + idx // cw, ci * cw + idx % cw]
        t16 = (tg * np.float32(64)).astype(np.float16).astype(np.float64)
        n = (0.5 * (t16 ** 2).sum(1)).astype(np.float32)
        h0 = n.astype(np.float16).astype(np.float32)
        h1 = (n - h0).astype(np.float16).astype(np.float32)
        h2 = (n - h0 - h1).astype(np.float16).astype(np.float32)
        nn = h0.astype(np.float64) + h1 + h2
        x0, x1 = max(0, cw * (ci - R)), min(W, cw * (ci + R + 1))
        y0, y1 = max(0, ch * (cj - R)), min(H, ch * (cj + R + 1))
        for tyi in range(g["tiles_y"]):
            for txi in range(g["tiles_x"]):
                qx0, qy0 = x0 + txi * g["tile_w"], y0 + tyi * g["tile_h"]
                item = (tyi * g["tiles_x"] + txi) * (ncx * ncy) + cell           # cell-minor work order
                if qx0 >= x1 or qy0 >= y1:
                    assert np.isnan(scores[item]).all()          # skipped work item
                    continue
                for row in [r for r in (0, 17, 127, 64, 128, 200, 255) if r < g["tile_w"] * g["tile_h"]]:
                    mt, rr = row // 128, row % 128               # MMA tile inside the item, row inside the tile
                    px, py = qx0 + mt * 16 + (rr & 15), qy0 + (rr >> 4)
                    if px >= W or py >= H:
                        continue                                  # zero-filled TMA rows
                    mq = np.float32(0.5 * (q16[py, px] ** 2).sum())
                    m0 = np.float16(mq).astype(np.float32)
                    m1 = np.float16(mq - m0).astype(np.float32)
                    m2 = np.float16(mq - m0 - m1).astype(np.float32)
                    want = nn - t16 @ q16[py, px] + (np.float64(m0) + m1 + m2)
                    got = scores[item, row, :T]
                    assert np.abs(got - want).max() < 2e-3, (cell, txi, tyi, row, np.abs(got - want).max())
                    assert (scores[item, row, T:] > 5e4).all()    # padding columns can never be selected
                    checked += 1
    assert checked > 100


def test_random_proposals_philox_statistics():
    """Seeded Philox draws: same acceptance rules, so the kept-count distribution must look like the
    reference's (about half of the 25 draws survive quirk Q4); reproducible for a fixed seed."""
    ops = pkg("ops")
    z = load_case("pair_a")
    p = flow_params(z["meta"])
    g1, g2 = dev(z["desc1"]), dev(z["desc2"])
    runs = []
    for seed in (7, 7, 8):
        pvec, lcost, nprop, labels = ops.knn_proposals(g1, g2, p)
        nn = nprop.clone()
        ops.random_proposals(g1, g2, p, pvec, lcost, nprop, labels, seed=seed)
        runs.append(((nprop - nn).cpu().numpy(), pvec.cpu().numpy()))
    assert np.array_equal(runs[0][0], runs[1][0]) and np.array_equal(runs[0][1], runs[1][1])
    assert not np.array_equal(runs[0][1], runs[2][1])
    kept = runs[0][0]
    assert kept.min() >= 0 and kept.max() <= 25
    # reference kept-count on this case (from the golden nprop): NN count is a multiple of 5 per pixel
    from oracle import proposals as oprop
    op = oracle_params(z["meta"])
    _, _, N0, _ = oprop.generisi(z["desc1"], z["desc2"], op)
    kept_ref = z["b0_nprop"] - N0
    assert abs(kept.mean() - kept_ref.mean()) < 1.5, (kept.mean(), kept_ref.mean())


# ---------------------------------------------------------------- BCD (A9-A11)
@pytest.mark.parametrize("name,dirs", [("pair_a", (0, 1)), ("pair_b", (0,))])
def test_bcd_fp64_golden(name, dirs):
    """float64 mode on the reference's float32-representable costs: labels equal after every sweep."""
    ops, ioc, lib = pkg("ops"), pkg("io_contract"), pkg("_lib")
    z = load_case(name)
    sweeps = int(z["meta"][5])
    for b in dirs:
        pvec = dev(ioc.pack_proposals(z[f"b{b}_proposals"]))
        nprop = dev(z[f"b{b}_nprop"], torch.int32)
        for mode, cost in ((lib.BCD_FP64_F32COST, dev(z[f"b{b}_lcosts"], torch.float32)),
                           (lib.BCD_FP64_F64COST, dev(z[f"b{b}_lcosts"], torch.float64))):
            labels = dev(z[f"b{b}_labels00"], torch.int32)
            snaps = ops.bcd(pvec, cost, nprop, labels, sweeps, mode=mode, per_sweep=True).cpu().numpy()
            for w in range(sweeps):
                assert np.array_equal(snaps[w], z[f"b{b}_labels{w + 1:02d}"]), (b, mode, w)
            assert np.array_equal(labels.cpu().numpy(), snaps[-1])
            yx, uvv = ops.flow_from_labels(pvec, labels)
            assert np.array_equal(yx.cpu().numpy(), z[f"b{b}_flow{sweeps:02d}"])


def test_bcd_int32_golden():
    """int32 mode on costs 20*m/2^12 against the unmodified reference's labels (bcd_q12 fixture)."""
    ops, ioc, lib = pkg("ops"), pkg("io_contract"), pkg("_lib")
    z = load_npz("bcd_q12")
    sweeps, shift = int(z["meta"][5]), int(z["meta"][6])
    pvec = dev(ioc.pack_proposals(z["proposals"]))
    labels = dev(z["labels00"], torch.int32)
    snaps = ops.bcd(pvec, dev(z["m"], torch.int32), dev(z["nprop"], torch.int32), labels, sweeps,
                    mode=lib.BCD_INT32, cost_shift=shift, per_sweep=True).cpu().numpy()
    for w in range(sweeps):
        assert np.array_equal(snaps[w], z[f"labels{w + 1:02d}"]), w


@pytest.mark.parametrize("H,W,K,tpsi,shift", [
    pytest.param(H, W, K, 8, 12, id=f"{H}-{W}-{K}")
    for H, W, K in ((37, 41, 150), (36, 64, 300), (48, 40, 500), (1, 40, 60), (40, 1, 60), (2, 2, 33))] + [
    # other tpsi and cost shifts; tpsi 0 and 9..32 and cost shifts below 4 run without K-set records
    (37, 41, 150, 0, 12), (20, 24, 300, 3, 12), (24, 20, 500, 12, 12), (37, 41, 150, 32, 12), (20, 24, 300, 8, 2)])
def test_bcd_vs_oracle_random(H, W, K, tpsi, shift):
    """Random proposal sets incl. degenerate shapes, ragged nprop, heavy ties (int costs), K up to 500, tpsi 0..32.
    The vectors come from a small square, so nearly every label's candidates overflow the build kernel's staging and
    most records are not stored: this tests the dense fallback.  test_gpu_bcd_records.py tests the record path."""
    from oracle import bcd as obcd
    ops, ioc, lib = pkg("ops"), pkg("io_contract"), pkg("_lib")
    rng = np.random.default_rng(H * 1000 + W + K)
    prop = rng.integers(-12, 13, (H, W, K, 2)).astype(np.int64)
    nprop = rng.integers(max(1, K // 3), K + 1, (H, W)).astype(np.int64)
    m = rng.integers(0, 513, (H, W, K)).astype(np.int64)
    lab0 = (rng.integers(0, 1 << 30, (H, W)) % nprop).astype(np.int64)
    lq = 20.0 * m / float(1 << shift)
    want = obcd.ceo_bcd(prop, lq, nprop, lab0, 2, tpsi=tpsi)
    pvec = dev(ioc.pack_proposals(prop))
    for mode, cost, kw in ((lib.BCD_INT32, dev(m, torch.int32), dict(cost_shift=shift)),
                           (lib.BCD_FP64_F64COST, dev(lq, torch.float64), {})):
        labels = dev(lab0, torch.int32)
        snaps = ops.bcd(pvec, cost, dev(nprop, torch.int32), labels, 2, mode=mode, tpsi=tpsi, per_sweep=True,
                        **kw).cpu().numpy()
        assert np.array_equal(snaps[0], want[0]) and np.array_equal(snaps[1], want[1]), mode
        if tpsi == 32:   # the largest tpsi accepted
            with pytest.raises(lib.FlowB200Error, match="unsupported"):
                ops.bcd(pvec, cost, dev(nprop, torch.int32), labels, 2, mode=mode, tpsi=33, **kw)


@pytest.mark.parametrize("extra", [0, 40 << 10, 400 << 10])
def test_bcd_int32_any_workspace_size(extra):
    """The K-set records are a cache: with no room for them (every step evaluated densely) or room for only some of
    them, the labels are the reference's (bcd_q12 fixture, unmodified `python bcd.py`)."""
    ops, ioc, lib = pkg("ops"), pkg("io_contract"), pkg("_lib")
    z = load_npz("bcd_q12")
    sweeps, shift = int(z["meta"][5]), int(z["meta"][6])
    pvec = dev(ioc.pack_proposals(z["proposals"]))
    H, W, K = pvec.shape
    nb = lib.load().flowb200_bcd_min_workspace_bytes(H, W, K) + extra
    assert nb < lib.load().flowb200_bcd_workspace_bytes(H, W, K)
    labels = dev(z["labels00"], torch.int32)
    snaps = ops.bcd(pvec, dev(z["m"], torch.int32), dev(z["nprop"], torch.int32), labels, sweeps,
                    mode=lib.BCD_INT32, cost_shift=shift, per_sweep=True, workspace_bytes=nb).cpu().numpy()
    for w in range(sweeps):
        assert np.array_equal(snaps[w], z[f"labels{w + 1:02d}"]), w


def test_bcd_int32_generic_kernel(monkeypatch):
    """Chains that have a step without a stored record are left by the 32-bit kernel to the fallback, the integer
    variant of the float64 kernel (exact double arithmetic on the int32 terms, dense steps).
    FLOWB200_KSET_FORCE_GENERIC sends every chain that way: the labels stay the reference's (bcd_q12 fixture); on the
    float32 costs of pair_a they equal the unforced run's and BCD_INT32's on the quantised costs (the fallback reads
    the data costs from the cost array, the 32-bit kernel from the records); and they are the oracle's on random
    proposal sets with large integer costs at cost shifts 12 and 8."""
    from oracle import bcd as obcd
    ops, ioc, lib = pkg("ops"), pkg("io_contract"), pkg("_lib")

    def force_generic(on):
        if on:
            monkeypatch.setenv("FLOWB200_KSET_FORCE_GENERIC", "1")
        else:
            monkeypatch.delenv("FLOWB200_KSET_FORCE_GENERIC", raising=False)

    force_generic(True)
    z = load_npz("bcd_q12")
    sweeps, shift = int(z["meta"][5]), int(z["meta"][6])
    labels = dev(z["labels00"], torch.int32)
    snaps = ops.bcd(dev(ioc.pack_proposals(z["proposals"])), dev(z["m"], torch.int32), dev(z["nprop"], torch.int32),
                    labels, sweeps, mode=lib.BCD_INT32, cost_shift=shift, per_sweep=True).cpu().numpy()
    for w in range(sweeps):
        assert np.array_equal(snaps[w], z[f"labels{w + 1:02d}"]), w

    z = load_case("pair_a")
    pvec = dev(ioc.pack_proposals(z["b0_proposals"]))
    nprop = dev(z["b0_nprop"], torch.int32)
    lc = dev(z["b0_lcosts"], torch.float32)
    lab0 = dev(z["b0_labels00"], torch.int32)
    forced = ops.bcd(pvec, lc, nprop, lab0.clone(), 2, mode=lib.BCD_INT32_F32COST, cost_shift=12, per_sweep=True)
    force_generic(False)
    unforced = ops.bcd(pvec, lc, nprop, lab0.clone(), 2, mode=lib.BCD_INT32_F32COST, cost_shift=12, per_sweep=True)
    quantised = ops.bcd(pvec, ops.quantise_costs(lc, 0.05, 12), nprop, lab0.clone(), 2, mode=lib.BCD_INT32,
                        cost_shift=12, per_sweep=True)
    assert torch.equal(forced, unforced) and torch.equal(forced, quantised)

    rng = np.random.default_rng(5)
    H, W, K = 38, 45, 96
    prop = rng.integers(-14, 15, (H, W, K, 2)).astype(np.int64)
    nprop = rng.integers(K // 2, K + 1, (H, W)).astype(np.int64)
    m = rng.integers(0, 60000, (H, W, K)).astype(np.int64)          # near the 16-bit limit of the data cost
    lab0 = (rng.integers(0, 1 << 30, (H, W)) % nprop).astype(np.int64)
    for shift in (12, 8):
        want = obcd.ceo_bcd(prop, 20.0 * m / float(1 << shift), nprop, lab0, 2)
        for force in (True, False):
            force_generic(force)
            labels = dev(lab0, torch.int32)
            snaps = ops.bcd(dev(ioc.pack_proposals(prop)), dev(m, torch.int32), dev(nprop, torch.int32), labels, 2,
                            mode=lib.BCD_INT32, cost_shift=shift, per_sweep=True).cpu().numpy()
            assert np.array_equal(snaps[0], want[0]) and np.array_equal(snaps[1], want[1]), (shift, force)


def test_bcd_fp64_ksets_equal_oracle_and_any_workspace():
    """The float64 modes run on the compiled K-sets too (what `bcd.py` uses on reference-written files).  They equal
    the C oracle after every sweep, with every record stored, none (dense steps) or some, on the reference's
    unquantised costs."""
    from oracle import cport
    ops, ioc, lib = pkg("ops"), pkg("io_contract"), pkg("_lib")
    z = load_case("pair_b")
    sweeps = 2
    pvec = dev(ioc.pack_proposals(z["b0_proposals"]))
    nprop = dev(z["b0_nprop"], torch.int32)
    lab0 = dev(z["b0_labels00"], torch.int32)
    H, W, K = pvec.shape
    L = lib.load()
    lo, hi = L.flowb200_bcd_min_workspace_bytes(H, W, K), L.flowb200_bcd_workspace_bytes(H, W, K)
    for mode, cost in ((lib.BCD_FP64_F32COST, dev(z["b0_lcosts"], torch.float32)),
                       (lib.BCD_FP64_F64COST, dev(z["b0_lcosts"] * 1.0000001, torch.float64))):
        # the oracle gets the same costs in float64 (float32 costs widened exactly)
        want = np.stack(cport.ceo_bcd(z["b0_proposals"], cost.double().cpu().numpy(), z["b0_nprop"], z["b0_labels00"],
                                      sweeps))
        for nb in (None, lo, lo + (hi - lo) // 7):
            got = ops.bcd(pvec, cost, nprop, lab0.clone(), sweeps, mode=mode, per_sweep=True, workspace_bytes=nb)
            assert np.array_equal(got.cpu().numpy(), want), (mode, nb)


def test_bcd_int32_on_float_costs_equals_quantise_then_int32():
    ops, ioc, lib = pkg("ops"), pkg("io_contract"), pkg("_lib")
    z = load_case("pair_a")
    pvec = dev(ioc.pack_proposals(z["b0_proposals"]))
    nprop = dev(z["b0_nprop"], torch.int32)
    lc = dev(z["b0_lcosts"], torch.float32)
    a = dev(z["b0_labels00"], torch.int32)
    b = a.clone()
    ops.bcd(pvec, ops.quantise_costs(lc, 0.05, 12), nprop, a, 2, mode=lib.BCD_INT32, cost_shift=12)
    ops.bcd(pvec, lc, nprop, b, 2, mode=lib.BCD_INT32_F32COST, cost_shift=12)
    assert torch.equal(a, b)


def test_quantise_costs():
    ops = pkg("ops")
    rng = np.random.default_rng(0)
    c = rng.uniform(0, 2.5, (9, 11, 20)).astype(np.float32)
    c[..., 15:] = 1000.0
    m = ops.quantise_costs(dev(c), 0.05, 12).cpu().numpy()
    want = np.where(c == 1000.0, 0, np.rint(0.05 * c.astype(np.float64) * 4096.0)).astype(np.int32)
    assert np.array_equal(m, want)


@pytest.mark.parametrize("shift", range(15))
def test_quantise_costs_every_shift(shift):
    """m = rint((lamda * c) * 2^S) in float64, 1000.0 (an unused slot) -> 0, at every shift: uniform costs, costs whose
    product lands exactly half-way (lamda 0.5, c = (2j+1) / 2^S: rint rounds half to even), the float32 neighbours of
    1000.0 (quantised), and n = 0, 1, 255, 257 (not a multiple of the block); shifts -1 and 15 are refused."""
    ops, lib = pkg("ops"), pkg("_lib")
    rng = np.random.default_rng(shift)
    S = float(1 << shift)
    c = rng.uniform(0, 2.5, (9, 11, 20)).astype(np.float32)
    c[..., 15:] = 1000.0
    ties = ((2 * np.arange(300) + 1) / S).astype(np.float32)
    thousand = np.array([np.nextafter(F32(1000), F32(0)), 1000.0, np.nextafter(F32(1000), F32(np.inf))], np.float32)
    arrays = [c, ties, thousand] + [rng.uniform(0, 3, n).astype(np.float32) for n in (0, 1, 255, 257)]
    for lamda in (0.05, 0.5, 1.0):
        for a in arrays:
            want = np.where(a == 1000.0, 0, np.rint((lamda * a.astype(np.float64)) * S)).astype(np.int32)
            m = ops.quantise_costs(dev(a), lamda, shift).cpu().numpy()
            assert m.shape == a.shape and np.array_equal(m, want), (lamda, a.shape)
    # j + 1/2 rounds to the even neighbour
    assert np.array_equal(ops.quantise_costs(dev(ties), 0.5, shift).cpu().numpy(), 2 * ((np.arange(300) + 1) // 2))
    m = torch.zeros(3, dtype=torch.int32, device="cuda")
    for bad in (-1, 15):
        rc = lib.load().flowb200_quantise_costs(C.c_void_p(dev(thousand).data_ptr()), C.c_void_p(m.data_ptr()), 3, 0.05,
                                                bad, C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == lib.EINVAL


def test_epe_metric_matches_error_image():
    from oracle import epe as oepe
    ops = pkg("ops")
    rng = np.random.default_rng(2)
    H, W = 77, 123
    t = np.concatenate([rng.normal(0, 5, (H, W, 2)), rng.random((H, W, 1)) > 0.2], -1).astype(np.float32)
    g = np.concatenate([t[..., :2] + rng.normal(0, 2, (H, W, 2)), rng.random((H, W, 1)) > 0.1], -1).astype(np.float32)
    want = oepe.error_image(t, g)
    got = ops.epe(dev(t), dev(g))
    assert got[2] == want[2]
    assert abs(got[0] - want[0]) <= 1e-5 * want[0] and abs(got[1] - want[1]) < 1e-9       # float64 vs float32 averaging
    assert ops.epe(dev(t * 0), dev(g * 0))[2] == 0


def test_epe_metric_golden():
    """flowb200_epe against visualization.errorImage itself (tests/golden/epe.npz, make_golden_extra.py)."""
    ops = pkg("ops")
    z = load_npz("epe")
    for k in range(3):
        mean, outl, n = ops.epe(dev(z[f"c{k}_test"]), dev(z[f"c{k}_gt"]))
        assert n == int(z[f"c{k}_nvalid"])
        assert abs(mean - float(z[f"c{k}_mean"])) <= 2e-6 * max(1.0, float(z[f"c{k}_mean"]))   # float64 vs float32 mean
        assert abs(outl - float(z[f"c{k}_outliers"])) < 1e-9


def test_pack_for_c_golden():
    """pakovanjeZaC (daisy i flann.py:321-398): flowb200_ksets_pack + stage1.pack_for_c against the four arrays the
    reference's own function wrote (tests/golden/zac.npz), inside the [:nprop[p], :nprop[q]] region."""
    from test_oracle_golden import assert_zac_equal
    ops, ioc, stage1 = pkg("ops"), pkg("io_contract"), pkg("stage1")
    z = load_npz("zac")
    H, W, _, _, _, K = (int(v) for v in z["meta"])
    pvec = np.full((H, W, K), -1, np.int32)
    pvec[...] = ioc.pack_proposals(z["proposals"].astype(np.int64))
    packed = ops.ksets_pack(dev(pvec), dev(z["nprop"], torch.int32)).cpu().numpy()
    assert_zac_equal(stage1.pack_for_c(packed, H, W), z)


# ---------------------------------------------------------------- whole path
def test_pipeline_matches_stagewise_and_oracle():
    """flow_pair (device resident) == the stages called one by one; EPE vs the oracle pipeline <= 0.01 px."""
    from oracle import bcd as obcd, consistency as ocons, daisy as od, epe as oepe, proposals as oprop
    ops, synth = pkg("ops"), pkg("synth")
    H, W, cw, ch = 48, 64, 16, 12
    img1, img2, fwd, bwd = synth.make_pair(H, W, 2, max_dx=6, max_dy=4, n_rect=2)
    p = pkg("params").FlowParams(H=H, W=W, cellw=cw, cellh=ch, n_gauss=0, maxnprop=125)
    out, raw_f, raw_b = ops.flow_pair(dev(img1), dev(img2), p, sweeps=2, directions=2, want_raw=True)
    # oracle pipeline on the oracle's own descriptors, no random proposals (n_gauss = 0: deterministic)
    op = oprop.Params(H, W, cw, ch, n_gauss=0, maxnprop=125)
    d1, d2 = od.daisy(img1), od.daisy(img2)
    flows = []
    for a, b in ((d1, d2), (d2, d1)):
        P, L, N, B = oprop.generisi(a, b, op)
        lab = obcd.ceo_bcd(P, L, N, B, 2)[-1]
        flows.append(oprop.final_flow(P, lab))
    want = ocons.post_processing(flows[0], flows[1], p.con_tresh)
    gt = synth.gt_uvv(fwd)
    e_got = oepe.error_image(out.cpu().numpy(), gt)
    e_want = oepe.error_image(want, gt)
    assert abs(e_got[0] - e_want[0]) <= 0.01, (e_got, e_want)       # north star: EPE within 0.01 px
    assert np.array_equal(raw_f.cpu().numpy(), ocons.ucitaj_flow(flows[0]))
    assert np.array_equal(out.cpu().numpy(), want)


# ---------------------------------------------------------------- single-huge-image mode (SURVEY 8e, configs[4])
@pytest.mark.parametrize("world", [2, 3])
def test_banded_search_on_device_merges_to_full(world):
    """Every band's search run on this one GPU in turn, merged with the slot-range copy plan: bit-identical to the
    full-image search (proposals, costs, nprop, bestlabels)."""
    ops, huge, params, synth = pkg("ops"), pkg("huge"), pkg("params"), pkg("synth")
    H, W = 150, 584
    p = params.for_k(150, H=H, W=W, knn_mode=1)
    a, b, _, _ = synth.make_pair(H, W, 3)
    d1, d2 = ops.daisy(dev(a)), ops.daisy(dev(b))
    want = ops.knn_proposals(d1, d2, p)
    bands = huge.band_plan(p, world)
    blocks = {}
    for bd in bands:
        if bd.ci_hi > bd.ci_lo:
            pv, lc, _, _ = ops.knn_proposals(d1[:, bd.sx0:bd.sx1].contiguous(), d2[:, bd.tx0:bd.tx1].contiguous(),
                                             huge.sub_params(p, bd))
            blocks[bd.rank] = (pv, lc)
    for rank in range(world):
        mine = blocks.get(rank, (None, None))
        got = huge.merge_bands(p, bands, rank, mine[0], mine[1], d1.device, blocks=blocks)
        for g, w in zip(got, want):
            assert torch.equal(g, w)


@pytest.mark.parametrize("world", [2, 5])
def test_slot_copy_kernel_equals_the_torch_slicing(world):
    """flowb200_slot_copy (one launch per pack / unpack) against pack_band / unpack_band evaluated with torch on the
    CPU, on random band blocks: merged proposals, costs, nprop and bestlabels bit-identical on every rank."""
    huge, params = pkg("huge"), pkg("params")
    H, W = 110, 657          # 9 cell columns, ragged cell rows (110 = 4 * 25 + 10)
    p = params.for_k(150, H=H, W=W, knn_mode=1)
    rng = np.random.default_rng(world)
    bands = huge.band_plan(p, world)
    cpu = {}
    for bd in bands:
        if bd.ci_hi > bd.ci_lo:
            pv = torch.from_numpy(rng.integers(-2 ** 31, 2 ** 31 - 1, (H, bd.width, p.maxnprop), dtype=np.int64).astype(np.int32))
            lc = torch.from_numpy(rng.random((H, bd.width, p.maxnprop), dtype=np.float32) * 3)
            cpu[bd.rank] = (pv, lc)
    gpu = {r: (a.cuda(), b.cuda()) for r, (a, b) in cpu.items()}
    for rank in range(world):
        want = huge.merge_bands(p, bands, rank, *cpu.get(rank, (None, None)), "cpu", blocks=cpu)
        got = huge.merge_bands(p, bands, rank, *gpu.get(rank, (None, None)), torch.device("cuda"), blocks=gpu)
        for g, w in zip(got, want):
            assert torch.equal(g.cpu(), w)


def test_two_ranks_nccl_flow_pair_equals_one_gpu(tmp_path):
    """torchrun, 2 ranks over NCCL: the sharded pair pipeline returns, on both ranks, exactly what one GPU computes."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import subprocess, sys, textwrap
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "w.py"
    script.write_text(textwrap.dedent(f"""
        import os, sys, torch, torch.distributed as dist
        sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "tests"))
        from helpers import pkg
        ops, huge, params, synth, lib = pkg("ops"), pkg("huge"), pkg("params"), pkg("synth"), pkg("_lib")
        local = int(os.environ["LOCAL_RANK"]); torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        rank, world = dist.get_rank(), dist.get_world_size()
        p = params.for_k(150, H=150, W=584, knn_mode=1)
        a, b, _, _ = synth.make_pair(150, 584, 4)
        g0, g1 = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
        got = huge.flow_pair_sharded(g0, g1, p, 2, 2, 7, lib.BCD_INT32, rank, world, dist)
        want = ops.flow_pair(g0, g1, p, 2, 2, seed=7, bcd_mode=lib.BCD_INT32)
        ok = torch.equal(got, want)
        open(os.path.join({str(tmp_path)!r}, f"ok{{rank}}"), "w").write(str(ok))
        dist.destroy_process_group()
    """))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29547", str(script)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    assert open(tmp_path / "ok0").read() == "True" and open(tmp_path / "ok1").read() == "True"


@pytest.mark.parametrize("nparts", [2, 3])
def test_bcd_in_pieces_equals_whole(nparts):
    """flowb200_bcd_prepare / flowb200_bcd_phase with the chains of every phase split into parts, the parts run one
    after the other on this GPU with their own workspaces and label replicas, differences summed as the all-reduce of
    huge.bcd_sharded does: the reference's labels (bcd_q12 fixture)."""
    ops, ioc, lib = pkg("ops"), pkg("io_contract"), pkg("_lib")
    z = load_npz("bcd_q12")
    sweeps, shift = int(z["meta"][5]), int(z["meta"][6])
    pvec = dev(ioc.pack_proposals(z["proposals"]))
    m, nprop = dev(z["m"], torch.int32), dev(z["nprop"], torch.int32)
    kw = dict(mode=lib.BCD_INT32, cost_shift=shift)
    wss = [ops.bcd_workspace(pvec, nparts).clone() for _ in range(nparts)]   # a part's share of the record arena
    for r in range(nparts):
        ops.bcd_prepare(pvec, m, nprop, wss[r], r, nparts, **kw)
    labels = dev(z["labels00"], torch.int32)
    for w in range(sweeps):
        for phase in range(4):
            total = torch.zeros_like(labels)
            for r in range(nparts):
                mine = labels.clone()
                ops.bcd_phase(pvec, m, nprop, mine, wss[r], phase, r, nparts, **kw)
                total += mine - labels
            labels = labels + total
        assert np.array_equal(labels.cpu().numpy(), z[f"labels{w + 1:02d}"]), w


def test_ctx_batch_of_host_pairs_equals_single_calls():
    """flowb200_ctx_flow_pairs_host (a rank's share of BASELINE configs[3], copies overlapped with the computation) returns,
    for every pair, exactly what flowb200_ctx_flow_pair_host returns for it with the same seed."""
    import ctypes as C
    ops, lib, synth, params = pkg("ops"), pkg("_lib"), pkg("synth"), pkg("params")
    L = lib.load()
    H, W = 52, 70
    p = params.FlowParams(H=H, W=W, cellw=16, cellh=12, n_gauss=10, maxnprop=140)
    cp = ops.cparams(p, bcd_mode=lib.BCD_INT32)
    ctx = L.flowb200_ctx_create(C.byref(cp))
    assert ctx
    try:
        for n in (1, 2, 5):
            pairs = [synth.make_pair(H, W, 20 + i, max_dx=5, max_dy=3, n_rect=1)[:2] for i in range(n)]
            want = []
            for i, (a, b) in enumerate(pairs):
                o = np.empty((H, W, 3), np.float32)
                lib.check(L.flowb200_ctx_flow_pair_host(ctx, a.ctypes.data, b.ctypes.data, 2, 2, 7 + i, o.ctypes.data), "single")
                want.append(o)
            outs = [np.full((H, W, 3), np.nan, np.float32) for _ in range(n)]
            Arr = C.c_void_p * n
            lib.check(L.flowb200_ctx_flow_pairs_host(ctx, Arr(*[a.ctypes.data for a, _ in pairs]),
                                                     Arr(*[b.ctypes.data for _, b in pairs]), n, 2, 2, 7,
                                                     Arr(*[o.ctypes.data for o in outs])), "batch")
            for i in range(n):
                assert np.array_equal(outs[i], want[i]), (n, i)
        assert L.flowb200_ctx_flow_pairs_host(ctx, None, None, 0, 2, 2, 0, None) == lib.EINVAL
    finally:
        L.flowb200_ctx_destroy(ctx)


def test_best_labels_kernel():
    """flowb200_best_labels = the first strict minimum of the first nprop data costs (daisy i flann.py:181-184), ties and
    empty pixels included; on a real proposal set it reproduces the labels the search itself returns."""
    ops, params, synth = pkg("ops"), pkg("params"), pkg("synth")
    rng = np.random.default_rng(8)
    H, W, K = 37, 53, 70
    lc = rng.integers(0, 6, (H, W, K)).astype(np.float32) * 0.25          # many ties
    npr = rng.integers(0, K + 1, (H, W)).astype(np.int32)
    want = np.zeros((H, W), np.int32)
    for y in range(H):
        for x in range(W):
            if npr[y, x]:
                want[y, x] = int(np.argmin(lc[y, x, :npr[y, x]]))
    got = ops.best_labels(dev(lc), dev(npr)).cpu().numpy()
    assert np.array_equal(got, want)
    p = params.FlowParams(H=61, W=90, cellw=16, cellh=12, n_gauss=0, maxnprop=125, knn_mode=1)
    a, b, _, _ = synth.make_pair(61, 90, 5, max_dx=5, max_dy=3, n_rect=2)
    d1, d2 = ops.daisy(dev(a)), ops.daisy(dev(b))
    pv, lcost, nprop, labels = ops.knn_proposals(d1, d2, p)
    assert torch.equal(ops.best_labels(lcost, nprop), labels)


@pytest.mark.parametrize("K", [1, 31, 32, 33, 64, 65, 512])
def test_best_labels_kernel_edges(K):
    """flowb200_best_labels = the first strict minimum of the first nprop data costs (daisy i flann.py:181-184), ties and
    empty pixels included, at K around the warp width: nprop 0, 1, 31, 32, 33 and K; equal minima 32 slots apart (one
    lane) and 1 apart (two lanes); a smaller cost at slot nprop (ignored); costs 0, 1e-45 (subnormal), 1000 and +inf.
    (Costs are >= 0 and not -0.0: the kernel orders them by their bits.)"""
    ops = pkg("ops")
    rng = np.random.default_rng(8 + K)
    H, W = 37, 53
    lc = rng.integers(0, 6, (H, W, K)).astype(np.float32) * 0.25          # many ties
    npr = np.where(rng.random((H, W)) < 0.5, rng.choice([0, 1, 31, 32, 33, K], (H, W)),
                   rng.integers(0, K + 1, (H, W))).clip(0, K).astype(np.int32)
    special = np.array([0.0, 1e-45, 1000.0, np.inf], np.float32)
    assert special[1] > 0                                                  # the smallest subnormal, not flushed
    flat_c, flat_n = lc.reshape(H * W, K), npr.reshape(H * W)
    for p in range(H * W):
        n, kind = int(flat_n[p]), p % 5
        if kind == 0 and n > 32:                     # equal minima at s and s + 32
            s = int(rng.integers(0, n - 32))
            flat_c[p, :n] = rng.uniform(1, 2, n)
            flat_c[p, [s, s + 32]] = 0.5
        elif kind == 1 and n > 1:                    # equal minima at s and s + 1
            s = int(rng.integers(0, n - 1))
            flat_c[p, :n] = rng.uniform(1, 2, n)
            flat_c[p, [s, s + 1]] = 0.5
        elif kind == 2 and n < K:                    # a smaller cost just past nprop
            flat_c[p, :n] = rng.uniform(1, 2, n)
            flat_c[p, n] = 0.0
        elif kind == 3:                              # special values inside nprop
            flat_c[p, :n] = special[rng.integers(0, 4, n)]
        elif kind == 4:                              # mostly 1000 / +inf, one subnormal
            flat_c[p, :n] = special[rng.integers(2, 4, n)]
            if n:
                flat_c[p, int(rng.integers(0, n))] = special[1]
    want = np.array([int(np.argmin(flat_c[p, :flat_n[p]])) if flat_n[p] else 0 for p in range(H * W)],
                    np.int32).reshape(H, W)
    got = ops.best_labels(dev(lc), dev(npr)).cpu().numpy()
    assert np.array_equal(got, want)
