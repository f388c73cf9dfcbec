"""Full-size (BASELINE.json configs[1]: 1024x436, K=300) checks, mostly through properties that do not need the CPU
oracle (the stage-by-stage oracle comparisons at this size are in test_gpu_baseline_configs.py; they take minutes):

* the tcgen05 search equals an independent float64 brute force (torch) on sampled (pixel, cell) tasks, and every
  block of k proposals is sorted by distance;
* the two BCD programmes (bcd_ksets.cu: int32 and float64) give the C oracle's labels after every sweep on costs
  quantised to 20*m/2^12 (the oracle's two sweeps take about 30 s on 8 host threads), and the int32 programme does not
  depend on how much of the record cache fits the workspace;
* the consistency check is idempotent.
"""
import numpy as np
import pytest

from helpers import pkg

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

H, W, K = 436, 1024, 300


@pytest.fixture(scope="module")
def stage1():
    ops, params, synth = pkg("ops"), pkg("params"), pkg("synth")
    p = params.for_k(K, H=H, W=W, knn_mode=1)
    a, b, _, _ = synth.make_pair(H, W, 5)
    d1, d2 = ops.daisy(torch.from_numpy(a).cuda()), ops.daisy(torch.from_numpy(b).cuda())
    pvec, lcost, nprop, labels, idx, _ = ops.knn_proposals(d1, d2, p, want_idx=True)
    return p, d1, d2, pvec, lcost, nprop, labels, idx


def test_search_equals_float64_brute_force_on_sampled_tasks(stage1):
    p, d1, d2, pvec, lcost, nprop, labels, idx = stage1
    rng = np.random.default_rng(0)
    R, k = p.cell_radius, p.k_cell
    for _ in range(300):
        y, x = int(rng.integers(0, H)), int(rng.integers(0, W))
        qx, qy = x // p.cellw, y // p.cellh
        cis = list(range(max(0, qx - R), min(p.ncellx - 1, qx + R) + 1))
        cjs = list(range(max(0, qy - R), min(p.ncelly - 1, qy + R) + 1))
        if not cis or not cjs:
            continue
        bi, bj = int(rng.integers(0, len(cis))), int(rng.integers(0, len(cjs)))
        ci, cj = cis[bi], cjs[bj]
        blk = bi * len(cjs) + bj
        t = d2[cj * p.cellh:(cj + 1) * p.cellh, ci * p.cellw:(ci + 1) * p.cellw].reshape(-1, 68).double()
        q = d1[y, x].double()
        dist = ((t - q) * (t - q)).sum(1)            # (float64 sum in torch's order: ties at 1e-16 level are not expected)
        order = torch.argsort(dist, stable=True)[:k]
        got = idx[y, x, blk].long()
        assert torch.equal(got, order), (y, x, ci, cj)
        assert bool((dist[got][1:] >= dist[got][:-1]).all())
        v = pvec[y, x, blk * k:(blk + 1) * k]
        dy, dx = (v << 16 >> 16), (v >> 16)
        assert torch.equal(dy.long(), cj * p.cellh + got // p.cellw - y) and torch.equal(dx.long(), ci * p.cellw + got % p.cellw - x)


def test_two_bcd_implementations_agree_and_cache_size_does_not_matter(stage1):
    from oracle import cport
    ops, lib, ioc = pkg("ops"), pkg("_lib"), pkg("io_contract")
    p, d1, d2, pvec, lcost, nprop, labels, _ = stage1
    pv, lc, npr = pvec.clone(), lcost.clone(), nprop.clone()
    ops.random_proposals(d1, d2, p, pv, lc, npr, labels, seed=3)
    m = ops.quantise_costs(lc, p.lamda, 12)
    lq = (m.double() * (20.0 / 4096.0))
    lq = torch.where(lc == 1000.0, torch.full_like(lq, 1000.0), lq)
    want = np.stack(cport.ceo_bcd(ioc.unpack_proposals(pv.cpu().numpy()), lq.cpu().numpy(), npr.cpu().numpy(),
                                  labels.cpu().numpy(), 2))
    a = labels.clone()
    sa = ops.bcd(pv, m, npr, a, 2, mode=lib.BCD_INT32, cost_shift=12, per_sweep=True).cpu().numpy()
    sb = ops.bcd(pv, lq, npr, labels.clone(), 2, mode=lib.BCD_FP64_F64COST, per_sweep=True).cpu().numpy()
    for w in range(2):
        assert np.array_equal(sa[w], want[w]), ("int32", w, float((sa[w] != want[w]).mean()))
        assert np.array_equal(sb[w], want[w]), ("float64", w, float((sb[w] != want[w]).mean()))
    assert float((a != labels).float().mean()) > 0.05          # the sweeps did something
    c = labels.clone()
    L = lib.load()
    small = L.flowb200_bcd_min_workspace_bytes(H, W, K) + (L.flowb200_bcd_workspace_bytes(H, W, K) -
                                                          L.flowb200_bcd_min_workspace_bytes(H, W, K)) // 3
    ops.bcd(pv, m, npr, c, 2, mode=lib.BCD_INT32, cost_shift=12, workspace_bytes=small)
    assert torch.equal(c, a)


def test_consistency_check_is_idempotent(stage1):
    ops = pkg("ops")
    p, d1, d2, pvec, lcost, nprop, labels, _ = stage1
    pb, lb, nb, labb = ops.knn_proposals(d2, d1, p)
    f = ops.flow_from_labels(pvec, labels, want_yx=False)[1]
    g = ops.flow_from_labels(pb, labb, want_yx=False)[1]
    once = ops.consistency(f.clone(), g, p.con_tresh)
    twice = ops.consistency(once.clone(), g, p.con_tresh)
    assert torch.equal(once, twice)
    assert 0.2 < float(once[..., 2].mean()) <= 1.0
