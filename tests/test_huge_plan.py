"""Single-huge-image mode, host logic on CPU: banded proposal search + slot-range merge reproduces the full-image
proposal set bit for bit (the CPU oracle stands in for the device search), in one process and over two gloo ranks."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from helpers import pkg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _descs(H, W, seed):
    rng = np.random.default_rng(seed)
    return (rng.random((H, W, 68), dtype=np.float32) * 0.05, rng.random((H, W, 68), dtype=np.float32) * 0.05)


def _full(p, d1, d2):
    from oracle import cport
    prop, lc, npr, best = cport.generisi(d1, d2, p)
    ioc = pkg("io_contract")
    return ioc.pack_proposals(prop), lc.astype(np.float32), npr.astype(np.int32), best.astype(np.int32)


def _band_block(p, b, d1, d2):
    import torch
    from oracle import cport
    huge, ioc = pkg("huge"), pkg("io_contract")
    sp = huge.sub_params(p, b)
    prop, lc, _, _ = cport.generisi(d1[:, b.sx0:b.sx1], d2[:, b.tx0:b.tx1], sp)
    return torch.from_numpy(ioc.pack_proposals(prop)), torch.from_numpy(lc.astype(np.float32))


@pytest.mark.parametrize("H,W,cw,ch,R,k,world", [(40, 70, 8, 6, 2, 3, 2), (40, 70, 8, 6, 2, 3, 3), (33, 95, 9, 7, 1, 2, 4),
                                                 (30, 26, 8, 6, 2, 2, 8), (36, 64, 8, 6, 2, 3, 1)])
def test_banded_search_merges_to_full(H, W, cw, ch, R, k, world):
    import torch
    params, huge = pkg("params"), pkg("huge")
    r = 2 * R + 1
    p = params.FlowParams(H=H, W=W, cellw=cw, cellh=ch, cell_radius=R, k_cell=k, n_gauss=0, maxnprop=r * r * k + 3)
    d1, d2 = _descs(H, W, H * W + world)
    want = _full(p, d1, d2)
    bands = huge.band_plan(p, world)
    assert [b.ci_lo for b in bands][0] == 0 and bands[-1].ci_hi == p.ncellx
    assert all(a.ci_hi == b.ci_lo for a, b in zip(bands, bands[1:]))
    blocks = {b.rank: _band_block(p, b, d1, d2) for b in bands if b.ci_hi > b.ci_lo}
    for rank in range(world):
        mine = blocks.get(rank, (None, None))
        pvec, lcost, nprop, labels = huge.merge_bands(p, bands, rank, mine[0], mine[1], "cpu", blocks=blocks)
        assert np.array_equal(pvec.numpy(), want[0])
        assert np.array_equal(lcost.numpy(), want[1])
        assert np.array_equal(nprop.numpy(), want[2])
        assert np.array_equal(labels.numpy(), want[3])


def _slot_copy_emul(table, vec, cost, flat, to_flat):
    """What include/flowb200.h says flowb200_slot_copy does, in numpy (cost as its int32 bit pattern)."""
    ci = cost.view(np.int32)
    for y0, y1, x0, x1, slot0, n, off_vec, off_cost in table:
        cnt = (y1 - y0) * (x1 - x0) * n
        if to_flat:
            flat[off_vec:off_vec + cnt] = vec[y0:y1, x0:x1, slot0:slot0 + n].reshape(-1)
            flat[off_cost:off_cost + cnt] = ci[y0:y1, x0:x1, slot0:slot0 + n].reshape(-1)
        else:
            vec[y0:y1, x0:x1, slot0:slot0 + n] = flat[off_vec:off_vec + cnt].reshape(y1 - y0, x1 - x0, n)
            ci[y0:y1, x0:x1, slot0:slot0 + n] = flat[off_cost:off_cost + cnt].reshape(y1 - y0, x1 - x0, n)


@pytest.mark.parametrize("H,W,cw,ch,R,k,world", [(40, 70, 8, 6, 2, 3, 3), (33, 95, 9, 7, 1, 2, 4), (30, 26, 8, 6, 2, 2, 8)])
def test_slot_copy_tables_describe_the_same_copies_as_the_torch_slicing(H, W, cw, ch, R, k, world):
    """The int64 tables handed to flowb200_slot_copy on the device (huge._plan_table), applied with the header's
    definition of the kernel, give what pack_band / unpack_band (the CPU path of merge_bands) give."""
    import torch
    params, huge = pkg("params"), pkg("huge")
    r = 2 * R + 1
    p = params.FlowParams(H=H, W=W, cellw=cw, cellh=ch, cell_radius=R, k_cell=k, n_gauss=0, maxnprop=r * r * k + 3)
    rng = np.random.default_rng(world)
    bands = huge.band_plan(p, world)
    sizes = [2 * huge._plan_elems(huge.copy_plan(p, b)) for b in bands]
    cap = max(max(sizes), 1)
    K = p.maxnprop
    blocks = {b.rank: (rng.integers(-9, 9, (H, b.width, K)).astype(np.int32), rng.random((H, b.width, K), dtype=np.float32))
              for b in bands if b.ci_hi > b.ci_lo}
    recv = np.zeros(world * cap, dtype=np.int32)
    for b in bands:
        if sizes[b.rank]:
            t = huge._plan_table(p, world, b.rank, cap, "cpu").numpy()
            send = np.zeros(cap, dtype=np.int32)
            _slot_copy_emul(t, blocks[b.rank][0], blocks[b.rank][1], send, True)
            want = torch.zeros(cap, dtype=torch.int32)
            huge.pack_band(p, b, torch.from_numpy(blocks[b.rank][0]), torch.from_numpy(blocks[b.rank][1]), want)
            assert np.array_equal(send, want.numpy())
            recv[b.rank * cap:(b.rank + 1) * cap] = send
    pvec, lcost = np.full((H, W, K), -1, dtype=np.int32), np.full((H, W, K), 1000.0, dtype=np.float32)
    _slot_copy_emul(huge._plan_table(p, world, -1, cap, "cpu").numpy(), pvec, lcost, recv, False)
    tb = {r_: (torch.from_numpy(a), torch.from_numpy(c)) for r_, (a, c) in blocks.items()}
    mine = tb.get(0, (None, None))
    want = huge.merge_bands(p, bands, 0, mine[0], mine[1], "cpu", blocks=tb)
    assert np.array_equal(pvec, want[0].numpy()) and np.array_equal(lcost, want[1].numpy())


def test_two_gloo_ranks_exchange_bands(tmp_path):
    pytest.importorskip("torch")
    script = tmp_path / "w.py"
    script.write_text(textwrap.dedent(f"""
        import importlib, os, sys
        import numpy as np, torch, torch.distributed as dist
        sys.path.insert(0, {ROOT!r}); sys.path.insert(0, os.path.join({ROOT!r}, "tests"))
        from helpers import pkg
        from oracle import cport
        params, huge, ioc = pkg("params"), pkg("huge"), pkg("io_contract")
        dist.init_process_group("gloo")
        rank, world = dist.get_rank(), dist.get_world_size()
        p = params.FlowParams(H=40, W=70, cellw=8, cellh=6, cell_radius=2, k_cell=3, n_gauss=0, maxnprop=80)
        rng = np.random.default_rng(5)
        d1 = rng.random((40, 70, 68), dtype=np.float32) * 0.05
        d2 = rng.random((40, 70, 68), dtype=np.float32) * 0.05
        bands = huge.band_plan(p, world)
        b = bands[rank]
        prop, lc, _, _ = cport.generisi(d1[:, b.sx0:b.sx1], d2[:, b.tx0:b.tx1], huge.sub_params(p, b))
        got = huge.merge_bands(p, bands, rank, torch.from_numpy(ioc.pack_proposals(prop)),
                               torch.from_numpy(lc.astype(np.float32)), "cpu", dist=dist)
        prop, lc, npr, best = cport.generisi(d1, d2, p)
        ok = (np.array_equal(got[0].numpy(), ioc.pack_proposals(prop)) and np.array_equal(got[1].numpy(), lc.astype(np.float32))
              and np.array_equal(got[2].numpy(), npr.astype(np.int32)) and np.array_equal(got[3].numpy(), best.astype(np.int32)))
        open(os.path.join({str(tmp_path)!r}, f"ok{{rank}}"), "w").write(str(ok))
    """))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29541", str(script)],
                       capture_output=True, text=True, timeout=300, env=dict(os.environ, OMP_NUM_THREADS="1"))
    assert r.returncode == 0, r.stderr[-3000:]
    assert open(tmp_path / "ok0").read() == "True" and open(tmp_path / "ok1").read() == "True"


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_bcd_phases_with_delta_exchange_equal_full_sweeps(world):
    """Splitting every phase's chains over `world` parts and summing the label differences (what huge.bcd_sharded
    does with an all-reduce) reproduces the oracle's full sweeps: the chains of a phase are independent."""
    from oracle import bcd as obcd
    rng = np.random.default_rng(world)
    H, W, K = 9, 11, 12
    prop = rng.integers(-6, 7, (H, W, K, 2)).astype(np.int64)
    nprop = rng.integers(3, K + 1, (H, W)).astype(np.int64)
    lc = 20.0 * rng.integers(0, 513, (H, W, K)) / 4096.0
    lab0 = (rng.integers(0, 1 << 20, (H, W)) % nprop).astype(np.int64)
    want = obcd.ceo_bcd(prop, lc, nprop, lab0, 2)[-1]
    phases = [(1, 0, [(0, x) for x in range(0, W, 2)]), (0, -1, [(y, W - 1) for y in range(0, H, 2)]),
              (-1, 0, [(H - 1, x) for x in range(1, W, 2)]), (0, 1, [(y, 0) for y in range(1, H, 2)])]
    labels = [lab0.copy() for _ in range(world)]          # every rank's replica
    for _ in range(2):
        for ys, xs, starts in phases:
            n = len(starts)
            deltas = []
            for r in range(world):
                mine = starts[n * r // world:n * (r + 1) // world]
                before = labels[r].copy()
                if mine:
                    obcd._phase(prop, lc, nprop, labels[r], 8, 0.05, ys, xs, mine)
                deltas.append(labels[r] - before)
                labels[r] = before
            total = sum(deltas)                           # the all-reduce
            for r in range(world):
                labels[r] = labels[r] + total
    for r in range(world):
        assert np.array_equal(labels[r], want)


class _OracleOps:
    """CPU stand-in for ops.bcd_workspace / bcd_prepare / bcd_phase: the oracle's _phase on the owned chains."""

    def __init__(self, prop, lc, nprop):
        self.prop, self.lc, self.nprop = prop, lc, nprop

    def bcd_workspace(self, pvec, nparts=1):
        return None

    def bcd_prepare(self, *a, **k):
        pass

    def bcd_phase(self, pvec, cost, nprop, labels, ws, phase, part, nparts, **kw):
        from oracle import bcd as obcd
        H, W = labels.shape
        geo = [(1, 0, [(0, x) for x in range(0, W, 2)]), (0, -1, [(y, W - 1) for y in range(0, H, 2)]),
               (-1, 0, [(H - 1, x) for x in range(1, W, 2)]), (0, 1, [(y, 0) for y in range(1, H, 2)])][phase]
        n = len(geo[2])
        mine = geo[2][n * part // nparts:n * (part + 1) // nparts]     # ksets_phase's chain range, csrc/bcd_ksets.cu
        if mine:
            lab = labels.numpy().astype(np.int64)
            obcd._phase(self.prop, self.lc, self.nprop, lab, 8, 0.05, geo[0], geo[1], mine)
            labels.copy_(__import__("torch").from_numpy(lab.astype(np.int32)))


def test_two_gloo_ranks_bcd_sharded(tmp_path):
    """huge.bcd_sharded itself (per-phase label difference all-reduce) over two gloo ranks, the oracle standing in
    for the device operators: both ranks end with the oracle's full sweeps."""
    pytest.importorskip("torch")
    script = tmp_path / "w.py"
    script.write_text(textwrap.dedent(f"""
        import os, sys
        import numpy as np, torch, torch.distributed as dist
        sys.path.insert(0, {ROOT!r}); sys.path.insert(0, os.path.join({ROOT!r}, "tests"))
        from helpers import pkg
        from oracle import bcd as obcd
        from test_huge_plan import _OracleOps
        params, huge = pkg("params"), pkg("huge")
        dist.init_process_group("gloo")
        rank, world = dist.get_rank(), dist.get_world_size()
        rng = np.random.default_rng(9)
        H, W, K = 8, 10, 10
        prop = rng.integers(-6, 7, (H, W, K, 2)).astype(np.int64)
        nprop = rng.integers(3, K + 1, (H, W)).astype(np.int64)
        lc = 20.0 * rng.integers(0, 513, (H, W, K)) / 4096.0
        lab0 = (rng.integers(0, 1 << 20, (H, W)) % nprop).astype(np.int64)
        want = obcd.ceo_bcd(prop, lc, nprop, lab0, 2)[-1]
        labels = torch.from_numpy(lab0.astype(np.int32))
        p = params.FlowParams(H=H, W=W, cellw=4, cellh=4, maxnprop=K, n_gauss=0, k_cell=1, cell_radius=0)
        huge.bcd_sharded(None, None, None, labels, 2, p, 3, rank, world, dist, ops=_OracleOps(prop, lc, nprop))
        open(os.path.join({str(tmp_path)!r}, f"ok{{rank}}"), "w").write(str(np.array_equal(labels.numpy(), want)))
    """))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29543", str(script)],
                       capture_output=True, text=True, timeout=300, env=dict(os.environ, OMP_NUM_THREADS="1"))
    assert r.returncode == 0, r.stderr[-3000:]
    assert open(tmp_path / "ok0").read() == "True" and open(tmp_path / "ok1").read() == "True"
