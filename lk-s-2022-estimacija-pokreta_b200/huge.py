"""Single-huge-image mode (BASELINE.json configs[4], SURVEY.md section 8e): one image pair on several GPUs.

The proposal search is the part that shards: the TARGET cells are partitioned into contiguous bands of cell
columns, one band per rank.  A rank searches only its band (plus nothing else: it crops the target descriptors to
its band and the source descriptors to the columns whose +-cell_radius window reaches the band, and runs the
ordinary per-cell exact search on that sub-image).  In the reference's slot order (daisy i flann.py:162-177: cell
column major, cell row minor, then rank) the proposals one source pixel gets from one band are ONE contiguous slot
range, so the "merge of per-GPU top-K lists" is not a comparison merge: every rank packs the slot ranges of its band,
one all-gather moves them, and every rank copies slot ranges into place (`merge_bands`, NCCL over NVLink; gloo in the
CPU tests).  BCD shards too: the
chains of a phase are independent, every rank runs a contiguous share of them and one all-reduce of the label
differences per phase gives every rank the phase's result (`bcd_sharded`).  DAISY, the random proposals and the
consistency check are cheap and run replicated, with identical results on every rank.

All functions here are host-side planning and torch.distributed plumbing; the arithmetic is the C-ABI kernels'.
"""
from dataclasses import dataclass
from functools import lru_cache

import numpy as np

from .params import FlowParams


@dataclass(frozen=True)
class Band:
    rank: int
    ci_lo: int        # target cell columns [ci_lo, ci_hi) searched by this rank
    ci_hi: int
    sx0: int          # source columns [sx0, sx1) of the sub-image (sx0 is a multiple of cellw)
    sx1: int
    tx0: int          # target columns of the sub-image = the same [sx0, sx1); only the band's cells are searched
    tx1: int          # (FlowParams.cell_x0 / cell_x1), the other slots stay unwritten and the merge ignores them

    @property
    def width(self):
        return self.sx1 - self.sx0


@lru_cache(maxsize=64)
def band_plan(p: FlowParams, world: int):
    """Contiguous, balanced bands of target cell columns.  Ranks beyond the number of cell columns get empty bands.
    (The plans of this module are pure functions of the frozen parameters and are cached: at 3840x2160 they cost the
    host more per call than the device needs for the copies they describe.)"""
    n, R, cw = p.ncellx, p.cell_radius, p.cellw
    bands = []
    for r in range(world):
        lo, hi = (n * r) // world, (n * (r + 1)) // world
        if hi <= lo:
            bands.append(Band(r, lo, lo, 0, 0, 0, 0))
            continue
        sx0 = max(0, lo - R) * cw
        sx1 = min(p.W, (hi + R) * cw)
        bands.append(Band(r, lo, hi, sx0, sx1, sx0, sx1))
    return bands


def sub_params(p: FlowParams, b: Band) -> FlowParams:
    """Parameters of the rank's sub-image problem (full height, columns [sx0, sx1)); only the band's own cell columns
    are searched (the sub-image also holds up to cell_radius halo columns on either side, which the source pixels of
    the band's edge need as SOURCES only)."""
    from dataclasses import replace
    c0 = b.ci_lo - b.sx0 // p.cellw
    return replace(p.with_shape(p.H, b.width), cell_x0=c0, cell_x1=c0 + (b.ci_hi - b.ci_lo))


@lru_cache(maxsize=64)
def _row_groups(p: FlowParams):
    """Maximal runs of image rows whose number of cell rows in range is the same: [(y0, y1, n_cj)]."""
    out = []
    y = 0
    while y < p.H:
        r = y // p.cellh
        n = max(0, min(p.ncelly - 1, r + p.cell_radius) - max(0, r - p.cell_radius) + 1)
        y1 = min(p.H, (r + 1) * p.cellh)
        if out and out[-1][2] == n:
            out[-1] = (out[-1][0], y1, n)
        else:
            out.append((y, y1, n))
        y = y1
    return out


@lru_cache(maxsize=256)
def copy_plan(p: FlowParams, b: Band):
    """Slot-range copies that place band `b`'s proposals into the full-image arrays:
    [(y0, y1, x0, x1, dst_slot0, src_slot0, nslots)] with dst[y0:y1, x0:x1, dst_slot0:+n] = src[y0:y1, x0-sx0:x1-sx0,
    src_slot0:+n].  Slot of the r-th neighbour from cell (ci, cj) at pixel (y, x): k*((ci-ci_min)*n_cj + (cj-cj_min)) + r
    (SURVEY.md appendix A); n_cj and cj_min are the same in the sub-image (full height), ci_min differs."""
    if b.ci_hi <= b.ci_lo:
        return []
    R, cw, k = p.cell_radius, p.cellw, p.k_cell
    sub_c0 = b.sx0 // cw
    plan = []
    q_last = (p.W - 1) // cw
    for q in range(q_last + 1):
        x0, x1 = max(q * cw, b.sx0), min(min(p.W, (q + 1) * cw), b.sx1)
        if x0 >= x1:
            continue
        g_lo, g_hi = max(0, q - R), min(p.ncellx - 1, q + R)
        c_lo, c_hi = max(b.ci_lo, g_lo), min(b.ci_hi - 1, g_hi)
        if c_lo > c_hi:
            continue
        s_lo = max(sub_c0, g_lo)
        for y0, y1, n_cj in _row_groups(p):
            if n_cj <= 0:
                continue
            plan.append((y0, y1, x0, x1, (c_lo - g_lo) * n_cj * k, (c_lo - s_lo) * n_cj * k, (c_hi - c_lo + 1) * n_cj * k))
    return plan


def nn_counts(p: FlowParams):
    """nprop after generisi: k * (cell columns in range) * (cell rows in range), int32 (H, W)."""
    R = p.cell_radius
    qx = np.arange(p.W) // p.cellw
    qy = np.arange(p.H) // p.cellh
    nx = np.maximum(0, np.minimum(p.ncellx - 1, qx + R) - np.maximum(0, qx - R) + 1)
    ny = np.maximum(0, np.minimum(p.ncelly - 1, qy + R) - np.maximum(0, qy - R) + 1)
    return (p.k_cell * ny[:, None] * nx[None, :]).astype(np.int32)


def nn_counts_on(p: FlowParams, device):
    """nn_counts evaluated on `device` with torch (no host pass over the image, no host-to-device copy)."""
    import torch
    R = p.cell_radius
    qx = torch.arange(p.W, device=device, dtype=torch.int32) // p.cellw
    qy = torch.arange(p.H, device=device, dtype=torch.int32) // p.cellh
    nx = ((qx + R).clamp(max=p.ncellx - 1) - (qx - R).clamp(min=0) + 1).clamp(min=0)
    ny = ((qy + R).clamp(max=p.ncelly - 1) - (qy - R).clamp(min=0) + 1).clamp(min=0)
    return (p.k_cell * ny[:, None] * nx[None, :]).to(torch.int32)


def _plan_elems(plan):
    return sum((y1 - y0) * (x1 - x0) * n for y0, y1, x0, x1, _, _, n in plan)


def pack_band(p: FlowParams, b: Band, sub_pvec, sub_lcost, out):
    """The slot ranges of band `b` that the merge needs (copy_plan order), vectors then costs (viewed as int32), into the
    flat int32 buffer `out`: what a rank sends instead of its whole (halo columns, unused slots) block."""
    plan = copy_plan(p, b)
    half = _plan_elems(plan)
    lc_i = sub_lcost.view(sub_pvec.dtype)
    o = 0
    for y0, y1, x0, x1, _, s0, n in plan:
        cnt = (y1 - y0) * (x1 - x0) * n
        out[o:o + cnt].view(y1 - y0, x1 - x0, n).copy_(sub_pvec[y0:y1, x0 - b.sx0:x1 - b.sx0, s0:s0 + n])
        out[half + o:half + o + cnt].view(y1 - y0, x1 - x0, n).copy_(lc_i[y0:y1, x0 - b.sx0:x1 - b.sx0, s0:s0 + n])
        o += cnt
    return 2 * half


def unpack_band(p: FlowParams, b: Band, flat, pvec, lcost):
    """Inverse of pack_band into the full-image arrays."""
    plan = copy_plan(p, b)
    half = _plan_elems(plan)
    lc_i = lcost.view(pvec.dtype)
    o = 0
    for y0, y1, x0, x1, d0, _, n in plan:
        cnt = (y1 - y0) * (x1 - x0) * n
        pvec[y0:y1, x0:x1, d0:d0 + n] = flat[o:o + cnt].view(y1 - y0, x1 - x0, n)
        lc_i[y0:y1, x0:x1, d0:d0 + n] = flat[half + o:half + o + cnt].view(y1 - y0, x1 - x0, n)
        o += cnt


def _best_labels(lcost, nprop):
    """bestlabels from the merged data costs: flowb200_best_labels on the device.  CPU tensors occur only in the gloo
    tests of this module's host logic (tests/test_huge_plan.py); for them the same definition is evaluated with torch."""
    import torch
    if lcost.is_cuda:
        from . import ops
        return ops.best_labels(lcost, nprop)
    K = lcost.shape[2]
    key = (lcost.contiguous().view(torch.int32).to(torch.int64) << 32) | torch.arange(K, dtype=torch.int64)
    key = torch.where(torch.arange(K)[None, None, :] < nprop[..., None], key, torch.full_like(key, 2 ** 62))
    labels = (key.min(dim=2).values & 0xFFFFFFFF).to(torch.int32)
    return torch.where(nprop > 0, labels, torch.zeros_like(labels))


_TABLES = {}


def _plan_table(p: FlowParams, world: int, which, cap: int, device):
    """The copy plans as the int64 table flowb200_slot_copy takes, on `device` (cached).  which = rank: that band's
    pack table (array = the rank's sub-image, flat = its send buffer); which = -1: the unpack table of ALL bands
    (array = the full image, flat = the all-gather result, band r at offset r * cap)."""
    import torch
    key = (p, world, which, cap, str(device))
    t = _TABLES.get(key)
    if t is None:
        rows = []
        for b in band_plan(p, world):
            if which >= 0 and b.rank != which:
                continue
            plan = copy_plan(p, b)
            half = _plan_elems(plan)
            o = 0
            for y0, y1, x0, x1, d0, s0, n in plan:
                if which >= 0:
                    rows.append((y0, y1, x0 - b.sx0, x1 - b.sx0, s0, n, o, half + o))
                else:
                    rows.append((y0, y1, x0, x1, d0, n, b.rank * cap + o, b.rank * cap + half + o))
                o += (y1 - y0) * (x1 - x0) * n
        t = torch.tensor(rows, dtype=torch.int64).reshape(-1, 8).to(device)
        if len(_TABLES) > 64:
            _TABLES.clear()
        _TABLES[key] = t
    return t


def merge_bands(p: FlowParams, bands, rank, sub_pvec, sub_lcost, device, dist=None, blocks=None):
    """Every rank contributes the slot ranges of its band (packed, no halo columns, no unused slots) to ONE all-gather;
    every rank unpacks all bands into the full proposal set.  On the device packing and unpacking are one
    flowb200_slot_copy launch each; CPU tensors (the gloo tests of this module) take the torch slicing of
    pack_band / unpack_band, which defines what the kernel does.

    sub_pvec int32 / sub_lcost float32: (H, band width, K) of THIS rank (None for an empty band).
    blocks (tests): {rank: (pvec, lcost)} of the other ranks, packed and unpacked locally instead of the all-gather.
    Returns (pvec (H,W,K) int32 filled -1, lcost (H,W,K) float32 filled 1000, nprop int32, labels int32) where
    labels is the first strict argmin of the data cost (daisy i flann.py:181-184)."""
    import torch
    H, W, K = p.H, p.W, p.maxnprop
    pvec = torch.full((H, W, K), -1, dtype=torch.int32, device=device)
    lcost = torch.full((H, W, K), 1000.0, dtype=torch.float32, device=device)
    sizes = [2 * _plan_elems(copy_plan(p, b)) for b in bands]
    cap = max(max(sizes), 1)
    world = len(bands)
    on_gpu = pvec.is_cuda
    if on_gpu:
        from . import ops

    def pack(b, pv, lc, out):
        if on_gpu:
            ops.slot_copy(_plan_table(p, world, b.rank, cap, device), pv, lc, out, True)
        else:
            pack_band(p, b, pv, lc, out)

    recv = torch.empty((world, cap), dtype=torch.int32, device=device)
    if blocks is not None or dist is None or world == 1:
        if sizes[rank]:
            pack(bands[rank], sub_pvec, sub_lcost, recv[rank])
        if blocks is not None:
            for b in bands:
                if b.rank != rank and sizes[b.rank]:
                    pack(b, blocks[b.rank][0], blocks[b.rank][1], recv[b.rank])
    else:
        send = torch.empty(cap, dtype=torch.int32, device=device)
        if sizes[rank]:
            pack(bands[rank], sub_pvec, sub_lcost, send)
        try:
            dist.all_gather_into_tensor(recv.view(-1), send)
        except (RuntimeError, AttributeError, NotImplementedError):
            dist.all_gather([recv[r] for r in range(world)], send)
    if on_gpu:
        ops.slot_copy(_plan_table(p, world, -1, cap, device), pvec, lcost, recv.view(-1), False)
    else:
        for b in bands:
            if sizes[b.rank]:
                unpack_band(p, b, recv[b.rank], pvec, lcost)
    nprop = nn_counts_on(p, device)
    labels = _best_labels(lcost, nprop)       # first strict argmin of the data costs (daisy i flann.py:181-184)
    return pvec, lcost, nprop, labels


def knn_proposals_sharded(desc_src, desc_tgt, p: FlowParams, rank, world, dist=None, knn_mode=None):
    """generisi for one direction with the target cells sharded over `world` ranks.  Same outputs as
    ops.knn_proposals on one device."""
    from . import ops
    if world == 1:   # nothing to merge: the ordinary search
        return ops.knn_proposals(desc_src, desc_tgt, p, knn_mode=knn_mode)
    bands = band_plan(p, world)
    b = bands[rank]
    sub_pvec = sub_lcost = None
    if b.ci_hi > b.ci_lo:
        sp = sub_params(p, b)
        s = desc_src[:, b.sx0:b.sx1].contiguous()
        t = desc_tgt[:, b.tx0:b.tx1].contiguous()
        sub_pvec, sub_lcost, _, _ = ops.knn_proposals(s, t, sp, knn_mode=knn_mode)
    return merge_bands(p, bands, rank, sub_pvec, sub_lcost, desc_src.device, dist)


def bcd_sharded(pvec, cost, nprop, labels, sweeps, p: FlowParams, mode, rank, world, dist=None, ops=None):
    """ceoBCD with every phase's chains split over the ranks.  The chains of a phase are independent (they read and
    write only their own pixels), so a rank runs its share and the ranks then exchange what changed: every rank holds
    the full label image, `new - old` is zero outside the rank's own chains, and one all-reduce(sum) of that difference
    per phase (4 bytes per pixel over NVLink) gives every rank the phase's result.
    `ops` (tests): a stand-in for the device operators with the same bcd_workspace / bcd_prepare / bcd_phase."""
    if ops is None:
        from . import ops
    ws = ops.bcd_workspace(pvec, world)
    kw = dict(mode=mode, lamda=p.lamda, tpsi=p.tpsi, cost_shift=p.cost_shift)
    ops.bcd_prepare(pvec, cost, nprop, ws, rank, world, **kw)
    for _ in range(sweeps):
        for phase in range(4):
            if dist is None or world == 1:
                ops.bcd_phase(pvec, cost, nprop, labels, ws, phase, rank, world, **kw)
                continue
            before = labels.clone()
            ops.bcd_phase(pvec, cost, nprop, labels, ws, phase, rank, world, **kw)
            delta = labels - before
            dist.all_reduce(delta)
            labels.copy_(before + delta)
    return labels


def flow_pair_sharded(bgr0, bgr1, p: FlowParams, sweeps, directions, seed, bcd_mode, rank, world, dist=None,
                      want_raw=False):
    """The whole path for ONE pair on `world` ranks: DAISY replicated, proposal search sharded by target cell band and
    merged over `dist`, the rest replicated.  Returns what ops.flow_pair returns, identical on every rank."""
    import torch
    from . import ops, _lib
    d = [ops.daisy(bgr0), ops.daisy(bgr1)]
    uvv = []
    for direction in range(directions):
        src, tgt = d[direction], d[1 - direction]
        pvec, lcost, nprop, labels = knn_proposals_sharded(src, tgt, p, rank, world, dist)
        ops.random_proposals(src, tgt, p, pvec, lcost, nprop, labels, seed=seed + direction)
        mrf = bcd_mode & _lib.BCD_MRF
        if (bcd_mode & ~_lib.BCD_MRF) in (_lib.BCD_INT32, _lib.BCD_INT32_F32COST):
            bcd_sharded(pvec, lcost, nprop, labels, sweeps, p, _lib.BCD_INT32_F32COST | mrf, rank, world, dist)
        else:   # the float64 programme is not split: replicated
            ops.bcd(pvec, lcost, nprop, labels, sweeps, mode=_lib.BCD_FP64_F32COST | mrf, lamda=p.lamda, tpsi=p.tpsi,
                    cost_shift=p.cost_shift)
        if p.flow_refine:
            uvv.append(ops.flow_subpixel(src, tgt, pvec, nprop, labels))
        else:
            uvv.append(ops.flow_from_labels(pvec, labels, want_yx=False)[1])
        del pvec, lcost
    out = uvv[0].clone()
    if directions == 2:
        ops.consistency(out, uvv[1], p.con_tresh)
    if want_raw:
        return out, uvv[0], (uvv[1] if directions == 2 else None)
    return out
