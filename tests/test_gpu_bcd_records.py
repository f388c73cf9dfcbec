"""The K-set records of the BCD programme (csrc/bcd_ksets.cu), read out of the workspace and compared entry by entry
with a host restatement, and the record path -- every chain step on a stored record, no chain left to the fallback --
at every tpsi, cost shift and chain width against the C oracle.

The label tests of test_gpu_parity.py draw their vectors from a small square, so nearly every record overflows the
build kernel's staging and their chains run on the dense fallback; the record path there only sees the real proposal
sets (tpsi 8, cost shift 12).  Here the proposal sets are made so that the records fit, and the module asserts that
they did: a case whose records were not stored would silently test the fallback instead.

Costs as in test_gpu_parity.py: integer m for BCD_INT32, 20 m / 2^S (exact in float32 and float64) for the other modes
and the oracle, so that every mode must give the oracle's labels exactly.
"""
import numpy as np
import pytest

from helpers import pkg

# ---------------------------------------------------------------- restated constants of csrc/bcd_ksets.cu
HASH_Y, HASH_X = 16, 64           # kHashY, kHashX: bucket coordinates offset by 8 / 32 and clamped
REC_HEADER = 16                   # kRecHeader
MAX_LIST = 124                    # kMaxList
NULL_ENTRY = 0x8FF8               # kNullEntry
COST_LIMIT = 1 << 16              # kCostLimit16
STAGE_PER_LABEL = 16              # kStagePerLabel
SLOT_PER_LABEL = 12               # kSlotPerLabel
FITS, STAGING, LIST, COST, SLOT = range(5)   # predicted outcome of a record (arena exhaustion aside)

MODES = ("BCD_INT32", "BCD_INT32_F32COST", "BCD_FP64_F64COST", "BCD_FP64_F32COST")


def lib():
    return pkg("_lib")


def align_up(v, a=256):
    return (v + a - 1) // a * a


def kset_layout(H, W, K, workspace_bytes=0):
    """kset_layout: byte offsets of the workspace's parts; workspace_bytes 0 = the recommended size."""
    Kpad, Kst, n = (K + 31) // 32 * 32, (K + 7) // 8 * 8, H * W
    col, row = (W + 1) // 2 * H, (H + 1) // 2 * W
    L, off = dict(Kpad=Kpad, Kst=Kst), 0
    for name, nbytes in (("bp", max(col, row) * Kpad * 2), ("sorig", n * Kst * 2), ("svec", n * Kst * 4),
                         ("desc", 2 * n * 8), ("cursor", 256), ("flags", (max(W, H) + 1) // 2 * 4)):
        L[name] = off
        off += align_up(nbytes)
    L["arena"] = off
    if workspace_bytes == 0:
        L["arena_bytes"] = 2 * n * (REC_HEADER + 16 + 10 * K + 18 * K)
    else:
        L["arena_bytes"] = (workspace_bytes - off) & ~15 if workspace_bytes > off else 0
    L["total"] = off + align_up(L["arena_bytes"])
    return L


def slot_bytes(Kpad):
    """kset_slot_bytes"""
    return (REC_HEADER + 2 * Kpad + 8 * Kpad + 2 * SLOT_PER_LABEL * Kpad + 127) & ~127


def bucket_shift(tpsi):
    b = 0
    while (1 << b) < tpsi:
        b += 1
    return b


def chain_width(K):
    """T of make_plan's FB_KS_CASE table and the chains per SM it aims at."""
    return next((T, mb) for T, mb in ((64, 8), (128, 6), (192, 5), (256, 4), (320, 4), (384, 3), (512, 2)) if K <= T)


def slot_shift(H, W, K):
    """make_plan: four record slots, or two when four would not leave `minb` chains of the shorter orientation
    resident on an SM (budget = 227 KB / minb - 1.5 KB; the 32-bit kernel's fixed part 4 KB pad + dp 4 KB + control
    384 B + 6 B per chain step, 128-aligned)."""
    _, mb = chain_width(K)
    budget = 227 * 1024 // mb - 1024 - 512
    fixed = (4096 + 384 + 6 * min(H, W) + 127) & ~127
    return 1 if 4096 + fixed + 4 * slot_bytes((K + 31) // 32 * 32) > budget else 2


def dp_bound_ok(H, W, tpsi, shift):
    """make_plan's bound of the int32 modes: a chain of max(H, W) steps, each adding at most a 16-bit data cost, two
    side terms and one pairwise term of at most tpsi << shift, stays below 0xFFFF0000."""
    return max(H, W) * ((3 * tpsi << shift) + 65535) < 0xFFFF0000


def prev_pixels(H, W, orient):
    """prev_pixel for every pixel (flat index, -1 at the start of a chain)."""
    y, x = np.divmod(np.arange(H * W), W)
    if orient == 0:
        yq = np.where(x & 1, y + 1, y - 1)
        return np.where((yq < 0) | (yq >= H), -1, yq * W + x)
    xq = np.where(y & 1, x - 1, x + 1)
    return np.where((xq < 0) | (xq >= W), -1, y * W + xq)


def owns_line(line, nlines, part, nparts):
    line = np.asarray(line)
    nch = np.where(line & 1, nlines // 2, (nlines + 1) // 2)
    c = line >> 1
    return (c >= nch * part // nparts) & (c < nch * (part + 1) // nparts)


def owned_tasks(H, W, part, nparts):
    """(2, H*W) bool: the records part `part` builds (column chains of its columns, row chains of its rows)."""
    y, x = np.divmod(np.arange(H * W), W)
    return np.stack([owns_line(x, W, part, nparts), owns_line(y, H, part, nparts)])


def bucket_yx(dy, dx, b):
    return np.clip((dy >> b) + HASH_Y // 2, 0, HASH_Y - 1), np.clip((dx >> b) + HASH_X // 2, 0, HASH_X - 1)


def pack(prop):
    return pkg("io_contract").pack_proposals(prop)


def quantised(m_or_cost, mode, shift):
    """the data cost field of a record: m (BCD_INT32), rint(0.05 * c * 2^S) (BCD_INT32_F32COST), 0 (float64 modes)"""
    if mode == "BCD_INT32":
        return np.asarray(m_or_cost, np.int64)
    if mode == "BCD_INT32_F32COST":
        return np.rint(0.05 * np.asarray(m_or_cost, np.float32).astype(np.float64) * float(1 << shift)).astype(np.int64)
    return np.zeros(np.shape(m_or_cost), np.int64)


# ---------------------------------------------------------------- host restatement of the records
def predict(prop, nprop, mq, tpsi, mode):
    """Every record kset_build_kernel would build, as the host sees it.

    prop int (H,W,K,2) [dy,dx]; nprop (H,W); mq (H,W,K) the data cost field (quantised()).  Returns a dict of arrays
    over the 2*H*W tasks (task = orient * H*W + pixel): status (FITS or the first reason it does not), bytes, and per
    task the list lengths (n,) and the sorted keys label << 16 | entry of every stored entry."""
    H, W, K, _ = prop.shape
    npix, Kpad, b = H * W, (K + 31) // 32 * 32, bucket_shift(tpsi)
    dy, dx = prop[..., 0].reshape(npix, K).astype(np.int64), prop[..., 1].reshape(npix, K).astype(np.int64)
    ky, kx = bucket_yx(dy, dx, b)
    by, bx = dy >> b, dx >> b
    ry0, ry1 = bucket_yx(by - 1 << b, bx - 1 << b, b)   # first bucket row / column of the 3 x 3 block
    ry2, ry3 = bucket_yx(by + 1 << b, bx + 1 << b, b)
    npr = nprop.reshape(npix).astype(np.int64)
    mq = mq.reshape(npix, K)
    status, nbytes, lens, keys = np.zeros(2 * npix, np.int64), np.zeros(2 * npix, np.int64), [None] * 2 * npix, \
        [None] * 2 * npix
    sb = slot_bytes(Kpad)
    for orient in (0, 1):
        prv = prev_pixels(H, W, orient)
        for p in range(npix):
            n, q = int(npr[p]), int(prv[p])
            task = orient * npix + p
            cost_ok = mode not in ("BCD_INT32", "BCD_INT32_F32COST") or bool(np.all((mq[p, :n] >= 0) &
                                                                                  (mq[p, :n] < COST_LIMIT)))
            if q >= 0:
                nq = int(npr[q])
                l1 = np.abs(dy[p, :n, None] - dy[q, None, :nq]) + np.abs(dx[p, :n, None] - dx[q, None, :nq])
                member = l1 < tpsi
                cand = ((ky[q, None, :nq] >= ry0[p, :n, None]) & (ky[q, None, :nq] <= ry2[p, :n, None]) &
                        (kx[q, None, :nq] >= ry1[p, :n, None]) & (kx[q, None, :nq] <= ry3[p, :n, None])).sum()
                ln = member.sum(1)
                j, k = np.nonzero(member)
                keys[task] = np.sort((j << 16) | (k << 3) | (l1[j, k] << 12))
            else:
                cand, ln, keys[task] = 0, np.zeros(n, np.int64), np.zeros(0, np.int64)
            lens[task] = ln
            eo = REC_HEADER + 2 * ((n + 7) & ~7) + 8 * n
            nbytes[task] = (eo + 8 * int(((ln + 3) // 4).sum()) + 15) & ~15
            if not cost_ok:
                status[task] = COST
            elif cand > STAGE_PER_LABEL * Kpad:
                status[task] = STAGING
            elif ln.max(initial=0) > MAX_LIST:
                status[task] = LIST
            elif nbytes[task] > sb:
                status[task] = SLOT
    return dict(status=status, bytes=nbytes, lens=lens, keys=keys)


# ---------------------------------------------------------------- the workspace, read back
class Workspace:
    """the workspace's sort output, descriptors, cursor and record arena, copied to the host as needed"""

    def __init__(self, ws, H, W, K):
        self.L = L = kset_layout(H, W, K, ws.numel())
        self.H, self.W, self.K, self.ws = H, W, K, ws
        n = H * W
        self.desc = self._bytes(L["desc"], 16 * n).view(np.uint64).astype(np.int64)
        self.cursor = int(self._bytes(L["cursor"], 8).view(np.uint64)[0])
        self._arena = None

    def _bytes(self, off, nbytes):
        return self.ws[off:off + nbytes].cpu().numpy()

    @property
    def sorig(self):
        return self._bytes(self.L["sorig"], 2 * self.H * self.W * self.L["Kst"]).view(np.uint16).reshape(
            self.H * self.W, -1)

    @property
    def svec(self):
        return self._bytes(self.L["svec"], 4 * self.H * self.W * self.L["Kst"]).view(np.int32).reshape(
            self.H * self.W, -1)

    @property
    def arena(self):
        if self._arena is None:
            self._arena = self._bytes(self.L["arena"], self.cursor)
        return self._arena

    def offsets(self):
        d = self.desc
        return (d & ((1 << 40) - 1)) << 4, (d >> 40) << 4

    def record(self, task):
        """decode one record: header, group offsets, structs, entries"""
        off, size = (int(x[task]) for x in self.offsets())
        rec = self.arena[off:off + size]
        n, groups, so, eo = (int(x) for x in rec[:16].view(np.uint32))
        st = rec[so:so + 8 * n].view(np.uint32).reshape(n, 2).astype(np.int64)
        return dict(size=size, n=n, groups=groups, so=so, eo=eo,
                    goff=rec[REC_HEADER:REC_HEADER + 2 * n].view(np.uint16).astype(np.int64),
                    vec=st[:, 0].astype(np.uint32).view(np.int32), cost=st[:, 1] & 0xFFFF,
                    label=(st[:, 1] >> 16) & 511, ng=st[:, 1] >> 25,
                    ents=rec[eo:eo + 8 * groups].view(np.uint16).astype(np.int64))


def check_sort(wsr, pvec, nprop, tpsi, pixels):
    """kset_sort_kernel: sorig[:n] is a permutation, svec = pvec[sorig], bucket keys do not decrease"""
    K, b = wsr.K, bucket_shift(tpsi)
    pv = pvec.reshape(-1, K)
    sorig, svec = wsr.sorig, wsr.svec
    for p in np.flatnonzero(pixels):
        n = int(nprop.reshape(-1)[p])
        so = sorig[p, :n].astype(np.int64)
        assert np.array_equal(np.sort(so), np.arange(n)), p
        sv = svec[p, :n]
        assert np.array_equal(sv, pv[p, so]), p
        dy, dx = ((sv.astype(np.int64) & 0xFFFF) ^ 0x8000) - 0x8000, sv.astype(np.int64) >> 16
        ky, kx = bucket_yx(dy, dx, b)
        assert np.all(np.diff(ky * HASH_X + kx) >= 0), p


def check_records(wsr, pvec, mq, pred, tasks=None, arena_full=True):
    """Every record against the host restatement (compared by label: the order among equal-length lists and inside a
    list comes from atomics).  tasks: bool (2*H*W,) of the records the part builds (others must have descriptor 0).
    Returns the number of stored records."""
    H, W, K = wsr.H, wsr.W, wsr.K
    npix = H * W
    tasks = np.ones(2 * npix, bool) if tasks is None else tasks
    want = tasks & (pred["status"] == FITS)
    if arena_full:
        assert np.array_equal(wsr.desc != 0, want), np.flatnonzero((wsr.desc != 0) != want)[:10]
        assert wsr.cursor == int(pred["bytes"][want].sum())
    else:
        assert not np.any((wsr.desc != 0) & ~want)
    off, size = wsr.offsets()
    stored = np.flatnonzero(wsr.desc)
    o = np.argsort(off[stored])
    ends = off[stored][o] + size[stored][o]
    assert np.all(ends[:-1] <= off[stored][o][1:]) and (len(ends) == 0 or ends[-1] <= wsr.L["arena_bytes"])
    pv = pvec.reshape(npix, K)
    mq = mq.reshape(npix, K)
    for task in stored:
        p = task % npix
        r = wsr.record(task)
        n, lens = r["n"], pred["lens"][task]
        assert n == len(lens) and r["size"] == pred["bytes"][task], task
        assert r["so"] == REC_HEADER + 2 * ((n + 7) & ~7) and r["eo"] == r["so"] + 8 * n, task
        assert r["size"] == (r["eo"] + 8 * r["groups"] + 15) & ~15, task
        lab = r["label"]
        assert np.array_equal(np.sort(lab), np.arange(n)), task
        assert np.array_equal(r["vec"], pv[p, lab]) and np.array_equal(r["cost"], mq[p, lab] & 0xFFFF), task
        ln = lens[lab]
        assert np.all(np.diff(ln) <= 0), task                       # non-increasing list length
        assert np.array_equal(r["ng"], (ln + 3) // 4), task
        starts = np.concatenate([[0], np.cumsum(r["ng"])[:-1]])    # disjoint, in position order, inside the header count
        assert np.array_equal(r["goff"], starts) and r["ng"].sum() == r["groups"], task
        pos = np.repeat(np.arange(n), r["ng"])
        within = ((np.arange(r["groups"]) - r["goff"][pos])[:, None] * 4 + np.arange(4)).reshape(-1)
        valid = within < np.repeat(ln, r["ng"] * 4)
        ents = r["ents"]
        assert np.all(ents[~valid] == NULL_ENTRY) and np.all(ents[valid] & 0x8000 == 0), task
        got = np.sort((np.repeat(lab, r["ng"] * 4)[valid] << 16) | ents[valid])
        assert np.array_equal(got, pred["keys"][task]), task
    return len(stored)


# ---------------------------------------------------------------- proposal sets whose records fit
def fitting_set(rng, H, W, K, tpsi, costs="wide", ragged=False, clusters=True, region=None):
    """Proposal vectors inside the unclamped hash box of tpsi's bucket shift: each pixel takes a window of K of one
    pool of 1.5 K vectors (neighbouring windows overlap), a quarter of them moved by less than tpsi.  Checkerboard
    clusters of repeated vectors (copies on even / odd pixels: 32 / 1, 14 / 1, 6 / 1, 3 / 2) give lists of 32, 14,
    6 and 3 entries; pool vectors far from every neighbour's give empty lists.

    Returns prop int32 (H,W,K,2) [dy,dx] (unused slots -1), nprop int64 (H,W), m int32 (H,W,K), lab0 int64 (H,W).
    costs: "wide" m in [0, 65535], "ties" m in [0, 3]."""
    b = bucket_shift(tpsi)
    ylo, yhi, xlo, xhi = region or (-(8 << b), (8 << b) - 1, -(32 << b), (32 << b) - 1)
    cl = [(32, 1), (14, 1), (6, 1), (3, 2)] if K >= 100 else [(14, 1), (6, 1), (3, 2)] if K >= 33 else []
    if not clusters:
        cl = []
    # cluster centres: one bucket row of the box, two buckets apart (their 3 x 3 blocks are disjoint)
    cy = np.full(len(cl), ylo)
    cx = xlo + (2 << b) * np.arange(len(cl)) + (1 << b)
    # pool: distinct vectors at least three bucket rows away from the cluster row
    py0 = ylo + (3 << b)
    G = K + K // 2
    cells = (yhi - py0 + 1) * (xhi - xlo + 1)
    assert cells >= G, (K, tpsi)
    flat = rng.choice(cells, G, replace=False)
    pool = np.stack([py0 + flat // (xhi - xlo + 1), xlo + flat % (xhi - xlo + 1)], 1)
    # vector table: the pool, then the cluster centres; slot s of a pixel's list before its rotation holds the
    # pixel's cluster copies (s < ncl), then a window of the pool
    table = np.concatenate([pool, np.stack([cy, cx], 1)]).astype(np.int32)
    slot_cl = [np.full(K, -1, np.int64), np.full(K, -1, np.int64)]     # cluster of slot s: even, odd pixels
    for par in (0, 1):
        s0 = 0
        for i, ac in enumerate(cl):
            slot_cl[par][s0:s0 + ac[par]] = G + i
            s0 += ac[par]
    npix = H * W
    y, x = np.divmod(np.arange(npix, dtype=np.int32), W)
    odd = ((y + x) % 2).astype(np.int32)
    ncl = np.array([sum(a for a, _ in cl), sum(c for _, c in cl)], np.int32)[odd]
    start = rng.integers(0, G, npix, dtype=np.int32)
    rot = rng.integers(0, K, npix, dtype=np.int32)
    j = np.arange(K, dtype=np.int32)
    s = (j[None, :] + rot[:, None]) % K                              # labels: the list rotated by a random amount
    idx = np.where(s < ncl[:, None], np.stack(slot_cl)[odd[:, None], s], (start[:, None] + s - ncl[:, None]) % G)
    v = table[idx]                                                   # (npix, K, 2)
    if tpsi > 1:   # a quarter of the pool vectors moved by an L1 distance of 0..tpsi-1
        offs = np.array([(a, sg * (d - abs(a))) for d in range(tpsi) for a in range(-d, d + 1) for sg in (-1, 1)],
                        np.int32)
        pick = rng.integers(0, 4 * len(offs), (npix, K), dtype=np.int32)
        moved = (pick < len(offs)) & (idx < G)
        v[moved] += offs[pick[moved]]
        np.clip(v[..., 0], py0, yhi, out=v[..., 0])
        np.clip(v[..., 1], xlo, xhi, out=v[..., 1])
    nprop = rng.integers(max(1, K - K // 4), K + 1, npix) if ragged else np.full(npix, K)
    v[j[None, :] >= nprop[:, None]] = -1
    m = rng.integers(0, 65536 if costs == "wide" else 4, (npix, K), dtype=np.int32)
    lab0 = rng.integers(0, 1 << 30, npix) % nprop
    return v.reshape(H, W, K, 2), nprop.reshape(H, W).astype(np.int64), m.reshape(H, W, K), lab0.reshape(H, W)


# ---------------------------------------------------------------- running the library
def dev(a, dtype):
    torch = pytest.importorskip("torch")
    return torch.from_numpy(np.ascontiguousarray(a)).to(dtype).cuda()


def mode_inputs(mode, m, shift):
    """cost tensor of `mode` for integer costs m: m itself (BCD_INT32) or 20 m / 2^S, exact in float32 and float64"""
    import torch
    lq = 20.0 * m / float(1 << shift)
    if mode == "BCD_INT32":
        return dev(m, torch.int32)
    return dev(lq, torch.float64 if mode == "BCD_FP64_F64COST" else torch.float32)


def oracle(prop, nprop, m, lab0, shift, sweeps, tpsi):
    from oracle import cport
    return np.stack(cport.ceo_bcd(prop, 20.0 * m / float(1 << shift), nprop, lab0, sweeps, tpsi=tpsi))


def workspace(H, W, K, nbytes=None):
    import torch
    L = lib().load()
    nb = L.flowb200_bcd_workspace_bytes(H, W, K) if nbytes is None else int(nbytes)
    return torch.zeros(nb, dtype=torch.uint8, device="cuda")


def run_bcd(pvec, cost, nprop, lab0, sweeps, mode, tpsi, shift, ws):
    """flowb200_bcd with a caller-owned workspace; labels after every sweep (sweeps, H, W)"""
    import torch
    ops, L = pkg("ops"), lib()
    H, W, K = pvec.shape
    labels = dev(lab0, torch.int32)
    snaps = torch.empty((sweeps, H, W), dtype=torch.int32, device="cuda")
    rc = L.load().flowb200_bcd(ops._ptr(pvec), ops._ptr(cost), ops._ptr(nprop), ops._ptr(labels), H, W, K,
                               getattr(L, mode), 0.05, int(tpsi), int(shift), int(sweeps), ops._ptr(snaps),
                               ops._ptr(ws), ws.numel(), ops._stream())
    L.check(rc, "flowb200_bcd")
    return snaps.cpu().numpy()


def run_phases(pvec, cost, nprop, lab0, sweeps, mode, tpsi, shift, ws, part=0, nparts=1):
    """bcd_prepare + bcd_phase (int32 modes): labels after every sweep, and the chain flags of every phase"""
    import torch
    ops, L = pkg("ops"), lib()
    H, W, K = pvec.shape
    kw = dict(mode=getattr(L, mode), lamda=0.05, tpsi=tpsi, cost_shift=shift)
    ops.bcd_prepare(pvec, cost, nprop, ws, part, nparts, **kw)
    labels = dev(lab0, torch.int32)
    Lw = kset_layout(H, W, K, ws.numel())
    snaps, flags = [], []
    for _ in range(sweeps):
        for phase in range(4):
            ops.bcd_phase(pvec, cost, nprop, labels, ws, phase, part, nparts, **kw)
            nch = ((W + 1) // 2, (H + 1) // 2, W // 2, H // 2)[phase]
            flags.append(ws[Lw["flags"]:Lw["flags"] + 4 * nch].cpu().numpy().view(np.int32).copy())
        snaps.append(labels.cpu().numpy())
    return np.stack(snaps), flags


def device_case(prop, nprop, m):
    import torch
    return dev(pack(prop), torch.int32), dev(nprop, torch.int32)


# ================================================================ CPU tests: the restatements
def test_layout_restatement_matches_the_library():
    """kset_layout restated: a layout change in bcd_ksets.cu fails here, not as garbage reads in the GPU tests."""
    L = lib().load()
    for H, W, K in ((1, 1, 1), (1, 40, 33), (40, 1, 64), (37, 41, 150), (662, 700, 300), (2, 16383, 40),
                    (436, 1024, 300), (17, 29, 511), (5, 6, 512)):
        ly = kset_layout(H, W, K)
        assert ly["arena"] == L.flowb200_bcd_min_workspace_bytes(H, W, K), (H, W, K)
        assert ly["total"] == L.flowb200_bcd_workspace_bytes(H, W, K), (H, W, K)


def test_make_plan_restatements():
    """the ring of two slots starts at min(H, W) = 662 at T = 320 and, at T = 192, at 1622 for K = 161..192 but 2390
    for K = 150 (the slot size follows Kpad: the 3840x2160 K = 150 workload keeps four slots); the dp bound admits
    chains of 9362 steps at shift 14 and 16383 at shift 13 (tpsi 8), one step fewer than refused"""
    assert slot_shift(1622, 1700, 192) == 1 and slot_shift(1621, 1700, 192) == 2
    assert slot_shift(2390, 2400, 150) == 1 and slot_shift(2389, 2400, 150) == 2 and slot_shift(2160, 3840, 150) == 2
    assert slot_shift(662, 700, 300) == 1 and slot_shift(661, 700, 300) == 2
    assert dp_bound_ok(2, 9362, 8, 14) and not dp_bound_ok(2, 9363, 8, 14)
    assert dp_bound_ok(2, 16383, 8, 13) and not dp_bound_ok(2, 16384, 8, 13)


@pytest.mark.parametrize("K", [33, 100, 511])
def test_fitting_set_fits_at_every_tpsi(K):
    """the generator's records all fit (predicted), at every tpsi, ragged nprop included; and its lists cover the
    lengths 0, 1..4, 5..8, 13..31 and 32 or more"""
    hist = np.zeros(MAX_LIST + 2, np.int64)
    for tpsi in range(1, 9):
        rng = np.random.default_rng(K * 10 + tpsi)
        prop, nprop, m, _ = fitting_set(rng, 5, 6, K, tpsi, ragged=tpsi % 2 == 0)
        pred = predict(prop, nprop, quantised(m, "BCD_INT32", 12), tpsi, "BCD_INT32")
        assert np.all(pred["status"] == FITS), (K, tpsi, np.bincount(pred["status"]))
        for ln in pred["lens"]:
            hist += np.bincount(ln, minlength=len(hist))[:len(hist)]
    assert hist[0] and hist[1:5].sum() and hist[5:9].sum() and hist[13:32].sum(), hist
    if K >= 100:
        assert hist[32:].sum(), hist


# ================================================================ GPU tests
@pytest.mark.gpu
@pytest.mark.parametrize("tpsi", range(1, 9))
def test_record_contents(tpsi):
    """Every record of the generator's sets equals the host restatement, in every mode; the sort agrees; the labels
    are the oracle's after every sweep.  Parts 2 and 3 build only the records of their own lines, the same ones."""
    H, W, K, shift, sweeps = 7, 9, 100, 12, 2
    rng = np.random.default_rng(100 + tpsi)
    prop, nprop, m, lab0 = fitting_set(rng, H, W, K, tpsi, costs="ties" if tpsi % 2 else "wide", ragged=tpsi > 4)
    pvec, npr = device_case(prop, nprop, m)
    pv = pack(prop)
    want = oracle(prop, nprop, m, lab0, shift, sweeps, tpsi)
    for mode in MODES:
        mq = quantised(m if mode == "BCD_INT32" else 20.0 * m / float(1 << shift), mode, shift)
        pred = predict(prop, nprop, mq, tpsi, mode)
        assert np.all(pred["status"] == FITS)
        cost = mode_inputs(mode, m, shift)
        ws = workspace(H, W, K)
        if mode.startswith("BCD_INT32"):
            got, flags = run_phases(pvec, cost, npr, lab0, sweeps, mode, tpsi, shift, ws)
            assert all(not f.any() for f in flags), mode
        else:
            got = run_bcd(pvec, cost, npr, lab0, sweeps, mode, tpsi, shift, ws)
        assert np.array_equal(got, want), mode
        wsr = Workspace(ws, H, W, K)
        check_sort(wsr, pv, nprop, tpsi, np.ones(H * W, bool))
        assert check_records(wsr, pv, mq, pred) == 2 * H * W
        if mode == "BCD_INT32":
            for nparts in (2, 3):
                for part in range(nparts):
                    wp = workspace(H, W, K)
                    pkg("ops").bcd_prepare(pvec, cost, npr, wp, part, nparts, mode=lib().BCD_INT32, tpsi=tpsi,
                                           cost_shift=shift)
                    own = owned_tasks(H, W, part, nparts)
                    wpr = Workspace(wp, H, W, K)
                    check_records(wpr, pv, mq, pred, tasks=own.reshape(-1))
                    check_sort(wpr, pv, nprop, tpsi, own[0] | own[1])


# ---- the record path at every tpsi, cost shift and chain width
PATH_CASES = [
    # H, W, K, tpsi, shift, int32 on float costs too
    (1, 40, 33, 1, 4, False), (40, 1, 40, 2, 7, True), (23, 31, 64, 3, 11, False), (17, 29, 65, 4, 12, True),
    (19, 27, 100, 5, 13, False), (21, 25, 129, 7, 14, True), (15, 33, 150, 8, 4, False), (13, 21, 193, 1, 7, False),
    (24, 17, 250, 2, 11, True), (11, 19, 257, 3, 12, False), (18, 13, 300, 4, 13, False), (9, 23, 321, 5, 14, True),
    (14, 15, 384, 7, 4, False), (12, 17, 511, 8, 12, True), (2, 2, 129, 8, 13, False), (31, 9, 33, 7, 14, False),
    (3, 37, 256, 1, 12, False), (25, 1, 384, 3, 7, True), (1, 1, 100, 4, 11, False), (16, 16, 192, 8, 14, False),
]


def test_path_cases_cover_every_tpsi_shift_and_width():
    tp = {c[3] for c in PATH_CASES}
    sh = {c[4] for c in PATH_CASES}
    ks = {c[2] for c in PATH_CASES}
    assert {1, 2, 3, 4, 5, 7, 8} <= tp and {4, 7, 11, 12, 13, 14} <= sh
    assert {33, 40, 64, 65, 100, 129, 150, 193, 250, 257, 300, 321, 384, 511} <= ks
    assert {chain_width(K)[0] for K in ks} == {64, 128, 192, 256, 320, 384, 512}
    assert any(c[0] == 1 for c in PATH_CASES) and any(c[1] == 1 for c in PATH_CASES)
    assert {c[3] for c in PATH_CASES if c[5]} >= {2, 4, 7, 8}   # BCD_INT32_F32COST in some cases


@pytest.mark.gpu
@pytest.mark.parametrize("H,W,K,tpsi,shift,f32", PATH_CASES, ids=[f"{c[0]}x{c[1]}-K{c[2]}-t{c[3]}-s{c[4]}"
                                                                  for c in PATH_CASES])
def test_record_path(H, W, K, tpsi, shift, f32):
    """Every record stored, every chain on the 32-bit kernel (no flag after any phase), the oracle's labels after
    every sweep; the float64 modes on the same records."""
    sweeps = 2
    rng = np.random.default_rng(H * 7919 + W * 31 + K + tpsi * 13 + shift)
    prop, nprop, m, lab0 = fitting_set(rng, H, W, K, tpsi, costs="ties" if (H + W) % 2 else "wide",
                                       ragged=K % 2 == 1)
    pvec, npr = device_case(prop, nprop, m)
    want = oracle(prop, nprop, m, lab0, shift, sweeps, tpsi)
    modes = ["BCD_INT32"] + (["BCD_INT32_F32COST"] if f32 else []) + ["BCD_FP64_F64COST", "BCD_FP64_F32COST"]
    for mode in modes:
        ws = workspace(H, W, K)
        cost = mode_inputs(mode, m, shift)
        if mode.startswith("BCD_INT32"):
            got, flags = run_phases(pvec, cost, npr, lab0, sweeps, mode, tpsi, shift, ws)
            assert all(not f.any() for f in flags), mode
        else:
            got = run_bcd(pvec, cost, npr, lab0, sweeps, mode, tpsi, shift, ws)
        desc = Workspace(ws, H, W, K).desc
        assert np.all(desc != 0), (mode, int((desc == 0).sum()))
        assert np.array_equal(got, want), mode


@pytest.mark.gpu
def test_arena_exhausted_at_an_exact_byte():
    """A workspace of min + the records' total stores every record; 16 bytes less stores all but one, whose chain
    alone is left to the fallback; the labels are the oracle's either way."""
    H, W, K, tpsi, shift, sweeps = 10, 12, 100, 8, 12, 2
    prop, nprop, m, lab0 = fitting_set(np.random.default_rng(7), H, W, K, tpsi)
    pvec, npr = device_case(prop, nprop, m)
    pv = pack(prop)
    pred = predict(prop, nprop, m, tpsi, "BCD_INT32")
    assert np.all(pred["status"] == FITS)
    total = int(pred["bytes"].sum())
    lo = lib().load().flowb200_bcd_min_workspace_bytes(H, W, K)
    want = oracle(prop, nprop, m, lab0, shift, sweeps, tpsi)
    cost = mode_inputs("BCD_INT32", m, shift)
    for short in (0, 16):
        ws = workspace(H, W, K, lo + total - short)
        got, flags = run_phases(pvec, cost, npr, lab0, sweeps, "BCD_INT32", tpsi, shift, ws)
        assert np.array_equal(got, want), short
        wsr = Workspace(ws, H, W, K)
        assert wsr.cursor == total                     # the record that did not fit was counted all the same
        check_records(wsr, pv, m, pred, arena_full=False)
        missing = np.flatnonzero(wsr.desc == 0)
        assert len(missing) == (short // 16), missing
        assert sum(int(f.sum()) for f in flags[:4]) == len(missing)
        if short:
            task = int(missing[0])
            orient, p = divmod(task, H * W)
            y, x = divmod(p, W)
            phase = (0 if x % 2 == 0 else 2) if orient == 0 else (1 if y % 2 == 0 else 3)
            assert flags[phase][(x if orient == 0 else y) // 2] == 1


@pytest.mark.gpu
def test_record_format_limits():
    """Records at the limits of the format, made by editing pixels of a fitting set (tpsi 8; the pool is kept in the
    lower rows of the hash box, the edits use the top rows): lists of 124 (stored) and 125 (not), data costs 65535
    (stored) and 65536 (not), a record of exactly a slot (stored) and 16 bytes more (not), staging overflow, and
    vectors beyond the hash range (negative ones on bucket edges, magnitudes in the thousands).  The predicted
    outcome of every record is the stored one, and the labels are the oracle's."""
    H, W, K, tpsi, shift, sweeps = 6, 12, 160, 8, 12, 2
    b = bucket_shift(tpsi)
    region = (-(8 << b) + (4 << b), (8 << b) - 1, -(32 << b), (32 << b) - 1)   # pool: bucket rows 4..15
    prop, nprop, m, lab0 = fitting_set(np.random.default_rng(11), H, W, K, tpsi, region=region, clusters=False)
    Ytop = -(8 << b)                                                          # bucket row 0
    col = lambda i: -(32 << b) + (2 << b) * i + 3                            # noqa: E731  two buckets apart
    # row 0 runs right to left: the previous pixel of (0, x) is (0, x + 1)
    prop[0, 1, :124] = (Ytop, col(0))                 # (0, 0): one label on 124 copies -> a list of 124
    prop[0, 0, 0] = (Ytop, col(0))
    prop[0, 3, :125] = (Ytop, col(2))                 # (0, 2): a list of 125
    prop[0, 2, 0] = (Ytop, col(2))
    # a record of exactly a slot: q holds 7 clusters of 16 copies and 4 of 12; p puts 6 labels on the 16s, 154 on
    # the 12s: 6 * 4 + 154 * 3 = 486 groups; 16 bytes more with 8 and 152 (488 groups)
    for px, a in ((4, 6), (6, 8)):
        q = [(Ytop, col(i)) for i in range(7) for _ in range(16)] + [(Ytop, col(7 + i)) for i in range(4) for _ in
                                                                     range(12)]
        prop[0, px + 1] = q
        prop[0, px] = [(Ytop, col(i % 7)) for i in range(a)] + [(Ytop, col(7 + i % 4)) for i in range(K - a)]
    # staging overflow: 160 x 160 candidates in one bucket pair, no member (L1 = 9)
    prop[0, 9] = (Ytop, col(20))
    prop[0, 8] = (Ytop, col(20) + 9)
    # vectors beyond the hash box and on bucket edges (row 2 runs right to left too; row 3 left to right)
    edges = [(-1, -1), (-1, 0), (0, -1), (-(1 << b), -(1 << b)), (-(1 << b) - 1, -(1 << b) - 1), (-(1 << b), 3),
             (-1, -(1 << b) - 1), (3000, -2500), (-4000, 2999), (2999, 4000), (-3001, -3005), (1 << 14, -(1 << 14))]
    for y, x in ((2, 5), (2, 6), (3, 5), (3, 6), (4, 6)):
        e = np.array(edges)
        jit = np.random.default_rng(y * 100 + x).integers(-1, 2, e.shape)
        prop[y, x, :len(edges)] = np.concatenate([e[:6], e[6:] + jit[6:]])
        prop[y, x, len(edges):2 * len(edges)] = e + jit
    npix = H * W
    m = m.copy()
    m[0, 10, 3] = 65535
    m[1, 10, 4] = 65536
    pred = predict(prop, nprop, m, tpsi, "BCD_INT32")
    st = pred["status"]
    task = lambda y, x, orient=1: orient * npix + y * W + x                   # noqa: E731
    assert int(pred["lens"][task(0, 0)].max()) == 124 and st[task(0, 0)] == FITS
    assert int(pred["lens"][task(0, 2)].max()) == 125 and st[task(0, 2)] == LIST
    Kpad = (K + 31) // 32 * 32
    assert pred["bytes"][task(0, 4)] == slot_bytes(Kpad) and st[task(0, 4)] == FITS
    assert pred["bytes"][task(0, 6)] == slot_bytes(Kpad) + 16 and st[task(0, 6)] == SLOT
    assert st[task(0, 8)] == STAGING
    assert st[task(0, 10, 0)] == FITS and st[task(0, 10, 1)] == FITS
    assert st[task(1, 10, 0)] == COST and st[task(1, 10, 1)] == COST
    edge_tasks = [task(y, x, o) for y, x in ((2, 5), (3, 5), (3, 6)) for o in (0, 1)]
    assert np.all(st[edge_tasks] == FITS), st[edge_tasks]
    assert (st == FITS).sum() > 0.9 * len(st)
    pvec, npr = device_case(prop, nprop, m)
    pv = pack(prop)
    want = oracle(prop, nprop, m, lab0, shift, sweeps, tpsi)
    for mode in ("BCD_INT32", "BCD_FP64_F64COST"):
        ws = workspace(H, W, K)
        cost = mode_inputs(mode, m, shift)
        if mode == "BCD_INT32":
            got, _ = run_phases(pvec, cost, npr, lab0, sweeps, mode, tpsi, shift, ws)
            mq = m
        else:
            got = run_bcd(pvec, cost, npr, lab0, sweeps, mode, tpsi, shift, ws)
            mq = np.zeros_like(m)
            pred = predict(prop, nprop, mq, tpsi, mode)
        assert np.array_equal(got, want), mode
        wsr = Workspace(ws, H, W, K)
        check_sort(wsr, pv, nprop, tpsi, np.ones(npix, bool))
        check_records(wsr, pv, mq, pred)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [511, 512])
def test_records_at_the_label_limit(K):
    """K = 511: entries reach label 510 and the 32-bit kernel runs every chain; K = 512: entries point at label 511,
    whose dp slot the 32-bit kernel keeps for the padding entries, so every chain is left to the fallback."""
    H, W, tpsi, shift, sweeps = 4, 5, 8, 12, 2
    prop, nprop, m, lab0 = fitting_set(np.random.default_rng(K), H, W, K, tpsi)
    # the last label of every pixel: one vector, shared by all pixels
    prop[:, :, K - 1] = (7, 9)
    pvec, npr = device_case(prop, nprop, m)
    pv = pack(prop)
    pred = predict(prop, nprop, m, tpsi, "BCD_INT32")
    assert np.all(pred["status"] == FITS)
    want = oracle(prop, nprop, m, lab0, shift, sweeps, tpsi)
    ws = workspace(H, W, K)
    got, flags = run_phases(pvec, mode_inputs("BCD_INT32", m, shift), npr, lab0, sweeps, "BCD_INT32", tpsi, shift, ws)
    assert np.array_equal(got, want)
    assert all(np.all(f == (1 if K == 512 else 0)) for f in flags)
    wsr = Workspace(ws, H, W, K)
    check_records(wsr, pv, m, pred)
    top = max(int(((k >> 3) & 511).max(initial=0)) for k in pred["keys"])
    assert top == K - 1
    got = run_bcd(pvec, mode_inputs("BCD_FP64_F64COST", m, shift), npr, lab0, sweeps, "BCD_FP64_F64COST", tpsi,
                  shift, workspace(H, W, K))
    assert np.array_equal(got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("W,shift", [(9362, 14), (16383, 13)])
def test_dp_bound(W, shift):
    """The longest chains make_plan admits, every step adding the most it can: empty K-sets (quirk Q1 adds tpsi),
    both side terms tpsi, data costs 65535 - (0..3); dp ends just under 0xFFFF0000.  One step longer is refused in
    the int32 modes and runs in the float64 ones."""
    H, K, tpsi, sweeps = 2, 40, 8, 1
    rng = np.random.default_rng(W)
    for Wc, ok in ((W, True), (W + 1, False)):
        y, x = np.divmod(np.arange(H * Wc), Wc)
        grp = ((y + x) % 2)[:, None, None]
        prop = rng.integers(-3, 4, (H * Wc, K, 2)) + grp * np.array([0, 200])
        prop = prop.reshape(H, Wc, K, 2).astype(np.int64)
        nprop = np.full((H, Wc), K, np.int64)
        m = (65535 - rng.integers(0, 4, (H, Wc, K))).astype(np.int64)
        lab0 = rng.integers(0, K, (H, Wc)).astype(np.int64)
        assert dp_bound_ok(H, Wc, tpsi, shift) == ok
        want = oracle(prop, nprop, m, lab0, shift, sweeps, tpsi)
        pvec, npr = device_case(prop, nprop, m)
        if ok:
            ws = workspace(H, Wc, K)
            got, flags = run_phases(pvec, mode_inputs("BCD_INT32", m, shift), npr, lab0, sweeps, "BCD_INT32", tpsi,
                                    shift, ws)
            assert all(not f.any() for f in flags)
            assert np.all(Workspace(ws, H, Wc, K).desc != 0)
            assert np.array_equal(got, want)
        else:
            for mode in ("BCD_INT32", "BCD_INT32_F32COST"):
                with pytest.raises(lib().FlowB200Error, match="unsupported"):
                    run_bcd(pvec, mode_inputs(mode, m, shift), npr, lab0, sweeps, mode, tpsi, shift,
                            workspace(H, Wc, K))
            got = run_bcd(pvec, mode_inputs("BCD_FP64_F64COST", m, shift), npr, lab0, sweeps, "BCD_FP64_F64COST",
                          tpsi, shift, workspace(H, Wc, K))
            assert np.array_equal(got, want)


@pytest.mark.gpu
def test_two_slot_ring():
    """T = 320 with the shorter chains 662 steps long: make_plan takes a ring of two record slots.  Every record
    stored, no chain flagged, the oracle's labels, in BCD_INT32 and BCD_FP64_F64COST."""
    H, W, K, tpsi, shift, sweeps = 662, 700, 300, 8, 12, 1
    assert chain_width(K)[0] == 320 and slot_shift(H, W, K) == 1
    prop, nprop, m, lab0 = fitting_set(np.random.default_rng(662), H, W, K, tpsi)
    pvec, npr = device_case(prop, nprop, m)
    want = oracle(prop, nprop, m, lab0, shift, sweeps, tpsi)
    ws = workspace(H, W, K)
    got, flags = run_phases(pvec, mode_inputs("BCD_INT32", m, shift), npr, lab0, sweeps, "BCD_INT32", tpsi, shift, ws)
    assert all(not f.any() for f in flags)
    assert np.all(Workspace(ws, H, W, K).desc != 0)
    assert np.array_equal(got, want)
    ws = workspace(H, W, K)
    got = run_bcd(pvec, mode_inputs("BCD_FP64_F64COST", m, shift), npr, lab0, sweeps, "BCD_FP64_F64COST", tpsi, shift,
                  ws)
    assert np.all(Workspace(ws, H, W, K).desc != 0)
    assert np.array_equal(got, want)
