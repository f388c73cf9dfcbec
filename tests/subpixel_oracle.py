"""Sub-pixel refinement of a label field (DESIGN section 4.8), restated in numpy float32.  TEST INFRASTRUCTURE.

For pixel p = (y, x) with label l and vector v = (dy, dx) = pvec[p][l], the cost of the target p + v + e is
    c(e) = sum68_numpy_order(|fl(d1(p)[i] - d2(p + v + e)[i])|)
(oracle.proposals.sum_f32_numpy_order: the NN data cost without the tphi truncation) for e in {(0,0), (0,-1), (0,+1),
(-1,0), (+1,0)}.  Per axis, with c-, c0, c+ along it:
    offset = (c- - c+) / (2 (c- - 2 c0 + c+))       every operation one float32 round-to-nearest, in this order,
applied only when the three targets lie inside the frame and c0 < c-, c0 < c+, then clamped to [-0.5, 0.5] (fmax / fmin:
a NaN offset becomes -0.5); otherwise 0.  Output: float32 (dx + ox, dy + oy, 1).
A label in [0, K) outside [0, nprop), and a (-1, -1) fill vector, give (dx, dy, 1) unrefined (what flowb200_flow_from_labels
writes); a label outside [0, K) names no slot and gives (0, 0, 0).
"""
import numpy as np

from oracle.proposals import sum_f32_numpy_order

F32 = np.float32
FILL = np.int32(-1)          # (-1, -1) packed: 0xFFFFFFFF
OFFSETS = ((0, 0), (0, -1), (0, 1), (-1, 0), (1, 0))


def unpack(v):
    """packed int32 vectors -> (dy, dx) int64 (include/flowb200.h)."""
    v = np.asarray(v, dtype=np.int32)
    dy = (v & 0xFFFF).astype(np.int16).astype(np.int64)
    dx = (v >> 16).astype(np.int64)
    return dy, dx


def pack(dy, dx):
    dy, dx = np.asarray(dy, np.int64), np.asarray(dx, np.int64)
    return ((dy & 0xFFFF) | ((dx & 0xFFFF) << 16)).astype(np.uint32).view(np.int32)


def costs(d1, d2, ys, xs, ty, tx, chunk=1 << 16):
    """c at source pixels (ys, xs) and targets (ty, tx), all in range: float32 (n,)."""
    out = np.empty(len(ys), np.float32)
    for s in range(0, len(ys), chunk):
        e = slice(s, s + chunk)
        out[e] = sum_f32_numpy_order(np.abs(d1[ys[e], xs[e]] - d2[ty[e], tx[e]]))
    return out


def axis_offset(cm, c0, cp):
    """The per-axis offset of three float32 costs (arrays) whose targets are all in the frame."""
    cm, c0, cp = (np.asarray(a, F32) for a in (cm, c0, cp))
    num = cm - cp
    den = F32(2) * ((cm - F32(2) * c0) + cp)
    with np.errstate(divide="ignore", invalid="ignore"):
        o = (num / den).astype(F32)
    o = np.fmin(np.fmax(o, F32(-0.5)), F32(0.5))
    return np.where((c0 < cm) & (c0 < cp), o, F32(0)).astype(F32)


def subpixel(desc_src, desc_tgt, pvec, nprop, labels):
    """float32 (H, W, 3) = (u, v, valid), what flowb200_flow_subpixel writes."""
    d1 = np.ascontiguousarray(desc_src, F32)
    d2 = np.ascontiguousarray(desc_tgt, F32)
    pvec = np.asarray(pvec, np.int32)
    H, W, K = pvec.shape
    lab = np.asarray(labels, np.int64).reshape(H, W)
    npr = np.minimum(np.asarray(nprop, np.int64).reshape(H, W), K)
    out = np.zeros((H, W, 3), F32)
    slot = (lab >= 0) & (lab < K)
    ys, xs = np.nonzero(slot)
    v = pvec[ys, xs, lab[ys, xs]]
    dy, dx = unpack(v)
    out[ys, xs, 0] = dx.astype(F32)
    out[ys, xs, 1] = dy.astype(F32)
    out[ys, xs, 2] = F32(1)
    ty, tx = ys + dy, xs + dx
    live = (lab[ys, xs] < npr[ys, xs]) & (v != FILL) & (ty >= 0) & (ty < H) & (tx >= 0) & (tx < W)
    ys, xs, dy, dx, ty, tx = (a[live] for a in (ys, xs, dy, dx, ty, tx))
    c0 = costs(d1, d2, ys, xs, ty, tx)
    for axis, (n, t, d, ch) in enumerate(((W, tx, dx, 0), (H, ty, dy, 1))):
        ok = (t - 1 >= 0) & (t + 1 < n)
        sel = np.nonzero(ok)[0]
        off = np.zeros(len(ys), F32)
        if len(sel):
            s_y, s_x, s_ty, s_tx = ys[sel], xs[sel], ty[sel], tx[sel]
            if axis == 0:
                cm = costs(d1, d2, s_y, s_x, s_ty, s_tx - 1)
                cp = costs(d1, d2, s_y, s_x, s_ty, s_tx + 1)
            else:
                cm = costs(d1, d2, s_y, s_x, s_ty - 1, s_tx)
                cp = costs(d1, d2, s_y, s_x, s_ty + 1, s_tx)
            off[sel] = axis_offset(cm, c0[sel], cp)
        out[ys, xs, ch] = (d.astype(F32) + off).astype(F32)
    return out
