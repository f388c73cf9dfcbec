"""Device-level operators of the flow hot path: torch CUDA tensors in, torch CUDA tensors out.

Every function enqueues hand-written sm_100a kernels from libflowb200.so on torch's current stream
through the C ABI (include/flowb200.h).  torch only owns the memory.  Device layouts:

  desc    float32 (H, W, 68)        DAISY descriptors                         (daisy i flann.py:69-77)
  pvec    int32   (H, W, K)         proposal vectors, (int16 dy) | (int16 dx) << 16; unused = -1
  lcost   float32 (H, W, K)         data costs, unused = 1000                 (daisy i flann.py:90)
  nprop   int32   (H, W)
  labels  int32   (H, W)            bestlabels
  uvv     float32 (H, W, 3)         (dx, dy, valid)                           (postprocessing.py:7-17)
"""
import ctypes as C
import math

import torch

from . import _lib
from .params import FlowParams


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t, dtype=None, name="tensor"):
    if t is None:
        return C.c_void_p(0)
    if not t.is_cuda:
        raise _lib.FlowB200Error(f"{name} must be a CUDA tensor (no CPU fallback)")
    if dtype is not None and t.dtype != dtype:
        raise TypeError(f"{name}: expected {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    return C.c_void_p(t.data_ptr())


def cparams(p: FlowParams, bcd_mode=_lib.BCD_FP64_F32COST, knn_mode=None):
    p.validate()
    if knn_mode is None:
        knn_mode = p.knn_mode
    return _lib.CParams(H=p.H, W=p.W, cellw=p.cellw, cellh=p.cellh, cell_radius=p.cell_radius, k_cell=p.k_cell,
                        n_gauss=p.n_gauss, sigma=p.sigma, maxnprop=p.maxnprop, tphi=p.tphi, tpsi=p.tpsi,
                        lamda=p.lamda, cost_shift=p.cost_shift, bcd_mode=bcd_mode, knn_mode=knn_mode,
                        con_tresh=p.con_tresh, cell_x0=p.cell_x0, cell_x1=p.cell_x1, flow_refine=p.flow_refine)


def _workspace(nbytes, device):
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


def daisy(bgr):
    """uint8 (H,W,3) BGR -> float32 (H,W,68).  izracunajDaisy, daisy i flann.py:69-77."""
    lib = _lib.load()
    H, W, ch = bgr.shape
    assert ch == 3
    desc = torch.empty((H, W, 68), dtype=torch.float32, device=bgr.device)
    nb = lib.flowb200_daisy_workspace_bytes(H, W)
    ws = _workspace(nb, bgr.device)
    _lib.check(lib.flowb200_daisy(_ptr(bgr, torch.uint8, "bgr"), H, W, _ptr(desc), _ptr(ws), ws.numel(), _stream()),
               "flowb200_daisy")
    return desc


def knn_proposals(desc_src, desc_tgt, p: FlowParams, want_idx=False, knn_mode=None):
    """napraviCD2 + generisi (daisy i flann.py:144-148, 157-189) with an exact search.

    Returns (pvec, lcost, nprop, labels[, knn_idx, stats])."""
    lib = _lib.load()
    cp = cparams(p, knn_mode=knn_mode)
    dev = desc_src.device
    H, W, K = p.H, p.W, p.maxnprop
    assert tuple(desc_src.shape) == (H, W, 68) and tuple(desc_tgt.shape) == (H, W, 68)
    pvec = torch.empty((H, W, K), dtype=torch.int32, device=dev)
    lcost = torch.empty((H, W, K), dtype=torch.float32, device=dev)
    nprop = torch.empty((H, W), dtype=torch.int32, device=dev)
    labels = torch.empty((H, W), dtype=torch.int32, device=dev)
    r = 2 * p.cell_radius + 1
    idx = torch.empty((H, W, r * r, p.k_cell), dtype=torch.int32, device=dev) if want_idx else None
    stats = torch.zeros(8, dtype=torch.int32, device=dev) if want_idx else None
    nb = lib.flowb200_knn_workspace_bytes(C.byref(cp))
    ws = _workspace(nb, dev)
    rc = lib.flowb200_knn_proposals(_ptr(desc_src, torch.float32, "desc_src"), _ptr(desc_tgt, torch.float32, "desc_tgt"),
                                    C.byref(cp), _ptr(pvec), _ptr(lcost), _ptr(nprop), _ptr(labels), _ptr(idx),
                                    _ptr(stats), _ptr(ws), ws.numel(), _stream())
    _lib.check(rc, "flowb200_knn_proposals")
    if want_idx:
        return pvec, lcost, nprop, labels, idx, stats
    return pvec, lcost, nprop, labels


def random_proposals(desc_src, desc_tgt, p: FlowParams, pvec, lcost, nprop, labels, draws=None, seed=0):
    """nasumicni (daisy i flann.py:205-233), in place on pvec/lcost/nprop.

    draws: optional int16 (H,W,n_gauss,2) accepted (tgy,tgx) samples to replay; None -> Philox."""
    lib = _lib.load()
    cp = cparams(p)
    rc = lib.flowb200_random_proposals(_ptr(desc_src, torch.float32), _ptr(desc_tgt, torch.float32), C.byref(cp),
                                       _ptr(pvec, torch.int32), _ptr(lcost, torch.float32), _ptr(nprop, torch.int32),
                                       _ptr(labels, torch.int32), _ptr(draws, torch.int16, "draws"),
                                       C.c_uint64(int(seed)), _stream())
    _lib.check(rc, "flowb200_random_proposals")


def ksets_pack(pvec, nprop, tpsi=8):
    """pakovanje (daisy i flann.py:256-309): uint8 (H,W,2,K*K//8+1).  Legacy export, small sizes only."""
    lib = _lib.load()
    H, W, K = pvec.shape
    out = torch.empty((H, W, 2, K * K // 8 + 1), dtype=torch.uint8, device=pvec.device)
    _lib.check(lib.flowb200_ksets_pack(_ptr(pvec, torch.int32), _ptr(nprop, torch.int32), H, W, K, int(tpsi),
                                       _ptr(out), _stream()), "flowb200_ksets_pack")
    return out


def quantise_costs(lcost, lamda=0.05, shift=12):
    lib = _lib.load()
    m = torch.empty(lcost.shape, dtype=torch.int32, device=lcost.device)
    _lib.check(lib.flowb200_quantise_costs(_ptr(lcost, torch.float32), _ptr(m), lcost.numel(), float(lamda), int(shift),
                                           _stream()), "flowb200_quantise_costs")
    return m


_BCD_COST_DTYPE = {_lib.BCD_FP64_F32COST: torch.float32, _lib.BCD_FP64_F64COST: torch.float64,
                   _lib.BCD_INT32: torch.int32, _lib.BCD_INT32_F32COST: torch.float32}


def _cost_dtype(mode):
    """dtype of the cost array of a BCD mode (the BCD_MRF flag does not change it)"""
    return _BCD_COST_DTYPE[mode & ~_lib.BCD_MRF]


def _bcd_args(pvec, cost, nprop, mode, lamda, tpsi, cost_shift, *labels):
    """The arguments the BCD entry points begin with: pvec, cost, nprop[, labels], H, W, K, mode, lamda, tpsi,
    cost_shift (flowb200_bcd_prepare takes no labels)."""
    H, W, K = pvec.shape
    ptrs = [_ptr(pvec, torch.int32, "pvec"), _ptr(cost, _cost_dtype(mode), "cost"), _ptr(nprop, torch.int32, "nprop")]
    ptrs += [_ptr(t, torch.int32, "labels") for t in labels]
    return (*ptrs, H, W, K, int(mode), float(lamda), int(tpsi), int(cost_shift))


def energy(pvec, cost, nprop, labels, mode=_lib.BCD_FP64_F32COST, lamda=0.05, tpsi=8, cost_shift=12):
    """The MRF energy of labels in the arithmetic of `mode` (flowb200_energy): (data, pairwise, total, n_bad), n_bad =
    pixels whose label is outside [0, nprop), left out of both terms.  Exact in the int32 modes."""
    lib = _lib.load()
    out = torch.empty(4, dtype=torch.float64, device=pvec.device)
    _lib.check(lib.flowb200_energy(*_bcd_args(pvec, cost, nprop, mode, lamda, tpsi, cost_shift, labels), _ptr(out),
                                   _stream()), "flowb200_energy")
    data, pair, total, bad = out.tolist()
    return data, pair, total, int(bad)


def bcd(pvec, cost, nprop, labels, sweeps, mode=_lib.BCD_FP64_F32COST, lamda=0.05, tpsi=8, cost_shift=12,
        per_sweep=False, workspace_bytes=None, energy_per_phase=False):
    """ceoBCD (python bcd.py:261-284): `sweeps` sweeps in place on labels.

    Returns int32 (sweeps,H,W) snapshots after every sweep when per_sweep, else None.
    energy_per_phase (int32 modes, which bcd_prepare / bcd_phase run): returns (snapshots, energies) instead, with
    energies the total energy (`energy`) before the first phase and after every phase, 1 + 4 * sweeps floats."""
    lib = _lib.load()
    H, W, K = pvec.shape
    snaps = torch.empty((sweeps, H, W), dtype=torch.int32, device=pvec.device) if per_sweep else None
    nb = lib.flowb200_bcd_workspace_bytes(H, W, K) if workspace_bytes is None else int(workspace_bytes)
    ws = _workspace(nb, pvec.device)[:nb]
    if energy_per_phase:
        if (mode & ~_lib.BCD_MRF) not in (_lib.BCD_INT32, _lib.BCD_INT32_F32COST):
            raise ValueError("energy_per_phase: int32 modes only (bcd_prepare / bcd_phase)")
        kw = dict(mode=mode, lamda=lamda, tpsi=tpsi, cost_shift=cost_shift)
        bcd_prepare(pvec, cost, nprop, ws, 0, 1, **kw)
        energies = [energy(pvec, cost, nprop, labels, **kw)[2]]
        for w in range(sweeps):
            for phase in range(4):
                bcd_phase(pvec, cost, nprop, labels, ws, phase, 0, 1, **kw)
                energies.append(energy(pvec, cost, nprop, labels, **kw)[2])
            if per_sweep:
                snaps[w].copy_(labels)
        return snaps, energies
    _lib.check(lib.flowb200_bcd(*_bcd_args(pvec, cost, nprop, mode, lamda, tpsi, cost_shift, labels), int(sweeps),
                                _ptr(snaps), _ptr(ws), ws.numel(), _stream()), "flowb200_bcd")
    return snaps


def bcd_workspace(pvec, nparts=1):
    """Workspace for flowb200_bcd / flowb200_bcd_prepare.  A part of `nparts` stores only the records of its own chains,
    so its record arena is the recommended size divided by nparts (plus slack); whatever does not fit is evaluated on
    the fly (any size between the minimum and the recommended one gives the same labels)."""
    lib = _lib.load()
    H, W, K = pvec.shape
    full = lib.flowb200_bcd_workspace_bytes(H, W, K)
    if nparts > 1:
        lo = lib.flowb200_bcd_min_workspace_bytes(H, W, K)
        full = min(full, lo + int((full - lo) * 1.3 / nparts) + (1 << 20))
    return _workspace(full, pvec.device)


def bcd_prepare(pvec, cost, nprop, ws, part=0, nparts=1, mode=_lib.BCD_INT32_F32COST, lamda=0.05, tpsi=8, cost_shift=12):
    """Compile the K-sets of the chains part `part` of `nparts` owns into the workspace `ws` (int32 modes)."""
    lib = _lib.load()
    _lib.check(lib.flowb200_bcd_prepare(*_bcd_args(pvec, cost, nprop, mode, lamda, tpsi, cost_shift), int(part),
                                        int(nparts), _ptr(ws), ws.numel(), _stream()), "flowb200_bcd_prepare")


def bcd_phase(pvec, cost, nprop, labels, ws, phase, part=0, nparts=1, mode=_lib.BCD_INT32_F32COST, lamda=0.05, tpsi=8,
              cost_shift=12):
    """Run the owned chains of one phase in place on labels (after bcd_prepare with the same workspace and part)."""
    lib = _lib.load()
    _lib.check(lib.flowb200_bcd_phase(*_bcd_args(pvec, cost, nprop, mode, lamda, tpsi, cost_shift, labels), int(phase),
                                      int(part), int(nparts), _ptr(ws), ws.numel(), _stream()), "flowb200_bcd_phase")


def best_labels(lcost, nprop):
    """bestlabels of generisi (daisy i flann.py:181-184) from the data costs: int32 (H,W)."""
    lib = _lib.load()
    H, W, K = lcost.shape
    labels = torch.empty((H, W), dtype=torch.int32, device=lcost.device)
    _lib.check(lib.flowb200_best_labels(_ptr(lcost, torch.float32, "lcost"), _ptr(nprop, torch.int32, "nprop"), H, W, K,
                                        _ptr(labels), _stream()), "flowb200_best_labels")
    return labels


def slot_copy(table, vec, cost, flat, to_flat):
    """flowb200_slot_copy: the slot ranges listed in `table` (int64 (n, 8), see include/flowb200.h) between the proposal
    arrays vec int32 / cost float32 (rows, width, K) and the flat int32 buffer; to_flat packs, otherwise unpacks."""
    lib = _lib.load()
    _, width, K = vec.shape
    assert cost.shape == vec.shape and table.dim() == 2 and table.shape[1] == 8
    _lib.check(lib.flowb200_slot_copy(_ptr(table, torch.int64, "table"), int(table.shape[0]), _ptr(vec, torch.int32, "vec"),
                                      _ptr(cost, torch.float32, "cost"), width, K, _ptr(flat, torch.int32, "flat"),
                                      1 if to_flat else 0, _stream()), "flowb200_slot_copy")


def flow_from_labels(pvec, labels, want_yx=True, want_uvv=True):
    """vratiKonacniFlow (+ FlowImage layout).  Returns (flow_yx float64 (H,W,2) | None, uvv float32 (H,W,3) | None)."""
    lib = _lib.load()
    H, W, K = pvec.shape
    yx = torch.empty((H, W, 2), dtype=torch.float64, device=pvec.device) if want_yx else None
    uvv = torch.empty((H, W, 3), dtype=torch.float32, device=pvec.device) if want_uvv else None
    _lib.check(lib.flowb200_flow_from_labels(_ptr(pvec, torch.int32), _ptr(labels, torch.int32), H, W, K, _ptr(yx),
                                             _ptr(uvv), _stream()), "flowb200_flow_from_labels")
    return yx, uvv


def flow_subpixel(desc_src, desc_tgt, pvec, nprop, labels):
    """flow_from_labels with every vector refined per axis to the vertex of the parabola through the data costs of the
    target and its two neighbours (DESIGN section 4.8).  Returns uvv float32 (H,W,3) = (dx + ox, dy + oy, 1)."""
    lib = _lib.load()
    H, W, K = pvec.shape
    assert tuple(desc_src.shape) == (H, W, 68) and tuple(desc_tgt.shape) == (H, W, 68)
    assert tuple(nprop.shape) == (H, W) and tuple(labels.shape) == (H, W)
    uvv = torch.empty((H, W, 3), dtype=torch.float32, device=pvec.device)
    _lib.check(lib.flowb200_flow_subpixel(_ptr(desc_src, torch.float32, "desc_src"),
                                          _ptr(desc_tgt, torch.float32, "desc_tgt"), _ptr(pvec, torch.int32, "pvec"),
                                          _ptr(nprop, torch.int32, "nprop"), _ptr(labels, torch.int32, "labels"), H, W,
                                          K, _ptr(uvv), _stream()), "flowb200_flow_subpixel")
    return uvv


def consistency(flow1, flow2, tresh, region=None):
    """fowardBackwardConsistency (postprocessing.py:114-117), in place on flow1 (float32 (A,B,3))."""
    lib = _lib.load()
    A, B, ch = flow1.shape
    assert ch == 3 and tuple(flow2.shape) == (A, B, 3)
    a0, a1, b0, b1 = region if region is not None else (0, A, 0, B)
    _lib.check(lib.flowb200_consistency(_ptr(flow1, torch.float32, "flow1"), _ptr(flow2, torch.float32, "flow2"), A, B,
                                        float(tresh), a0, a1, b0, b1, _stream()), "flowb200_consistency")
    return flow1


def remove_small_segments(flow, tresh, min_segment_size, workspace=None):
    """removeSmallSegments (postprocessing.py:29-76), in place on flow (float32 (A,B,3) device tensor)."""
    lib = _lib.load()
    A, B, ch = flow.shape
    assert ch == 3
    need = int(lib.flowb200_segments_workspace_bytes(A, B))
    if workspace is None:
        workspace = torch.empty(need, dtype=torch.uint8, device=flow.device)
    _lib.check(lib.flowb200_remove_small_segments(_ptr(flow, torch.float32, "flow"), A, B, float(tresh),
                                                  int(min_segment_size), _ptr(workspace), workspace.numel(),
                                                  _stream()), "flowb200_remove_small_segments")
    return flow


def canny_edges(bgr, low=100, high=200, workspace=None):
    """edge.canny_ivice (edge.py:19-35) without the file I/O: uint8 (H,W,3) device tensor -> float32 (H,W),
    0.0 on an edge, 1.0 elsewhere.  `low` and `high` are floored like cv2.Canny's thresholds and may come in either
    order (the smaller one is the low threshold)."""
    lib = _lib.load()
    H, W, ch = bgr.shape
    assert ch == 3
    out = torch.empty((H, W), dtype=torch.float32, device=bgr.device)
    if workspace is None:
        workspace = torch.empty(int(lib.flowb200_edges_workspace_bytes(H, W)), dtype=torch.uint8, device=bgr.device)
    _lib.check(lib.flowb200_canny_edges(_ptr(bgr, torch.uint8, "bgr"), H, W, math.floor(low), math.floor(high),
                                        _ptr(out), _ptr(workspace), workspace.numel(), _stream()),
               "flowb200_canny_edges")
    return out


def epe(test_uvv, gt_uvv, abs_thresh=3.0):
    """visualization.errorImage (visualization.py:128-152): (mean EPE, outlier %, n_valid) over pixels valid in both."""
    lib = _lib.load()
    H, W, _ = test_uvv.shape
    out = torch.empty(3, dtype=torch.float64, device=test_uvv.device)
    _lib.check(lib.flowb200_epe(_ptr(test_uvv, torch.float32), _ptr(gt_uvv, torch.float32), H, W, float(abs_thresh),
                                _ptr(out), _stream()), "flowb200_epe")
    s, no, nv = out.tolist()
    if nv == 0:
        return float("nan"), float("nan"), 0
    return s / nv, 100.0 * no / nv, int(nv)


def flow_pair(bgr0, bgr1, p: FlowParams, sweeps, directions=2, seed=0, bcd_mode=_lib.BCD_FP64_F32COST,
              want_raw=False, workspace=None):
    """Whole device-resident path.  Returns checked forward field float32 (H,W,3) (and raw fwd/bwd fields)."""
    lib = _lib.load()
    cp = cparams(p, bcd_mode=bcd_mode)
    dev = bgr0.device
    out = torch.empty((p.H, p.W, 3), dtype=torch.float32, device=dev)
    raw_f = torch.empty_like(out) if want_raw else None
    raw_b = torch.empty_like(out) if want_raw and directions == 2 else None
    if workspace is None:
        workspace = _workspace(lib.flowb200_pair_workspace_bytes(C.byref(cp)), dev)
    rc = lib.flowb200_flow_pair(_ptr(bgr0, torch.uint8, "bgr0"), _ptr(bgr1, torch.uint8, "bgr1"), C.byref(cp),
                                int(sweeps), int(directions), C.c_uint64(int(seed)), _ptr(out), _ptr(raw_f),
                                _ptr(raw_b), _ptr(workspace), workspace.numel(), _stream())
    _lib.check(rc, "flowb200_flow_pair")
    if want_raw:
        return out, raw_f, raw_b
    return out


def pair_workspace(p: FlowParams, device, bcd_mode=_lib.BCD_FP64_F32COST):
    lib = _lib.load()
    cp = cparams(p, bcd_mode=bcd_mode)
    return _workspace(lib.flowb200_pair_workspace_bytes(C.byref(cp)), device)


def knn_debug_scores(desc_src, desc_tgt, p: FlowParams):
    """Diagnostics of the tcgen05 prefilter: (scores float32 [n_items][tile_w*tile_h][Tpad], geom dict).

    item = tile * n_cells + cell (cell-minor work order); a work item is tile_w x tile_h query pixels stored as
    tile_w/16 consecutive 16 x tile_h MMA tiles of 128 rows each (row = 16-wide x index + 16 * y)."""
    import numpy as np
    lib = _lib.load()
    cp = cparams(p, knn_mode=_lib.KNN_TCGEN05)
    geom = np.zeros(8, dtype=np.int32)
    _lib.check(lib.flowb200_knn_debug_scores(_ptr(desc_src, torch.float32), _ptr(desc_tgt, torch.float32), C.byref(cp),
                                             C.c_void_p(0), C.c_void_p(geom.ctypes.data), C.c_void_p(0), 0, _stream()),
               "flowb200_knn_debug_scores(geom)")
    names = ("Tpad", "stride_s", "tiles_x", "tiles_y", "n_items", "tile_w", "tile_h", "max_cand")
    g = {k: int(v) for k, v in zip(names, geom)}
    scores = torch.full((g["n_items"], g["tile_w"] * g["tile_h"], g["Tpad"]), float("nan"), dtype=torch.float32,
                        device=desc_src.device)
    ws = _workspace(lib.flowb200_knn_workspace_bytes(C.byref(cp)), desc_src.device)
    _lib.check(lib.flowb200_knn_debug_scores(_ptr(desc_src, torch.float32), _ptr(desc_tgt, torch.float32), C.byref(cp),
                                             _ptr(scores), C.c_void_p(geom.ctypes.data), _ptr(ws), ws.numel(), _stream()),
               "flowb200_knn_debug_scores")
    return scores, g
