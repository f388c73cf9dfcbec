"""Stage 2 drop-in: `bcd.py <pair> <backward> <bcd_times>` (reference python bcd.py:13-17, 67-81, 261-293).

Loads the stage-1 files (written by this repository's stage 1 or by the reference's), runs bcd_times sweeps
of chain Viterbi on the GPU, and writes flow + labels after every sweep under the reference's file names.
`packedksets.npy` is NOT read: it is a pure function of proposals/nprop (daisy i flann.py:256-309) and the
kernels evaluate the same predicate on the fly.
Arithmetic mode is chosen from the data so that labels equal the reference's float64 programme bit for bit:
  float32-representable costs -> FP64 mode on float32 costs; anything else -> FP64 mode on float64 costs;
  FLOWB200_BCD_INT32=1 requests the int32 mode and is honoured only if lamda*lcost*2^S is integral.
FLOWB200_BCD_MRF=1 runs block coordinate descent on the MRF energy (include/flowb200.h FLOWB200_BCD_MRF) in whichever
mode was chosen: the files written then differ from the reference's by design.
"""
import os
import sys

import numpy as np

from . import _lib
from . import io_contract as ioc


def run(picindex, backward, bcd_times, in_dir=".", out_dir=".", lamda=0.05, tpsi=8, cost_shift=12, log=print):
    import torch
    from . import ops
    picindex = ioc.pad2(picindex)
    backward = int(backward)
    bcd_times = int(bcd_times)
    ld = lambda name: np.load(os.path.join(in_dir, name))
    proposals = ld(ioc.stage1_file(picindex, backward, "proposals_nakon_gausa"))          # :73
    lcosts = ld(ioc.stage1_file(picindex, backward, "lcosts_nakon_gausa"))                # :74
    nprop = ld(ioc.stage1_file(picindex, backward, "nprop"))                              # :75
    labels = ld(ioc.labels_file(picindex, backward, 0))                                   # :78-81 (pastw = 0)
    H, W, K, _ = proposals.shape
    pvec = torch.from_numpy(ioc.pack_proposals(proposals)).cuda()
    g_nprop = torch.from_numpy(nprop.astype(np.int32)).cuda()
    g_lab = torch.from_numpy(labels.astype(np.int32)).cuda()
    mode, cost = _lib.BCD_FP64_F64COST, None
    if os.environ.get("FLOWB200_BCD_INT32") == "1":
        m = ioc.quantised_m(lcosts, lamda, cost_shift)
        if m is not None:
            mode, cost = _lib.BCD_INT32, torch.from_numpy(m).cuda()
    if cost is None:
        f32 = ioc.lcosts_to_f32(lcosts)
        if f32 is not None:
            mode, cost = _lib.BCD_FP64_F32COST, torch.from_numpy(f32).cuda()
        else:
            cost = torch.from_numpy(np.ascontiguousarray(lcosts, dtype=np.float64)).cuda()
    if os.environ.get("FLOWB200_BCD_MRF") == "1":
        mode |= _lib.BCD_MRF
    snaps = ops.bcd(pvec, cost, g_nprop, g_lab, bcd_times, mode=mode, lamda=lamda, tpsi=tpsi, cost_shift=cost_shift,
                    per_sweep=True)
    for w in range(1, bcd_times + 1):
        lab_w = snaps[w - 1].contiguous()
        flow, _ = ops.flow_from_labels(pvec, lab_w, want_uvv=False)
        np.save(os.path.join(out_dir, ioc.flow_file(picindex, backward, w)), flow.cpu().numpy())            # :282
        np.save(os.path.join(out_dir, ioc.labels_file(picindex, backward, w)),
                lab_w.cpu().numpy().astype(np.int64))                                                       # :283
        log("BCD", w)
    return 0


def main(argv=None):
    argv = sys.argv if argv is None else argv
    return run(argv[1], argv[2], int(argv[3]))
