"""Cost and effect of the sub-pixel refinement (flowb200_flow_subpixel, DESIGN section 4.8) on the device, in one call:

  kernel     CUDA-event time over many launches at 1024x436 (the search's proposals and the BCD's labels of four
             synthetic pairs, 4 x 243 MB of descriptors, cycled) and 3840x2160 (both directions of a synthetic pair, its
             ground-truth flow rounded as the vectors; 4.5 GB of descriptors), inputs several times the 126 MB L2;
             achieved bytes/s of the algorithmic 1656 B/pixel (source row 272 + five target rows 1360 + label, vector, nprop 12 + output 12);
  flow_pair  ms per pair at the bench configuration (1024x436, fwd+bwd, K = 300, INT32_F32COST, 4 sweeps) with
             flow_refine 0 and 1 alternating;
  EPE        of the raw forward and the checked field, integer and sub-pixel, on the synthetic pairs 5 and 6;
  card       name, power limit and maximum SM clock (nvidia-smi, read only).

The refined field of the first 1024x436 input set is compared with tests/subpixel_oracle.py bit for bit.  Prints one
JSON object; --out FILE also writes it there.

    python tests/tools/subpixel_time.py [--out FILE]
"""
import argparse
import dataclasses
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]
P = "lk-s-2022-estimacija-pokreta_b200"
ops, lib, params, synth = (importlib.import_module(f"{P}.{m}") for m in ("ops", "_lib", "params", "synth"))
import subpixel_oracle as so                     # noqa: E402
from oracle import epe as oepe                   # noqa: E402

BYTES_PER_PIXEL = 272 + 5 * 272 + 4 + 4 + 4 + 12


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def events_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def time_kernel(sets, H, W, K, reps=200):
    """sets: list of (desc_src, desc_tgt, pvec, nprop, labels, out) device tensors, used round robin."""
    L = lib.load()
    st = torch.cuda.current_stream().cuda_stream

    def launch(i):
        s = sets[i % len(sets)]
        rc = L.flowb200_flow_subpixel(*[ops._ptr(t) for t in s[:5]], H, W, K, ops._ptr(s[5]), ops.C.c_void_p(st))
        assert rc == 0
    for i in range(2 * len(sets)):
        launch(i)
    torch.cuda.synchronize()
    runs = [events_ms(launch, reps) for _ in range(3)]
    ms = min(runs)
    n = H * W
    distinct = {t.data_ptr(): t.numel() * t.element_size() for s in sets for t in s}
    return {"H": H, "W": W, "K": K, "input_sets": len(sets), "bytes_cycled": sum(distinct.values()),
            "ms_per_launch": round(ms, 4), "ms_runs": [round(r, 4) for r in runs],
            "algorithmic_bytes": n * BYTES_PER_PIXEL,
            "achieved_GBps": round(n * BYTES_PER_PIXEL / ms / 1e6, 1)}


def real_inputs_1024(p, pair, seed):
    img1, img2, fwd, _ = synth.make_pair(p.H, p.W, pair)
    d = [ops.daisy(dev(img1)), ops.daisy(dev(img2))]
    pvec, lcost, nprop, labels = ops.knn_proposals(d[0], d[1], p)
    ops.random_proposals(d[0], d[1], p, pvec, lcost, nprop, labels, seed=seed)
    ops.bcd(pvec, lcost, nprop, labels, 4, mode=lib.BCD_INT32_F32COST, cost_shift=p.cost_shift)
    del lcost
    return d[0], d[1], pvec, nprop, labels


def gt_inputs(H, W, pair):
    """Both directions of one synthetic pair, each with its ground-truth flow rounded as the only proposal (K = 1)."""
    img1, img2, fwd, bwd = synth.make_pair(H, W, pair)
    d = [ops.daisy(dev(img1)), ops.daisy(dev(img2))]
    sets = []
    for k, f in enumerate((fwd, bwd)):
        v = np.rint(f).astype(np.int64)
        sets.append((d[k], d[1 - k], dev(so.pack(v[..., 0], v[..., 1]).reshape(H, W, 1)),
                     dev(np.ones((H, W), np.int32)), dev(np.zeros((H, W), np.int32)),
                     torch.empty((H, W, 3), dtype=torch.float32, device="cuda")))
    return sets


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    out = {"card": card()}
    p = params.for_k(300, H=436, W=1024, knn_mode=1)
    # ---- kernel at 1024x436: four real input sets (4 x 243 MB of descriptors)
    sets, exact = [], True
    for i in range(4):
        s = real_inputs_1024(p, 5 + i, 10 * i)
        sets.append(s + (torch.empty((p.H, p.W, 3), dtype=torch.float32, device="cuda"),))
    got = ops.flow_subpixel(*sets[0][:5]).cpu().numpy()
    want = so.subpixel(*(t.cpu().numpy() for t in sets[0][:5]))
    exact &= bool(np.array_equal(got.view(np.uint32), want.view(np.uint32)))
    out["kernel_1024x436"] = time_kernel(sets, p.H, p.W, p.maxnprop)
    del sets
    torch.cuda.empty_cache()
    # ---- kernel at 3840x2160: both directions of one pair, vectors = rounded ground truth, K = 1
    H4, W4 = 2160, 3840
    sets = gt_inputs(H4, W4, 5)
    out["kernel_3840x2160"] = time_kernel(sets, H4, W4, 1, reps=50)
    del sets
    torch.cuda.empty_cache()
    out["kernel_equal_to_oracle_1024x436"] = exact
    # ---- flow_pair at the bench configuration, option off and on alternating
    img1, img2, _, _ = synth.make_pair(p.H, p.W, 0)
    g0, g1 = dev(img1), dev(img2)
    ws = ops.pair_workspace(p, "cuda", bcd_mode=lib.BCD_INT32_F32COST)
    cfg = {r: dataclasses.replace(p, flow_refine=r) for r in (0, 1)}

    def pair(r):
        return ops.flow_pair(g0, g1, cfg[r], sweeps=4, directions=2, seed=0, bcd_mode=lib.BCD_INT32_F32COST,
                             workspace=ws)
    for r in (0, 1, 0, 1):
        pair(r)
    torch.cuda.synchronize()
    ms = {0: [], 1: []}
    for rnd in range(4):
        for r in ((0, 1) if rnd % 2 == 0 else (1, 0)):
            ms[r].append(round(events_ms(lambda i: pair(r), 10), 3))
    out["flow_pair_ms"] = {"config": "1024x436 fwd+bwd K=300 INT32_F32COST 4 sweeps, 10 pairs per sample",
                           "flow_refine_0": ms[0], "flow_refine_1": ms[1],
                           "median_0": float(np.median(ms[0])), "median_1": float(np.median(ms[1]))}
    # ---- EPE both ways on the synthetic pairs of the CPU accuracy check
    out["epe"] = {}
    for pr in (5, 6):
        a, b, fwd, _ = synth.make_pair(p.H, p.W, pr)
        gt = synth.gt_uvv(fwd)
        e = {}
        for r in (0, 1):
            chk, raw, _ = ops.flow_pair(dev(a), dev(b), cfg[r], sweeps=4, directions=2, seed=0,
                                        bcd_mode=lib.BCD_INT32_F32COST, want_raw=True)
            er, ec = oepe.error_image(raw.cpu().numpy(), gt), oepe.error_image(chk.cpu().numpy(), gt)
            e["subpixel" if r else "integer"] = {"raw_fwd_epe": round(er[0], 4), "checked_epe": round(ec[0], 4),
                                                 "checked_outliers_pct": round(ec[1], 3), "checked_valid": ec[2]}
        out["epe"][str(pr)] = e
    out["card_after"] = card()
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(out, fh, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
