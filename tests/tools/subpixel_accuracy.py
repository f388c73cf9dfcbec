"""CPU-oracle EPE of integer against sub-pixel flow (DESIGN section 4.8) on synthetic pairs, no GPU.

For every pair: oracle DAISY of both frames, then per direction the exact search (cport.generisi), the random
proposals on replayed draws (cport.nasumicni, the draws of tests/test_gpu_baseline_configs.py) and 4 sweeps of the
float64 BCD (cport.ceo_bcd); the final labels give the integer field (oracle.consistency.ucitaj_flow of
vratiKonacniFlow) and the refined field (tests/subpixel_oracle.py).  Prints one JSON line: the EPE of the raw forward
field and of the checked forward field (con_tresh 10), both ways.

    python tests/tools/subpixel_accuracy.py [--pairs 5 6] [--size 436 1024] [--K 300] [--out file.json]
"""
import argparse
import importlib
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]
P = "lk-s-2022-estimacija-pokreta_b200"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, nargs="+", default=[5, 6])
    ap.add_argument("--size", type=int, nargs=2, default=[436, 1024], metavar=("H", "W"))
    ap.add_argument("--K", type=int, default=300)
    ap.add_argument("--sweeps", type=int, default=4)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from oracle import consistency as ocons, cport, daisy as od, epe as oepe, proposals as oprop
    import subpixel_oracle as so
    from test_gpu_baseline_configs import make_draws
    params, synth, ioc = (importlib.import_module(f"{P}.{m}") for m in ("params", "synth", "io_contract"))
    H, W = a.size
    p = params.for_k(a.K, H=H, W=W)
    op = oprop.Params(H, W, p.cellw, p.cellh, k_cell=p.k_cell, n_gauss=p.n_gauss, maxnprop=a.K)
    res = {"what": "CPU oracle, synthetic pairs (synth.make_pair), float64 BCD labels", "H": H, "W": W, "K": a.K,
           "sweeps": a.sweeps, "con_tresh": p.con_tresh, "host_threads": cport.num_threads(), "pairs": {}}
    for pair in a.pairs:
        t0 = time.time()
        img1, img2, gt_fwd, _ = synth.make_pair(H, W, pair)
        desc = [od.daisy(img1), od.daisy(img2)]
        flows = {}
        for d in (0, 1):
            s, t = desc[d], desc[1 - d]
            Pr, L, N, B = cport.generisi(s, t, op)
            Pr, L, N = cport.nasumicni(s, t, Pr, L, N, B, op, draws=make_draws(H, W, p.n_gauss, p.sigma, 77 + d))
            lab = cport.ceo_bcd(Pr, L, N, B, a.sweeps)[-1]
            pvec = ioc.pack_proposals(Pr)
            flows[d] = (ocons.ucitaj_flow(oprop.final_flow(Pr, lab)), so.subpixel(s, t, pvec, N, lab))
        gt = synth.gt_uvv(gt_fwd)
        r = {}
        for k, name in ((0, "integer"), (1, "subpixel")):
            raw = flows[0][k]
            checked = ocons.forward_backward_consistency(raw, flows[1][k], p.con_tresh)
            e_raw, e_chk = oepe.error_image(raw, gt), oepe.error_image(checked, gt)
            r[name] = {"raw_fwd_epe": round(e_raw[0], 4), "raw_fwd_outliers_pct": round(e_raw[1], 3),
                       "checked_epe": round(e_chk[0], 4), "checked_outliers_pct": round(e_chk[1], 3),
                       "checked_valid": e_chk[2]}
        fr = flows[0][1][..., :2] - flows[0][0][..., :2]
        r["refined_fraction_fwd"] = round(float((fr != 0).any(axis=-1).mean()), 4)
        r["seconds"] = round(time.time() - t0, 1)
        res["pairs"][str(pair)] = r
        print(f"pair {pair}: {json.dumps(r)}", file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
