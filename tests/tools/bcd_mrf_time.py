"""The reference programme (INT32_F32COST) against block coordinate descent on the MRF energy (INT32_F32COST | BCD_MRF)
on the bench workloads (BASELINE.json configs[1] and configs[2]): CUDA-event time of every column and row phase, the
energy (flowb200_energy, exact) before the first phase and after every phase, and the EPE of the checked forward field
(both directions, forward/backward check) against the synthetic ground truth.  One JSON line per configuration and
mode, after a line naming the card and its power limit.
   python tests/tools/bcd_mrf_time.py"""
import importlib, json, os, subprocess, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from oracle import epe as oepe
P = "lk-s-2022-estimacija-pokreta_b200"
ops, params, synth, lib = (importlib.import_module(f"{P}.{m}") for m in ("ops", "params", "synth", "_lib"))

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                      text=True).stdout.strip().splitlines()
print(json.dumps({"gpu": card[torch.cuda.current_device()] if card else None}))
CONFIGS = (("1024x436_K300_bcd4", 436, 1024, 300, 4), ("1242x375_K500_bcd8", 375, 1242, 500, 8))
MODES = (("reference", lib.BCD_INT32_F32COST), ("mrf", lib.BCD_INT32_F32COST | lib.BCD_MRF))


def ev():
    return torch.cuda.Event(enable_timing=True)


for name, H, W, K, sweeps in CONFIGS:
    p = params.for_k(K, H=H, W=W, knn_mode=1)
    img1, img2, gt, _ = synth.make_pair(H, W, 5)
    d = [ops.daisy(torch.from_numpy(img1).cuda()), ops.daisy(torch.from_numpy(img2).cuda())]
    sets = []
    for direction in (0, 1):
        pv, lc, npr, lab = ops.knn_proposals(d[direction], d[1 - direction], p)
        ops.random_proposals(d[direction], d[1 - direction], p, pv, lc, npr, lab, seed=1 + direction)
        sets.append((pv, lc, npr, lab))
    for mname, mode in MODES:
        kw = dict(mode=mode, lamda=p.lamda, tpsi=p.tpsi, cost_shift=p.cost_shift)
        pv, lc, npr, lab = sets[0]
        ws = ops.bcd_workspace(pv)
        for rep in range(3):   # the last repetition is reported
            l2 = lab.clone()
            torch.cuda.synchronize()
            e = [ev() for _ in range(2 + 4 * sweeps)]
            e[0].record()
            ops.bcd_prepare(pv, lc, npr, ws, 0, 1, **kw)
            e[1].record()
            for w in range(sweeps):
                for ph in range(4):
                    ops.bcd_phase(pv, lc, npr, l2, ws, ph, 0, 1, **kw)
                    e[2 + 4 * w + ph].record()
            torch.cuda.synchronize()
            t = [e[i].elapsed_time(e[i + 1]) for i in range(len(e) - 1)]
        ph = np.array(t[1:]).reshape(sweeps, 4)
        l3 = lab.clone()
        _, energies = ops.bcd(pv, lc, npr, l3, sweeps, energy_per_phase=True, **kw)
        assert torch.equal(l3, l2)
        flows = []
        for direction, (pv_, lc_, npr_, lab_) in enumerate(sets):
            ld = l2 if direction == 0 else lab_.clone()
            if direction:
                ops.bcd(pv_, lc_, npr_, ld, sweeps, **kw)
            flows.append(ops.flow_from_labels(pv_, ld, want_yx=False)[1])
        checked = ops.consistency(flows[0].clone(), flows[1], p.con_tresh).cpu().numpy()
        e_chk = oepe.error_image(checked, synth.gt_uvv(gt))
        e_raw = oepe.error_image(flows[0].cpu().numpy(), synth.gt_uvv(gt))
        rises = int(sum(b > a for a, b in zip(energies, energies[1:])))
        print(json.dumps({
            "config": name, "mode": mname, "sweeps": sweeps, "prepare_ms": round(t[0], 3),
            "col_phase_ms": round(float(ph[:, [0, 2]].mean()), 3), "row_phase_ms": round(float(ph[:, [1, 3]].mean()), 3),
            "chains_ms": round(float(ph.sum()), 3), "per_phase_ms": [[round(float(v), 3) for v in r] for r in ph],
            "energy_per_phase": energies, "energy_rises": rises,
            "epe_checked": round(e_chk[0], 4), "outliers_checked_pct": round(e_chk[1], 3), "n_valid_checked": e_chk[2],
            "epe_raw_forward": round(e_raw[0], 4)}))
