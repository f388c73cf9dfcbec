"""Times the proposal search (flowb200_knn_proposals, both search modes) on the bench frame and on the same frame with
its top third flat (1024x436, K = 300).  In a flat cell every query ties with all 1825 targets, so every such (query,
cell) task overflows the candidate list and is redone by brute force: the flat frame has over 2^20 of them, more than
the fallback list holds.  CUDA events, one warm-up call, best of 5.  The tensor-core result is checked against the
float64 search on each frame.  Prints one JSON line."""
import importlib, json, os, subprocess, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
P = "lk-s-2022-estimacija-pokreta_b200"
ops, params, synth = (importlib.import_module(f"{P}.{m}") for m in ("ops", "params", "synth"))

H, W = 436, 1024
p = params.for_k(300, H=H, W=W)
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
out = {"H": H, "W": W, "K": 300, "gpu": smi, "frames": {}}
for name in ("bench", "flat_top_third"):
    a, b, _, _ = synth.make_pair(H, W, 0)
    if name == "flat_top_third":
        a[:H // 3] = 128
        b[:H // 3] = 128
    d1, d2 = ops.daisy(torch.from_numpy(a).cuda()), ops.daisy(torch.from_numpy(b).cuda())
    rec = {}
    res = {}
    for mode in (1, 0):
        ts = []
        for it in range(6):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = ops.knn_proposals(d1, d2, p, want_idx=(it == 0), knn_mode=mode)
            e1.record()
            torch.cuda.synchronize()
            if it == 0:
                res[mode] = r
            else:
                ts.append(e0.elapsed_time(e1))
        rec[f"mode{mode}_ms_best"] = round(min(ts), 3)
        rec[f"mode{mode}_ms_median"] = round(sorted(ts)[len(ts) // 2], 3)
    rec["fallback_tasks"] = int(res[1][5][0])
    rec["tcgen05_equals_float64"] = all(torch.equal(x, y) for x, y in zip(res[1][:5], res[0][:5]))
    out["frames"][name] = rec
print(json.dumps(out))
