"""Per-kernel GPU time of one direction's tensor-core proposal search (flowb200_knn_proposals, knn_mode 1) on the bench
frame (1024x436, K = 300) and on the same frame with its top third flat, from torch.profiler: operand preparation,
selection (knn_select_kernel), re-rank, fallback.  One warm-up call, then 5 profiled calls; each kernel's time is the
median over the calls.  The proposals are checked against the float64 search on each frame.  Prints one JSON line."""
import importlib, json, os, subprocess, sys
import torch
from torch.profiler import ProfilerActivity, profile
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
P = "lk-s-2022-estimacija-pokreta_b200"
ops, params, synth = (importlib.import_module(f"{P}.{m}") for m in ("ops", "params", "synth"))

KERNELS = ("knn_prep_query", "knn_prep_target", "knn_select", "knn_rerank", "knn_fallback", "labels_from_best")
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
    ref = ops.knn_proposals(d1, d2, p, want_idx=True, knn_mode=0)
    got = ops.knn_proposals(d1, d2, p, want_idx=True, knn_mode=1)
    same = all(torch.equal(x, y) for x, y in zip(got[:5], ref[:5]))
    del ref, got
    torch.cuda.synchronize()
    times = {k: [] for k in KERNELS}
    for it in range(5):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ops.knn_proposals(d1, d2, p, knn_mode=1)
            torch.cuda.synchronize()
        acc = dict.fromkeys(KERNELS, 0.0)
        for ev in prof.events():
            if ev.device_type == torch.autograd.DeviceType.CUDA:
                for k in KERNELS:
                    if k in ev.name:
                        acc[k] += ev.device_time / 1000.0
        for k in KERNELS:
            times[k].append(acc[k])
    rec = {f"{k}_ms": round(sorted(v)[len(v) // 2], 3) for k, v in times.items()}
    rec["tcgen05_equals_float64"] = same
    out["frames"][name] = rec
print(json.dumps(out))
