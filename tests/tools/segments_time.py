"""Times removeSmallSegments (flowb200_remove_small_segments) on the checked forward field of the bench workload
(1024x436, K=300, 4 sweeps), on a synthetic island field and on noise, all through the one replay path; checks every
result against the C oracle.  Writes gpurun_out/segments_time.json.  (The oracle is used as the checker only.)"""
import importlib, json, os, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
P = "lk-s-2022-estimacija-pokreta_b200"
ops, params, synth, lib = (importlib.import_module(f"{P}.{m}") for m in ("ops", "params", "synth", "_lib"))
from oracle import cport
from helpers import segment_test_field

H, W = 436, 1024
p = params.for_k(300, H=H, W=W, knn_mode=1)
img1, img2, fwd, _ = synth.make_pair(H, W, 0)
checked = ops.flow_pair(torch.from_numpy(img1).cuda(), torch.from_numpy(img2).cuda(), p, 4, seed=1,
                        bcd_mode=lib.BCD_INT32_F32COST)
gt = torch.from_numpy(synth.gt_uvv(fwd)).cuda()
fields = {"bench_checked_forward": checked.cpu().numpy(),
          "synthetic_islands": segment_test_field(np.random.default_rng(5), H, W, "smooth"),
          "noise": segment_test_field(np.random.default_rng(6), H, W, "noise")}
out = {"H": H, "W": W, "tresh": 10, "min_segment_size": 100, "fields": {}}
for name, f in fields.items():
    t0 = time.perf_counter()
    want, nrem = cport.remove_small_segments(f, 10, 100, want_count=True)
    cpu_ms = (time.perf_counter() - t0) * 1e3
    rec = {"segments_removed": nrem, "valid_before": int(f[..., 2].sum()), "valid_after": int(want[..., 2].sum()),
           "oracle_cpu_ms_1_thread": round(cpu_ms, 3)}
    src = torch.from_numpy(f).cuda()
    ws = torch.empty(int(lib.load().flowb200_segments_workspace_bytes(H, W)), dtype=torch.uint8, device="cuda")
    ts = []
    for it in range(4):
        t = src.clone()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ops.remove_small_segments(t, 10, 100, workspace=ws)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    rec["gpu_ms"] = round(min(ts[1:]), 3)
    rec["equal_to_oracle"] = bool(np.array_equal(t.cpu().numpy(), want))
    if name == "bench_checked_forward":
        rec["epe_before"] = ops.epe(torch.from_numpy(f).cuda(), gt)[:2]
        rec["epe_after"] = ops.epe(torch.from_numpy(want).cuda(), gt)[:2]
    out["fields"][name] = rec
os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
with open(os.path.join(ROOT, "gpurun_out", "segments_time.json"), "w") as fh:
    json.dump(out, fh, indent=1)
print(json.dumps(out))
