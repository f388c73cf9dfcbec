"""BCD stage on the bench workload, piece by piece: CUDA-event time of the K-set preparation (sort + build) and of
every phase launch (32-bit chain kernel + the fallback launch behind it, whose blocks return at once when no chain is
flagged), and a full-size regression check of the labels against the C oracle (oracle/flow_oracle.c) on costs quantised
to 20*m/2^S.  Then the time of the whole call with every chain forced through the fallback (FLOWB200_KSET_FORCE_GENERIC;
its labels must equal the unforced run's), and of the float64 programme.
   python tests/tools/bcd_phase_time.py [K] [sweeps] [H] [W]"""
import importlib, json, os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from oracle import cport
P = "lk-s-2022-estimacija-pokreta_b200"
ops, params, synth, lib, ioc = (importlib.import_module(f"{P}.{m}") for m in ("ops", "params", "synth", "_lib",
                                                                              "io_contract"))
K = int(sys.argv[1]) if len(sys.argv) > 1 else 300
sweeps = int(sys.argv[2]) if len(sys.argv) > 2 else 4
H = int(sys.argv[3]) if len(sys.argv) > 3 else 436
W = int(sys.argv[4]) if len(sys.argv) > 4 else 1024
p = params.for_k(K, H=H, W=W, knn_mode=1)
img1, img2, _, _ = synth.make_pair(H, W, 0)
d1, d2 = ops.daisy(torch.from_numpy(img1).cuda()), ops.daisy(torch.from_numpy(img2).cuda())
pv, lc, npr, lab = ops.knn_proposals(d1, d2, p)
ops.random_proposals(d1, d2, p, pv, lc, npr, lab, seed=1)
ws = ops.bcd_workspace(pv)
kw = dict(mode=lib.BCD_INT32_F32COST, cost_shift=p.cost_shift)


def ev():
    return torch.cuda.Event(enable_timing=True)


def bcd_ms(labels, **k):
    torch.cuda.synchronize()
    e0, e1 = ev(), ev()
    e0.record()
    ops.bcd(pv, lc, npr, labels, sweeps, **k)
    e1.record()
    torch.cuda.synchronize()
    return round(e0.elapsed_time(e1), 3)


res = {}
for rep in range(3):
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
    res = {"K": K, "H": H, "W": W, "sweeps": sweeps, "nprop_mean": float(npr.float().mean()),
           "prepare_ms": round(t[0], 3), "col_phase_ms": round(float(ph[:, [0, 2]].mean()), 3),
           "row_phase_ms": round(float(ph[:, [1, 3]].mean()), 3), "chains_ms": round(float(ph.sum()), 3),
           "total_ms": round(float(sum(t)), 3), "per_phase_ms": [[round(float(v), 3) for v in r] for r in ph]}
print(json.dumps(res))
whole = lab.clone()
ops.bcd(pv, lc, npr, whole, sweeps, **kw)
assert torch.equal(whole, l2), "flowb200_bcd differs from prepare + phases"
m = ops.quantise_costs(lc, p.lamda, p.cost_shift)
lq = torch.where(lc == 1000.0, torch.full_like(lc, 1000.0, dtype=torch.float64), m.double() * (20.0 / (1 << p.cost_shift)))
ref = cport.ceo_bcd(ioc.unpack_proposals(pv.cpu().numpy()), lq.cpu().numpy(), npr.cpu().numpy(), lab.cpu().numpy(),
                    sweeps, tpsi=p.tpsi, lamda=p.lamda)[-1]
ok = np.array_equal(ref, l2.cpu().numpy())
print("labels equal to the C oracle:", ok, "| moved", float((l2 != lab).float().mean()))
assert ok
# every chain through the int32 fallback (the variable is read at every phase call); the second run is reported
os.environ["FLOWB200_KSET_FORCE_GENERIC"] = "1"
for rep in range(2):
    forced = lab.clone()
    forced_ms = bcd_ms(forced, **kw)
del os.environ["FLOWB200_KSET_FORCE_GENERIC"]
assert torch.equal(forced, whole), "the forced fallback differs from the unforced run"
print(json.dumps({"forced_fallback_total_ms": forced_ms, "sweeps": sweeps, "labels_equal_unforced": True}))
# the float64 programme on the K-set records (what bcd.py runs on reference-written files)
f64 = lab.clone()
print(json.dumps({"fp64_ksets_total_ms": bcd_ms(f64, mode=lib.BCD_FP64_F32COST), "sweeps": sweeps}))
