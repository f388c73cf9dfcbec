#!/usr/bin/env python
"""Benchmark of the flow hot path (BASELINE.json metric: flow Mpix/s & pairs/s, DAISY+kNN+BCD+consistency).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl flowb200|reference] [--workload NAME]
                  [--dump-outputs DIR]

One step = one synthetic image pair through the whole path: 2 x DAISY, per direction exact per-cell kNN
proposals + random-neighbour proposals + `sweeps` BCD sweeps, then the forward/backward check.
Workload (default) = BASELINE.json configs[1]: 1024x436, forward+backward+consistencyCheck(10), K=300,
bcd_times=4.  With N GPUs every rank processes its own pair per step (pairs are independent, README.md:40):
weak scaling, no data-path collective; value = N pairs / max-over-ranks time.

value  : device-resident (images already in HBM), CUDA events, max over ranks.
e2e    : the same through the host-buffer C ABI (flowb200_ctx_flow_pair_host): pinned H2D of both images,
         D2H of the checked field, inside the timed region.
roofline: the dominant KERNEL (kset_chain32_kernel, one launch per BCD phase): algorithmic bytes per launch (DESIGN.md)
         / its own CUDA-event duration measured here phase by phase; the stage times and fractions are beside it.
cpu_baseline: the CPU oracle (oracle/, C + numpy, all host threads) on a bounded crop of the same workload.
huge   : (unless --no-huge) a short run of the single-huge-image mode (configs[4], 3840x2160, huge.py) on the same
         ranks: ms per pair, and whether the sharded result is bit-identical to one GPU's.
--workload 99pairs_...: configs[3] as written: 99 distinct host-resident pairs dealt round robin over the ranks
         (dist.shard_units), each rank's share through flowb200_ctx_flow_pairs_host (copies overlapped).
--impl reference: the CPU oracle alone, same metric/config (the reference itself is pure Python that
         needs opencv-contrib + pyflann, absent offline; its unmodified source runs only on tiny crops).
--dump-outputs DIR: the outputs of the last timed step as .npy files (dump_outputs); the inputs are seeded, so two
         builds run with the same arguments can be compared output for output.  With N ranks each rank writes its own
         files (suffix _rank<r>), except in the huge mode, where every rank holds the same field.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries exactly one JSON line.  Libraries write there too (NCCL prints "NCCL version ..." on stdout when
# the environment sets NCCL_DEBUG=VERSION, as the GPU boxes do): file descriptor 1 is pointed at stderr for the whole
# run and the JSON line goes to a duplicate of the original stdout.
_JSON_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(line):
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()
PKG = "lk-s-2022-estimacija-pokreta_b200"

WORKLOADS = {
    # name: (H, W, K, sweeps, directions)
    "1024x436_fwd_K150_bcd4": (436, 1024, 150, 4, 1),            # configs[0]
    "1024x436_fwdbwd_K300_bcd4": (436, 1024, 300, 4, 2),         # configs[1]  (metric is quoted on this)
    "1242x375_fwdbwd_K500_bcd8": (375, 1242, 500, 8, 2),         # configs[2]
    # configs[4]: ONE pair on all ranks, target cells sharded, NCCL merge (huge.py); strong scaling
    "3840x2160_huge_K150_bcd4": (2160, 3840, 150, 4, 2),
    "1920x1080_huge_K150_bcd4": (1080, 1920, 150, 4, 2),
    # configs[3]: 99 pairs x 2 directions dealt over the ranks, host buffers in, host fields out
    "99pairs_1024x436_fwdbwd_K300_bcd4": (436, 1024, 300, 4, 2),
}
HUGE_IN_BENCH = "3840x2160_huge_K150_bcd4"
DEFAULT_WORKLOAD = "1024x436_fwdbwd_K300_bcd4"
METRIC = "flow Mpix/s (DAISY+kNN+BCD+consistency)"


def mod(name):
    return importlib.import_module(PKG + "." + name)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm": d["hbm_gbs"], "tensor_burst": d["bf16_tflops"], "tensor": d["bf16_tflops_sustained"],
                "src": "measured"}
    return {"hbm": 6650.0, "tensor_burst": 1590.0, "tensor": 1400.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(len(r) >= 7 and r[3 + j].lower() == "active" for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


DUMP_BYTES = 64_000_000          # all files of one --dump-outputs run together
NPY_HEADER_BYTES = 4096          # upper bound of an .npy header (numpy pads it to a multiple of 64 bytes)


def dump_outputs(dirname, arrays, suffix="", budget=DUMP_BYTES):
    """Writes every array of `arrays` (name -> what a caller of the timed path received in its last step) as
    <dirname>/<name><suffix>.npy, float64 kept and anything else as float32; the files, headers included, take at
    most `budget` bytes.  When the arrays do not fit, every array is cut down to the same fixed, seeded sample of its
    pixels (rows over its last axis), and <name>_index<suffix>.npy holds the flat indices of the pixels kept, so that
    two builds can be compared element for element on identical inputs."""
    os.makedirs(dirname, exist_ok=True)
    arrays = {k: np.asarray(v.cpu() if hasattr(v, "cpu") else v) for k, v in arrays.items()}
    arrays = {k: v if v.dtype == np.float64 else v.astype(np.float32) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    sample = total + NPY_HEADER_BYTES * len(arrays) > budget
    payload = budget - 2 * NPY_HEADER_BYTES * len(arrays)        # a data and an index file per array
    for name, a in arrays.items():
        if sample:
            rows = a.reshape(-1, a.shape[-1])
            row_bytes = rows.shape[1] * rows.itemsize + 8          # the pixel and its float64 index
            k = max(1, int(payload * a.nbytes / total) // row_bytes)
            idx = np.sort(np.random.default_rng(0).choice(rows.shape[0], size=min(k, rows.shape[0]), replace=False))
            # float64 because every dump file is float32 or float64; flat indices are exact in it below 2^53
            np.save(os.path.join(dirname, f"{name}_index{suffix}.npy"), idx.astype(np.float64))
            a = rows[idx]
        np.save(os.path.join(dirname, f"{name}{suffix}.npy"), a)


def make_params(workload, knn_mode):
    H, W, K, sweeps, directions = WORKLOADS[workload]
    P = mod("params")
    p = P.for_k(K, H=H, W=W, knn_mode=knn_mode)
    return p, sweeps, directions


def algorithmic_work(p, sweeps, directions):
    """Per-step algorithmic bytes / FLOPs of every stage (DESIGN.md 'Measurement', SURVEY.md section 8d)."""
    N = p.H * p.W
    T = p.cellw * p.cellh
    R = p.cell_radius
    q = 0
    for ci in range(p.ncellx):
        bw = min(p.W, p.cellw * (ci + R + 1)) - max(0, p.cellw * (ci - R))
        for cj in range(p.ncelly):
            bh = min(p.H, p.cellh * (cj + R + 1)) - max(0, p.cellh * (cj - R))
            q += bw * bh
    K = p.maxnprop
    return {
        "daisy": ("hbm", 2 * N * (3 + 68 * 4)),
        "knn": ("tensor", directions * 2 * 68 * q * T),
        "random": ("hbm", directions * N * (2 * 272 + p.n_gauss * 16)),
        "bcd": ("hbm", directions * sweeps * 2 * N * (K * 8 + 12)),
        "consistency": ("hbm", (directions - 1) * N * 28 + directions * N * 16),
    }


def stage_breakdown(ops, lib, p, sweeps, directions, g0, g1, bcd_mode, reps=2):
    """CUDA-event time of every stage, the same C-ABI calls flowb200_flow_pair makes, on torch's stream."""
    import torch
    acc = {k: 0.0 for k in ("daisy", "knn", "random", "bcd", "consistency")}

    def timed(key, fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        r = fn()
        b.record()
        b.synchronize()
        acc[key] += a.elapsed_time(b)
        return r
    for rep in range(reps + 1):
        if rep == 1:
            acc = {k: 0.0 for k in acc}          # first pass is warm-up
        d = timed("daisy", lambda: (ops.daisy(g0), ops.daisy(g1)))
        uv = []
        for di in range(directions):
            src, tgt = d[di], d[1 - di]
            pv, lc, npr, lab = timed("knn", lambda: ops.knn_proposals(src, tgt, p))
            timed("random", lambda: ops.random_proposals(src, tgt, p, pv, lc, npr, lab, seed=di))

            def run_bcd():
                mode = lib.BCD_INT32_F32COST if bcd_mode == lib.BCD_INT32 else bcd_mode   # as flowb200_flow_pair does
                ops.bcd(pv, lc, npr, lab, sweeps, mode=mode, lamda=p.lamda, tpsi=p.tpsi, cost_shift=p.cost_shift)
            timed("bcd", run_bcd)
            uv.append(timed("consistency", lambda: ops.flow_from_labels(pv, lab, want_yx=False)[1]))
        if directions == 2:
            timed("consistency", lambda: ops.consistency(uv[0], uv[1], p.con_tresh))
    return {k: v / reps for k, v in acc.items()}


def chain_kernel_times(ops, lib, p, sweeps, g0, g1, reps=2):
    """CUDA-event duration of every launch of the dominant kernel: flowb200_bcd_prepare (kset_sort + kset_build) and then
    flowb200_bcd_phase once per phase (kset_chain32_kernel; the generic kernel launched behind it returns at once when no
    chain is flagged), on the forward direction of one pair.  flowb200_bcd is exactly this sequence."""
    import torch
    d0, d1 = ops.daisy(g0), ops.daisy(g1)
    pv, lc, npr, lab = ops.knn_proposals(d0, d1, p)
    ops.random_proposals(d0, d1, p, pv, lc, npr, lab, seed=0)
    ws = ops.bcd_workspace(pv)
    kw = dict(mode=lib.BCD_INT32_F32COST, lamda=p.lamda, tpsi=p.tpsi, cost_shift=p.cost_shift)
    prep, col, row = [], [], []
    for rep in range(reps + 1):
        l2 = lab.clone()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 + 4 * sweeps)]
        torch.cuda.synchronize()
        ev[0].record()
        ops.bcd_prepare(pv, lc, npr, ws, 0, 1, **kw)
        ev[1].record()
        for w in range(sweeps):
            for ph in range(4):
                ops.bcd_phase(pv, lc, npr, l2, ws, ph, 0, 1, **kw)
                ev[2 + 4 * w + ph].record()
        torch.cuda.synchronize()
        if rep == 0:
            continue                               # warm-up
        t = [ev[i].elapsed_time(ev[i + 1]) for i in range(len(ev) - 1)]
        prep.append(t[0])
        col += [t[1 + 4 * w + ph] for w in range(sweeps) for ph in (0, 2)]
        row += [t[1 + 4 * w + ph] for w in range(sweeps) for ph in (1, 3)]
    return {"prepare_ms": float(np.mean(prep)), "column_phase_ms": float(np.mean(col)), "row_phase_ms": float(np.mean(row)),
            "ms_per_launch": float(np.mean(col + row))}


def cpu_oracle_pipeline(img1, img2, op, sweeps, directions, con_tresh, seed=0):
    """The whole path on the CPU oracle (numpy DAISY + C generisi/nasumicni/BCD/consistency)."""
    from oracle import consistency as ocons, cport, daisy as od, proposals as oprop
    d = (od.daisy(img1), od.daisy(img2))
    flows = []
    for di in range(directions):
        a, b = d[di], d[1 - di]
        P, L, N, B = cport.generisi(a, b, op)
        P, L, N = cport.nasumicni(a, b, P, L, N, B, op, seed=seed + di)
        lab = cport.ceo_bcd(P, L, N, B, sweeps, tpsi=op.tpsi, lamda=op.lamda)[-1]
        flows.append(oprop.final_flow(P, lab))
    if directions == 2:
        return ocons.forward_backward_consistency(ocons.ucitaj_flow(flows[0]), ocons.ucitaj_flow(flows[1]), con_tresh)
    return ocons.ucitaj_flow(flows[0])


def cpu_sample(p, sweeps, directions, steps=1):
    """Bounded sample of the workload for the CPU oracle: a crop of 5x5 cells (the centre cell's pixels see the
    full 5x5-cell search window), same K / sweeps / directions, all host threads (torchrun sets
    OMP_NUM_THREADS=1, so the thread count is set explicitly)."""
    from oracle import cport
    from oracle.proposals import Params
    synth = mod("synth")
    cport.set_num_threads(os.cpu_count() or 1)
    Hs, Ws = min(p.H, 5 * p.cellh), min(p.W, 5 * p.cellw)
    op = Params(Hs, Ws, p.cellw, p.cellh, p.cell_radius, p.k_cell, p.n_gauss, p.sigma, p.maxnprop, p.tphi, p.tpsi,
                p.lamda)
    img1, img2, _, _ = synth.make_pair(Hs, Ws, 0)
    cpu_oracle_pipeline(img1[:p.cellh * 1 + 20, :p.cellw + 20], img2[:p.cellh + 20, :p.cellw + 20],
                        Params(p.cellh + 20, p.cellw + 20, p.cellw, p.cellh, p.cell_radius, p.k_cell, p.n_gauss,
                               p.sigma, p.maxnprop, p.tphi, p.tpsi, p.lamda), 1, directions, p.con_tresh)   # warm-up
    ts = []
    for s in range(steps):
        t0 = time.perf_counter()
        out = cpu_oracle_pipeline(img1, img2, op, sweeps, directions, p.con_tresh, seed=s)
        ts.append(time.perf_counter() - t0)
    t = float(np.mean(ts))

    def cells_per_pixel(H, W):
        tot = 0
        for ci in range(W // p.cellw):
            bw = min(W, p.cellw * (ci + p.cell_radius + 1)) - max(0, p.cellw * (ci - p.cell_radius))
            for cj in range(H // p.cellh):
                tot += bw * (min(H, p.cellh * (cj + p.cell_radius + 1)) - max(0, p.cellh * (cj - p.cell_radius)))
        return tot / float(H * W)
    c_crop, c_full = cells_per_pixel(Hs, Ws), cells_per_pixel(p.H, p.W)
    return {"value": Hs * Ws / 1e6 / t, "unit": "Mpix/s", "cores": cport.num_threads(), "kind": "port",
            "crop": True, "extrapolated": False,
            "cells_in_range_per_pixel": {"crop": round(c_crop, 2), "workload": round(c_full, 2)},
            "note": "Mpix/s of the crop itself, not extrapolated: a pixel of the full workload searches "
                    f"{c_full:.1f} cells on average against {c_crop:.1f} in the crop, so the full-size CPU figure would "
                    "be lower (the exact search is ~60 % of the CPU time)",
            "sample": f"{steps} x {Ws}x{Hs} crop (5x5 cells of {p.cellw}x{p.cellh}), K={p.maxnprop}, bcd_times={sweeps}, "
                      f"{directions} direction(s), {t:.2f} s/step; C oracle with OpenMP + numpy DAISY",
            "seconds_per_step": t, "output": out}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    p, sweeps, directions = make_params(args.workload, 0)
    steps = args.steps
    r = cpu_sample(p, sweeps, directions, steps=steps)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"flow": r["output"]})
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "Mpix/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": 1, "ms_per_step": r["seconds_per_step"] * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": args.workload, "H": p.H, "W": p.W, "K": p.maxnprop, "k_cell": p.k_cell,
                       "n_gauss": p.n_gauss, "bcd_times": sweeps, "directions": directions,
                       "parallelism": "CPU oracle on rank 0, all host threads; every step is the bounded sample "
                                      "named in cpu_baseline.sample"},
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "crop", "extrapolated",
                                               "cells_in_range_per_pixel", "note")},
            "e2e": {"value": r["value"], "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def run_huge(args):
    """configs[4]: one image pair on all ranks (huge.flow_pair_sharded).  value = H*W / step time, strong scaling."""
    import torch
    import torch.distributed as dist
    lib, ops, synth, huge = mod("_lib"), mod("ops"), mod("synth"), mod("huge")
    lib.load()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    W_ = max(args.warmup, 3)
    p, sweeps, directions = make_params(args.workload, mod("params").DEFAULT_KNN_MODE)
    bcd_mode = lib.BCD_INT32 if args.bcd_mode == "int32" else lib.BCD_FP64_F32COST
    a, b, _, _ = synth.make_pair(p.H, p.W, 0)           # every rank holds the same pair
    ha, hb = torch.from_numpy(a).pin_memory(), torch.from_numpy(b).pin_memory()
    g0, g1 = ha.cuda(), hb.cuda()
    D = dist if world > 1 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(i, host=False):
        x0, x1 = (ha.cuda(non_blocking=True), hb.cuda(non_blocking=True)) if host else (g0, g1)
        out = huge.flow_pair_sharded(x0, x1, p, sweeps, directions, i, bcd_mode, rank, world, D)
        return out.cpu() if host else out

    for i in range(W_):
        step(i)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    L0 = lib.load().flowb200_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        out = step(W_ + i)
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = lib.load().flowb200_launch_count() - L0
    if args.dump_outputs and rank == 0:       # the same field on every rank
        dump_outputs(args.dump_outputs, {"flow": out})
    del out
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(i, host=True)
    torch.cuda.synchronize()
    t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e = p.H * p.W / 1e6 / (float(t.item()) / args.steps)
    # the sharded stage alone (search + merge), CUDA events, max over ranks
    d0, d1 = ops.daisy(g0), ops.daisy(g1)
    barrier()
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k0.record()
    huge.knn_proposals_sharded(d0, d1, p, rank, world, D)
    k1.record()
    barrier()
    t = torch.tensor([k0.elapsed_time(k1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    knn_ms = float(t.item())
    if rank == 0:
        pk = peaks()
        flops = algorithmic_work(p, sweeps, 1)["knn"][1]
        ach = flops / (knn_ms / 1e3) / 1e12
        line = {"metric": METRIC, "value": p.H * p.W / 1e6 / (ms_step / 1e3), "unit": "Mpix/s", "n_gpus": world,
                "steps": args.steps, "warmup": W_, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "int32" if bcd_mode == lib.BCD_INT32 else "f64", "data": "synthetic",
                "pairs_per_s": 1e3 / ms_step,
                "config": {"workload": args.workload, "H": p.H, "W": p.W, "K": p.maxnprop, "k_cell": p.k_cell,
                           "n_gauss": p.n_gauss, "bcd_times": sweeps, "directions": directions,
                           "parallelism": f"1 pair on {world} rank(s): proposal search sharded by target cell columns (broadcast + slot-range merge), BCD chains of every phase split (all-reduce of label differences); DAISY, random proposals, check replicated",
                           "l2": "working set (GBs of proposals) exceeds L2"},
                "e2e": {"value": e2e, "unit": "Mpix/s", "h2d_bytes_per_step": 2 * p.H * p.W * 3,
                        "d2h_bytes_per_step": p.H * p.W * 12},
                "gpu_launches": int(launches), "clocks": clocks,
                "roofline": {"kernel": "knn_select_kernel (+ re-rank, band merge)", "stage": "knn (one direction, sharded)",
                             "bound": "tensor", "achieved": ach, "peak": pk["tensor"] * world, "unit": "TFLOP/s",
                             "frac": ach / (pk["tensor"] * world), "traffic": None, "ms": knn_ms,
                             "peak_source": pk["src"] + " (MEASURED_PEAKS.json) x n_gpus",
                             "note": "algorithmic FLOPs of the full-image search / max-over-ranks time of search + merge"},
                "cpu_baseline": None}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def huge_extra(rank, world, local, steps=2):
    """Single-huge-image mode on the ranks of this run (the NCCL data plane the pair-sharded benchmark does not have):
    ms per 3840x2160 pair (max over ranks), and whether the sharded result equals one GPU's bit for bit."""
    import torch
    import torch.distributed as dist
    lib, ops, synth, huge = mod("_lib"), mod("ops"), mod("synth"), mod("huge")
    p, sweeps, directions = make_params(HUGE_IN_BENCH, mod("params").DEFAULT_KNN_MODE)
    a, b, _, _ = synth.make_pair(p.H, p.W, 0)
    g0, g1 = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
    D = dist if world > 1 else None

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    out = huge.flow_pair_sharded(g0, g1, p, sweeps, directions, 0, lib.BCD_INT32, rank, world, D)      # warm-up
    sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        out = huge.flow_pair_sharded(g0, g1, p, sweeps, directions, 1 + i, lib.BCD_INT32, rank, world, D)
    e1.record()
    sync()
    t = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    equal = None
    if world > 1:      # the same pair and seed on this rank's GPU alone (the same code as one part, no exchange:
                       # flowb200_flow_pair's own workspace layout would not fit 180 GB at this size)
        torch.cuda.empty_cache()
        want = huge.flow_pair_sharded(g0, g1, p, sweeps, directions, steps, lib.BCD_INT32, 0, 1, None)
        ok = torch.tensor([1.0 if torch.equal(out, want) else 0.0], dtype=torch.float64, device="cuda")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        equal = bool(ok.item() == 1.0)
    return {"workload": HUGE_IN_BENCH, "ms_per_pair": float(t.item()), "mpix_per_s": p.H * p.W / 1e6 / (float(t.item()) / 1e3),
            "n_gpus": world, "steps": steps, "scaling": "strong", "bit_equal_to_single_gpu": equal,
            "exchange": "target cell columns sharded: one all-gather of packed slot ranges per direction; BCD chains of "
                        "every phase split: one all-reduce of label differences per phase (huge.py)"}


def run_batch(args):
    """configs[3] as written: 99 distinct host-resident pairs x 2 directions, dealt round robin over the ranks
    (dist.shard_units), every rank's share through flowb200_ctx_flow_pairs_host (host buffers in, host fields out,
    the copies of pair i+1 / result i-1 overlapped with the computation of pair i).  value = 99 pairs / max-over-ranks
    wall time of one pass over the share; steps = passes."""
    import ctypes as C
    import torch
    import torch.distributed as dist
    lib, ops, synth, dm = mod("_lib"), mod("ops"), mod("synth"), mod("dist")
    L = lib.load()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    p, sweeps, directions = make_params(args.workload, mod("params").DEFAULT_KNN_MODE)
    n_pairs = 99
    mine = dm.shard_units(n_pairs, rank, world)
    # distinct pairs: picindex 0..98 (README.md:8) -> synthetic pair of that number
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max_workers=max(1, (os.cpu_count() or 8) // max(1, world))) as ex:   # (scipy releases the GIL)
        pairs = list(ex.map(lambda i: synth.make_pair(p.H, p.W, i)[:2], mine))
    outs = [np.empty((p.H, p.W, 3), dtype=np.float32) for _ in mine]
    cp = ops.cparams(p, bcd_mode=lib.BCD_INT32)
    ctx = L.flowb200_ctx_create(C.byref(cp))
    if not ctx:
        raise RuntimeError("flowb200_ctx_create failed: " + L.flowb200_last_cuda_error().decode())
    PtrArr = C.c_void_p * len(mine)
    a0 = PtrArr(*[a.ctypes.data for a, _ in pairs])
    a1 = PtrArr(*[b.ctypes.data for _, b in pairs])
    ao = PtrArr(*[o.ctypes.data for o in outs])

    def one_pass(seed0):
        lib.check(L.flowb200_ctx_flow_pairs_host(ctx, a0, a1, len(mine), sweeps, directions, seed0, ao),
                  "flowb200_ctx_flow_pairs_host")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    lib.check(L.flowb200_ctx_flow_pairs_host(ctx, a0, a1, min(3, len(mine)), sweeps, directions, 0, ao), "warm-up")
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    L0 = L.flowb200_launch_count()
    t0 = time.perf_counter()
    for s_ in range(args.steps):
        one_pass(1000 * s_)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / args.steps
    launches = L.flowb200_launch_count() - L0
    t = torch.tensor([dt], dtype=torch.float64, device="cuda")
    tmin = t.clone()
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    L.flowb200_ctx_destroy(ctx)
    if args.dump_outputs:      # this rank's pairs, in the order of dist.shard_units
        dump_outputs(args.dump_outputs, {"flow": np.stack(outs)}, f"_rank{rank}" if world > 1 else "",
                     DUMP_BYTES // world)
    secs = float(t.item())
    if rank == 0:
        val = n_pairs * p.H * p.W / 1e6 / secs
        emit({"metric": METRIC, "value": val, "unit": "Mpix/s", "n_gpus": world, "steps": args.steps, "warmup": 1,
              "ms_per_step": secs * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
              "dtype": "int32", "data": "synthetic", "pairs_per_s": n_pairs / secs,
              "config": {"workload": args.workload, "H": p.H, "W": p.W, "K": p.maxnprop, "k_cell": p.k_cell,
                         "n_gauss": p.n_gauss, "bcd_times": sweeps, "directions": directions, "pairs": n_pairs,
                         "pairs_per_rank": [len(dm.shard_units(n_pairs, r, world)) for r in range(world)],
                         "parallelism": f"99 pairs dealt round robin over {world} rank(s), no collective on the data path",
                         "l2": "every pair is distinct; per-pair working set (>1 GB) exceeds L2",
                         "timing": "wall clock around the blocking host API (a step = one pass over the 99 pairs), max over "
                                   "ranks; the fastest rank needed %.3f s" % float(tmin.item())},
              "e2e": {"value": val, "unit": "Mpix/s", "h2d_bytes_per_step": n_pairs * 2 * p.H * p.W * 3,
                      "d2h_bytes_per_step": n_pairs * p.H * p.W * 12},
              "gpu_launches": int(launches), "clocks": clocks, "roofline": None, "cpu_baseline": None})
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="flowb200", choices=["flowb200", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--knn-mode", type=int, default=None)
    ap.add_argument("--bcd-mode", default="int32", choices=["int32", "fp64"])
    ap.add_argument("--inflight", type=int, default=1,
                    help="pairs of one rank processed concurrently per step (own stream, workspace and host thread "
                         "each; pairs are independent, README.md:40).  1 = one pair after the other (default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-breakdown", action="store_true")
    ap.add_argument("--no-huge", action="store_true", help="skip the short single-huge-image run (key 'huge')")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the timed path returned in its last step as DIR/<name>.npy "
                         "(float32 / float64, at most 64 MB = 64,000,000 bytes in all, over all ranks: "
                         "a fixed, seeded sample of larger outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    if "huge" in args.workload:
        return run_huge(args)
    if args.workload.startswith("99pairs"):
        return run_batch(args)

    import ctypes as C
    import torch
    import torch.distributed as dist
    lib, ops, synth = mod("_lib"), mod("ops"), mod("synth")
    L = lib.load()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    W_ = max(args.warmup, 3)
    knn_mode = args.knn_mode if args.knn_mode is not None else mod("params").DEFAULT_KNN_MODE
    p, sweeps, directions = make_params(args.workload, knn_mode)
    bcd_mode = lib.BCD_INT32 if args.bcd_mode == "int32" else lib.BCD_FP64_F32COST
    cp = ops.cparams(p, bcd_mode=bcd_mode)

    # a few distinct synthetic pairs per rank, cycled (the per-step working set, ~GBs of proposals, is far
    # larger than L2, so steps do not warm each other)
    inflight = max(1, args.inflight)
    npairs = max(2, inflight)
    pairs = [synth.make_pair(p.H, p.W, 10 * rank + i) for i in range(npairs)]
    dev_pairs = [(torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()) for a, b, _, _ in pairs]
    ws = ops.pair_workspace(p, "cuda", bcd_mode)

    def step_one(i):
        g0, g1 = dev_pairs[i % npairs]
        return ops.flow_pair(g0, g1, p, sweeps, directions, seed=i, bcd_mode=bcd_mode, workspace=ws)

    if inflight > 1:
        # a step = `inflight` independent pairs, each on its own stream, workspace and host thread (the library keeps
        # one auxiliary stream per host thread for the backward direction).  The side streams start after the
        # current stream's position and the current stream waits for all of them, so CUDA events recorded on the
        # current stream bracket the whole batch.
        import threading
        side = [torch.cuda.Stream() for _ in range(inflight)]
        wss = [ws] + [ops.pair_workspace(p, "cuda", bcd_mode) for _ in range(inflight - 1)]

        def step_batch(i):
            cur = torch.cuda.current_stream()
            start = torch.cuda.Event()
            start.record(cur)
            outs, errs = [None] * inflight, []

            def work(j):
                try:
                    torch.cuda.set_device(local)
                    side[j].wait_event(start)
                    with torch.cuda.stream(side[j]):
                        g0, g1 = dev_pairs[(i * inflight + j) % npairs]
                        outs[j] = ops.flow_pair(g0, g1, p, sweeps, directions, seed=i * inflight + j,
                                                bcd_mode=bcd_mode, workspace=wss[j])
                except Exception as e:     # re-raised on the main thread below
                    errs.append(e)
            th = [threading.Thread(target=work, args=(j,)) for j in range(inflight)]
            for t_ in th:
                t_.start()
            for t_ in th:
                t_.join()
            if errs:
                raise errs[0]
            for s_ in side:
                cur.wait_stream(s_)
            return outs
    step = step_batch if inflight > 1 else step_one

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(W_):
        out = step(i)
    barrier()
    launches0 = L.flowb200_launch_count()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        out = step(W_ + i)
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = (L.flowb200_launch_count() - launches0)
    if args.dump_outputs:      # the checked forward field of every pair of the last step
        outs = out if inflight > 1 else [out]
        names = ["flow"] if inflight == 1 else [f"flow_{j}" for j in range(inflight)]
        dump_outputs(args.dump_outputs, dict(zip(names, outs)), f"_rank{rank}" if world > 1 else "",
                     DUMP_BYTES // world)
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_step = ms_total / args.steps
    mpix = world * inflight * p.H * p.W / 1e6 / (ms_step / 1e3)

    # ---- e2e: host buffers through the C-ABI context, H2D + D2H inside the timed region
    ctx = L.flowb200_ctx_create(C.byref(cp))
    if not ctx:
        raise RuntimeError("flowb200_ctx_create failed: " + L.flowb200_last_cuda_error().decode())
    host_out = np.empty((p.H, p.W, 3), dtype=np.float32)

    def e2e_step(i):
        a, b, _, _ = pairs[i % npairs]
        lib.check(L.flowb200_ctx_flow_pair_host(ctx, a.ctypes.data, b.ctypes.data, sweeps, directions, i,
                                                host_out.ctypes.data), "flowb200_ctx_flow_pair_host")
    e2e_step(0)
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        e2e_step(1 + i)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_mpix = world * p.H * p.W / 1e6 / (float(t.item()) / args.steps)
    L.flowb200_ctx_destroy(ctx)
    huge_res = None
    if not args.no_huge and args.workload == DEFAULT_WORKLOAD:
        del ws
        torch.cuda.empty_cache()
        huge_res = huge_extra(rank, world, local)
        ws = ops.pair_workspace(p, "cuda", bcd_mode)

    if rank == 0:
        pk = peaks()
        work = algorithmic_work(p, sweeps, directions)
        roof, stages = None, None
        if not args.no_breakdown:
            stages = stage_breakdown(ops, lib, p, sweeps, directions, dev_pairs[0][0], dev_pairs[0][1], bcd_mode)
            kt = chain_kernel_times(ops, lib, p, sweeps, dev_pairs[0][0], dev_pairs[0][1])
            # the dominant kernel: kset_chain32_kernel, one launch per BCD phase.  Algorithmic bytes per launch =
            # N * (8 K + 12) (SURVEY.md 8d: 2 N (8 K + 12) per sweep, every pixel visited once by a column and once by a
            # row phase, i.e. half of the pixels per phase x 2 ... = a quarter of a sweep per launch)
            n_launch = directions * sweeps * 4
            per_launch = work["bcd"][1] / n_launch
            ach = per_launch / (kt["ms_per_launch"] / 1e3) / 1e9
            traffic, tsrc = None, None
            tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
            if os.path.isfile(tpath):
                with open(tpath) as f:
                    tj = json.load(f)
                traffic = tj["kernels"].get("kset_chain32_kernel", {}).get("mean_dram_bytes_per_launch")
                tsrc = "profiles/r02_traffic.json: " + tj.get("source", "")
            roof = {"kernel": "kset_chain32_kernel", "stage": "bcd", "bound": "hbm", "achieved": ach, "peak": pk["hbm"],
                    "unit": "GB/s", "frac": ach / pk["hbm"], "traffic": traffic, "traffic_source": tsrc,
                    "peak_source": pk["src"] + " (MEASURED_PEAKS.json)", "launches_per_step": n_launch,
                    "algorithmic_per_launch": per_launch, "ms_per_launch": kt["ms_per_launch"],
                    "kernel_ms": {k: round(v, 4) for k, v in kt.items()},
                    "note": "ms_per_launch = CUDA events around every flowb200_bcd_phase call of one direction run alone "
                            "(column and row phases averaged); the kernel is bound by instruction issue and step "
                            "latency, not by HBM (DESIGN.md 4.4)",
                    "stage_ms": {k: round(v, 4) for k, v in stages.items()},
                    "stage_note": "stage = the stage's C-ABI calls of both directions one after the other, CUDA events",
                    "stage_frac_of_roofline": {
                        k: round((work[k][1] / (v / 1e3) / (1e9 if work[k][0] == "hbm" else 1e12)) /
                                 (pk["hbm"] if work[k][0] == "hbm" else pk["tensor"]), 5) if v > 0 else None
                        for k, v in stages.items()}}
        # accuracy on the synthetic pair (known ground-truth flow), visualization.errorImage's definition, untimed
        gt = torch.from_numpy(synth.gt_uvv(pairs[0][2])).cuda()
        chk, raw_f, _ = ops.flow_pair(dev_pairs[0][0], dev_pairs[0][1], p, sweeps, directions, seed=0, bcd_mode=bcd_mode,
                                      want_raw=True, workspace=ws)
        e_raw, e_chk = ops.epe(raw_f, gt), ops.epe(chk, gt)
        accuracy = {"epe_px_forward_raw": e_raw[0], "outlier_pct_forward_raw": e_raw[1],
                    "epe_px_after_consistency": e_chk[0], "outlier_pct_after_consistency": e_chk[1],
                    "kept_frac_after_consistency": e_chk[2] / max(1, e_raw[2]),
                    "definition": "visualization.py:128-152 (EPE > 3 px = outlier), vs the synthetic ground truth"}
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            r = cpu_sample(p, sweeps, directions, steps=2)
            cpu = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "crop", "extrapolated",
                                     "cells_in_range_per_pixel", "note")}
        line = {"metric": METRIC, "value": mpix, "unit": "Mpix/s", "n_gpus": world, "steps": args.steps, "warmup": W_,
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "int32" if bcd_mode == lib.BCD_INT32 else "f64", "data": "synthetic",
                "pairs_per_s": world * inflight / (ms_step / 1e3),
                "config": {"workload": args.workload, "H": p.H, "W": p.W, "K": p.maxnprop, "k_cell": p.k_cell,
                           "n_gauss": p.n_gauss, "bcd_times": sweeps, "directions": directions,
                           "knn_mode": knn_mode, "bcd_mode": args.bcd_mode, "parallelism": f"pairs x{world}",
                           "pairs_in_flight_per_gpu": inflight,
                           "l2": "per-step working set (proposals+costs, >1 GB) exceeds L2; 2 pairs cycled"},
                "e2e": {"value": e2e_mpix, "unit": "Mpix/s", "h2d_bytes_per_step": 2 * p.H * p.W * 3,
                        "d2h_bytes_per_step": p.H * p.W * 12},
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
                "accuracy": accuracy, "huge": huge_res}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
