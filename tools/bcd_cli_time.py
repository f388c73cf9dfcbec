"""The drop-in `bcd.py <pair> <backward> <bcd_times>` on reference-format stage-1 files at the reference's own size
(1241x375, K=150): wall time of the whole script (file I/O included) and CUDA-event time of the BCD call inside it.
Stage 1 is this repository's `daisy i flann.py` on a synthetic pair (it writes the reference's int64 / float64 files).
   python tools/bcd_cli_time.py [bcd_times]   ->  one JSON line"""
import importlib, json, os, subprocess, sys, tempfile, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
P = "lk-s-2022-estimacija-pokreta_b200"
synth = importlib.import_module(f"{P}.synth")
sweeps = int(sys.argv[1]) if len(sys.argv) > 1 else 4
H, W = 375, 1241
with tempfile.TemporaryDirectory() as tmp:
    synth.write_dataset(os.path.join(tmp, "data_scene_flow"), H, W, [6])
    work = os.path.join(tmp, "work")
    os.makedirs(work)
    env = dict(os.environ, FLOWB200_SKIP_KSETS="1")          # no 2.6 GB packedksets.npy: bcd.py does not read it
    t0 = time.time()
    subprocess.run([sys.executable, os.path.join(ROOT, "daisy i flann.py"), "6", "0", "1"], cwd=work, env=env, check=True,
                   stdout=subprocess.DEVNULL)
    t1 = time.time()
    out = {}
    code = (f"import sys, time, torch; sys.path.insert(0, {ROOT!r}); import importlib;"
            f"st = importlib.import_module('{P}.stage2'); ops = importlib.import_module('{P}.ops');"
            "orig = ops.bcd\n"
            "def timed(*a, **k):\n"
            "    torch.cuda.synchronize(); e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)\n"
            "    e0.record(); r = orig(*a, **k); e1.record(); torch.cuda.synchronize()\n"
            "    print('BCD_MS', e0.elapsed_time(e1), 'MODE', k.get('mode')); return r\n"
            "ops.bcd = timed\n"
            f"t = time.time(); st.run('6', '0', {sweeps}, log=lambda *a: None); print('RUN_S', time.time() - t)")
    r = subprocess.run([sys.executable, "-c", code], cwd=work, capture_output=True, text=True, check=True)
    for line in r.stdout.splitlines():
        f = line.split()
        if f and f[0] == "BCD_MS":
            out["ksets_bcd_ms"] = round(float(f[1]), 2)
            out["bcd_mode"] = int(f[3])
        if f and f[0] == "RUN_S":
            out["ksets_script_s"] = round(float(f[1]), 2)
    out.update(H=H, W=W, K=150, bcd_times=sweeps, stage1_script_s=round(t1 - t0, 2),
               note="bcd_mode 0 = FP64_F32COST (reference-written costs are float32 sums); script time includes np.load "
                    "of 1.7 GB of int64/float64 files and the np.save calls after every sweep")
    print(json.dumps(out))
