"""Generate tests/golden/*.npz by executing the reference's own source (oracle/ref_harness.py).

Run in the build container only (needs /root/reference):   python tests/golden/make_golden.py
The fixtures are what pins the oracle restatements; the GPU box only ever reads the .npz files.
Arrays are stored in compact dtypes (values are exactly representable); `load_case` in
tests/helpers.py restores the reference dtypes.
"""
import importlib
import os
import sys
import tempfile
import zipfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import helpers                                # noqa: E402
from oracle import ref_harness as rh          # noqa: E402
from oracle import daisy as odaisy            # noqa: E402

synth = importlib.import_module("lk-s-2022-estimacija-pokreta_b200.synth")
OUT = os.path.dirname(os.path.abspath(__file__))


def compact(r):
    out = {}
    for k, v in r.items():
        if k in ("proposals", "draws"):
            out[k] = v.astype(np.int16)
        elif k in ("nprop", "labels00") or k.startswith("labels"):
            out[k] = v.astype(np.int16)
        elif k == "lcosts":
            f = v.astype(np.float32)
            assert np.array_equal(f.astype(np.float64), v), "lcosts not float32-representable"
            out[k] = f
        elif k.startswith("flow"):
            out[k] = v.astype(np.int16) if np.array_equal(v, np.round(v)) else v
        else:
            out[k] = v
    return out


def stage_case(name, H, W, cw, ch, pair, sweeps, seed, both_dirs, thresholds=()):
    img1, img2, fwd, bwd = synth.make_pair(H, W, pair, max_dx=6, max_dy=4, n_rect=2)
    pp = rh.reference_postprocessing() if thresholds else None
    data = {"img1": img1, "img2": img2, "gt_fwd": fwd, "gt_bwd": bwd,
            "meta": np.array([H, W, cw, ch, pair, sweeps, seed], dtype=np.int64),
            "desc1": odaisy.daisy(img1), "desc2": odaisy.daisy(img2)}
    flows_final = {}
    for b in ((0, 1) if both_dirs else (0,)):
        wd = tempfile.mkdtemp(prefix=f"golden_{name}_{b}_")
        src, tgt = (img1, img2) if b == 0 else (img2, img1)
        r = rh.run_stage1(wd, src, tgt, pair, b, True, cw, ch, seed=seed + b)
        labs, flows = rh.run_stage2(wd, H, W, pair, b, sweeps)
        r = compact(r)
        for k, v in r.items():
            data[f"b{b}_{k}"] = v
        for w, (l, f) in enumerate(zip(labs, flows), 1):
            data[f"b{b}_labels{w:02d}"] = l.astype(np.int16)
            data[f"b{b}_flow{w:02d}"] = f.astype(np.int16)
        flows_final[b] = os.path.join(wd, f"Gotova flow slika 1{pair:02d} backward={b} posle {sweeps:02d} BCD.npy")
        print(name, "dir", b, "nprop", r["nprop"].min(), r["nprop"].max())
    for thr in thresholds:
        out = os.path.join(tempfile.mkdtemp(), "sparse_field.npy")
        fi = pp.postProcessing(flows_final[0], flows_final[1], thr, out)
        data[f"sparse_thr{thr}"] = np.load(out)
        assert np.array_equal(fi.flow, data[f"sparse_thr{thr}"])
        print(name, "thr", thr, "valid", float(data[f"sparse_thr{thr}"][..., 2].mean()))
    save_case(os.path.join(OUT, name + ".npz"), data)
    return data


def save_case(path, data):
    """Writes a stage case with the stage-1 proposals, costs and K-set bits of every direction replaced by digests
    (tests/helpers.load_case recomputes them with the oracle and checks them against the digests), LZMA-compressed:
    the full arrays would make the file several MB."""
    data = dict(data)
    K = int(data[[k for k in data if k.endswith("_proposals")][0]].shape[2])
    for b in (0, 1):
        if f"b{b}_proposals" not in data:
            continue
        nprop = data[f"b{b}_nprop"].astype(np.int64)
        data[f"b{b}_proposals_sha256"] = helpers.digest(data.pop(f"b{b}_proposals").astype(np.int64))
        data[f"b{b}_lcosts_sha256"] = helpers.digest(data.pop(f"b{b}_lcosts").astype(np.float64))
        data[f"b{b}_packedksets_sha256"] = helpers.ksets_digest(data.pop(f"b{b}_packedksets"), nprop, K)
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_LZMA) as zf:
        for k, v in data.items():
            with zf.open(k + ".npy", "w") as f:
                np.lib.format.write_array(f, np.asanyarray(v))


def bcd_quantised_case(name, z, sweeps, shift):
    """Reference BCD on costs quantised to 20*m/2^S (exact in float64): pins the int32 mode.  z: what stage_case
    returned, i.e. the reference's own stage-1 arrays (the saved case keeps only their digests)."""
    H, W, cw, ch, pair, _, _ = (int(v) for v in z["meta"])
    lc = z["b0_lcosts"].astype(np.float64)
    m = np.rint(0.05 * lc * (1 << shift)).astype(np.int64)
    m[z["b0_lcosts"] == 1000.0] = 0
    lq = 20.0 * m / float(1 << shift)
    lq[z["b0_lcosts"] == 1000.0] = 1000.0
    assert np.array_equal(0.05 * lq[lq != 1000.0], (m / float(1 << shift))[lq != 1000.0])
    wd = tempfile.mkdtemp(prefix=f"golden_{name}_")
    rh.write_stage1_files(wd, pair, 0, z["b0_proposals"], lq, z["b0_nprop"], z["b0_labels00"], z["b0_packedksets"])
    labs, _ = rh.run_stage2(wd, H, W, pair, 0, sweeps)
    data = {"meta": np.array([H, W, cw, ch, pair, sweeps, shift], dtype=np.int64), "m": m.astype(np.int32),
            "proposals": z["b0_proposals"], "nprop": z["b0_nprop"], "labels00": z["b0_labels00"]}
    for w, l in enumerate(labs, 1):
        data[f"labels{w:02d}"] = l.astype(np.int16)
        print(name, "sweep", w, "changed", int((l != z["b0_labels00"]).sum()))
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **data)


def consistency_cases():
    """Reference postprocessing on hand-made flows: quirk Q5, non-integer flow, thresholds."""
    pp = rh.reference_postprocessing()
    rng = np.random.default_rng(11)
    data = {}
    H, W = 20, 30
    f = np.zeros((H, W, 2)); f[..., 1] = 3
    g = np.zeros((H, W, 2)); g[..., 1] = -3
    cases = {"const": (f, g, 10)}
    f2 = rng.integers(-6, 7, size=(H, W, 2)).astype(np.float64)
    g2 = -f2 + rng.integers(-2, 3, size=(H, W, 2))
    cases["randint"] = (f2, g2, 2)
    f3 = rng.normal(0, 4, size=(37, 23, 2))
    g3 = rng.normal(0, 4, size=(37, 23, 2))
    cases["real"] = (f3, g3, 5)
    for k, (a, b, thr) in cases.items():
        d = tempfile.mkdtemp()
        np.save(os.path.join(d, "a.npy"), a)
        np.save(os.path.join(d, "b.npy"), b)
        pp.postProcessing(os.path.join(d, "a.npy"), os.path.join(d, "b.npy"), thr, os.path.join(d, "o.npy"))
        data[k + "_fwd"], data[k + "_bwd"], data[k + "_thr"] = a, b, np.array(thr)
        data[k + "_out"] = np.load(os.path.join(d, "o.npy"))
        print("consistency", k, "valid", float(data[k + "_out"][..., 2].mean()))
    np.savez_compressed(os.path.join(OUT, "consistency.npz"), **data)


def parovi_case():
    """The reference's napravi_parove.parovi on the 'real' consistency output -> tests/golden/parovi_real.txt."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("_ref_parovi", os.path.join(rh.REF, "napravi_parove.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    z = np.load(os.path.join(OUT, "consistency.npz"))
    d = tempfile.mkdtemp()
    np.save(os.path.join(d, "f.npy"), z["real_out"])
    mod.parovi(os.path.join(d, "f.npy"), os.path.join(OUT, "parovi_real.txt"))


if __name__ == "__main__":
    assert rh.available(), "reference source not found"
    consistency_cases()
    parovi_case()
    pair_a = stage_case("pair_a", 40, 48, 12, 10, pair=3, sweeps=2, seed=5, both_dirs=True, thresholds=(10, 2))
    stage_case("pair_b", 44, 50, 12, 10, pair=7, sweeps=1, seed=9, both_dirs=False)
    bcd_quantised_case("bcd_q12", pair_a, sweeps=3, shift=12)
