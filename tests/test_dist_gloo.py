"""N > 1 host logic on CPU: two gloo ranks shard the pair list without overlap, and the timing reduction is the max."""
import os
import subprocess
import sys
import textwrap

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_shard_units_partition():
    from helpers import pkg
    d = pkg("dist")
    for n in (0, 1, 7, 99, 198):
        for ws in (1, 2, 4, 8):
            shards = [d.shard_units(n, r, ws) for r in range(ws)]
            flat = sorted(u for s in shards for u in s)
            assert flat == list(range(n))
            assert max(len(s) for s in shards) - min(len(s) for s in shards) <= 1
    with pytest.raises(ValueError):
        d.shard_units(4, 2, 2)


def test_two_gloo_ranks(tmp_path):
    pytest.importorskip("torch")
    script = tmp_path / "w.py"
    script.write_text(textwrap.dedent(f"""
        import importlib, json, os, sys
        sys.path.insert(0, {ROOT!r})
        d = importlib.import_module("lk-s-2022-estimacija-pokreta_b200.dist")
        rank, ws, local = d.init(backend="gloo")
        units = d.shard_units(99, rank, ws)
        d.barrier()
        t = d.max_over_ranks(10.0 + rank)            # rank 1 is the slow one
        n = d.sum_over_ranks(len(units))
        json.dump({{"rank": rank, "ws": ws, "units": units, "t": t, "n": n}}, open(os.path.join({str(tmp_path)!r}, f"r{{rank}}.json"), "w"))
    """))
    # --standalone: the rendezvous takes a free local port, so runs of the suite that overlap on one host do not collide
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node=2", str(script)],
                       capture_output=True, text=True, timeout=300, env=dict(os.environ, OMP_NUM_THREADS="1"))
    assert r.returncode == 0, r.stderr[-3000:]
    import json
    outs = [json.load(open(tmp_path / f"r{k}.json")) for k in (0, 1)]
    assert outs[0]["ws"] == outs[1]["ws"] == 2
    assert sorted(outs[0]["units"] + outs[1]["units"]) == list(range(99))
    assert not set(outs[0]["units"]) & set(outs[1]["units"])
    assert outs[0]["t"] == outs[1]["t"] == 11.0
    assert outs[0]["n"] == outs[1]["n"] == 99.0
