"""The tensor-core selection's candidate sets, through the counters the search reports.  GPU only.

knn_select_kernel writes, per (query, cell) task, every target whose score is within the bound, in ascending position.
Its candidate sets are fixed by that bound: a rewrite of the selection must not move it by one bit, even where the
exact re-rank would hide the difference in the proposals.  The six counters of `knn_proposals(..., want_idx=True)`
(tasks redone by brute force, list overflows, the 64-bit sum of the candidate counts) are compared with the values
the selection gave before its pass-1 compare was rewritten (packed subtractions and sign bits instead of set.le),
measured on a B200.  Running this file prints the counters of the current build.
"""
import numpy as np
import pytest

from helpers import pkg

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


def _synth_descriptors(H, W, flat_top=False):
    ops, synth = pkg("ops"), pkg("synth")
    a, b, _, _ = synth.make_pair(H, W, 0)
    if flat_top:
        a[:H // 3] = 128
        b[:H // 3] = 128
    return ops.daisy(torch.from_numpy(a).cuda()), ops.daisy(torch.from_numpy(b).cuda())


# name -> (H, W, K, cell size or None for the default 73 x 25, flat top third)
CASES = {
    "bench_k10": (436, 1024, 300, None, False),          # the benchmark's frame and search
    "flat_top_k10": (436, 1024, 300, None, True),        # over 2^20 overflowed tasks (test_gpu_knn_edges)
    "k5": (250, 511, 150, None, False),
    "k12_t320": (160, 240, 500, (20, 16), False),        # T = 320: the last chunk is part padding
}

# stats[0..5] recorded from the selection before the rewrite, NVIDIA B200 (profiles/r05_knn_select_stats.log: the
# build before and the build after, one session)
EXPECTED = {
    "bench_k10": [405, 0, 405, 0, 123069261, 0],
    "flat_top_k10": [2871033, 0, 2871033, 0, 84504907, 0],
    "k12_t320": [271356, 0, 271356, 0, 12259400, 0],
    "k5": [1, 0, 1, 0, 16063398, 0],
}


def run_case(name):
    params, ops = pkg("params"), pkg("ops")
    H, W, K, cell, flat_top = CASES[name]
    kw = dict(H=H, W=W, knn_mode=1)
    if cell:
        kw.update(cellw=cell[0], cellh=cell[1])
    p = params.for_k(K, **kw)
    d1, d2 = _synth_descriptors(H, W, flat_top)
    stats = ops.knn_proposals(d1, d2, p, want_idx=True, knn_mode=1)[5].cpu().numpy()
    return [int(v) for v in stats[:6]]


@pytest.mark.parametrize("name", sorted(CASES))
def test_select_counters_unchanged(name):
    got = run_case(name)
    want = EXPECTED[name]
    assert got == want, (name, got, want)
    total = (got[5] & 0xffffffff) << 32 | (got[4] & 0xffffffff)
    assert total > 0, (name, total)


if __name__ == "__main__":
    import json
    import os
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    print(json.dumps({name: run_case(name) for name in sorted(CASES)}))
