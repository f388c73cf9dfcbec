"""CPU oracles of FLOWB200_BCD_MRF: block coordinate descent on the MRF energy (include/flowb200.h).  TEST
INFRASTRUCTURE, next to the reference programme's oracles in oracle/ (which it does not change).

numpy (`ceo_bcd`, `run_phase`) and C (`ceo_bcd_c`, tests/mrf_oracle.c, compiled on first use into a cache directory
under the system's temporary directory) restate the same programme, independently of the kernels' two-candidate form:
the phases of ceoBCD (python bcd.py:261-284) with
  side neighbours ACROSS the chain axis: (y, x+1), (y, x-1) of a column chain; (y+1, x), (y-1, x) of a row chain,
    with their current labels (lines of the other parity, which the phase does not write);
  dp0(l) = (psi_plus + psi_minus) + lamda*lcost,  U(l) = (lamda*lcost + psi_plus) + psi_minus   (the reference's order);
  m = min over every k < nprop[prev] of dp_{i-1}(k) + min(L1, tpsi), back = lowest such k (no quirk Q1);
  end: lowest-index argmin of the last dp, backtrack.
Each chain's Viterbi is then the exact minimum of the energy (oracle.bcd.energy) over the chain, the rest fixed.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

PHASES = ((1, 0), (0, -1), (-1, 0), (0, 1))   # (ystep, xstep) of phases A, B, C, D (:265-277)


def phase_starts(phase, H, W):
    """chain starts of phase 0..3: even columns down, even rows right to left, odd columns up, odd rows left to right"""
    return ([(0, x) for x in range(0, W, 2)],
            [(y, W - 1) for y in range(0, H, 2)],
            [(H - 1, x) for x in range((W // 2) * 2 - 1, -1, -2)],
            [(y, 0) for y in range((H // 2) * 2 - 1, -1, -2)])[phase]


def _phase(proposals, lcosts, nprop, labels, tpsi, lamda, ystep, xstep, starts):
    """all chains `starts` of one phase, vectorised over the chains; labels in place"""
    H, W, K, _ = proposals.shape
    C_ = len(starts)
    if C_ == 0:
        return
    sy = np.array([s[0] for s in starts])
    sx = np.array([s[1] for s in starts])
    L = H if ystep != 0 else W
    yside, xside = (1, 0) if ystep == 0 else (0, 1)    # across the chain axis
    old = labels.copy()
    lab_idx = np.arange(K)
    dp_prev = None
    back = np.zeros((L, C_, K), dtype=np.int64)
    for i in range(L):
        y = sy + i * ystep
        x = sx + i * xstep
        v = proposals[y, x]                               # (C,K,2)
        n = nprop[y, x]
        cost = lcosts[y, x]

        def side(dy, dx):
            yy, xx = y + dy, x + dx
            ok = (yy >= 0) & (yy < H) & (xx >= 0) & (xx < W)
            yc, xc = np.clip(yy, 0, H - 1), np.clip(xx, 0, W - 1)
            nb = proposals[yc, xc, old[yc, xc]]           # (C,2)
            l1 = np.abs(v[..., 0] - nb[..., None, 0]) + np.abs(v[..., 1] - nb[..., None, 1])
            return np.where(ok[..., None], np.minimum(tpsi, l1), 0)
        psi_p = side(yside, xside)
        psi_m = side(-yside, -xside)
        if i == 0:
            dp = (psi_p + psi_m) + lamda * cost
        else:
            small = (lamda * cost + psi_p) + psi_m
            u = proposals[y - ystep, x - xstep]
            pn = nprop[y - ystep, x - xstep]
            l1 = np.abs(v[:, :, None, 0] - u[:, None, :, 0]) + np.abs(v[:, :, None, 1] - u[:, None, :, 1])
            kvalid = lab_idx[None, None, :] < pn[:, None, None]
            cand = np.where(kvalid, dp_prev[:, None, :] + np.minimum(l1, tpsi), np.inf)
            back[i] = cand.argmin(axis=2)
            dp = cand.min(axis=2) + small
        dp_prev = np.where(lab_idx[None, :] < n[:, None], dp, np.inf)
    lab = dp_prev.argmin(axis=1)
    for i in range(L - 1, -1, -1):
        labels[sy + i * ystep, sx + i * xstep] = lab
        if i > 0:
            lab = back[i, np.arange(C_), lab]


def run_phase(proposals, lcosts, nprop, labels, phase, tpsi=8, lamda=0.05, chain_chunk=64):
    """one phase (0..3), labels (int64) in place"""
    H, W = labels.shape
    starts = phase_starts(phase, H, W)
    for s in range(0, len(starts), chain_chunk):
        _phase(proposals, lcosts, nprop, labels, tpsi, lamda, *PHASES[phase], starts[s:s + chain_chunk])


def ceo_bcd(proposals, lcosts, nprop, labels, sweeps, tpsi=8, lamda=0.05):
    """list of the int64 label images after every sweep (oracle.bcd.ceo_bcd's contract)"""
    labels = labels.astype(np.int64).copy()
    out = []
    for _ in range(sweeps):
        for phase in range(4):
            run_phase(proposals, lcosts, nprop, labels, phase, tpsi, lamda)
        out.append(labels.copy())
    return out


_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def _load():
    """compile tests/mrf_oracle.c (the flags of oracle/Makefile) into a directory keyed by the source's hash"""
    global _lib
    if _lib is None:
        src = os.path.join(_HERE, "mrf_oracle.c")
        with open(src, "rb") as f:
            key = hashlib.sha256(f.read()).hexdigest()[:16]
        out = os.path.join(tempfile.gettempdir(), f"flowb200_mrf_oracle_{os.getuid()}", f"{key}.so")
        if not os.path.isfile(out):
            os.makedirs(os.path.dirname(out), exist_ok=True)
            tmp = f"{out}.{os.getpid()}"
            subprocess.run(["gcc", "-O3", "-march=x86-64-v3", "-fopenmp", "-fPIC", "-std=c11", "-Wall",
                            "-ffp-contract=off", "-shared", "-o", tmp, src, "-lm"], check=True)
            os.replace(tmp, out)
        _lib = C.CDLL(out)
    return _lib


def ceo_bcd_c(proposals, lcosts, nprop, labels, sweeps, tpsi=8, lamda=0.05, phases=4):
    """the C restatement: list of the int64 label images after every sweep; phases < 4 stops the last sweep after
    that many phases (its snapshot is then taken there)"""
    prop = np.ascontiguousarray(proposals, dtype=np.int32)
    lc = np.ascontiguousarray(lcosts, dtype=np.float64)
    npr = np.ascontiguousarray(nprop, dtype=np.int32)
    lab = np.array(labels, dtype=np.int32, copy=True)
    H, W, K, _ = prop.shape
    snaps = np.empty((sweeps, H, W), dtype=np.int32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
    rc = _load().mrf_bcd(p(prop), p(lc), p(npr), p(lab), H, W, K, C.c_double(lamda), int(tpsi), int(sweeps),
                         int(phases), p(snaps))
    if rc:
        raise RuntimeError(f"mrf_bcd failed: {rc}")
    return [s.astype(np.int64) for s in snaps]
