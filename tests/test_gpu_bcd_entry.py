"""The argument checks of the four BCD entry points (flowb200_bcd, flowb200_bcd_prepare, flowb200_bcd_phase,
flowb200_energy): one row per class of invalid input and entry point, each with the exact return code.

The entry points differ in what they check and in which order (check_args in csrc/bcd_ksets.cu), and the differences
are kept as they are: prepare / phase check the cost shift before the mode, so a float64 mode with a bad
shift is EINVAL there rather than EUNSUPPORTED; they refuse stray flag bits as EUNSUPPORTED where flowb200_bcd says
EINVAL; their tpsi range is make_plan's (EUNSUPPORTED); part / nparts / phase are checked after the mode; and
flowb200_energy has no limit on K or on H, W (only on H * W).

Every non-null pointer is a real device buffer sized for the shape its row declares, holding a valid problem (every
proposal (0, 0), nprop = K, labels 0, zero costs, a zeroed workspace), so that a row that a regression accepted
would run on memory it owns.
"""
import ctypes as C

import pytest

from helpers import pkg

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

H0, W0, K0 = 4, 5, 8
INT32, F32C, FP64, FP64_F64, MRF = 2, 3, 0, 1, 16
OK, EINVAL, EWORKSPACE, EUNSUPPORTED = 0, -1, -2, -4

DEFAULTS = dict(H=H0, W=W0, K=K0, mode=INT32, lamda=0.05, tpsi=8, shift=12, sweeps=1, part=0, nparts=1, phase=0,
                ws_bytes=None)
POINTERS = {"bcd": ("pvec", "cost", "nprop", "labels", "ws"), "prepare": ("pvec", "cost", "nprop", "ws"),
            "phase": ("pvec", "cost", "nprop", "labels", "ws"), "energy": ("pvec", "cost", "nprop", "labels", "out4")}
BCD3 = ("bcd", "prepare", "phase")


def rows():
    """(entry, overrides of DEFAULTS or a null pointer name, expected return code)"""
    R = []
    for e in POINTERS:
        R.append((e, {}, OK))
        R += [(e, {"null": p}, EINVAL) for p in POINTERS[e]]
        R += [(e, {k: 0}, EINVAL) for k in ("H", "W", "K")]
        R += [(e, {k: -3}, EINVAL) for k in ("H", "W", "K")]
        big = OK if e == "energy" else EINVAL   # flowb200_energy: no limit on K or on H, W
        R += [(e, {"K": 513}, big), (e, {"H": 16385, "W": 2, "K": 1}, big), (e, {"H": 2, "W": 16385, "K": 1}, big)]
        # the cost shift: checked in the int32 modes; prepare / phase check it in every mode, before the mode
        for s in (-1, 15):
            R.append((e, {"shift": s}, EINVAL))
            R.append((e, {"shift": s, "mode": FP64}, EINVAL if e in ("prepare", "phase") else OK))
            R.append((e, {"shift": s, "mode": FP64_F64 | MRF}, EINVAL if e in ("prepare", "phase") else OK))
        # tpsi: flowb200_bcd and flowb200_energy refuse < 0; the K-set plan refuses > 32 and, in prepare / phase, < 0
        R.append((e, {"tpsi": -1}, EUNSUPPORTED if e in ("prepare", "phase") else EINVAL))
        R.append((e, {"tpsi": 33}, OK if e == "energy" else EUNSUPPORTED))
        # modes and flags
        R += [(e, {"mode": m}, EUNSUPPORTED if e in ("prepare", "phase") else EINVAL)
              for m in (32, INT32 | 32, INT32 | MRF | 64, -1)]
        R += [(e, {"mode": m}, OK) for m in (INT32 | MRF, F32C, F32C | MRF)]
        R += [(e, {"mode": m}, EUNSUPPORTED if e in ("prepare", "phase") else OK)
              for m in (FP64, FP64 | MRF, FP64_F64, FP64_F64 | MRF)]
    R.append(("bcd", {"sweeps": -1}, EINVAL))
    R.append(("bcd", {"sweeps": 0}, OK))
    R.append(("bcd", {"sweeps": 0, "tpsi": 33}, EUNSUPPORTED))   # sweeps 0: the plan only
    for e in ("prepare", "phase"):
        R += [(e, {"part": 1, "nparts": 1}, EINVAL), (e, {"part": -1}, EINVAL), (e, {"nparts": 0}, EINVAL),
              (e, {"part": 2, "nparts": 2}, EINVAL), (e, {"part": 1, "nparts": 2}, OK)]
        R.append((e, {"nparts": 0, "mode": FP64}, EUNSUPPORTED))   # part / nparts after the mode
        R.append((e, {"nparts": 0, "tpsi": 33}, EINVAL))           # ... and before the plan
    R += [("phase", {"phase": 4}, EINVAL), ("phase", {"phase": -1}, EINVAL), ("phase", {"phase": 3}, OK),
          ("phase", {"phase": 4, "mode": FP64}, EUNSUPPORTED)]
    # the dp bound of the int32 modes (tpsi 8, shift 14: chains of 9362 steps; the float64 modes have none)
    for e in BCD3:
        R += [(e, {"H": 2, "W": 9363, "K": 1, "shift": 14}, EUNSUPPORTED),
              (e, {"H": 9363, "W": 2, "K": 1, "shift": 14}, EUNSUPPORTED),
              (e, {"H": 2, "W": 9362, "K": 1, "shift": 14}, OK)]
    R.append(("bcd", {"H": 2, "W": 9363, "K": 1, "shift": 14, "mode": FP64}, OK))
    R.append(("energy", {"H": 2, "W": 9363, "K": 1, "shift": 14}, OK))
    # a workspace smaller than the fixed part; the fixed part alone is enough
    for e in BCD3:
        R += [(e, {"ws_bytes": "min-1"}, EWORKSPACE), (e, {"ws_bytes": "min"}, OK)]
    R.append(("bcd", {"ws_bytes": "min-1", "mode": FP64}, EWORKSPACE))
    return R


ROWS = rows()


def row_id(r):
    e, ov, rc = r
    return f"{e}-" + ("-".join(f"{k}={v}" for k, v in ov.items()) or "defaults") + f"-rc{rc}"


def call(entry, ov):
    L = pkg("_lib")
    lib = L.load()
    a = dict(DEFAULTS, **{k: v for k, v in ov.items() if k != "null"})
    H, W, K = a["H"], a["W"], a["K"]
    npix, n = max(H, 1) * max(W, 1), max(H, 1) * max(W, 1) * max(K, 1)
    base = a["mode"] & ~MRF if a["mode"] >= 0 else -1
    cdtype = {FP64_F64: torch.float64, INT32: torch.int32}.get(base, torch.float32)
    ws_min = lib.flowb200_bcd_min_workspace_bytes(H, W, K)
    ws_bytes = {None: lib.flowb200_bcd_workspace_bytes(H, W, K), "min": ws_min,
                "min-1": ws_min - 1}[a["ws_bytes"]]
    buf = dict(pvec=torch.zeros(n, dtype=torch.int32, device="cuda"),
               cost=torch.zeros(n, dtype=cdtype, device="cuda"),
               nprop=torch.full((npix,), max(K, 1), dtype=torch.int32, device="cuda"),
               labels=torch.zeros(npix, dtype=torch.int32, device="cuda"),
               ws=torch.zeros(max(ws_bytes, 256), dtype=torch.uint8, device="cuda"),
               out4=torch.zeros(4, dtype=torch.float64, device="cuda"))
    P = {k: C.c_void_p(0 if ov.get("null") == k else t.data_ptr()) for k, t in buf.items()}
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    head = (a["mode"], a["lamda"], a["tpsi"], a["shift"])
    if entry == "bcd":
        rc = lib.flowb200_bcd(P["pvec"], P["cost"], P["nprop"], P["labels"], H, W, K, *head, a["sweeps"], None,
                              P["ws"], ws_bytes, s)
    elif entry == "prepare":
        rc = lib.flowb200_bcd_prepare(P["pvec"], P["cost"], P["nprop"], H, W, K, *head, a["part"], a["nparts"],
                                      P["ws"], ws_bytes, s)
    elif entry == "phase":
        rc = lib.flowb200_bcd_phase(P["pvec"], P["cost"], P["nprop"], P["labels"], H, W, K, *head, a["phase"],
                                    a["part"], a["nparts"], P["ws"], ws_bytes, s)
    else:
        rc = lib.flowb200_energy(P["pvec"], P["cost"], P["nprop"], P["labels"], H, W, K, *head, P["out4"], s)
    torch.cuda.synchronize()
    return rc


@pytest.mark.parametrize("entry,ov,rc", ROWS, ids=[row_id(r) for r in ROWS])
def test_entry_return_code(entry, ov, rc):
    assert call(entry, ov) == rc
