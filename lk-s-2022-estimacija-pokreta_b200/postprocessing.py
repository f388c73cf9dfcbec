"""Drop-in for the reference's `postprocessing` module (postprocessing.py:1-142), hot-path part.

Same names, arguments, in-place semantics and output as the reference:
  FlowImage().ucitajFlow(path)                       :5-17     .npy only; [dy,dx] -> (dx, dy, 1) float32
  removeSmallSegments(flow, tresh, min_segment_size) :29-76    in place on flow (disabled in the reference's own
                                                               postProcessing, :132; SURVEY 8f row 1)
  consistencyCheck(flow1, flow2, u1, v1, tresh)      :79-110   one pixel, in place on flow1
  fowardBackwardConsistency(flow1, flow2, tresh)     :114-117  every pixel of flow1
  postProcessing(filename1, filename2, con_tresh, npysave) -> FlowImage   :123-135
`flow`, `flow1`, `flow2` are float32 (H,W,3) arrays = (dx, dy, valid) as in the reference, whose callers pass
`FlowImage.flow` (:133); a FlowImage itself is accepted too.  The work runs on the GPU through
flowb200_consistency_host / flowb200_remove_small_segments_host (quirk Q5 and the scan-order effects of
removeSmallSegments reproduced); there is no CPU fallback.
"""
import math
import os
import sys

import numpy as np

from . import _lib


class FlowImage:
    def __init__(self):
        self.flow = np.zeros((1, 1, 3), dtype=np.float32)
        self.height = 1
        self.width = 1

    def ucitajFlow(self, flow_file):
        ext = os.path.splitext(flow_file)[1]
        if ext == ".npy":
            img = np.load(flow_file)
            self.height, self.width = int(img.shape[0]), int(img.shape[1])
            self.flow = np.zeros((self.height, self.width, 3), dtype=np.float32)
            self.flow[:, :, 0] = img[:, :, 1]
            self.flow[:, :, 1] = img[:, :, 0]
            self.flow[:, :, 2] = 1
        else:
            print("Unknown file format!")


def _field(flow, name):
    """The (H,W,3) array behind an argument: the array itself (what the reference's callers pass) or FlowImage.flow."""
    f = flow.flow if isinstance(flow, FlowImage) else flow
    if not isinstance(f, np.ndarray) or f.ndim != 3 or f.shape[2] != 3:
        raise TypeError(f"{name} must be an (H,W,3) array or a FlowImage")
    return f


def _inplace_field(flow, name):
    f = _field(flow, name)
    if f.dtype != np.float32 or not f.flags.c_contiguous or not f.flags.writeable:
        raise TypeError(f"{name} is modified in place: it must be a writeable C-contiguous float32 array")
    return f


def removeSmallSegments(flow, tresh, min_segment_size):
    """In place on flow, returns None like the reference (:29-76).

    A segment of `count` pixels is removed when `count > 1 and count < min_segment_size` (:73).  With an integer count
    a fractional bound acts like its ceiling, clamped to [0, 2**31 - 1]; NaN and -inf remove nothing (bound 0) and
    +inf removes every segment of two or more pixels (bound 2**31 - 1), as that comparison implies."""
    f = _inplace_field(flow, "flow")
    L = _lib.load()
    try:
        bound = max(0, min(int(math.ceil(min_segment_size)), 2**31 - 1))
    except ValueError:      # NaN: the comparison is always false
        bound = 0
    except OverflowError:   # +inf: every count of two or more is below it; -inf: none is
        bound = 2**31 - 1 if min_segment_size > 0 else 0
    _lib.check(L.flowb200_remove_small_segments_host(f.ctypes.data, f.shape[0], f.shape[1], float(tresh), bound),
               "flowb200_remove_small_segments_host")


def _match_shape(f1, f2, a0, a1, b0, b1):
    """flow2 of another shape than flow1.  The reference indexes flow2[u2][v2] with 0 <= u2 < A, 0 <= v2 < B
    (flow1's shape, :80, :87-90) by flow2's OWN shape: rows/columns beyond (A, B) are never read, and a target
    beyond flow2's extent raises IndexError (:97).  The device call takes one shape, so flow2 is cropped / zero
    padded to (A, B) here, after the same IndexError test."""
    A, B = f1.shape[0], f1.shape[1]
    A2, B2 = f2.shape[0], f2.shape[1]
    if A2 < A or B2 < B:
        r = f1[a0:a1, b0:b1]
        with np.errstate(invalid="ignore", over="ignore"):
            u2 = np.trunc(r[:, :, 0] + np.arange(a0, a1, dtype=np.float32)[:, None])
            v2 = np.trunc(r[:, :, 1] + np.arange(b0, b1, dtype=np.float32)[None, :])
        inside = (r[:, :, 2] > 0.5) & (u2 >= 0) & (v2 >= 0) & (u2 < A) & (v2 < B)
        if np.any(inside & ((u2 >= A2) | (v2 >= B2))):
            raise IndexError(f"flow2 of shape {f2.shape} is indexed out of bounds by flow1 of shape {f1.shape}")
    out = np.zeros((A, B, 3), dtype=np.float32)
    out[:min(A, A2), :min(B, B2)] = f2[:min(A, A2), :min(B, B2)]
    return out


def _check_region(flow1, flow2, a0, a1, b0, b1, tresh):
    f1 = _inplace_field(flow1, "flow1")
    f2 = np.ascontiguousarray(_field(flow2, "flow2"), dtype=np.float32)
    A, B = f1.shape[0], f1.shape[1]
    if f2.shape[:2] != f1.shape[:2]:
        f2 = _match_shape(f1, f2, a0, a1, b0, b1)
    if f2 is f1 or np.shares_memory(f1, f2):
        f2 = f2.copy()
    L = _lib.load()
    _lib.check(L.flowb200_consistency_host(f1.ctypes.data, f2.ctypes.data, A, B, float(tresh), a0, a1, b0, b1),
               "flowb200_consistency_host")


def consistencyCheck(flow1, flow2, u1, v1, tresh):
    """One pixel (u1, v1) = (row, col) of flow1, in place; returns None like the reference."""
    shp = _field(flow1, "flow1").shape
    if u1 < 0 or v1 < 0 or u1 >= shp[0] or v1 >= shp[1]:
        raise IndexError("index out of bounds")
    _check_region(flow1, flow2, int(u1), int(u1) + 1, int(v1), int(v1) + 1, tresh)


def fowardBackwardConsistency(flow1, flow2, tresh):
    shp = _field(flow1, "flow1").shape
    _check_region(flow1, flow2, 0, shp[0], 0, shp[1], tresh)


def postProcessing(filename1, filename2, con_tresh, npysave):
    flow1 = FlowImage()
    flow1.ucitajFlow(filename1)
    flow2 = FlowImage()
    flow2.ucitajFlow(filename2)
    # removeSmallSegments(flow1.flow, 10, 100) is commented out in the reference (:132)
    fowardBackwardConsistency(flow1.flow, flow2.flow, con_tresh)
    np.save(npysave, flow1.flow)
    return flow1


if __name__ == "__main__":
    postProcessing(sys.argv[1], sys.argv[2], float(sys.argv[3]), sys.argv[4])
