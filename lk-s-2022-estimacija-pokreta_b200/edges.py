"""Drop-in for the reference's `edge` module (edge.py), the Canny part: EpicFlow's edge input.

  canny_ivice(fileslike, binfile)   edge.py:19-35   image file -> raw float32 [H][W] file, 0.0 on an edge, 1.0 elsewhere
  sed_ivice(fileslike, binfile)     edge.py:4-17    structured edge detection: needs opencv-contrib `ximgproc` and a
                                                    trained `model.yml`, neither of which exists offline - not provided

The edge map is computed on the GPU (flowb200_canny_edges_host), bit-identical to cv2.Canny on the blurred gray
image; there is no CPU fallback.  Image decoding stays with cv2.imread as in the reference.
"""
import math

import numpy as np

from . import _lib


def canny_edges(img_bgr, threshold1=100, threshold2=200):
    """uint8 (H,W,3) BGR array -> float32 (H,W) `(255 - cv2.Canny(...)) / 255` (edge.py:21-29).  The thresholds
    may come in either order, as for cv2.Canny: the smaller one is the low threshold."""
    img = np.ascontiguousarray(img_bgr, dtype=np.uint8)
    if img.ndim != 3 or img.shape[2] != 3:
        raise TypeError("expected an (H,W,3) uint8 BGR image")
    H, W = img.shape[:2]
    out = np.empty((H, W), dtype=np.float32)
    L = _lib.load()
    # cv::Canny compares the integer L1 magnitude with cvFloor of both thresholds (the library swaps them if needed)
    _lib.check(L.flowb200_canny_edges_host(img.ctypes.data, H, W, math.floor(threshold1), math.floor(threshold2),
                                           out.ctypes.data), "flowb200_canny_edges_host")
    return out


def canny_ivice(fileslike, binfile):
    import cv2
    img = cv2.imread(fileslike)              # None makes cv2.cvtColor raise in the reference (:21)
    if img is None:
        raise TypeError(f"cv2.imread could not read {fileslike!r}")
    inverted_edges1 = canny_edges(img, 100, 200)
    with open(binfile, "wb") as f:
        f.write(inverted_edges1)


def sed_ivice(fileslike, binfile):
    raise NotImplementedError("sed_ivice needs cv2.ximgproc (opencv-contrib) and a trained model.yml; "
                              "only canny_ivice is provided")
