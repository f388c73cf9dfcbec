"""Canny edge map oracle (numpy).  TEST INFRASTRUCTURE — see oracle/__init__.py.

Restates `edge.py`:19-35 (`canny_ivice`): BGR2GRAY -> GaussianBlur(3x3, sigma 0) -> cv2.Canny(100, 200) ->
`(255 - edges) / 255` as float32 (0.0 on an edge, 1.0 elsewhere), the edge input of EpicFlow.  The arithmetic is
OpenCV's main module (imgproc), which IS installed here: tests/test_oracle_edges.py pins every step against cv2
itself (4.13) and against the output of the reference's own function (tests/golden/edges.npz).

OpenCV's integer arithmetic as restated here (8-bit input, aperture 3, L2gradient=False):
  blur     (sum of the 3x3 neighbourhood weighted 1 2 1 / 2 4 2 / 1 2 1  + 8) >> 4, border REFLECT_101
  Sobel    3x3, int16, border REPLICATE (what cv::Canny asks for)
  mag      |dx| + |dy|, zero outside the image
  NMS      a pixel with mag > low survives when it is a maximum along its quantised gradient direction, with
           OpenCV's asymmetric comparisons: horizontal (|dy| << 15 < |dx| * 13573): m > left and m >= right;
           vertical (|dy| << 15 > |dx| * 13573 + (|dx| << 16)): m > up and m >= down; diagonal: m > both
           neighbours on the diagonal the signs of dx, dy select
  hysteresis  survivors with mag > high are edges; survivors 8-connected to an edge are edges
  thresholds  floored; swapped when low > high (cv::Canny takes them in either order)
"""
import numpy as np

from .daisy import gray_u8

TG22 = 13573          # (int)(0.41421356237309504 * (1 << 15) + 0.5)
SHIFT = 15


def blur3(gray):
    """cv2.GaussianBlur(gray, (3, 3), 0) on uint8."""
    g = np.pad(gray.astype(np.int32), 1, mode="reflect")     # numpy 'reflect' == BORDER_REFLECT_101
    if gray.shape[0] == 1:
        g[0], g[2] = g[1], g[1]
    if gray.shape[1] == 1:
        g[:, 0], g[:, 2] = g[:, 1], g[:, 1]
    h = g[:, :-2] + 2 * g[:, 1:-1] + g[:, 2:]
    s = h[:-2] + 2 * h[1:-1] + h[2:]
    return ((s + 8) >> 4).astype(np.uint8)


def sobel3(img):
    """cv2.Sobel(img, CV_16S, 1, 0, 3) and (0, 1, 3) with BORDER_REPLICATE -> (dx, dy) int32."""
    p = np.pad(img.astype(np.int32), 1, mode="edge")
    sm_v = p[:-2] + 2 * p[1:-1] + p[2:]          # smooth over rows, all columns
    dx = sm_v[:, 2:] - sm_v[:, :-2]
    sm_h = p[:, :-2] + 2 * p[:, 1:-1] + p[:, 2:]
    dy = sm_h[2:] - sm_h[:-2]
    return dx, dy


def nms_map(dx, dy, low, high):
    """0 = survivor below `high`, 2 = survivor above `high`, 1 = no edge (cv::Canny's map values)."""
    H, W = dx.shape
    mag = np.zeros((H + 2, W + 2), dtype=np.int64)
    mag[1:-1, 1:-1] = np.abs(dx) + np.abs(dy)
    m = mag[1:-1, 1:-1]
    x = np.abs(dx).astype(np.int64)
    y = np.abs(dy).astype(np.int64) << SHIFT
    tg22x = x * TG22
    tg67x = tg22x + (x << (SHIFT + 1))
    left, right = mag[1:-1, :-2], mag[1:-1, 2:]
    up, down = mag[:-2, 1:-1], mag[2:, 1:-1]
    ul, ur, dl, dr = mag[:-2, :-2], mag[:-2, 2:], mag[2:, :-2], mag[2:, 2:]
    horiz = y < tg22x
    vert = ~horiz & (y > tg67x)
    diag = ~horiz & ~vert
    neg = (dx.astype(np.int64) ^ dy.astype(np.int64)) < 0      # s = -1: compare up-right and down-left
    keep = (horiz & (m > left) & (m >= right)) | (vert & (m > up) & (m >= down)) | \
           (diag & np.where(neg, (m > ur) & (m > dl), (m > ul) & (m > dr)))
    keep &= m > low
    out = np.ones((H, W), dtype=np.uint8)
    out[keep] = 0
    out[keep & (m > high)] = 2
    return out


def hysteresis(pmap):
    """Edges = strong survivors and every survivor 8-connected to one (flood fill from the strong ones)."""
    H, W = pmap.shape
    edge = pmap == 2
    cand = pmap != 1
    stack = list(zip(*np.nonzero(edge)))
    while stack:
        i, j = stack.pop()
        for di in (-1, 0, 1):
            for dj in (-1, 0, 1):
                a, b = i + di, j + dj
                if 0 <= a < H and 0 <= b < W and cand[a, b] and not edge[a, b]:
                    edge[a, b] = True
                    stack.append((a, b))
    return edge


def canny(img_u8, low=100, high=200):
    """cv2.Canny(img, low, high) -> uint8 {0, 255}.  Like cv::Canny, the thresholds are floored and taken in either
    order: when low > high the two are swapped (floor is monotonic, so swapping before or after it is the same)."""
    dx, dy = sobel3(img_u8)
    lo, hi = int(np.floor(low)), int(np.floor(high))
    if lo > hi:
        lo, hi = hi, lo
    return hysteresis(nms_map(dx, dy, lo, hi)).astype(np.uint8) * 255


def canny_ivice(bgr, low=100, high=200):
    """edge.py:19-35 without the file I/O: float32 (H,W), 0.0 on an edge, 1.0 elsewhere."""
    edges = canny(blur3(gray_u8(bgr)), low, high)
    return np.array((255 - edges) / 255, dtype="float32")
