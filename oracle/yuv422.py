"""numpy restatement of cv2.cvtColor(COLOR_YUV2BGR_YUY2 / COLOR_YUV2BGR_UYVY) on cv2's packed 4:2:2 frames.

A (H, W, 2) uint8 frame holds, in each row, W/2 groups of 4 bytes, one per horizontal pixel pair (x = 2i, 2i + 1): YUY2 Y0 U Y1 V,
UYVY U Y0 V Y1.  The two pixels of a pair share its (U, V); the arithmetic is that of oracle/yuv420.py (BT.601 video range, 20-bit fixed
point), which csrc/rv_yuv422.cu computes too.
"""
import numpy as np

from .yuv420 import CUB, CUG, CVG, CVR, CY, SHIFT

# byte offsets of Y0, U, Y1, V in a pixel pair's group
ORDER = {"YUY2": (0, 1, 2, 3), "UYVY": (1, 0, 3, 2)}


def planes(frame, layout):
    """(Y (H,W), U (H,W/2), V (H,W/2)) of one (H, W, 2) frame; layout "YUY2" or "UYVY"."""
    h, w, _ = frame.shape
    g = frame.reshape(h, w // 2, 4)
    y0, u, y1, v = (g[..., k] for k in ORDER[layout])
    return np.stack([y0, y1], -1).reshape(h, w), u, v


def from_planes(y, u, v, layout):
    """The (H, W, 2) frame of planes Y (H,W), U and V (H,W/2)."""
    h, w = y.shape
    yp = y.reshape(h, w // 2, 2)
    g = np.empty((h, w // 2, 4), np.uint8)
    for k, p in zip(ORDER[layout], (yp[..., 0], u, yp[..., 1], v)):
        g[..., k] = p
    return g.reshape(h, w, 2)


def yuv422_to_bgr(frame, layout):
    """(H, W, 2) uint8 -> (H, W, 3) uint8 BGR, as cv2."""
    y, u, v = planes(frame, layout)
    u = np.repeat(u.astype(np.int32) - 128, 2, 1)
    v = np.repeat(v.astype(np.int32) - 128, 2, 1)
    half = 1 << (SHIFT - 1)
    ruv, guv, buv = half + CVR * v, half + CVG * v + CUG * u, half + CUB * u
    yy = np.maximum(0, y.astype(np.int32) - 16) * CY
    return np.stack([np.clip((yy + t) >> SHIFT, 0, 255) for t in (buv, guv, ruv)], -1).astype(np.uint8)


def every_triple(layout):
    """One 4096 x 4096 frame that holds each of the 2^24 (Y, U, V) triples exactly once: pixel pair k (row-major over the 4096 x 2048
    pairs) carries U = k & 255, V = (k >> 8) & 255 and Y = 2 (k >> 16) + (0, 1)."""
    k = np.arange(1 << 23, dtype=np.int64).reshape(4096, 2048)
    y = np.stack([2 * (k >> 16), 2 * (k >> 16) + 1], -1).reshape(4096, 4096)
    return from_planes(y.astype(np.uint8), (k & 255).astype(np.uint8), ((k >> 8) & 255).astype(np.uint8), layout)
