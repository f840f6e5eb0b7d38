"""numpy restatement of cv2.cvtColor(COLOR_YUV2BGR_NV12 / COLOR_YUV2BGR_I420) on cv2's single-array 4:2:0 frames.

A (3H/2, W) uint8 frame holds H rows of Y and then the chroma: NV12 interleaves U, V bytes (U first) in H/2 rows of the same pitch;
I420 packs W*H/4 bytes of U and then W*H/4 bytes of V.  Every 2 x 2 block of Y shares one (U, V) pair; the arithmetic is BT.601 video
range in 20-bit fixed point, all of it within int32 (csrc/rv_yuv.cu computes the same).
"""
import numpy as np

CY, CUB, CUG, CVG, CVR, SHIFT = 1220542, 2116026, -409993, -852492, 1673527, 20


def planes(frame, layout):
    """(Y (H,W), U (H/2,W/2), V (H/2,W/2)) of one (3H/2, W) frame; layout "NV12" or "I420"."""
    rows, w = frame.shape
    h = rows // 3 * 2
    y = frame[:h]
    if layout == "NV12":
        uv = frame[h:].reshape(h // 2, w // 2, 2)
        return y, uv[..., 0], uv[..., 1]
    c = np.ascontiguousarray(frame[h:]).reshape(-1)
    q = (h // 2) * (w // 2)
    return y, c[:q].reshape(h // 2, w // 2), c[q:].reshape(h // 2, w // 2)


def from_planes(y, u, v, layout):
    """The (3H/2, W) frame of planes Y (H,W), U and V (H/2,W/2)."""
    h, w = y.shape
    if layout == "NV12":
        chroma = np.stack([u, v], -1).reshape(h // 2, w)
    else:
        chroma = np.concatenate([u.reshape(-1), v.reshape(-1)]).reshape(h // 2, w)
    return np.concatenate([y, chroma]).astype(np.uint8)


def yuv420_to_bgr(frame, layout):
    """(3H/2, W) uint8 -> (H, W, 3) uint8 BGR, as cv2."""
    y, u, v = planes(frame, layout)
    u = np.repeat(np.repeat(u.astype(np.int32) - 128, 2, 0), 2, 1)
    v = np.repeat(np.repeat(v.astype(np.int32) - 128, 2, 0), 2, 1)
    half = 1 << (SHIFT - 1)
    ruv, guv, buv = half + CVR * v, half + CVG * v + CUG * u, half + CUB * u
    yy = np.maximum(0, y.astype(np.int32) - 16) * CY
    return np.stack([np.clip((yy + t) >> SHIFT, 0, 255) for t in (buv, guv, ruv)], -1).astype(np.uint8)


def every_triple(layout):
    """One 4096 x 4096 frame that holds each of the 2^24 (Y, U, V) triples exactly once: chroma block k (row-major over the 2048 x
    2048 blocks) carries U = k & 255, V = (k >> 8) & 255 and the four Y values 4 (k >> 16) + (0, 1, 2, 3)."""
    k = np.arange(1 << 22, dtype=np.int64).reshape(2048, 2048)
    u, v, g = k & 255, (k >> 8) & 255, k >> 16
    y = np.empty((4096, 4096), np.int64)
    for dy in (0, 1):
        for dx in (0, 1):
            y[dy::2, dx::2] = 4 * g + 2 * dy + dx
    return from_planes(y, u, v, layout)
