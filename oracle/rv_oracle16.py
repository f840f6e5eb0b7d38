"""numpy restatement of the chain on 16-bit frames (cv2's CV_16U path) -- TEST INFRASTRUCTURE ONLY.

The reference hands uint16 BGR frames to cv2 unchanged (src/preprocess/ops/clahe_dehaze.py:19-30, ops/median_derain.py:10-14,
pipeline.py:24-30), and cv2 runs the stock chain in 16-bit arithmetic.  Restated here as the executable spec of the 16-bit path;
tests/test_u16.py pins every function against the live cv2:

  BGR2YCrCb   Y = D(1868 B + 9617 G + 4899 R), Cr = sat16(D((R - Y) 11682 + (32768 << 14))), Cb = sat16(D((B - Y) 9241 + (32768 << 14)))
  YCrCb2BGR   B = sat16(Y + D((Cb - 32768) 29049)), G = sat16(Y + D((Cb - 32768)(-5636) + (Cr - 32768)(-11698))),
              R = sat16(Y + D((Cr - 32768) 22987));  D(x) = (x + 8192) >> 14
  BGR2GRAY    (3735 B + 19235 G + 9798 R + 16384) >> 15 (the 8-bit coefficients of SURVEY.md A.5)
  CLAHE       SURVEY.md A.3 with histSize 65536: clip = max(1, int(clip_limit * area / 65536)) when clip_limit > 0,
              batch = clipped / 65536, step = max(65536 / residual, 1), lutScale = float32(65535) / float32(area), 16-bit saturation
  medianBlur  exact k x k median per channel, BORDER_REPLICATE, k in {3, 5} (cv2 has no 16-bit k 7 / 9)

The CLAHE never materialises the grid^2 x 65,536 table (512 MB at grid 64): a tile's LUT at value v is its clipped cumulative
histogram, which is the capped counts of the values present up to v (one sorted array over all tiles) plus the closed forms of the
uniform batch, batch * (v + 1), and of the residual redistribution, min(v / step + 1, residual).  All float32 operations are
numpy's, each rounded on its own (no FMA contraction), as cv2's scalar code.
"""
import numpy as np

HIST = 65536


def _d(x):
    return (x + 8192) >> 14


def _u16(a):
    a = np.asarray(a)
    if a.dtype != np.uint16:
        raise TypeError("uint16 expected")
    return a


def bgr2ycrcb16(img):
    img = _u16(img)
    B, G, R = (img[..., i].astype(np.int64) for i in range(3))
    Y = _d(1868 * B + 9617 * G + 4899 * R)
    Cr = np.clip(_d((R - Y) * 11682 + (32768 << 14)), 0, 65535)
    Cb = np.clip(_d((B - Y) * 9241 + (32768 << 14)), 0, 65535)
    return np.stack([Y, Cr, Cb], -1).astype(np.uint16)


def ycrcb2bgr16(img):
    img = _u16(img)
    Y, Cr, Cb = (img[..., i].astype(np.int64) for i in range(3))
    Cr, Cb = Cr - 32768, Cb - 32768
    b = Y + _d(Cb * 29049)
    g = Y + _d(Cb * -5636 + Cr * -11698)
    r = Y + _d(Cr * 22987)
    return np.clip(np.stack([b, g, r], -1), 0, 65535).astype(np.uint16)


def bgr2gray16(img):
    img = _u16(img)
    B, G, R = (img[..., i].astype(np.int64) for i in range(3))
    return ((3735 * B + 19235 * G + 9798 * R + 16384) >> 15).astype(np.uint16)


def gray_span16(img):
    g = bgr2gray16(img)
    return int(g.max()) - int(g.min())


def _reflect101(p, n):
    """OpenCV borderInterpolate(p, n, BORDER_REFLECT_101) for an index array."""
    p = np.asarray(p, np.int64)
    if n == 1:
        return np.zeros_like(p)
    period = 2 * (n - 1)
    p = np.abs(p) % period
    return np.where(p >= n, period - p, p)


def clahe_geometry(H, W, grid):
    """clahe.cpp: both dimensions are padded when either is not divisible by the grid (A.3)"""
    eh, ew = H, W
    if W % grid or H % grid:
        ew, eh = W + (grid - W % grid), H + (grid - H % grid)
    return ew // grid, eh // grid


class _Luts:
    """The LUTs of every tile of a plane, evaluated on demand at (tile, value) pairs."""

    def __init__(self, plane, grid, clip_limit):
        H, W = plane.shape
        tw, th = clahe_geometry(H, W, grid)
        self.grid, area = grid, tw * th
        ys, xs = _reflect101(np.arange(grid * th), H), _reflect101(np.arange(grid * tw), W)
        ext = plane[ys][:, xs].astype(np.int64)
        tid = (np.arange(grid * th) // th)[:, None] * grid + (np.arange(grid * tw) // tw)[None, :]
        self.keys, cnt = np.unique(tid * HIST + ext, return_counts=True)
        T = grid * grid
        tile_of = self.keys // HIST
        clip = max(1, int(clip_limit * area / HIST)) if clip_limit > 0 else 0
        capped = np.minimum(cnt, clip) if clip else cnt
        clipped = np.bincount(tile_of, weights=(cnt - capped).astype(np.float64), minlength=T).astype(np.int64)
        self.batch = clipped // HIST
        self.residual = clipped - self.batch * HIST
        self.step = np.maximum(HIST // np.maximum(self.residual, 1), 1)
        self.cc = np.cumsum(capped)
        self.first = np.searchsorted(self.keys, np.arange(T, dtype=np.int64) * HIST)
        self.base = np.where(self.first > 0, self.cc[np.maximum(self.first - 1, 0)], 0)
        self.scale = np.float32(65535) / np.float32(area)

    def __call__(self, t, v):
        t, v = np.asarray(t, np.int64), np.asarray(v, np.int64)
        idx = np.searchsorted(self.keys, t * HIST + v, side="right") - 1
        s = np.where(idx >= self.first[t], self.cc[np.maximum(idx, 0)] - self.base[t], 0)
        s = s + self.batch[t] * (v + 1)
        res = self.residual[t]
        s = s + np.where(res > 0, np.minimum(v // self.step[t] + 1, res), 0)
        return np.clip(np.rint(s.astype(np.float32) * self.scale), 0, 65535).astype(np.int64)


def clahe16_tile_lut(plane, grid, clip_limit, ty, tx):
    """The 65,536-entry u16 LUT of tile (ty, tx) that cv2's 16-bit CLAHE builds (and never exposes)."""
    plane = _u16(plane)
    luts = _Luts(plane, grid, clip_limit)
    return luts(np.full(HIST, ty * grid + tx), np.arange(HIST)).astype(np.uint16)


def _axis(n, tiles, size):
    """A.3 interpolation terms along one axis, float32 with every operation rounded: (i1, i2, a, a1)"""
    inv = np.float32(1.0) / np.float32(size)
    f = np.arange(n).astype(np.float32) * inv
    f = f - np.float32(0.5)
    i1 = np.floor(f).astype(np.int64)
    a = f - i1.astype(np.float32)
    a1 = np.float32(1.0) - a
    return np.maximum(i1, 0), np.minimum(i1 + 1, tiles - 1), a, a1


def clahe16_plane(plane, clip_limit, grid):
    """cv2.createCLAHE(clip_limit, (grid, grid)).apply(plane) for a uint16 plane"""
    plane = _u16(plane)
    H, W = plane.shape
    tw, th = clahe_geometry(H, W, grid)
    luts = _Luts(plane, grid, clip_limit)
    ty1, ty2, ya, ya1 = _axis(H, grid, th)
    tx1, tx2, xa, xa1 = _axis(W, grid, tw)
    v = plane.astype(np.int64)
    l00 = luts(ty1[:, None] * grid + tx1[None, :], v).astype(np.float32)
    l01 = luts(ty1[:, None] * grid + tx2[None, :], v).astype(np.float32)
    l10 = luts(ty2[:, None] * grid + tx1[None, :], v).astype(np.float32)
    l11 = luts(ty2[:, None] * grid + tx2[None, :], v).astype(np.float32)
    top = l00 * xa1[None, :] + l01 * xa[None, :]
    bot = l10 * xa1[None, :] + l11 * xa[None, :]
    res = top * ya1[:, None] + bot * ya[:, None]
    return np.clip(np.rint(res), 0, 65535).astype(np.uint16)


def median16(img, k):
    """cv2.medianBlur(img, k) for uint16 (H,W) or (H,W,C), k in {3, 5}"""
    if k not in (3, 5):
        raise ValueError("cv2 has a 16-bit median for k = 3 and 5 only")
    img = _u16(img)
    squeeze = img.ndim == 2
    a = img[..., None] if squeeze else img
    r = k // 2
    pad = np.pad(a, ((r, r), (r, r), (0, 0)), mode="edge")
    out = np.empty_like(a)
    for y0 in range(0, a.shape[0], 64):            # bounded memory: 64 output rows at a time
        y1 = min(y0 + 64, a.shape[0])
        win = np.lib.stride_tricks.sliding_window_view(pad[y0:y1 + 2 * r], (k, k), axis=(0, 1))
        win = win.reshape(y1 - y0, a.shape[1], a.shape[2], k * k)
        out[y0:y1] = np.partition(win, k * k // 2, axis=-1)[..., k * k // 2]
    return out[..., 0] if squeeze else out


def clahe_dehaze16(img, clip_limit, grid):
    """CLAHEDehaze (YCrCb) on a uint16 BGR frame"""
    ycc = bgr2ycrcb16(img)
    ycc[..., 0] = clahe16_plane(np.ascontiguousarray(ycc[..., 0]), clip_limit, grid)
    return ycrcb2bgr16(ycc)


def chain16(img, clip_limit, grid, ksize):
    """CLAHEDehaze (YCrCb) -> MedianDerain on a uint16 BGR frame; ksize 0 = no median"""
    if ksize not in (0, 3, 5):
        raise ValueError("cv2 has a 16-bit median for k = 3 and 5 only")
    out = clahe_dehaze16(img, clip_limit, grid)
    return median16(out, ksize) if ksize else out
