"""The reference's six OpenCV calls, restated -- TEST INFRASTRUCTURE ONLY.

The reference's CPU implementation of the path *is* this sequence of cv2 calls
(src/preprocess/ops/clahe_dehaze.py:13-32 and ops/median_derain.py:10-14); the reference is
not part of this repository, so the sequence is restated here and tests/test_oracle.py and
tests/test_reference_equivalence.py check it against outputs and coercions recorded from the reference's own classes.  Used as the live ground truth in tests and as the
`--impl reference` / cpu_baseline arm of bench.py.
"""
import cv2
import numpy as np


def coerce_clahe_params(params):
    """clahe_dehaze.py:14-17"""
    space = str(params.get("space", "YCrCb")).upper()
    clip_limit = float(params.get("clip_limit", 2.0))
    grid = max(2, int(params.get("tile_grid", 8)))
    return space, clip_limit, grid


def coerce_ksize(params):
    """median_derain.py:11-13"""
    k = int(params.get("ksize", 3))
    if k % 2 == 0:
        k += 1
    return max(3, min(k, 9))


def clahe_dehaze(image, space="YCrCb", clip_limit=2.0, tile_grid=8):
    """clahe_dehaze.py:19-30"""
    clahe = cv2.createCLAHE(clipLimit=float(clip_limit), tileGridSize=(int(tile_grid), int(tile_grid)))
    if space == "LAB":
        lab = cv2.cvtColor(image, cv2.COLOR_BGR2LAB)
        l, a, b = cv2.split(lab)
        return cv2.cvtColor(cv2.merge([clahe.apply(l), a, b]), cv2.COLOR_LAB2BGR)
    ycc = cv2.cvtColor(image, cv2.COLOR_BGR2YCrCb)
    y, cr, cb = cv2.split(ycc)
    return cv2.cvtColor(cv2.merge([clahe.apply(y), cr, cb]), cv2.COLOR_YCrCb2BGR)


def median_derain(image, ksize=3):
    """median_derain.py:14"""
    return cv2.medianBlur(image, int(ksize))


def chain(image, space="YCrCb", clip_limit=2.0, tile_grid=8, ksize=3):
    """pipeline.py:42-44 over [CLAHEDehaze, MedianDerain]; ksize 0 skips the median."""
    out = clahe_dehaze(image, space, clip_limit, tile_grid)
    return median_derain(out, ksize) if ksize else out


def low_contrast(image, thresh=20.0):
    """pipeline.py:24-30"""
    gray = cv2.cvtColor(image, cv2.COLOR_BGR2GRAY)
    return (int(gray.max()) - int(gray.min())) < float(thresh)


def letterbox_f16(image, size=640, pad_value=114):
    """Detector input as ultralytics prepares it inside model.predict (yolo_ultralytics.py:28-35): LetterBox (cv2.resize
    INTER_LINEAR + cv2.copyMakeBorder 114), BGR->RGB, HWC->CHW, /255, half.  ultralytics itself is not installed; the
    geometry follows its LetterBox with auto=False, scaleup=True, center=True."""
    h, w = image.shape[:2]
    r = min(size / h, size / w)
    nw, nh = max(1, int(round(w * r))), max(1, int(round(h * r)))
    dw, dh = (size - nw) / 2, (size - nh) / 2
    img = cv2.resize(image, (nw, nh), interpolation=cv2.INTER_LINEAR) if (w, h) != (nw, nh) else image
    top, bottom = int(round(dh - 0.1)), int(round(dh + 0.1))
    left, right = int(round(dw - 0.1)), int(round(dw + 0.1))
    img = cv2.copyMakeBorder(img, top, bottom, left, right, cv2.BORDER_CONSTANT, value=(pad_value,) * 3)
    return (np.ascontiguousarray(img[:, :, ::-1].transpose(2, 0, 1)).astype(np.float32) / np.float32(255)).astype(np.float16)
