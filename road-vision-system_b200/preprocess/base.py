"""Operator base class -- same contract as /root/reference/src/preprocess/base.py:4-16."""
from abc import ABC, abstractmethod
from typing import Any

import numpy as np


class PreprocessOp(ABC):
    """`op(image) -> image`; image is BGR (H,W,3) uint8 (or uint16); unknown params are kept and ignored."""

    def __init__(self, **params: Any):
        self.params = params

    @abstractmethod
    def __call__(self, image):
        pass


def as_bgr_u8(image):
    """Validate the per-frame contract (SURVEY.md 8b): (H,W,3) uint8, any strides.

    The reference hands the array to cv2, which accepts strided / read-only / Fortran-order
    views and fails with cv2.error on other shapes or dtypes; here those failures are
    ValueError / TypeError raised before anything touches the GPU.
    """
    if not isinstance(image, np.ndarray):
        raise TypeError(f"image must be a numpy.ndarray, got {type(image).__name__}")
    if image.dtype != np.uint8:
        raise ValueError(f"image must be uint8, got {image.dtype}")
    if image.ndim != 3 or image.shape[2] != 3:
        raise ValueError(f"image must have shape (H,W,3), got {image.shape}")
    if image.shape[0] < 1 or image.shape[1] < 1:
        raise ValueError("empty image")
    return np.ascontiguousarray(image)


def as_bgr_frame(image):
    """as_bgr_u8, but also admitting (H,W,3) uint16 frames (HDR sensors, cv2.imread(..., IMREAD_ANYDEPTH)), which the reference
    hands to cv2's 16-bit path unchanged.  Any strides; returns a C-contiguous array of the input's dtype."""
    if isinstance(image, np.ndarray) and image.dtype == np.uint16:
        if image.ndim != 3 or image.shape[2] != 3:
            raise ValueError(f"image must have shape (H,W,3), got {image.shape}")
        if image.shape[0] < 1 or image.shape[1] < 1:
            raise ValueError("empty image")
        return np.ascontiguousarray(image)
    return as_bgr_u8(image)


def as_frame(image):
    """as_bgr_frame, but also admitting what cv2 accepts beyond BGR: (H,W,4) BGRA / BGRx frames (cv2.imread(..., IMREAD_UNCHANGED) on
    PNGs with alpha, video decoder surfaces) and single-channel (H,W) or (H,W,1) frames (monochrome, NIR and thermal cameras), uint8
    or uint16, any strides.  Returns a C-contiguous (H,W,C) array (a single channel as (H,W,1)) of the input's dtype."""
    if isinstance(image, np.ndarray) and image.dtype in (np.uint8, np.uint16) and \
            (image.ndim == 2 or (image.ndim == 3 and image.shape[2] in (1, 4))):
        if image.shape[0] < 1 or image.shape[1] < 1:
            raise ValueError("empty image")
        return np.ascontiguousarray(image.reshape(image.shape[0], image.shape[1], -1))
    return as_bgr_frame(image)
