"""CLAHEDehaze -- drop-in for /root/reference/src/preprocess/ops/clahe_dehaze.py:4-32.

Same name, params and per-frame contract; the cv2.cvtColor / split / createCLAHE().apply /
merge / cvtColor sequence (:19-30) runs as the sm_100a kernels behind rv_clahe_dehaze.
"""
from ..._native import Params, check_frame_params, default_context
from ..base import PreprocessOp, as_frame


def coerce(params):
    """clahe_dehaze.py:14-17 -- evaluated on every call, so mutating op.params takes effect."""
    space = str(params.get("space", "YCrCb")).upper()
    clip_limit = float(params.get("clip_limit", 2.0))
    grid = max(2, int(params.get("tile_grid", 8)))
    return ("LAB" if space == "LAB" else "YCrCb"), clip_limit, grid


class CLAHEDehaze(PreprocessOp):
    """CLAHE on the luminance channel. params: space "YCrCb"|"LAB", clip_limit float, tile_grid int.

    uint16 frames run cv2's 16-bit chain (65,536-bin histograms) in YCrCb with tile_grid <= 64; LAB raises ValueError there, as
    cv2 has no 16-bit LAB.  (H,W,4) BGRA frames give a (H,W,3) result, as cv2.cvtColor ignores and drops alpha; single-channel
    frames raise ValueError (cv2 has no colour conversion for them)."""

    def __call__(self, image):
        space, clip_limit, grid = coerce(self.params)
        img = as_frame(image)
        # LAB / grid > 64 at 16 bits, a single channel: before the GPU
        check_frame_params(Params.make(space, clip_limit, grid, 0, clahe=True), img.dtype, img.shape[2])
        ctx = default_context(self.params.get("device"))
        return ctx.clahe_dehaze(img[None], space, clip_limit, grid)[0]
