"""MedianDerain -- drop-in for /root/reference/src/preprocess/ops/median_derain.py:4-14."""
from ..._native import Params, check_frame_params, default_context
from ..base import PreprocessOp, as_frame


def coerce(params):
    """median_derain.py:11-13: int, even -> +1, clamp to [3, 9]."""
    k = int(params.get("ksize", 3))
    if k % 2 == 0:
        k += 1
    return max(3, min(k, 9))


class MedianDerain(PreprocessOp):
    """k x k median per channel, BORDER_REPLICATE (cv2.medianBlur semantics). params: ksize 3/5/7/9 (3/5 on uint16 frames, as cv2).
    BGR, BGRA (alpha filtered too) and single-channel frames; a single channel comes back as (H,W), as from cv2."""

    def __call__(self, image):
        k = coerce(self.params)
        img = as_frame(image)
        check_frame_params(Params.make(ksize=k, clahe=False), img.dtype, img.shape[2])        # k 7 / 9 at 16 bits: before the GPU
        ctx = default_context(self.params.get("device"))
        out = ctx.median(img[None], k)[0]
        return out[..., 0] if out.shape[2] == 1 else out
