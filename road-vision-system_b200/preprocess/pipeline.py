"""PreprocessPipeline -- drop-in for /root/reference/src/preprocess/pipeline.py:7-45.

Same constructor (`enabled`, `chain`, `auto_gate`), same `pipeline(image, ts=None)` call.
Differences are internal: an adjacent CLAHEDehaze -> MedianDerain pair is dispatched as ONE
fused GPU pass (the ops stay individually callable), and `process_batch` is the new
multi-frame entry (no reference counterpart; the reference loop keeps one frame in flight,
main_preview.py:88-142).
"""
from typing import Any, Dict

import numpy as np

from .._native import (DeviceArray, Params, _check_torch_out, _torch_stream, check_bgr_for_yuv, check_frame_params, check_out_yuv,
                       check_u16_params, check_yuv_frames, default_context)
from .base import as_bgr_frame, as_frame
from .ops import CLAHEDehaze, MedianDerain
from .ops import clahe_dehaze as _clahe
from .ops import median_derain as _median
from .registry import get_op_class


def _is_cuda_tensor(x):
    return type(x).__module__.startswith("torch") and hasattr(x, "is_cuda") and x.is_cuda


class PreprocessPipeline:
    def __init__(self, config: Dict[str, Any], context=None):
        """`config`: the reference's `preprocess:` dict (pipeline.py:13-22).  `context` (new, optional): the rvb200.Context
        this pipeline runs on -- give every camera stream / worker thread its own (a context is not thread-safe);
        without it the process-wide default context of `config["device"]` is used."""
        self._context = context
        self._snap = None
        self.enabled = bool(config.get("enabled", True))
        self.chain_cfg = config.get("chain", []) or []
        self.auto_gate_cfg = config.get("auto_gate", {}) or {}
        self.device = config.get("device")          # optional new key; the stock YAML does not set it
        self.ops = []
        for node in self.chain_cfg:
            name = node.get("name")
            params = node.get("params", {})
            cls = get_op_class(name)
            self.ops.append(cls(**params))

    # -- helpers -------------------------------------------------------------------------
    def _ctx(self):
        return self._context if self._context is not None else default_context(self.device)

    def _gate(self):
        enable = bool(self.auto_gate_cfg.get("enable_low_contrast_gate", False))
        return enable, float(self.auto_gate_cfg.get("contrast_thresh", 20.0))

    def _low_contrast(self, image) -> bool:
        """pipeline.py:24-30: gray span < thresh (gray = cv2 BGR2GRAY fixed point, computed on the GPU; BGRA: alpha ignored)."""
        span = int(self._ctx().gray_span(as_frame(image)[None])[0])
        return span < self._gate()[1]

    def _segments(self):
        """Fold the op list into fused GPU passes: [(Params | op)].  Params are re-read on every call, like the reference
        (clahe_dehaze.py:14-17, median_derain.py:11-13: mutating `op.params` between frames takes effect); the folded result
        is reused for as long as the op objects and their params dicts compare equal to the snapshot it was built from."""
        snap = self._snap
        ops = self.ops
        if snap is not None and len(snap[0]) == len(ops):
            for (op0, params0), op in zip(snap[0], ops):
                if op0 is not op or params0 != op.params:
                    break
            else:
                for sg in snap[1]:
                    if isinstance(sg, Params):
                        sg.gate_enable = 0
                return snap[1]
        segs = self._fold()
        self._snap = ([(op, dict(op.params)) for op in ops], segs)
        return segs

    def _fold(self):
        segs, i = [], 0
        while i < len(self.ops):
            op = self.ops[i]
            nxt = self.ops[i + 1] if i + 1 < len(self.ops) else None
            if type(op).__call__ is CLAHEDehaze.__call__ and nxt is not None and type(nxt).__call__ is MedianDerain.__call__:
                space, clip, grid = _clahe.coerce(op.params)
                segs.append(Params.make(space, clip, grid, _median.coerce(nxt.params), clahe=True))
                i += 2
            elif type(op).__call__ is CLAHEDehaze.__call__:
                space, clip, grid = _clahe.coerce(op.params)
                segs.append(Params.make(space, clip, grid, 0, clahe=True))
                i += 1
            elif type(op).__call__ is MedianDerain.__call__:
                segs.append(Params.make(ksize=_median.coerce(op.params), clahe=False))
                i += 1
            else:
                segs.append(op)         # foreign operator: called as in the reference
                i += 1
        return segs

    @staticmethod
    def _check_u16(segs):
        """16-bit frames: every fused GPU pass must have a 16-bit path (YCrCb, k 3 / 5, grid <= 64) -- checked before any frame
        reaches the GPU, so that a LAB / k 7 / 9 chain fails with ValueError instead of after the gate or a foreign operator ran."""
        for sg in segs:
            if isinstance(sg, Params):
                check_u16_params(sg)

    def _check_channels(self, segs, dtype, channels):
        """What cv2 would reject on (..., channels) frames -- the gate or a CLAHE pass on a single channel -- raises ValueError before
        any frame reaches the GPU.  Channel counts are followed through the GPU passes (CLAHE gives 3) up to the first foreign
        operator, whose output is unknown until it runs.  Returns the channel count after the passes, or None if a foreign op
        decides it."""
        if self._gate()[0]:
            check_frame_params(Params.make(clahe=False, ksize=3, gate=True), dtype, channels)
        for sg in segs:
            if not isinstance(sg, Params):
                return None
            channels = check_frame_params(sg, dtype, channels)
        return channels

    def _pass(self, image, seg, **kw):
        """One fused GPU pass on one frame; a single-channel result comes back as (H,W), as from cv2."""
        out = self._ctx().chain(as_frame(image)[None], seg, **kw)[0]
        return out[..., 0] if out.shape[2] == 1 else out

    # -- per-frame contract --------------------------------------------------------------
    def __call__(self, image: np.ndarray, ts: float = None) -> np.ndarray:
        if not self.enabled or not self.ops:
            return image
        segs = self._segments()
        if isinstance(image, np.ndarray) and image.dtype != np.uint8 and image.dtype == np.uint16:
            self._check_u16(segs)
        frame = image
        if self._gate()[0] or isinstance(segs[0], Params):
            frame = as_frame(image)
            self._check_channels(segs, frame.dtype, frame.shape[2])
        if self._gate()[0]:
            if len(segs) == 1 and isinstance(segs[0], Params):
                # one fused pass: the gate's gray span comes out of the histogram pass of the same upload
                seg = segs[0]
                seg.gate_enable, seg.gate_thresh = 1, self._gate()[1]
                flag = np.ones(1, np.int32)
                out = self._pass(frame, seg, processed=flag)
                return out if flag[0] else image          # skipped: the input object itself, as pipeline.py:39-40
            if not self._low_contrast(frame):
                return image
        out = image
        for seg in segs:
            if isinstance(seg, Params):
                out = self._pass(out, seg)
            else:
                out = seg(out)
        return out

    # -- new: batched multi-frame entry --------------------------------------------------
    def process_batch(self, frames: np.ndarray, out: np.ndarray = None, yuv: str = None, out_yuv: str = None) -> np.ndarray:
        """(B,H,W,3) uint8 -> (B,H,W,3) uint8; equals B per-frame calls bit for bit.  uint16 frames give uint16 results (cv2's
        16-bit chain: YCrCb only, median k 3 / 5, tile_grid <= 64).

        `yuv="NV12"` / `"I420"`: `frames` are a decoder's (B,3H/2,W) uint8 4:2:0 frames; the result is exactly that of this call on
        their cv2.cvtColor(COLOR_YUV2BGR_NV12 / _I420) conversion, (B,H,W,3) BGR.  The conversion runs on the GPU; with the stock
        chain (one fused pass, with or without the gate) only the YUV bytes cross PCIe.

        `yuv="YUY2"` / `"UYVY"`: `frames` are a camera's (B,H,W,2) uint8 packed 4:2:2 frames (the array cv2.cvtColor takes; each row
        holds W/2 groups of 4 bytes, one per pixel pair: YUY2 Y0 U Y1 V, UYVY U Y0 V Y1); the result is exactly that of this call on
        their cv2.cvtColor(COLOR_YUV2BGR_YUY2 / _UYVY) conversion.  W must be even, H may be odd.  Routed as the 4:2:0 input is: with
        the stock chain only their 2 bytes per pixel cross PCIe.

        `out_yuv="NV12"` / `"I420"` (8-bit BGR or `yuv=` frames): the result comes back as (B,3H/2,W) uint8 4:2:0 frames for a video
        encoder, exactly cv2.cvtColor(COLOR_BGR2YUV_I420) of the BGR result this call returns without it (NV12: its U and V planes
        interleaved, U first) -- frames the gate skips included, so a 4:2:0 frame that is not processed comes back re-encoded, not as
        its input bytes.  The conversion runs on the GPU; with the stock chain only the 4:2:0 bytes cross PCIe on the way back.

        `frames` / `out` may be pinned arrays from `Context.pinned_empty` (fastest: H2D, kernels
        and D2H of consecutive chunks overlap).  Frames the low-contrast gate skips are copied
        through unchanged.  `out="device"` keeps the result on the GPU (a `DeviceArray`, usable from torch / cupy through
        `__cuda_array_interface__`): nothing is copied back, which is what a detector on the same GPU wants
        (main_preview.py:99).
        """
        if out_yuv is not None:
            return self._process_batch_yuv_out(frames, out, yuv, out_yuv)
        if yuv is not None:
            return self._process_batch_yuv(frames, out, yuv)
        if _is_cuda_tensor(frames):
            return self._process_batch_device(frames, out)
        if isinstance(out, str):
            if out != "device":
                raise ValueError('out must be an array, None or "device"')
            return self._process_batch_keep(frames)
        if not isinstance(frames, np.ndarray) or frames.ndim != 4 or frames.shape[3] not in (1, 3, 4) or \
                (frames.dtype != np.uint8 and frames.dtype != np.uint16):
            raise ValueError("frames must be a (B,H,W,C) uint8 or uint16 numpy array with C = 1 (gray), 3 (BGR) or 4 (BGRA) (or a torch "
                             "CUDA tensor of that shape)")
        if frames.dtype == np.uint16 and self.enabled and self.ops:
            self._check_u16(self._segments())
        if self.enabled and self.ops:
            self._check_batch_channels(self._segments(), frames.dtype, frames.shape[3])
        if not self.enabled or not self.ops:
            if out is None:
                return frames
            np.copyto(out, frames)
            return out
        ctx = self._ctx()
        gate, thresh = self._gate()
        cur = frames
        segs = self._segments()
        if gate and not (len(segs) == 1 and isinstance(segs[0], Params)):
            # general case: decide per frame up front, run the chain on the selected frames only
            span = ctx.gray_span(np.ascontiguousarray(frames))
            sel = np.flatnonzero(span < thresh)
            res = np.array(frames, copy=True) if out is None else out
            if out is not None:
                np.copyto(out, frames)
            if len(sel):
                sub = np.ascontiguousarray(frames[sel])
                for seg in segs:
                    sub = ctx.chain(sub, seg) if isinstance(seg, Params) else np.stack([seg(f) for f in sub])
                res[sel] = sub
            return res
        for idx, seg in enumerate(segs):
            last = idx == len(segs) - 1
            if isinstance(seg, Params):
                if gate:
                    seg.gate_enable, seg.gate_thresh = 1, thresh
                cur = ctx.chain(cur, seg, out=out if last else None)
            else:
                cur = np.stack([seg(f) for f in cur])
                if last and out is not None:
                    np.copyto(out, cur)
                    cur = out
        return cur

    def _fused_segment(self):
        """The single fused GPU pass the chain folds to (the stock config), or None."""
        segs = self._segments() if (self.enabled and self.ops) else []
        return segs[0] if len(segs) == 1 and isinstance(segs[0], Params) else None

    def _device_ctx(self, frames):
        return self._context if (self._context is not None and self._context.device == frames.device.index) \
            else default_context(frames.device.index)

    def _process_batch_yuv(self, frames, out, yuv):
        """process_batch on (B,3H/2,W) 4:2:0 or (B,H,W,2) 4:2:2 frames.  One fused pass: host frames go through rv_submit_io_fmt (the
        YUV bytes are uploaded and converted in the pipeline's BGR workspace).  Anything else converts on the GPU first and takes the
        BGR path."""
        if _is_cuda_tensor(frames):
            import torch
            _, b, h, w = check_yuv_frames(frames.shape, frames.dtype == torch.uint8, yuv)
            if not frames.is_contiguous():
                raise ValueError("frames must be a contiguous CUDA tensor")
            # everything the device path would refuse is refused before the conversion is enqueued
            self._check_device_chain()
            _check_torch_out(out, (b, h, w, 3), torch.uint8, frames.device,
                             f"out must be a contiguous uint8 CUDA tensor of shape {(b, h, w, 3)} on the input's device")
            return self._process_batch_device(self._device_ctx(frames)._convert(frames, yuv, None), out)
        if isinstance(out, str) and out != "device":
            raise ValueError('out must be an array, None or "device"')
        if not isinstance(frames, np.ndarray):
            raise ValueError(f"yuv={yuv!r} takes a uint8 numpy array or torch CUDA tensor")
        _, b, h, w = check_yuv_frames(frames.shape, frames.dtype == np.uint8, yuv)
        shape = (b, h, w, 3)
        if out is not None and not isinstance(out, str) and not (isinstance(out, np.ndarray) and out.shape == shape and
                                                                 out.dtype == np.uint8 and out.flags.c_contiguous):
            raise ValueError(f"out must be a C-contiguous uint8 array of shape {shape}")
        ctx = self._ctx()
        seg = self._fused_segment()
        if seg is None:
            bgr = ctx._convert(frames, yuv, None)
            return self._process_batch_keep(bgr) if isinstance(out, str) else self.process_batch(bgr, out)
        gate, thresh = self._gate()
        if gate:
            seg.gate_enable, seg.gate_thresh = 1, thresh
        if isinstance(out, str):
            res = DeviceArray(ctx, shape)
        elif out is not None:
            res = out
        else:
            res = ctx._host_result(shape)
        ctx.submit_io(np.ascontiguousarray(frames), seg, out=res, yuv=yuv)
        ctx.wait()
        return res

    def _process_batch_yuv_out(self, frames, out, yuv, out_yuv):
        """process_batch with 4:2:0 results.  Host frames with the stock chain (one fused pass) go through rv_submit_io_fmt: each
        chunk's BGR result is converted on the GPU and only the 4:2:0 bytes are copied back.  Anything else computes the BGR result as
        process_batch does and converts it on the GPU.  Every refusal comes before a context is made or work is enqueued."""
        check_out_yuv(out_yuv)
        tensor = _is_cuda_tensor(frames)
        if not tensor and not isinstance(frames, np.ndarray):
            raise ValueError("frames must be a numpy array or a torch CUDA tensor")
        if tensor:
            import torch
            u8 = frames.dtype == torch.uint8
        else:
            u8 = frames.dtype == np.uint8
        if yuv is not None:
            _, b, h, w = check_yuv_frames(frames.shape, u8, yuv)
            if h % 2:           # (4:2:2 frames may have an odd height)
                raise ValueError(f"4:2:0 output needs an even height and width, got {h}x{w}")
        else:
            _, b, h, w = check_bgr_for_yuv(frames.shape, u8, out_yuv)
        shape = (b, h * 3 // 2, w)
        if tensor:
            if not frames.is_contiguous():
                raise ValueError("frames must be a contiguous CUDA tensor")
            _check_torch_out(out, shape, torch.uint8, frames.device,
                             f"out must be a contiguous uint8 CUDA tensor of shape {shape} on the input's device")
            self._check_device_chain()
            ctx = self._device_ctx(frames)
            bgr = ctx._convert(frames, yuv, None) if yuv is not None else frames
            return ctx.bgr_to_yuv420(self._process_batch_device(bgr), out_yuv, out=out)
        if isinstance(out, str) and out != "device":
            raise ValueError('out must be an array, None or "device"')
        if out is not None and not isinstance(out, str) and not (isinstance(out, np.ndarray) and out.shape == shape and
                                                                 out.dtype == np.uint8 and out.flags.c_contiguous):
            raise ValueError(f"out must be a C-contiguous uint8 array of shape {shape}")
        ctx = self._ctx()
        seg = self._fused_segment()
        if seg is None:
            if isinstance(out, str):
                return ctx.bgr_to_yuv420(self.process_batch(frames, out="device", yuv=yuv), out_yuv)
            return ctx.bgr_to_yuv420(self.process_batch(frames, yuv=yuv), out_yuv, out=out)
        gate, thresh = self._gate()
        if gate:
            seg.gate_enable, seg.gate_thresh = 1, thresh
        if isinstance(out, str):
            res = DeviceArray(ctx, shape)
        elif out is not None:
            res = out
        else:
            res = ctx._host_result(shape)
        ctx.submit_io(np.ascontiguousarray(frames), seg, out=res, yuv=yuv, out_yuv=out_yuv)
        ctx.wait()
        return res

    def _check_batch_channels(self, segs, dtype, channels):
        """_check_channels for a batch, which must have one result shape: with the gate, a CLAHE pass on BGRA frames would give
        3-channel processed frames next to 4-channel skipped ones."""
        self._check_channels(segs, dtype, channels)
        if self._gate()[0] and channels == 4 and any(isinstance(sg, Params) and sg.clahe for sg in segs):
            raise ValueError("the low-contrast gate with CLAHEDehaze on BGRA batches would mix 3-channel (processed) and 4-channel "
                             "(skipped) frames; call the pipeline per frame, or drop alpha first")

    def _process_batch_keep(self, frames):
        """Host frames in, result left on the GPU (no D2H at all)."""
        if not isinstance(frames, np.ndarray) or frames.ndim != 4 or frames.shape[3] not in (1, 3, 4) or \
                (frames.dtype != np.uint8 and frames.dtype != np.uint16):
            raise ValueError("frames must be a (B,H,W,C) uint8 or uint16 numpy array with C = 1, 3 or 4")
        segs = self._segments() if (self.enabled and self.ops) else []
        if frames.dtype == np.uint16:
            self._check_u16(segs)
        self._check_batch_channels(segs, frames.dtype, frames.shape[3])
        ctx = self._ctx()
        frames = np.ascontiguousarray(frames)
        if not segs or self._gate()[0] or not all(isinstance(sg, Params) for sg in segs):
            # identity, gated or foreign operators: compute on the host path, then upload
            res = self.process_batch(frames)
            dev = DeviceArray(ctx, res.shape, res.dtype)
            ctx._ck(ctx._lib.rv_memcpy(ctx._h, dev.ptr, np.ascontiguousarray(res).ctypes.data, dev.nbytes, 0))
            return dev
        if frames.shape[3] != 3:
            # gray / BGRA: upload once, then every pass runs device to device (CLAHE passes give 3 channels)
            b, h, w, c = frames.shape
            cur = DeviceArray(ctx, frames.shape, frames.dtype)
            ctx._ck(ctx._lib.rv_memcpy(ctx._h, cur.ptr, frames.ctypes.data, cur.nbytes, 0))
            for sg in segs:
                oc = 3 if sg.clahe else c
                dst = DeviceArray(ctx, (b, h, w, oc), frames.dtype)
                ctx.chain_ex_device(cur.ptr, dst.ptr, b, h, w, sg, 8 * frames.dtype.itemsize, c)
                cur, c = dst, oc
            return cur
        if frames.dtype == np.uint16:
            # upload once, then every pass runs device to device
            b, h, w, _ = frames.shape
            cur = DeviceArray(ctx, frames.shape, np.uint16)
            ctx._ck(ctx._lib.rv_memcpy(ctx._h, cur.ptr, frames.ctypes.data, cur.nbytes, 0))
            for sg in segs:
                dst = DeviceArray(ctx, frames.shape, np.uint16)
                ctx.chain_u16_device(cur.ptr, dst.ptr, b, h, w, sg)
                cur = dst
            return cur
        cur = frames
        for sg in segs:
            dst = DeviceArray(ctx, frames.shape)
            ctx.submit_io(cur, sg, shape=frames.shape[:3], out=dst)
            ctx.wait()
            cur = dst
        return cur

    def _check_device_chain(self):
        """What device-resident batches do not support -- the gate, foreign operators -- raises ValueError.  A disabled or empty
        pipeline passes (its result is its input)."""
        if not self.enabled or not self.ops:
            return
        if self._gate()[0]:
            raise ValueError("the low-contrast gate is not supported for device-resident batches; use numpy frames")
        if not all(isinstance(sg, Params) for sg in self._segments()):
            raise ValueError("device-resident batches support only CLAHEDehaze / MedianDerain chains")

    def _process_batch_device(self, frames, out=None):
        """Device-resident batch: a contiguous torch CUDA uint8 / uint16 tensor (B,H,W,C), C = 1, 3 or 4, in, a tensor of the same
        kind out (3 channels after a CLAHE pass).  Work is enqueued on torch's current stream (no host synchronisation): use the
        result with torch as usual."""
        import torch
        if (frames.dtype != torch.uint8 and frames.dtype != torch.uint16) or frames.dim() != 4 or frames.shape[3] not in (1, 3, 4) or \
                not frames.is_contiguous():
            raise ValueError("frames must be a contiguous (B,H,W,C) uint8 or uint16 CUDA tensor with C = 1, 3 or 4")
        wide = frames.dtype == torch.uint16
        if wide and self.enabled and self.ops:
            self._check_u16(self._segments())
        final = tuple(frames.shape)
        if self.enabled and self.ops:
            self._check_batch_channels(self._segments(), np.uint16 if wide else np.uint8, frames.shape[3])
            if any(isinstance(sg, Params) and sg.clahe for sg in self._segments()):
                final = final[:3] + (3,)
        _check_torch_out(out, final, frames.dtype, frames.device,
                         f"out must be a contiguous CUDA tensor of shape {final} and the input's dtype and device")
        if not self.enabled or not self.ops:
            return frames if out is None else out.copy_(frames)
        self._check_device_chain()
        ctx = self._device_ctx(frames)
        b, h, w, _ = frames.shape
        segs = self._segments()
        cur = frames
        for idx, sg in enumerate(segs):
            c = cur.shape[3]
            oc = 3 if sg.clahe else c
            last = idx == len(segs) - 1 and out is not None
            if c != 3:
                dst = out if last else torch.empty((b, h, w, oc), dtype=frames.dtype, device=frames.device)
                ctx.chain_ex_device(cur.data_ptr(), dst.data_ptr(), b, h, w, sg, 16 if wide else 8, c, stream=_torch_stream(frames.device))
                cur = dst
                continue
            dst = out if last else torch.empty_like(cur)
            stream = _torch_stream(frames.device)
            if wide:
                ctx.chain_u16_device(cur.data_ptr(), dst.data_ptr(), b, h, w, sg, stream=stream)
            elif stream is None:        # legacy default stream: run on the context's stream, synchronously
                ctx.chain_device(cur.data_ptr(), dst.data_ptr(), b, h, w, sg)
            else:
                ctx.submit_device(cur.data_ptr(), dst.data_ptr(), b, h, w, sg, stream=stream)
            cur = dst
        return cur

    # -- new: chain fused with the detector-input stage (SURVEY.md 8f-1) ------------------------
    def process_batch_to_tensor(self, frames: np.ndarray, size: int = 640, pad_value: int = 114, want_frames: bool = False,
                                out=None, padding_present: bool = False, yuv: str = None):
        """(B,H,W,3) uint8 -> ((B,3,size,size) float16 network input, processed frames or None).

        `out`: optional (B,3,size,size) float16 array for the tensor (pinned, from `Context.pinned_empty(shape, np.float16)`, for
        the overlapped H2D / kernels / D2H pipeline), or "device" to leave the tensor on the GPU (a `DeviceArray`): with pinned
        `frames` the only PCIe traffic is then the upload of the frames.
        `padding_present=True`: `out` already holds the letterbox padding rows (`Context.fill_tensor_padding`, done once per buffer
        of a ring), so only the image rows come back over PCIe -- 56 % of the tensor for 1080p frames.

        The tensor is what the detector stage builds from `proc` right after the chain (main_preview.py:99 ->
        yolo_ultralytics.py:28-35: letterbox, BGR->RGB, HWC->CHW, /255, half).  When the chain is the stock
        CLAHEDehaze -> MedianDerain pair and the down-scale is an exact integer (1080p -> 640), the resize happens inside
        the chain kernel and the full-resolution frames are only written if `want_frames` is set.

        `yuv="NV12"` / `"I420"` / `"YUY2"` / `"UYVY"`: `frames` are (B,3H/2,W) uint8 4:2:0 or (B,H,W,2) uint8 4:2:2 frames, as in
        process_batch; the processed frames are BGR.
        """
        if yuv is not None:
            return self._to_tensor_yuv(frames, size, pad_value, want_frames, out, padding_present, yuv)
        if isinstance(frames, np.ndarray) and frames.dtype == np.uint16:
            raise ValueError("process_batch_to_tensor takes uint8 frames: the detector input is built from 8-bit frames "
                             "(run process_batch on uint16 frames and convert them to 8 bits first)")
        if not isinstance(frames, np.ndarray) or frames.ndim != 4 or frames.shape[3] != 3 or frames.dtype != np.uint8:
            raise ValueError("frames must be a (B,H,W,3) uint8 numpy array")
        ctx = self._ctx()
        segs = self._segments() if (self.enabled and self.ops) else []
        keep = isinstance(out, str)
        if keep and out != "device":
            raise ValueError('out must be an array, None or "device"')
        if out is not None and not keep and (out.shape != (frames.shape[0], 3, size, size) or out.dtype != np.float16
                                             or not out.flags.c_contiguous):
            raise ValueError("out must be a C-contiguous (B,3,size,size) float16 array")
        if self._gate()[0] or len(segs) != 1 or not isinstance(segs[0], Params):
            proc = self.process_batch(frames)
            t = ctx.letterbox_f16(proc, size, pad_value)
            if keep:
                dev = DeviceArray(ctx, t.shape, np.float16)
                ctx._ck(ctx._lib.rv_memcpy(ctx._h, dev.ptr, t.ctypes.data, dev.nbytes, 0))
                t = dev
            elif out is not None:
                np.copyto(out, t)
                t = out
            return t, (proc if want_frames else None)
        if keep:
            frames = np.ascontiguousarray(frames)
            dev = DeviceArray(ctx, (frames.shape[0], 3, size, size), np.float16)
            full = ctx._host_result(frames.shape) if want_frames else None
            ctx.submit_io(frames, segs[0], out=full, tensor=dev, size=size, pad_value=pad_value)
            ctx.wait()
            return dev, full
        return ctx.chain_letterbox(frames, segs[0], size, pad_value, want_full=want_frames, out=out,
                                   padding_present=bool(padding_present and out is not None))

    def _to_tensor_yuv(self, frames, size, pad_value, want_frames, out, padding_present, yuv):
        """process_batch_to_tensor on (B,3H/2,W) 4:2:0 or (B,H,W,2) 4:2:2 host frames: where the BGR call takes its fused path (one
        pass, no gate) the frames go through rv_submit_io_fmt; otherwise they are converted on the GPU and take the BGR call."""
        if not isinstance(frames, np.ndarray):
            raise ValueError(f"yuv={yuv!r} takes a uint8 numpy array")
        _, b, h, w = check_yuv_frames(frames.shape, frames.dtype == np.uint8, yuv)
        keep = isinstance(out, str)
        if keep and out != "device":
            raise ValueError('out must be an array, None or "device"')
        if out is not None and not keep and (out.shape != (b, 3, size, size) or out.dtype != np.float16 or not out.flags.c_contiguous):
            raise ValueError("out must be a C-contiguous (B,3,size,size) float16 array")
        ctx = self._ctx()
        seg = self._fused_segment()
        if seg is None or self._gate()[0]:
            return self.process_batch_to_tensor(ctx._convert(frames, yuv, None), size, pad_value, want_frames, out, padding_present)
        if keep:
            t = DeviceArray(ctx, (b, 3, size, size), np.float16)
        else:
            t = np.empty((b, 3, size, size), np.float16) if out is None else out
        full = ctx._host_result((b, h, w, 3)) if want_frames else None
        ctx.submit_io(np.ascontiguousarray(frames), seg, out=full, tensor=t, size=size, pad_value=pad_value,
                      padding_present=bool(padding_present and out is not None and not keep), yuv=yuv)
        ctx.wait()
        return t, full
