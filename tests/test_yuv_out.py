"""Processed frames returned as YUV 4:2:0 (NV12, I420) for a video encoder, converted on the GPU exactly as cv2.cvtColor does.

The 4:2:0 result of a batch is cv2.cvtColor(R, COLOR_BGR2YUV_I420) of the BGR result R that the same call returns without out_yuv,
re-laid out as NV12 (U and V interleaved, U first) on request.  CPU tests pin a numpy restatement of cv2's integer conversion on the
live cv2 over all 2^24 BGR triples and check that malformed calls raise before a context exists.  GPU tests compare every entry with
cv2 to the last bit.
"""
import ctypes as C
import itertools
import os
import re

import cv2
import numpy as np
import pytest

from oracle import cv2_chain
from oracle import yuv420 as Y

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LAYOUTS = ["NV12", "I420"]
STOCK = [{"name": "CLAHEDehaze", "params": {"clip_limit": 2.0, "tile_grid": 8}}, {"name": "MedianDerain", "params": {"ksize": 5}}]
TO_BGR = {"NV12": cv2.COLOR_YUV2BGR_NV12, "I420": cv2.COLOR_YUV2BGR_I420}

# cv2's COLOR_BGR2YUV_I420 in 20-bit fixed point (BT.601 video range); chroma from the top-left pixel of each 2 x 2 block
CRY, CGY, CBY, CRU, CGU, CBU, CGV, CBV = 269484, 528482, 102760, -155188, -305135, 460324, -385875, -74448


def bgr_to_yuv420(bgr, layout):
    """(H,W,3) uint8 BGR -> (3H/2,W) uint8 4:2:0, as cv2 (NV12: cv2's I420 with U and V interleaved)."""
    b, g, r = (bgr[..., i].astype(np.int32) for i in range(3))          # every term fits in int32, as on the GPU
    y = (CRY * r + CGY * g + CBY * b + (1 << 19) + (16 << 20)) >> 20
    b, g, r = b[::2, ::2], g[::2, ::2], r[::2, ::2]
    u = (CRU * r + CGU * g + CBU * b + (1 << 19) + (128 << 20)) >> 20
    v = (CBU * r + CGV * g + CBV * b + (1 << 19) + (128 << 20)) >> 20
    return Y.from_planes(y, u, v, layout)


def cv2_yuv(bgr, layout):
    """cv2's own conversion of one frame or a batch, re-laid out as NV12 when asked."""
    if bgr.ndim == 4:
        return np.stack([cv2_yuv(f, layout) for f in bgr])
    i420 = cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420)
    return i420 if layout == "I420" else Y.from_planes(*Y.planes(i420, "I420"), "NV12")


def bgr_batch(n, h, w, seed=0):
    """n BGR frames: road scenes (rvb200.synth) where the size allows, random bytes otherwise; the last frame is random."""
    from rvb200 import synth
    rng = np.random.default_rng(seed + 131 * h + w)
    out = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
    if h >= 16 and w >= 16 and n > 1:
        pool = synth.frame_pool(h, w, min(n - 1, 8), base_seed=seed)
        for i in range(n - 1):
            out[i] = pool[i % len(pool)]
    return out


def _pipe(chain, gate=False, thresh=20.0, enabled=True, context=None):
    import rvb200
    return rvb200.PreprocessPipeline({"enabled": enabled, "chain": chain,
                                      "auto_gate": {"enable_low_contrast_gate": gate, "contrast_thresh": thresh}}, context=context)


# ---------------------------------------------------------------- CPU
def test_oracle_equals_cv2_on_every_triple_as_a_top_left_pixel():
    c = np.arange(1 << 24, dtype=np.uint32)
    img = np.stack([(c >> 16) & 255, (c >> 8) & 255, c & 255], -1).astype(np.uint8).reshape(4096, 4096, 3)
    big = np.repeat(np.repeat(img, 2, 0), 2, 1)                     # every colour is the top-left pixel of a 2 x 2 block
    want = cv2.cvtColor(big, cv2.COLOR_BGR2YUV_I420)
    got = bgr_to_yuv420(big, "I420")
    assert np.array_equal(got, want)
    nv12 = bgr_to_yuv420(big, "NV12")
    assert np.array_equal(nv12, Y.from_planes(*Y.planes(want, "I420"), "NV12"))


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("h,w", [(270, 482), (6, 10), (2, 2), (2, 4098), (134, 2)])
def test_oracle_equals_cv2_on_ragged_sizes(layout, h, w):
    bgr = np.random.default_rng(h * w).integers(0, 256, (h, w, 3), dtype=np.uint8)
    assert np.array_equal(bgr_to_yuv420(bgr, layout), cv2_yuv(bgr, layout))


def test_cv2_refuses_an_odd_height_and_an_odd_width():
    for shape in ((3, 4, 3), (4, 3, 3)):
        with pytest.raises(cv2.error):
            cv2.cvtColor(np.zeros(shape, np.uint8), cv2.COLOR_BGR2YUV_I420)


def test_malformed_yuv_output_calls_raise_before_a_context_exists(monkeypatch):
    from rvb200 import _native
    from rvb200.preprocess import pipeline as P

    def no_context(*a, **k):
        raise AssertionError("a context was created")
    monkeypatch.setattr(P, "default_context", no_context)
    monkeypatch.setattr(_native, "default_context", no_context)
    monkeypatch.setattr(_native.Context, "__init__", no_context)
    good = np.zeros((2, 6, 10, 3), np.uint8)
    nv12 = np.zeros((2, 9, 10), np.uint8)
    cases = [(good, None, "NV21", None, "out_yuv must be"), (good, None, "nv12", None, "out_yuv must be"),
             (good, None, "", None, "out_yuv must be"), (np.zeros((2, 5, 10, 3), np.uint8), None, "NV12", None, "even height"),
             (np.zeros((2, 6, 9, 3), np.uint8), None, "I420", None, "even height"),
             (good.astype(np.uint16), None, "NV12", None, "uint8"), (np.zeros((2, 6, 10, 1), np.uint8), None, "I420", None, "BGR"),
             (np.zeros((2, 6, 10, 4), np.uint8), None, "NV12", None, "BGR"), (np.zeros((6, 10, 3), np.uint8), None, "NV12", None, "BGR"),
             (np.zeros((2, 0, 10, 3), np.uint8), None, "NV12", None, "empty"),
             (good, np.zeros((2, 6, 10, 3), np.uint8), "NV12", None, "out must be"),
             (good, np.zeros((2, 9, 10), np.int16), "NV12", None, "out must be"),
             (good, np.zeros((2, 9, 20), np.uint8)[:, :, ::2], "I420", None, "out must be"),
             (good, "host", "NV12", None, "out must be"), (good.tolist(), None, "NV12", None, "numpy"),
             (np.zeros((2, 9, 9), np.uint8), None, "I420", "NV12", "even width"),
             (nv12, None, "I420", "NV21", "yuv must be"), (nv12, np.zeros((2, 6, 10, 3), np.uint8), "NV12", "NV12", "out must be")]
    for chain, gate, enabled in ((STOCK, False, True), (STOCK, True, True), (STOCK[1:] * 2, False, True), ([], False, True),
                                 (STOCK, False, False)):
        pipe = _pipe(chain, gate=gate, enabled=enabled)
        for frames, out, out_yuv, yuv, msg in cases:
            with pytest.raises(ValueError, match=re.escape(msg)):
                pipe.process_batch(frames, out=out, yuv=yuv, out_yuv=out_yuv)
    with pytest.raises(ValueError, match="out_yuv must be"):
        _native.check_out_yuv("YV12")
    assert _native.check_bgr_for_yuv((5, 1080, 1920, 3), True, "I420") == (2, 5, 1080, 1920)


def test_header_declares_and_library_exports_the_yuv_output_entries():
    from rvb200 import _native
    header = open(os.path.join(ROOT, "include", "rv_b200.h")).read()
    lib = _native.load_library()
    for name in ("rv_bgr_to_yuv420", "rv_submit_io_fmt"):
        assert re.search(rf"\bint {name}\(", header) and name in _native.EXPORTS and hasattr(lib, name)
    buf = np.zeros(64, np.uint8)
    io = _native.IO()
    p = _native.Params.make()
    assert lib.rv_bgr_to_yuv420(None, buf.ctypes.data, buf[32:].ctypes.data, 1, 2, 2, 6, 2, 1, 0, None) == -1
    assert lib.rv_submit_io_fmt(None, C.byref(io), 0, 1, 1, 2, 2, C.byref(p)) == -1
    assert lib.rv_submit_io_fmt(None, None, 0, 0, 1, 2, 2, C.byref(p)) == -1


# ---------------------------------------------------------------- GPU
def _ctx():
    import rvb200
    return rvb200.default_context(0)


def _torch(x):
    import torch
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


STAGE_SHAPES = [(8192, 8192), (2, 2), (6, 10), (270, 482), (540, 4098), (134, 2), (1080, 1920), (2160, 3840)]


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("h,w", STAGE_SHAPES)
def test_gpu_stage_pageable_pinned_device_and_side_stream(h, w, layout):
    import torch
    ctx = _ctx()
    if (h, w) == (8192, 8192):                                       # all 2^24 colours as top-left pixels
        c = np.arange(1 << 24, dtype=np.uint32)
        img = np.stack([(c >> 16) & 255, (c >> 8) & 255, c & 255], -1).astype(np.uint8).reshape(4096, 4096, 3)
        frames = np.repeat(np.repeat(img, 2, 0), 2, 1)[None]
    else:
        frames = bgr_batch(3, h, w, seed=h)
    want = cv2_yuv(frames, layout)
    assert np.array_equal(ctx.bgr_to_yuv420(frames, layout), want)
    pin, pout = ctx.pinned_empty(frames.shape), ctx.pinned_empty(want.shape)
    pin[...] = frames
    assert ctx.bgr_to_yuv420(pin, layout, out=pout) is pout and np.array_equal(pout, want)
    side = torch.cuda.Stream()
    t = _torch(frames)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        got = ctx.bgr_to_yuv420(t, layout).cpu()
    assert np.array_equal(got.numpy(), want)
    assert np.array_equal(ctx.bgr_to_yuv420(t, layout).cpu().numpy(), want)      # torch's default stream


@pytest.mark.gpu
def test_gpu_stage_pitches_offsets_and_refusals():
    """BGR device frames at an odd pitch one byte into their allocation, NV12 out at an odd pitch, on a side stream; I420 at widths
    that are not multiples of 8 and from an odd offset (the byte-wise path); host memory with pitches; the C entry's refusals."""
    import torch
    from rvb200 import _native as N
    ctx = _ctx()
    n, h = 3, 134
    for layout, w, op in (("NV12", 246, 246 + 3), ("I420", 246, 246), ("I420", 244, 244), ("NV12", 248, 251)):
        frames = bgr_batch(n, h, w, seed=5)
        want = cv2_yuv(frames, layout)
        ip = 3 * w + 5
        padded = np.zeros((n, h, ip), np.uint8)
        padded[..., :3 * w] = frames.reshape(n, h, 3 * w)
        din = torch.zeros(padded.size + 1, dtype=torch.uint8, device="cuda")
        din[1:] = _torch(padded.reshape(-1))
        dout = torch.zeros(n * op * h * 3 // 2 + 1, dtype=torch.uint8, device="cuda")
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        ctx._ck(ctx._lib.rv_bgr_to_yuv420(ctx._h, C.c_void_p(din.data_ptr() + 1), C.c_void_p(dout.data_ptr() + 1), n, h, w, ip, op,
                                          N.YUV_LAYOUTS[layout], N.MEM_DEVICE, C.c_void_p(side.cuda_stream)))
        side.synchronize()
        got = dout[1:].cpu().numpy().reshape(n, h * 3 // 2, op)[:, :, :w]
        assert np.array_equal(got, want), (layout, w)
        hout = np.zeros((n, h * 3 // 2, op), np.uint8)
        ctx._ck(ctx._lib.rv_bgr_to_yuv420(ctx._h, padded.ctypes.data, hout.ctypes.data, n, h, w, ip, op, N.YUV_LAYOUTS[layout],
                                          N.MEM_HOST, None))
        assert np.array_equal(hout[:, :, :w], want), (layout, w)
    buf = np.zeros(4096, np.uint8)
    out = np.zeros(4096, np.uint8)
    for (h, w, ip, op, layout) in ((5, 4, 12, 4, 1), (4, 5, 15, 5, 1), (0, 4, 12, 4, 1), (4, 0, 12, 4, 2), (4, 4, 11, 4, 1),
                                   (4, 4, 12, 3, 1), (4, 4, 12, 6, 2), (4, 4, 12, 4, 0), (4, 4, 12, 4, 3), (4, 4, 12, 4, -1)):
        assert ctx._lib.rv_bgr_to_yuv420(ctx._h, buf.ctypes.data, out.ctypes.data, 1, h, w, ip, op, layout, N.MEM_HOST, None) == -1
        assert not out.any()
    assert ctx._lib.rv_bgr_to_yuv420(ctx._h, buf.ctypes.data, buf[20:].ctypes.data, 1, 4, 4, 12, 4, 1, N.MEM_HOST, None) == -1
    assert ctx._lib.rv_bgr_to_yuv420(ctx._h, buf[10:].ctypes.data, buf.ctypes.data, 1, 4, 4, 12, 4, 1, N.MEM_HOST, None) == -1
    for kind in (N.MEM_HOST, N.MEM_PINNED):
        l0 = ctx.launch_count
        assert ctx._lib.rv_bgr_to_yuv420(ctx._h, buf.ctypes.data, None, 1, 4, 4, 12, 4, 1, kind, None) == -1
        assert ctx._lib.rv_bgr_to_yuv420(ctx._h, None, out.ctypes.data, 1, 4, 4, 12, 4, 1, kind, None) == -1
        assert ctx.launch_count == l0
    io = N.IO()
    io.in_, io.in_pitch, io.out, io.out_pitch = buf.ctypes.data, 12, out.ctypes.data, 4
    p = N.Params.make()
    for il, ol in ((0, 3), (3, 1), (0, -1)):
        assert ctx._lib.rv_submit_io_fmt(ctx._h, C.byref(io), il, ol, 1, 4, 4, C.byref(p)) == -1
    assert ctx._lib.rv_submit_io_fmt(ctx._h, C.byref(io), 0, 2, 1, 5, 4, C.byref(p)) == -1
    assert ctx._lib.rv_submit_io_fmt(ctx._h, C.byref(io), 0, 2, 1, 4, 4, C.byref(p)) == 0
    ctx.wait()
    io.out_pitch = 6
    assert ctx._lib.rv_submit_io_fmt(ctx._h, C.byref(io), 0, 2, 1, 4, 4, C.byref(p)) == -1        # I420 out needs out_pitch == w
    assert ctx._lib.rv_submit_io_fmt(ctx._h, C.byref(io), 0, 1, 1, 4, 4, C.byref(p)) == 0         # NV12 out takes a wider pitch
    ctx.wait()


def _chain_ref(bgr, space, clip, grid, k):
    return np.stack([cv2_chain.chain(f, space, clip, grid, k) for f in bgr])


def _inputs(bgr, yuv):
    """The frames a call takes: BGR, or their NV12 / I420 form (then the BGR they stand for is cv2's conversion of it)."""
    if yuv is None:
        return bgr, bgr
    frames = cv2_yuv(bgr, yuv)
    return frames, np.stack([cv2.cvtColor(f, TO_BGR[yuv]) for f in frames])


@pytest.mark.gpu
@pytest.mark.parametrize("yuv", [None, "NV12", "I420"])
@pytest.mark.parametrize("out_yuv", LAYOUTS)
def test_gpu_process_batch_parameter_matrix(yuv, out_yuv):
    frames, bgr = _inputs(bgr_batch(3, 96, 130, seed=2), yuv)
    bad = []
    for space, grid, clip, k in itertools.product(("YCrCb", "LAB"), (2, 8, 16), (0.0, 2.0), (3, 5, 7, 9)):
        chain = [{"name": "CLAHEDehaze", "params": {"space": space, "clip_limit": clip, "tile_grid": grid}},
                 {"name": "MedianDerain", "params": {"ksize": k}}]
        got = _pipe(chain).process_batch(frames, yuv=yuv, out_yuv=out_yuv)
        if not np.array_equal(got, cv2_yuv(_chain_ref(bgr, space, clip, grid, k), out_yuv)):
            bad.append((space, grid, clip, k))
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("out_yuv", LAYOUTS)
def test_gpu_gate_at_the_threshold(out_yuv):
    """Exactly at the threshold a frame is skipped and comes back as the conversion of its BGR; one unit above it is processed.  One
    fused pass and two passes, host and "device" results, BGR and NV12 in."""
    ctx = _ctx()
    for yuv in (None, "NV12"):
        frames, bgr = _inputs(bgr_batch(4, 64, 96, seed=11), yuv)
        spans = ctx.gray_span(bgr)
        t = float(sorted(spans)[1])
        for chain, ref in ((STOCK, lambda f: cv2_chain.chain(f, "YCrCb", 2.0, 8, 5)),
                           (STOCK[1:] * 2, lambda f: cv2.medianBlur(cv2.medianBlur(f, 5), 5))):
            for thresh in (t, t + 1, t - 0.5):
                want = cv2_yuv(np.stack([ref(f) if s < thresh else f for f, s in zip(bgr, spans)]), out_yuv)
                pipe = _pipe(chain, gate=True, thresh=thresh)
                assert np.array_equal(pipe.process_batch(frames, yuv=yuv, out_yuv=out_yuv), want), (yuv, len(chain), thresh)
                dev = pipe.process_batch(frames, out="device", yuv=yuv, out_yuv=out_yuv)
                assert np.array_equal(dev.numpy(), want), (yuv, len(chain), thresh)


@pytest.mark.gpu
@pytest.mark.parametrize("out_yuv", LAYOUTS)
def test_gpu_disabled_empty_and_foreign_operator(out_yuv):
    """What these pipelines return as BGR, re-encoded: for 4:2:0 input that is not the input bytes."""
    import rvb200

    class Flip(rvb200.PreprocessOp):
        def __call__(self, im):
            return np.ascontiguousarray(im[:, ::-1])
    for yuv in (None, "NV12", "I420"):
        frames, bgr = _inputs(bgr_batch(2, 120, 200, seed=13), yuv)
        want = cv2_yuv(bgr, out_yuv)
        for pipe in (_pipe(STOCK, enabled=False), _pipe([]), _pipe(STOCK, gate=True, enabled=False)):
            assert np.array_equal(pipe.process_batch(frames, yuv=yuv, out_yuv=out_yuv), want)
            out = np.zeros_like(want)
            assert pipe.process_batch(frames, out=out, yuv=yuv, out_yuv=out_yuv) is out and np.array_equal(out, want)
            assert np.array_equal(pipe.process_batch(frames, out="device", yuv=yuv, out_yuv=out_yuv).numpy(), want)
            assert np.array_equal(pipe.process_batch(_torch(frames), yuv=yuv, out_yuv=out_yuv).cpu().numpy(), want)
        if yuv is not None:
            assert not np.array_equal(_pipe([]).process_batch(frames, yuv=yuv, out_yuv=yuv), frames)     # not the identity
        pipe = _pipe(STOCK[::-1])
        pipe.ops.insert(1, Flip())
        ref = cv2_yuv(np.stack([cv2_chain.clahe_dehaze(np.ascontiguousarray(cv2.medianBlur(f, 5)[:, ::-1]), "YCrCb", 2.0, 8)
                                for f in bgr]), out_yuv)
        assert np.array_equal(pipe.process_batch(frames, yuv=yuv, out_yuv=out_yuv), ref)
        assert np.array_equal(pipe.process_batch(frames, out="device", yuv=yuv, out_yuv=out_yuv).numpy(), ref)


@pytest.mark.gpu
def test_gpu_device_refusals_come_before_anything_is_enqueued():
    import torch
    import rvb200

    class Flip(rvb200.PreprocessOp):
        def __call__(self, im):
            return np.ascontiguousarray(im[:, ::-1])
    ctx = _ctx()
    foreign = _pipe(STOCK)
    foreign.ops.insert(1, Flip())
    for frames, yuv in ((_torch(bgr_batch(2, 32, 48, seed=1)), None), (_torch(cv2_yuv(bgr_batch(2, 32, 48, seed=1), "NV12")), "NV12")):
        cases = [(_pipe(STOCK, gate=True), None, "gate"), (foreign, None, "CLAHEDehaze / MedianDerain"),
                 (_pipe(STOCK), torch.empty((2, 32, 48, 3), dtype=torch.uint8, device="cuda"), "out must be"),
                 (_pipe(STOCK), torch.empty((2, 48, 48), dtype=torch.uint8), "out must be")]
        for pipe, out, msg in cases:
            l0 = ctx.launch_count
            with pytest.raises(ValueError, match=msg):
                pipe.process_batch(frames, out=out, yuv=yuv, out_yuv="NV12")
            assert ctx.launch_count == l0, msg
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("out_yuv", LAYOUTS)
def test_gpu_outputs_numpy_pinned_device_and_torch_side_stream(out_yuv):
    import torch
    ctx = _ctx()
    for yuv in (None, "NV12", "I420"):
        frames, bgr = _inputs(bgr_batch(5, 270, 482, seed=3), yuv)
        for chain in (STOCK, STOCK[::-1]):
            pipe = _pipe(chain)
            ref = _chain_ref(bgr, "YCrCb", 2.0, 8, 5) if chain is STOCK else \
                np.stack([cv2_chain.clahe_dehaze(cv2.medianBlur(f, 5), "YCrCb", 2.0, 8) for f in bgr])
            want = cv2_yuv(ref, out_yuv)
            pin, pout = ctx.pinned_empty(frames.shape), ctx.pinned_empty(want.shape)
            pin[...] = frames
            assert pipe.process_batch(pin, out=pout, yuv=yuv, out_yuv=out_yuv) is pout and np.array_equal(pout, want)
            assert np.array_equal(pipe.process_batch(pin, yuv=yuv, out_yuv=out_yuv), want)
            out = np.zeros_like(want)
            assert pipe.process_batch(frames, out=out, yuv=yuv, out_yuv=out_yuv) is out and np.array_equal(out, want)
            assert np.array_equal(pipe.process_batch(frames[:, ::-1][:, ::-1], yuv=yuv, out_yuv=out_yuv), want)
            dev = pipe.process_batch(pin, out="device", yuv=yuv, out_yuv=out_yuv)
            assert dev.shape == want.shape and np.array_equal(dev.numpy(), want)
            side = torch.cuda.Stream()
            t = _torch(frames)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                res = pipe.process_batch(t, yuv=yuv, out_yuv=out_yuv)
                tout = torch.empty(want.shape, dtype=torch.uint8, device="cuda")
                res2 = pipe.process_batch(t, out=tout, yuv=yuv, out_yuv=out_yuv)
                host = res.cpu()
            side.synchronize()
            assert res2 is tout and np.array_equal(host.numpy(), want) and np.array_equal(tout.cpu().numpy(), want), (yuv, len(chain))


@pytest.mark.gpu
@pytest.mark.parametrize("out_yuv", LAYOUTS)
def test_gpu_64_frames_1080p(out_yuv):
    """64 x 1080p through the host pipeline's chunks (tapered first and last ones), BGR and NV12 in, checked against cv2."""
    ctx = _ctx()
    for yuv in (None, "NV12"):
        frames, bgr = _inputs(bgr_batch(64, 1080, 1920, seed=21), yuv)
        pin = ctx.pinned_empty(frames.shape)
        pin[...] = frames
        got = _pipe(STOCK).process_batch(pin, yuv=yuv, out_yuv=out_yuv)
        bad = [i for i in range(64) if not np.array_equal(got[i], cv2_yuv(cv2_chain.chain(bgr[i], "YCrCb", 2.0, 8, 5), out_yuv))]
        assert not bad, (yuv, bad)


@pytest.mark.gpu
@pytest.mark.parametrize("out_yuv", LAYOUTS)
def test_gpu_300_tiny_frames_cross_every_chunk_boundary(out_yuv):
    import rvb200
    ctx = rvb200.Context(0)
    ctx.set_option("chunk_frames", 7)
    try:
        for yuv in (None, "I420"):
            frames, bgr = _inputs(bgr_batch(301, 4, 6, seed=4), yuv)
            spans = [int(g.max()) - int(g.min()) for g in (cv2.cvtColor(f, cv2.COLOR_BGR2GRAY) for f in bgr)]
            for gate in (False, True):
                pipe = _pipe(STOCK, gate=gate, thresh=120.0, context=ctx)
                want = cv2_yuv(np.stack([cv2_chain.chain(f, "YCrCb", 2.0, 8, 5) if (not gate or s < 120) else f
                                         for f, s in zip(bgr, spans)]), out_yuv)
                assert np.array_equal(pipe.process_batch(frames, yuv=yuv, out_yuv=out_yuv), want), (yuv, gate)
        assert len(rvb200.chunk_schedule(301, 7)) > 40
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("out_yuv", LAYOUTS)
def test_gpu_yuv_out_job_is_the_bgr_job_plus_one_conversion_per_chunk(out_yuv):
    """A job with a 4:2:0 frame output is the BGR-out job plus exactly one conversion launch per chunk, with the same gate flags and
    tensor, and its frames are the conversion of the BGR job's; for BGR and 4:2:0 input, with a tensor and with the gate, with host
    and device outputs."""
    import torch
    import rvb200
    ctx = _ctx()
    for yuv in (None, "NV12"):
        frames, bgr = _inputs(bgr_batch(40, 90, 160, seed=6), yuv)
        n, h, w, _ = bgr.shape
        chunks = len(rvb200.chunk_schedule(n, min(n, (24 << 20) // (3 * w * h))))
        for kw in ({"tensor": True}, {"gate": True}):
            p = rvb200.Params.make("YCrCb", 2.0, 8, 5, gate=kw.get("gate", False), gate_thresh=200.0)
            res = {}
            for oy in (None, out_yuv):
                out = np.zeros((n, h * 3 // 2, w) if oy else (n, h, w, 3), np.uint8)
                tensor = np.zeros((n, 3, 640, 640), np.float16) if "tensor" in kw else None
                processed = np.zeros(n, np.int32)
                l0 = ctx.launch_count
                ctx.submit_io(frames, p, out=out, tensor=tensor, processed=processed, yuv=yuv, out_yuv=oy)
                ctx.wait()
                res[oy] = (ctx.launch_count - l0, out, tensor, processed)
            (lb, ob, tb, pb), (ly, oy_, ty, py) = res[None], res[out_yuv]
            assert ly - lb == chunks, (yuv, kw, lb, ly, chunks)
            assert np.array_equal(oy_, cv2_yuv(ob, out_yuv)) and np.array_equal(pb, py), (yuv, kw)
            assert tb is None or np.array_equal(tb.view(np.uint16), ty.view(np.uint16)), (yuv, kw)
            runs = [cv2_chain.low_contrast(f, 200.0) if "gate" in kw else True for f in bgr]
            assert list(pb) == [int(r) for r in runs], kw
            dout = torch.zeros((n, h * 3 // 2, w), dtype=torch.uint8, device="cuda")      # device 4:2:0 output, written in place
            td = np.zeros_like(tb) if tb is not None else None
            torch.cuda.synchronize()
            l0 = ctx.launch_count
            ctx.submit_io(frames, p, out=dout, tensor=td, yuv=yuv, out_yuv=out_yuv)
            ctx.wait()
            assert ctx.launch_count - l0 == ly, (yuv, kw)
            assert np.array_equal(dout.cpu().numpy(), oy_) and (td is None or np.array_equal(td.view(np.uint16), tb.view(np.uint16)))
        # tensor only, with a 4:2:0 layout named for the absent frame output: the BGR job's tensor, no conversion
        p = rvb200.Params.make("YCrCb", 2.0, 8, 5)
        t1, t2 = np.zeros((n, 3, 640, 640), np.float16), np.zeros((n, 3, 640, 640), np.float16)
        ctx.submit_io(frames, p, tensor=t1, yuv=yuv)
        ctx.wait()
        ctx.submit_io(frames, p, tensor=t2, yuv=yuv, out_yuv=out_yuv)
        ctx.wait()
        assert np.array_equal(t1.view(np.uint16), t2.view(np.uint16))
