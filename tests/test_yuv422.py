"""Packed YUV 4:2:2 camera frames (YUY2, UYVY) in the batch entries, converted to BGR on the GPU exactly as cv2.cvtColor does.

CPU tests pin the numpy restatement of the conversion (oracle/yuv422.py) on the live cv2 over all 2^24 (Y, U, V) triples and ragged
sizes, and check that malformed batches raise ValueError before a context exists.  GPU tests require rv_yuv422_to_bgr, the 4:2:2 input of
rv_submit_io_fmt and every Python entry built on them to give, to the last bit, what the same call gives on the cv2-converted BGR frames.
"""
import ctypes as C
import itertools
import os
import re

import cv2
import numpy as np
import pytest

from oracle import cv2_chain
from oracle import rv_oracle as O
from oracle import yuv422 as Y

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CODES = {"YUY2": cv2.COLOR_YUV2BGR_YUY2, "UYVY": cv2.COLOR_YUV2BGR_UYVY}
TO_422 = {"YUY2": cv2.COLOR_BGR2YUV_YUY2, "UYVY": cv2.COLOR_BGR2YUV_UYVY}
LAYOUTS = ["YUY2", "UYVY"]
STOCK = [{"name": "CLAHEDehaze", "params": {"clip_limit": 2.0, "tile_grid": 8}}, {"name": "MedianDerain", "params": {"ksize": 5}}]


def yuv_batch(n, h, w, layout, seed=0):
    """n (h, w, 2) frames: road scenes (rvb200.synth, at most 8 distinct ones) through cv2's BGR -> 4:2:2 where the size allows, random
    bytes otherwise; the chroma of the last frame is random."""
    from rvb200 import synth
    rng = np.random.default_rng(seed + 131 * h + w)
    if h >= 16 and w >= 16:
        pool = [cv2.cvtColor(f, TO_422[layout]) for f in synth.frame_pool(h, w, min(n, 8), base_seed=seed)]
        out = np.stack([pool[i % len(pool)] for i in range(n)])
        y, _, _ = Y.planes(out[-1], layout)
        out[-1] = Y.from_planes(y, *rng.integers(0, 256, (2, h, w // 2), dtype=np.uint8), layout)
        return out
    return rng.integers(0, 256, (n, h, w, 2), dtype=np.uint8)


def bgr_of(frames, layout):
    return np.stack([cv2.cvtColor(f, CODES[layout]) for f in frames])


def _pipe(chain, gate=False, thresh=20.0, enabled=True, context=None):
    import rvb200
    return rvb200.PreprocessPipeline({"enabled": enabled, "chain": chain,
                                      "auto_gate": {"enable_low_contrast_gate": gate, "contrast_thresh": thresh}}, context=context)


# ---------------------------------------------------------------- CPU
@pytest.mark.parametrize("layout", LAYOUTS)
def test_oracle_equals_cv2_on_every_triple(layout):
    frame = Y.every_triple(layout)
    y, u, v = Y.planes(frame, layout)
    up = lambda p: np.repeat(p.astype(np.int64), 2, 1)         # noqa: E731
    assert len(np.unique((y.astype(np.int64) << 16) | (up(u) << 8) | up(v))) == 1 << 24
    assert np.array_equal(Y.yuv422_to_bgr(frame, layout), cv2.cvtColor(frame, CODES[layout]))


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("h,w", [(270, 482), (135, 246), (2, 4098), (7, 10), (5, 4), (1, 2), (33, 2050)])
def test_oracle_equals_cv2_on_ragged_sizes(layout, h, w):
    rng = np.random.default_rng(h * w)
    frame = rng.integers(0, 256, (h, w, 2), dtype=np.uint8)
    assert np.array_equal(Y.yuv422_to_bgr(frame, layout), cv2.cvtColor(frame, CODES[layout]))
    assert np.array_equal(Y.from_planes(*Y.planes(frame, layout), layout), frame)


def test_cv2_refuses_an_odd_width_and_takes_an_odd_height():
    for code in CODES.values():
        with pytest.raises(cv2.error):
            cv2.cvtColor(np.zeros((4, 5, 2), np.uint8), code)
        assert cv2.cvtColor(np.zeros((5, 4, 2), np.uint8), code).shape == (5, 4, 3)


def test_malformed_yuv422_batches_raise_before_a_context_exists(monkeypatch):
    import rvb200
    from rvb200 import _native
    from rvb200.preprocess import pipeline as P

    def no_context(*a, **k):
        raise AssertionError("a context was created")
    monkeypatch.setattr(P, "default_context", no_context)
    monkeypatch.setattr(_native, "default_context", no_context)
    monkeypatch.setattr(_native.Context, "__init__", no_context)
    good = np.zeros((2, 5, 10, 2), np.uint8)
    cases = [(np.zeros((5, 10, 2), np.uint8), "YUY2", "(B,H,W,2)"), (np.zeros((2, 5, 10), np.uint8), "UYVY", "(B,H,W,2)"),
             (np.zeros((2, 5, 10, 3), np.uint8), "YUY2", "(B,H,W,2)"), (np.zeros((2, 5, 10, 1), np.uint8), "UYVY", "(B,H,W,2)"),
             (good.astype(np.uint16), "YUY2", "uint8"), (good.astype(np.float32), "UYVY", "uint8"),
             (np.zeros((2, 5, 9, 2), np.uint8), "YUY2", "even width"), (np.zeros((2, 0, 10, 2), np.uint8), "UYVY", "empty"),
             (np.zeros((2, 5, 0, 2), np.uint8), "YUY2", "empty"), (good, "YUYV", "NV12"), (good, "yuy2", "NV12"), (good, "YVYU", "NV12")]
    for chain, gate in ((STOCK, False), (STOCK, True), (STOCK[1:] * 2, False), ([], False)):
        pipe = _pipe(chain, gate=gate)
        for frames, yuv, msg in cases:
            for call in (lambda: pipe.process_batch(frames, yuv=yuv), lambda: pipe.process_batch(frames, out="device", yuv=yuv),
                         lambda: pipe.process_batch_to_tensor(frames, yuv=yuv),
                         lambda: pipe.process_batch(frames, yuv=yuv, out_yuv="NV12")):
                with pytest.raises(ValueError, match=re.escape(msg)):
                    call()
        # an odd height is a 4:2:2 frame, but not one that 4:2:0 output can take
        with pytest.raises(ValueError, match="even height"):
            pipe.process_batch(good, yuv="YUY2", out_yuv="I420")
        with pytest.raises(ValueError, match="out_yuv must be"):
            pipe.process_batch(np.zeros((2, 6, 10, 2), np.uint8), yuv="YUY2", out_yuv="YUY2")
    with pytest.raises(ValueError):
        _pipe(STOCK).process_batch(good, out=np.zeros((2, 5, 10, 3), np.uint8)[:, ::-1], yuv="UYVY")
    with pytest.raises(ValueError):
        _pipe(STOCK).process_batch(good, out=np.zeros((2, 5, 10, 2), np.uint8), yuv="UYVY")
    with pytest.raises(ValueError):
        _pipe(STOCK).process_batch_to_tensor(good, out=np.zeros((2, 3, 64, 64), np.float32), yuv="YUY2")
    assert _native.check_yuv_frames((5, 1080, 1920, 2), True, "UYVY") == (17, 5, 1080, 1920)
    assert _native.check_yuv_frames((5, 135, 246, 2), True, "YUY2") == (16, 5, 135, 246)
    with pytest.raises(ValueError, match="yuv422_to_bgr"):
        _native.Context.yuv420_to_bgr(None, good, "YUY2")
    with pytest.raises(ValueError, match="'YUY2' or 'UYVY'"):
        _native.Context.yuv422_to_bgr(None, good, "NV12")
    assert rvb200.PreprocessPipeline({"chain": STOCK})._fused_segment() is not None


def test_header_declares_and_library_exports_the_yuv422_entry():
    from rvb200 import _native
    header = open(os.path.join(ROOT, "include", "rv_b200.h")).read()
    lib = _native.load_library()
    assert re.search(r"\bint rv_yuv422_to_bgr\(", header) and "rv_yuv422_to_bgr" in _native.EXPORTS and hasattr(lib, "rv_yuv422_to_bgr")
    assert "enum rv_yuv422 { RV_YUV_YUY2 = 16, RV_YUV_UYVY = 17 };" in header
    assert _native.YUV422_LAYOUTS == {"YUY2": 16, "UYVY": 17} and _native.YUV_LAYOUTS == {"NV12": 1, "I420": 2}
    buf = np.zeros(64, np.uint8)
    assert lib.rv_yuv422_to_bgr(None, buf.ctypes.data, buf[32:].ctypes.data, 1, 2, 2, 4, 6, 16, 0, None) == -1


# ---------------------------------------------------------------- GPU
def _ctx():
    import rvb200
    return rvb200.default_context(0)


def _torch(x):
    import torch
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _chain_ref(bgr, space, clip, grid, k, clahe=True):
    if not clahe:
        return np.stack([cv2.medianBlur(f, k) for f in bgr])
    if k == 0:
        return np.stack([cv2_chain.clahe_dehaze(f, space, clip, grid) for f in bgr])
    return np.stack([cv2_chain.chain(f, space, clip, grid, k) for f in bgr])


STAGE_SHAPES = [(4096, 4096), (2, 2), (7, 10), (135, 246), (270, 482), (1080, 1920), (2160, 3840)]


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("h,w", STAGE_SHAPES)
def test_gpu_stage_pageable_pinned_and_device(h, w, layout):
    import torch
    ctx = _ctx()
    if (h, w) == (4096, 4096):
        frames = Y.every_triple(layout)[None]
    else:
        frames = yuv_batch(3, h, w, layout, seed=h)
    want = bgr_of(frames, layout)
    assert np.array_equal(ctx.yuv422_to_bgr(frames, layout), want)
    pin, pout = ctx.pinned_empty(frames.shape), ctx.pinned_empty(want.shape)
    pin[...] = frames
    assert ctx.yuv422_to_bgr(pin, layout, out=pout) is pout and np.array_equal(pout, want)
    t = _torch(frames)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        got = ctx.yuv422_to_bgr(t, layout).cpu()
    assert np.array_equal(got.numpy(), want)
    got = ctx.yuv422_to_bgr(t, layout)                               # torch's default stream: synchronous on the context's stream
    assert np.array_equal(got.cpu().numpy(), want)


@pytest.mark.gpu
def test_gpu_stage_pitches_offsets_and_refusals():
    """Device frames at an odd pitch starting one byte into their allocation (the byte-wise path), output at an odd pitch, on a side
    stream; host memory with pitches; the C entries' refusals (RV_ERR_ARG, nothing written, nothing launched)."""
    import torch
    from rvb200 import _native as N
    ctx = _ctx()
    n, h, w = 3, 135, 246
    for layout in LAYOUTS:
        L = N.YUV422_LAYOUTS[layout]
        frames = yuv_batch(n, h, w, layout, seed=5)
        want = bgr_of(frames, layout)
        ip, op = 2 * w + 3, 3 * w + 5
        padded = np.zeros((n, h, ip), np.uint8)
        padded[..., :2 * w] = frames.reshape(n, h, 2 * w)
        din = torch.zeros(padded.size + 1, dtype=torch.uint8, device="cuda")
        din[1:] = _torch(padded.reshape(-1))
        dout = torch.zeros(n * h * op, dtype=torch.uint8, device="cuda")
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        ctx._ck(ctx._lib.rv_yuv422_to_bgr(ctx._h, C.c_void_p(din.data_ptr() + 1), C.c_void_p(dout.data_ptr()), n, h, w, ip, op, L,
                                          N.MEM_DEVICE, C.c_void_p(side.cuda_stream)))
        side.synchronize()
        got = dout.cpu().numpy().reshape(n, h, op)[:, :, :3 * w].reshape(n, h, w, 3)
        assert np.array_equal(got, want), layout
        hout = np.zeros((n, h, op), np.uint8)                          # host memory with pitches
        ctx._ck(ctx._lib.rv_yuv422_to_bgr(ctx._h, padded.ctypes.data, hout.ctypes.data, n, h, w, ip, op, L, N.MEM_HOST, None))
        assert np.array_equal(hout[:, :, :3 * w].reshape(n, h, w, 3), want), layout
    buf = np.zeros(4096, np.uint8)
    out = np.zeros(4096, np.uint8)
    dbuf = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    refused = [(5, 3, 6, 9, 16), (5, 0, 8, 12, 16), (0, 4, 8, 12, 17), (5, 4, 7, 12, 16), (5, 4, 8, 11, 17)] + \
              [(5, 4, 8, 12, layout) for layout in (0, 1, 2, 3, 15, 18)]
    for kind, src in ((N.MEM_HOST, buf.ctypes.data), (N.MEM_PINNED, buf.ctypes.data), (N.MEM_DEVICE, dbuf.data_ptr())):
        for h, w, ip, op, layout in refused:
            l0 = ctx.launch_count
            assert ctx._lib.rv_yuv422_to_bgr(ctx._h, C.c_void_p(src), out.ctypes.data, 1, h, w, ip, op, layout, kind, None) == -1, \
                (h, w, ip, op, layout)
            assert ctx.launch_count == l0 and not out.any()
        for layout in (16, 17):
            l0 = ctx.launch_count
            assert ctx._lib.rv_yuv422_to_bgr(ctx._h, C.c_void_p(src), None, 1, 5, 4, 8, 12, layout, kind, None) == -1
            assert ctx._lib.rv_yuv422_to_bgr(ctx._h, None, out.ctypes.data, 1, 5, 4, 8, 12, layout, kind, None) == -1
            assert ctx.launch_count == l0 and not out.any()
    assert ctx._lib.rv_yuv422_to_bgr(ctx._h, buf.ctypes.data, buf[30:].ctypes.data, 1, 5, 4, 8, 12, 16, N.MEM_HOST, None) == -1
    assert ctx._lib.rv_yuv422_to_bgr(ctx._h, buf.ctypes.data, buf[40:].ctypes.data, 1, 5, 4, 8, 12, 16, N.MEM_HOST, None) == 0
    for layout in (16, 17):                                            # the 4:2:0 entries keep their contract
        assert ctx._lib.rv_yuv420_to_bgr(ctx._h, buf.ctypes.data, out.ctypes.data, 1, 4, 4, 4, 12, layout, N.MEM_HOST, None) == -1
        assert b"bad YUV layout" in ctx._lib.rv_last_error(ctx._h) and not out.any()
    io = N.IO()
    io.in_, io.in_pitch, io.out, io.out_pitch = buf.ctypes.data, 8, out.ctypes.data, 12
    p = N.Params.make()
    for layout in (16, 17):
        l0 = ctx.launch_count
        assert ctx._lib.rv_submit_io_yuv(ctx._h, C.byref(io), layout, 1, 4, 4, C.byref(p)) == -1
        assert ctx.launch_count == l0 and not out.any()
        assert ctx._lib.rv_submit_io_fmt(ctx._h, C.byref(io), layout, 0, 1, 5, 4, C.byref(p)) == 0       # odd h, BGR out
        ctx.wait()
        io.out_pitch = 4
        assert ctx._lib.rv_submit_io_fmt(ctx._h, C.byref(io), layout, 1, 1, 5, 4, C.byref(p)) == -1      # odd h, NV12 out
        assert ctx._lib.rv_submit_io_fmt(ctx._h, C.byref(io), layout, 3, 1, 4, 4, C.byref(p)) == -1
        assert ctx._lib.rv_submit_io_fmt(ctx._h, C.byref(io), layout, 2, 1, 4, 4, C.byref(p)) == 0       # I420 out
        ctx.wait()
        io.in_pitch = 7
        assert ctx._lib.rv_submit_io_fmt(ctx._h, C.byref(io), layout, 2, 1, 4, 4, C.byref(p)) == -1      # in_pitch < 2w
        io.in_pitch, io.out_pitch = 8, 12
        out[:] = 0


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
def test_gpu_process_batch_parameter_matrix(layout):
    frames = yuv_batch(3, 97, 130, layout, seed=2)
    bgr = bgr_of(frames, layout)
    bad = []
    for space, k in itertools.product(("YCrCb", "LAB"), (0, 3, 5, 7, 9)):
        chain = [{"name": "CLAHEDehaze", "params": {"space": space, "clip_limit": 2.0, "tile_grid": 8}}]
        if k:
            chain.append({"name": "MedianDerain", "params": {"ksize": k}})
        if not np.array_equal(_pipe(chain).process_batch(frames, yuv=layout), _chain_ref(bgr, space, 2.0, 8, k)):
            bad.append((space, k))
    for k in (3, 5, 7, 9):
        if not np.array_equal(_pipe([{"name": "MedianDerain", "params": {"ksize": k}}]).process_batch(frames, yuv=layout),
                              _chain_ref(bgr, None, 0, 0, k, clahe=False)):
            bad.append(("median", k))
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
def test_gpu_gate_at_the_threshold(layout):
    """Exactly at the threshold a frame is skipped and comes back as its converted BGR; one unit above, it is processed.  One fused
    pass (the gate decided in the pipeline's histogram pass) and two passes (decided up front)."""
    ctx = _ctx()
    frames = yuv_batch(4, 63, 96, layout, seed=11)
    bgr = bgr_of(frames, layout)
    spans = ctx.gray_span(bgr)
    assert list(spans) == [int(g.max()) - int(g.min()) for g in (cv2.cvtColor(f, cv2.COLOR_BGR2GRAY) for f in bgr)]
    t = float(sorted(spans)[1])
    for chain, ref in ((STOCK, lambda f: cv2_chain.chain(f, "YCrCb", 2.0, 8, 5)),
                       (STOCK[1:] * 2, lambda f: cv2.medianBlur(cv2.medianBlur(f, 5), 5))):
        for thresh in (t, t + 1, t - 0.5):
            want = np.stack([ref(f) if s < thresh else f for f, s in zip(bgr, spans)])
            pipe = _pipe(chain, gate=True, thresh=thresh)
            assert np.array_equal(pipe.process_batch(frames, yuv=layout), want), (len(chain), thresh)
            assert np.array_equal(pipe.process_batch(frames, out="device", yuv=layout).numpy(), want), (len(chain), thresh)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
def test_gpu_disabled_empty_and_foreign_operator(layout):
    import rvb200

    class Flip(rvb200.PreprocessOp):
        def __call__(self, im):
            return np.ascontiguousarray(im[:, ::-1])
    frames = yuv_batch(2, 121, 200, layout, seed=13)
    bgr = bgr_of(frames, layout)
    for pipe in (_pipe(STOCK, enabled=False), _pipe([]), _pipe(STOCK, gate=True, enabled=False)):
        assert np.array_equal(pipe.process_batch(frames, yuv=layout), bgr)
        out = np.zeros_like(bgr)
        assert pipe.process_batch(frames, out=out, yuv=layout) is out and np.array_equal(out, bgr)
        assert np.array_equal(pipe.process_batch(frames, out="device", yuv=layout).numpy(), bgr)
        assert np.array_equal(pipe.process_batch(_torch(frames), yuv=layout).cpu().numpy(), bgr)
    pipe = _pipe(STOCK[::-1])
    pipe.ops.insert(1, Flip())
    want = np.stack([cv2_chain.clahe_dehaze(np.ascontiguousarray(cv2.medianBlur(f, 5)[:, ::-1]), "YCrCb", 2.0, 8) for f in bgr])
    assert np.array_equal(pipe.process_batch(frames, yuv=layout), want)
    assert np.array_equal(pipe.process_batch(frames, out="device", yuv=layout).numpy(), want)


@pytest.mark.gpu
def test_gpu_device_yuv422_refusals_come_before_the_conversion():
    """A torch CUDA 4:2:2 batch that the device path refuses (the gate, a foreign operator, a wrong `out`) raises ValueError before any
    kernel is enqueued."""
    import torch
    import rvb200

    class Flip(rvb200.PreprocessOp):
        def __call__(self, im):
            return np.ascontiguousarray(im[:, ::-1])
    ctx = _ctx()
    t = _torch(yuv_batch(2, 33, 48, "YUY2", seed=1))
    foreign = _pipe(STOCK)
    foreign.ops.insert(1, Flip())
    cases = [(_pipe(STOCK, gate=True), None, "gate"), (foreign, None, "CLAHEDehaze / MedianDerain"),
             (_pipe(STOCK), torch.empty((2, 33, 48, 2), dtype=torch.uint8, device="cuda"), "out must be"),
             (_pipe(STOCK), torch.empty((2, 33, 48, 3), dtype=torch.uint8), "out must be")]
    for pipe, out, msg in cases:
        l0 = ctx.launch_count
        with pytest.raises(ValueError, match=msg):
            pipe.process_batch(t, out=out, yuv="YUY2")
        assert ctx.launch_count == l0, msg
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
def test_gpu_outputs_pinned_device_and_torch_side_stream(layout):
    import torch
    ctx = _ctx()
    frames = yuv_batch(5, 270, 482, layout, seed=3)
    bgr = bgr_of(frames, layout)
    for chain in (STOCK, STOCK[::-1]):
        pipe = _pipe(chain)
        ref = _chain_ref(bgr, "YCrCb", 2.0, 8, 5) if chain is STOCK else \
            np.stack([cv2_chain.clahe_dehaze(cv2.medianBlur(f, 5), "YCrCb", 2.0, 8) for f in bgr])
        pin, pout = ctx.pinned_empty(frames.shape), ctx.pinned_empty(ref.shape)
        pin[...] = frames
        assert pipe.process_batch(pin, out=pout, yuv=layout) is pout and np.array_equal(pout, ref)
        assert np.array_equal(pipe.process_batch(pin, yuv=layout), ref)
        assert np.array_equal(pipe.process_batch(np.ascontiguousarray(frames[:, ::-1])[:, ::-1], yuv=layout), ref)
        dev = pipe.process_batch(pin, out="device", yuv=layout)
        assert dev.shape == ref.shape and np.array_equal(dev.numpy(), ref)
        side = torch.cuda.Stream()
        t = _torch(frames)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            res = pipe.process_batch(t, yuv=layout)
            tout = torch.empty(ref.shape, dtype=torch.uint8, device="cuda")
            res2 = pipe.process_batch(t, out=tout, yuv=layout)
            host = res.cpu()
        side.synchronize()
        assert res2 is tout and np.array_equal(host.numpy(), ref) and np.array_equal(tout.cpu().numpy(), ref)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
def test_gpu_64_frames_1080p(layout):
    """64 x 1080p: the host pipeline's chunks and its tapered first and last chunks, frames checked against cv2."""
    ctx = _ctx()
    frames = yuv_batch(64, 1080, 1920, layout, seed=21)
    bgr = bgr_of(frames, layout)
    pin = ctx.pinned_empty(frames.shape)
    pin[...] = frames
    got = _pipe(STOCK).process_batch(pin, yuv=layout)
    bad = [i for i in range(64) if not np.array_equal(got[i], cv2_chain.chain(bgr[i], "YCrCb", 2.0, 8, 5))]
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
def test_gpu_300_tiny_frames_cross_every_chunk_boundary(layout):
    import rvb200
    ctx = rvb200.Context(0)
    ctx.set_option("chunk_frames", 7)
    try:
        frames = yuv_batch(301, 5, 6, layout, seed=4)
        bgr = bgr_of(frames, layout)
        spans = [int(g.max()) - int(g.min()) for g in (cv2.cvtColor(f, cv2.COLOR_BGR2GRAY) for f in bgr)]
        for gate in (False, True):
            pipe = _pipe(STOCK, gate=gate, thresh=120.0, context=ctx)
            want = np.stack([cv2_chain.chain(f, "YCrCb", 2.0, 8, 5) if (not gate or s < 120) else f for f, s in zip(bgr, spans)])
            assert np.array_equal(pipe.process_batch(frames, yuv=layout), want), gate
        assert len(rvb200.chunk_schedule(301, 7)) > 40
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("h,w", [(1080, 1920), (270, 482)])
def test_gpu_process_batch_to_tensor(h, w, layout):
    """Equals the BGR call on the converted frames and letterbox(process_batch(bgr)): with and without want_frames and
    padding_present, host and "device", and with the gate (which takes the converted-first path)."""
    ctx = _ctx()
    frames = yuv_batch(5, h, w, layout, seed=8)
    bgr = bgr_of(frames, layout)
    proc = _chain_ref(bgr, "YCrCb", 2.0, 8, 5)
    want_t = np.stack([O.letterbox_f16(f, 640) for f in proc])
    for gate in (False, True):
        pipe = _pipe(STOCK, gate=gate, thresh=1e9)
        for want_frames in (False, True):
            t, full = pipe.process_batch_to_tensor(frames, want_frames=want_frames, yuv=layout)
            tb, fb = pipe.process_batch_to_tensor(bgr, want_frames=want_frames)
            assert np.array_equal(t.view(np.uint16), tb.view(np.uint16)) and np.array_equal(t.view(np.uint16), want_t.view(np.uint16))
            assert (full is None) == (not want_frames) and (full is None or (np.array_equal(full, fb) and np.array_equal(full, proc)))
            dev, full = pipe.process_batch_to_tensor(frames, want_frames=want_frames, out="device", yuv=layout)
            assert np.array_equal(dev.numpy().view(np.uint16), want_t.view(np.uint16))
            assert full is None or np.array_equal(full, proc)
            pinned = ctx.pinned_empty(want_t.shape, np.float16)
            ctx.fill_tensor_padding(pinned, h, w)
            t, _ = pipe.process_batch_to_tensor(frames, want_frames=want_frames, out=pinned, padding_present=True, yuv=layout)
            assert t is pinned and np.array_equal(pinned.view(np.uint16), want_t.view(np.uint16))


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("out_yuv", ["NV12", "I420"])
def test_gpu_4_2_0_output_from_4_2_2_input(layout, out_yuv):
    """out_yuv= with 4:2:2 input equals the 4:2:0 conversion of the BGR result, for the stock chain (rv_submit_io_fmt), two passes and
    the gate; numpy, pinned, "device" and torch."""
    import torch
    ctx = _ctx()
    frames = yuv_batch(4, 270, 482, layout, seed=9)
    bgr = bgr_of(frames, layout)
    for pipe in (_pipe(STOCK), _pipe(STOCK[::-1]), _pipe(STOCK, gate=True, thresh=1e9)):
        want = ctx.bgr_to_yuv420(pipe.process_batch(bgr), out_yuv)
        assert np.array_equal(pipe.process_batch(frames, yuv=layout, out_yuv=out_yuv), want)
        pin, pout = ctx.pinned_empty(frames.shape), ctx.pinned_empty(want.shape)
        pin[...] = frames
        assert pipe.process_batch(pin, out=pout, yuv=layout, out_yuv=out_yuv) is pout and np.array_equal(pout, want)
        assert np.array_equal(pipe.process_batch(frames, out="device", yuv=layout, out_yuv=out_yuv).numpy(), want)
        if not pipe._gate()[0]:
            assert np.array_equal(pipe.process_batch(_torch(frames), yuv=layout, out_yuv=out_yuv).cpu().numpy(), want)
    i420 = cv2.cvtColor(_pipe(STOCK).process_batch(bgr)[0], cv2.COLOR_BGR2YUV_I420)
    if out_yuv == "I420":
        assert np.array_equal(_pipe(STOCK).process_batch(frames, yuv=layout, out_yuv="I420")[0], i420)
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
def test_gpu_yuv422_job_is_the_bgr_job_plus_one_conversion_per_chunk(layout):
    """A 4:2:2 host job equals the BGR job on the converted frames, output for output, gate flag for gate flag and tensor for tensor,
    and launches exactly one conversion kernel per chunk more; with a tensor and with the gate, over several chunks; device input is
    read in place."""
    import torch
    import rvb200
    ctx = rvb200.Context(0)
    ctx.set_option("chunk_frames", 8)
    try:
        frames = yuv_batch(40, 91, 160, layout, seed=6)
        bgr = bgr_of(frames, layout)
        n, h, w, _ = bgr.shape
        chunks = len(rvb200.chunk_schedule(n, 8))
        for kw in ({"tensor": True}, {"gate": True}):
            p = rvb200.Params.make("YCrCb", 2.0, 8, 5, gate=kw.get("gate", False), gate_thresh=200.0)
            res = {}
            for src, yuv in ((bgr, None), (frames, layout)):
                out = np.zeros_like(bgr)
                tensor = np.zeros((n, 3, 640, 640), np.float16) if "tensor" in kw else None
                processed = np.zeros(n, np.int32)
                l0 = ctx.launch_count
                ctx.submit_io(src, p, out=out, tensor=tensor, processed=processed, yuv=yuv)
                ctx.wait()
                res[yuv] = (ctx.launch_count - l0, out, tensor, processed)
            (lb, ob, tb, pb), (ly, oy, ty, py) = res[None], res[layout]
            assert chunks > 1 and ly - lb == chunks, (kw, lb, ly, chunks)
            runs = [cv2_chain.low_contrast(f, 200.0) if "gate" in kw else True for f in bgr]
            assert list(pb) == [int(r) for r in runs], kw
            assert all(np.array_equal(ob[i], cv2_chain.chain(bgr[i], "YCrCb", 2.0, 8, 5)) for i in range(n) if pb[i])
            assert all(np.array_equal(ob[i], bgr[i]) for i in range(n) if not pb[i])
            assert np.array_equal(ob, oy) and np.array_equal(pb, py) and (tb is None or np.array_equal(tb.view(np.uint16), ty.view(np.uint16)))
            dy = _torch(frames)                                        # device input, read in place
            torch.cuda.synchronize()
            od = np.zeros_like(bgr)
            td = np.zeros_like(tb) if tb is not None else None
            l0 = ctx.launch_count
            ctx.submit_io(dy, p, shape=(n, h, w), out=od, tensor=td, yuv=layout)
            ctx.wait()
            assert ctx.launch_count - l0 == ly and np.array_equal(od, ob), kw
            assert td is None or np.array_equal(td.view(np.uint16), tb.view(np.uint16)), kw
    finally:
        ctx.close()


@pytest.mark.gpu
def test_gpu_batch_feeder_of_yuy2_frames_to_process_batch():
    """A capture loop of raw YUY2 frames: BatchFeeder(shape=(H, W, 2)) over a pinned ring hands its batches straight to
    process_batch(yuv="YUY2"), which equals the chain on the cv2-converted frames; the last batch is partial."""
    import rvb200
    from rvb200.io_video.capture import SyntheticReader
    h, w = 135, 240
    pool = list(yuv_batch(5, h, w, "YUY2", seed=400))
    nframes, batch = 19, 8
    pctx = rvb200.Context(0)
    try:
        pl = _pipe(STOCK, context=pctx)
        vs = rvb200.VideoSource(reader=SyntheticReader(pool, limit=nframes))
        feeder = rvb200.BatchFeeder(vs, batch=batch, shape=(h, w, 2), alloc=pctx.pinned_empty, depth=3)
        want = [cv2_chain.chain(cv2.cvtColor(f, cv2.COLOR_YUV2BGR_YUY2), "YCrCb", 2.0, 8, 5) for f in pool]
        out = pctx.pinned_empty((batch, h, w, 3))
        seen, counts = 0, []
        for b in feeder:
            assert pctx.mem_kind(b.frames) == rvb200._native.MEM_PINNED and b.frames.shape[1:] == (h, w, 2)
            res = pl.process_batch(b.frames, out=out[:b.count], yuv="YUY2")
            for i in range(b.count):
                assert np.array_equal(res[i], want[(seen + i) % len(pool)]), (seen, i)
            counts.append(b.count)
            seen += b.count
            feeder.release(b)
        assert seen == nframes and counts == [8, 8, 3]
    finally:
        pctx.close()
