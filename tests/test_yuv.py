"""YUV 4:2:0 (NV12, I420) decoder frames in the batch entries, converted to BGR on the GPU exactly as cv2.cvtColor does.

CPU tests pin the numpy restatement of the conversion (oracle/yuv420.py) on the live cv2 over all 2^24 (Y, U, V) triples, and check
that malformed batches raise ValueError before a context exists.  GPU tests require rv_yuv420_to_bgr, rv_submit_io_yuv and every
Python entry built on them to give, to the last bit, what the same call gives on the cv2-converted BGR frames.
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
from oracle import yuv420 as Y

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CODES = {"NV12": cv2.COLOR_YUV2BGR_NV12, "I420": cv2.COLOR_YUV2BGR_I420}
LAYOUTS = ["NV12", "I420"]
STOCK = [{"name": "CLAHEDehaze", "params": {"clip_limit": 2.0, "tile_grid": 8}}, {"name": "MedianDerain", "params": {"ksize": 5}}]


def to_yuv(bgr, layout):
    """cv2's own BGR -> I420 (re-laid out as NV12 when asked): decoder-like frames with smooth road content."""
    i420 = cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420)
    return i420 if layout == "I420" else Y.from_planes(*Y.planes(i420, "I420"), "NV12")


def yuv_batch(n, h, w, layout, seed=0):
    """n frames: road scenes (rvb200.synth, at most 8 distinct ones) where the size allows, random bytes otherwise; the chroma of the
    last frame is random."""
    from rvb200 import synth
    rng = np.random.default_rng(seed + 131 * h + w)
    if h >= 16 and w >= 16:
        pool = [to_yuv(f, layout) for f in synth.frame_pool(h, w, min(n, 8), base_seed=seed)]
        out = np.stack([pool[i % len(pool)] for i in range(n)])
        out[-1, h:] = rng.integers(0, 256, out[-1, h:].shape, dtype=np.uint8)
        return out
    return rng.integers(0, 256, (n, h * 3 // 2, w), dtype=np.uint8)


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
    up = lambda p: np.repeat(np.repeat(p.astype(np.int64), 2, 0), 2, 1)         # noqa: E731
    assert len(np.unique((y.astype(np.int64) << 16) | (up(u) << 8) | up(v))) == 1 << 24
    assert np.array_equal(Y.yuv420_to_bgr(frame, layout), cv2.cvtColor(frame, CODES[layout]))


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("h,w", [(270, 482), (6, 10), (2, 2), (2, 4098), (134, 2)])
def test_oracle_equals_cv2_on_ragged_sizes(layout, h, w):
    rng = np.random.default_rng(h * w)
    frame = rng.integers(0, 256, (h * 3 // 2, w), dtype=np.uint8)
    assert np.array_equal(Y.yuv420_to_bgr(frame, layout), cv2.cvtColor(frame, CODES[layout]))
    assert np.array_equal(Y.from_planes(*Y.planes(frame, layout), layout), frame)


def test_cv2_refuses_an_odd_width():
    with pytest.raises(cv2.error):
        cv2.cvtColor(np.zeros((6, 9), np.uint8), cv2.COLOR_YUV2BGR_NV12)


def test_malformed_yuv_batches_raise_before_a_context_exists(monkeypatch):
    import rvb200
    from rvb200 import _native
    from rvb200.preprocess import pipeline as P

    def no_context(*a, **k):
        raise AssertionError("a context was created")
    monkeypatch.setattr(P, "default_context", no_context)
    monkeypatch.setattr(_native, "default_context", no_context)
    monkeypatch.setattr(_native.Context, "__init__", no_context)
    good = np.zeros((2, 6, 10), np.uint8)
    cases = [(np.zeros((6, 10), np.uint8), "NV12", "ndim"), (np.zeros((2, 4, 6, 10), np.uint8), "NV12", "(B,H,W,C)"),
             (np.zeros((2, 4, 10, 3), np.uint8), "I420", "(B,H,W,C)"), (good.astype(np.uint16), "NV12", "uint8"),
             (good.astype(np.float32), "I420", "uint8"), (np.zeros((2, 7, 10), np.uint8), "NV12", "multiple of 3"),
             (np.zeros((2, 6, 9), np.uint8), "I420", "even width"), (np.zeros((2, 0, 10), np.uint8), "NV12", "empty"),
             (np.zeros((2, 6, 0), np.uint8), "I420", "empty"), (good, "NV21", "NV12"), (good, "nv12", "NV12"), (good, "", "NV12")]
    for chain, gate in ((STOCK, False), (STOCK, True), (STOCK[1:] * 2, False), ([], False)):
        pipe = _pipe(chain, gate=gate)
        for frames, yuv, msg in cases:
            msg = "shape" if msg == "ndim" else msg
            for call in (lambda: pipe.process_batch(frames, yuv=yuv), lambda: pipe.process_batch(frames, out="device", yuv=yuv),
                         lambda: pipe.process_batch_to_tensor(frames, yuv=yuv)):
                with pytest.raises(ValueError, match=re.escape(msg)):
                    call()
    with pytest.raises(ValueError):
        _pipe(STOCK).process_batch(good, out="host", yuv="NV12")
    with pytest.raises(ValueError):
        _pipe(STOCK).process_batch(good, out=np.zeros((2, 4, 10, 3), np.uint8)[:, ::-1], yuv="NV12")
    with pytest.raises(ValueError):
        _pipe(STOCK).process_batch_to_tensor(good, out=np.zeros((2, 3, 64, 64), np.float32), yuv="NV12")
    assert _native.check_yuv_frames((5, 1080 * 3 // 2, 1920), True, "I420") == (2, 5, 1080, 1920)
    assert rvb200.PreprocessPipeline({"chain": STOCK})._fused_segment() is not None


def test_header_declares_and_library_exports_the_yuv_entries():
    from rvb200 import _native
    header = open(os.path.join(ROOT, "include", "rv_b200.h")).read()
    lib = _native.load_library()
    for name in ("rv_yuv420_to_bgr", "rv_submit_io_yuv"):
        assert re.search(rf"\bint {name}\(", header) and name in _native.EXPORTS and hasattr(lib, name)
    assert "enum rv_yuv { RV_YUV_NV12 = 1, RV_YUV_I420 = 2 };" in header and _native.YUV_LAYOUTS == {"NV12": 1, "I420": 2}
    buf = np.zeros(64, np.uint8)
    io = _native.IO()
    p = _native.Params.make()
    assert lib.rv_yuv420_to_bgr(None, buf.ctypes.data, buf.ctypes.data, 1, 2, 2, 2, 6, 1, 0, None) == -1
    assert lib.rv_submit_io_yuv(None, C.byref(io), 1, 1, 2, 2, C.byref(p)) == -1


# ---------------------------------------------------------------- GPU
def _ctx():
    import rvb200
    return rvb200.default_context(0)


def _torch(x):
    import torch
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


STAGE_SHAPES = [(4096, 4096), (2, 2), (6, 10), (270, 482), (540, 4098), (1080, 1920), (2160, 3840)]


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
    assert np.array_equal(ctx.yuv420_to_bgr(frames, layout), want)
    pin, pout = ctx.pinned_empty(frames.shape), ctx.pinned_empty(want.shape)
    pin[...] = frames
    assert ctx.yuv420_to_bgr(pin, layout, out=pout) is pout and np.array_equal(pout, want)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        got = ctx.yuv420_to_bgr(_torch(frames), layout).cpu()
    assert np.array_equal(got.numpy(), want)
    got = ctx.yuv420_to_bgr(_torch(frames), layout)                  # torch's default stream: synchronous on the context's stream
    assert np.array_equal(got.cpu().numpy(), want)


@pytest.mark.gpu
def test_gpu_stage_pitches_offsets_side_stream_and_refusals():
    """NV12 device frames at an odd pitch starting one byte into their allocation, output at an odd pitch, on a side stream; I420
    from an odd offset; the C entry's refusals (RV_ERR_ARG, nothing written)."""
    import torch
    from rvb200 import _native as N
    ctx = _ctx()
    n, h, w = 3, 134, 246
    for layout, ip in (("NV12", w + 3), ("I420", w)):
        frames = yuv_batch(n, h, w, layout, seed=5)
        want = bgr_of(frames, layout)
        padded = np.zeros((n, h * 3 // 2, ip), np.uint8)
        padded[..., :w] = frames
        op = 3 * w + 5
        din = torch.zeros(padded.size + 1, dtype=torch.uint8, device="cuda")
        din[1:] = _torch(padded.reshape(-1))
        dout = torch.zeros(n * h * op, dtype=torch.uint8, device="cuda")
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        ctx._ck(ctx._lib.rv_yuv420_to_bgr(ctx._h, C.c_void_p(din.data_ptr() + 1), C.c_void_p(dout.data_ptr()), n, h, w, ip, op,
                                          N.YUV_LAYOUTS[layout], N.MEM_DEVICE, C.c_void_p(side.cuda_stream)))
        side.synchronize()
        got = dout.cpu().numpy().reshape(n, h, op)[:, :, :3 * w].reshape(n, h, w, 3)
        assert np.array_equal(got, want), layout
        hout = np.zeros((n, h, op), np.uint8)                          # host memory with pitches
        ctx._ck(ctx._lib.rv_yuv420_to_bgr(ctx._h, padded.ctypes.data, hout.ctypes.data, n, h, w, ip, op, N.YUV_LAYOUTS[layout],
                                          N.MEM_HOST, None))
        assert np.array_equal(hout[:, :, :3 * w].reshape(n, h, w, 3), want), layout
    buf = np.zeros(4096, np.uint8)
    out = np.zeros(4096, np.uint8)
    for (h, w, ip, op, layout) in ((5, 4, 4, 12, 1), (4, 5, 5, 15, 1), (0, 4, 4, 12, 1), (4, 0, 4, 12, 2), (4, 4, 3, 12, 1),
                                   (4, 4, 4, 11, 1), (4, 4, 6, 12, 2), (4, 4, 4, 12, 0), (4, 4, 4, 12, 3)):
        assert ctx._lib.rv_yuv420_to_bgr(ctx._h, buf.ctypes.data, out.ctypes.data, 1, h, w, ip, op, layout, N.MEM_HOST, None) == -1
        assert not out.any()
    assert ctx._lib.rv_yuv420_to_bgr(ctx._h, buf.ctypes.data, buf[20:].ctypes.data, 1, 4, 4, 4, 12, 1, N.MEM_HOST, None) == -1
    dbuf = torch.zeros(64, dtype=torch.uint8, device="cuda")
    for kind, src in ((N.MEM_HOST, buf.ctypes.data), (N.MEM_PINNED, buf.ctypes.data), (N.MEM_DEVICE, dbuf.data_ptr())):
        for layout in (1, 2):                                          # no output: refused, nothing launched
            l0 = ctx.launch_count
            assert ctx._lib.rv_yuv420_to_bgr(ctx._h, C.c_void_p(src), None, 1, 4, 4, 4, 12, layout, kind, None) == -1
            assert ctx.launch_count == l0 and b"null frame pointer" in ctx._lib.rv_last_error(ctx._h)
    torch.cuda.synchronize()
    io = N.IO()
    io.in_, io.in_pitch, io.out, io.out_pitch = buf.ctypes.data, 4, out.ctypes.data, 12
    assert ctx._lib.rv_submit_io_yuv(ctx._h, C.byref(io), 0, 1, 4, 4, C.byref(N.Params.make())) == -1
    assert ctx._lib.rv_submit_io_yuv(ctx._h, C.byref(io), 2, 1, 4, 4, C.byref(N.Params.make())) == 0
    ctx.wait()
    io.in_pitch = 6
    assert ctx._lib.rv_submit_io_yuv(ctx._h, C.byref(io), 2, 1, 4, 4, C.byref(N.Params.make())) == -1


def _chain_ref(bgr, space, clip, grid, k, clahe=True):
    if not clahe:
        return np.stack([cv2.medianBlur(f, k) for f in bgr])
    return np.stack([cv2_chain.chain(f, space, clip, grid, k) for f in bgr])


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
def test_gpu_process_batch_parameter_matrix(layout):
    frames = yuv_batch(3, 96, 130, layout, seed=2)
    bgr = bgr_of(frames, layout)
    bad = []
    for space, grid, clip, k in itertools.product(("YCrCb", "LAB"), (2, 8, 16), (0.0, 2.0), (3, 5, 7, 9)):
        chain = [{"name": "CLAHEDehaze", "params": {"space": space, "clip_limit": clip, "tile_grid": grid}},
                 {"name": "MedianDerain", "params": {"ksize": k}}]
        if not np.array_equal(_pipe(chain).process_batch(frames, yuv=layout), _chain_ref(bgr, space, clip, grid, k)):
            bad.append((space, grid, clip, k))
    assert not bad, bad
    for k in (3, 5, 7, 9):
        assert np.array_equal(_pipe([{"name": "MedianDerain", "params": {"ksize": k}}]).process_batch(frames, yuv=layout),
                              _chain_ref(bgr, None, 0, 0, k, clahe=False)), k
    for space in ("YCrCb", "LAB"):
        got = _pipe([{"name": "CLAHEDehaze", "params": {"space": space}}]).process_batch(frames, yuv=layout)
        assert np.array_equal(got, np.stack([cv2_chain.clahe_dehaze(f, space, 2.0, 8) for f in bgr])), space


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
def test_gpu_gate_at_the_threshold(layout):
    """Exactly at the threshold a frame is skipped and comes back as its converted BGR; one unit above, it is processed.  One fused
    pass (the gate decided in the pipeline's histogram pass) and two passes (decided up front)."""
    ctx = _ctx()
    frames = yuv_batch(4, 64, 96, layout, seed=11)
    bgr = bgr_of(frames, layout)
    spans = ctx.gray_span(bgr)
    spans_cv2 = [int(g.max()) - int(g.min()) for g in (cv2.cvtColor(f, cv2.COLOR_BGR2GRAY) for f in bgr)]
    assert list(spans) == spans_cv2
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
    frames = yuv_batch(2, 120, 200, layout, seed=13)
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
    two = _pipe(STOCK[::-1])
    assert np.array_equal(two.process_batch(frames, yuv=layout),
                          np.stack([cv2_chain.clahe_dehaze(cv2.medianBlur(f, 5), "YCrCb", 2.0, 8) for f in bgr]))


@pytest.mark.gpu
def test_gpu_device_yuv_refusals_come_before_the_conversion():
    """A torch CUDA YUV batch that the device path refuses (the gate, a foreign operator, a wrong `out`) raises ValueError before any
    kernel is enqueued."""
    import torch
    import rvb200

    class Flip(rvb200.PreprocessOp):
        def __call__(self, im):
            return np.ascontiguousarray(im[:, ::-1])
    ctx = _ctx()
    t = _torch(yuv_batch(2, 32, 48, "NV12", seed=1))
    foreign = _pipe(STOCK)
    foreign.ops.insert(1, Flip())
    cases = [(_pipe(STOCK, gate=True), None, "gate"), (foreign, None, "CLAHEDehaze / MedianDerain"),
             (_pipe(STOCK), torch.empty((2, 32, 48, 4), dtype=torch.uint8, device="cuda"), "out must be"),
             (_pipe(STOCK), torch.empty((2, 32, 48, 3), dtype=torch.uint8), "out must be")]
    for pipe, out, msg in cases:
        l0 = ctx.launch_count
        with pytest.raises(ValueError, match=msg):
            pipe.process_batch(t, out=out, yuv="NV12")
        assert ctx.launch_count == l0, msg
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
def test_gpu_outputs_pinned_device_and_torch_side_stream(layout):
    import torch
    ctx = _ctx()
    frames = yuv_batch(5, 270, 482, layout, seed=3)
    want = _chain_ref(bgr_of(frames, layout), "YCrCb", 2.0, 8, 5)
    for chain in (STOCK, STOCK[::-1]):
        pipe = _pipe(chain)
        ref = want if chain is STOCK else np.stack([cv2_chain.clahe_dehaze(cv2.medianBlur(f, 5), "YCrCb", 2.0, 8)
                                                    for f in bgr_of(frames, layout)])
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
    """64 x 1080p: the host pipeline's 4-frame chunks and its tapered first and last chunks, frames checked against cv2."""
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
        frames = yuv_batch(301, 4, 6, layout, seed=4)
        bgr = bgr_of(frames, layout)
        for gate in (False, True):
            pipe = _pipe(STOCK, gate=gate, thresh=120.0, context=ctx)
            spans = [int(g.max()) - int(g.min()) for g in (cv2.cvtColor(f, cv2.COLOR_BGR2GRAY) for f in bgr)]
            want = np.stack([cv2_chain.chain(f, "YCrCb", 2.0, 8, 5) if (not gate or s < 120) else f for f, s in zip(bgr, spans)])
            assert np.array_equal(pipe.process_batch(frames, yuv=layout), want), gate
        assert len(rvb200.chunk_schedule(301, 7)) > 40
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("h,w", [(1080, 1920), (270, 482)])
def test_gpu_process_batch_to_tensor(h, w, layout):
    """Equals the BGR call on the converted frames (itself pinned to letterbox(process_batch(bgr))): with and without want_frames and
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
def test_gpu_yuv_job_is_the_bgr_job_plus_one_conversion_per_chunk(layout):
    """A YUV host job equals the BGR job on the converted frames, output for output, and launches exactly one conversion kernel per
    chunk more; with a tensor and with the gate.  The BGR job equals cv2 and rv_chain_u8 and launches what the build before the YUV
    input launched for it (4 with the tensor, 6 with the gate: one chunk), so adding the YUV input left it alone."""
    import torch
    import rvb200
    from rvb200 import _native as N
    ctx = _ctx()
    frames = yuv_batch(40, 90, 160, layout, seed=6)
    bgr = bgr_of(frames, layout)
    n, h, w, _ = bgr.shape
    chunks = len(rvb200.chunk_schedule(n, min(n, (24 << 20) // (3 * w * h))))
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
        assert chunks == 1 and lb == (4 if "tensor" in kw else 6), (kw, lb)
        assert ly - lb == chunks, (kw, lb, ly, chunks)
        runs = [cv2_chain.low_contrast(f, 200.0) if "gate" in kw else True for f in bgr]
        assert list(pb) == [int(r) for r in runs], kw
        assert all(np.array_equal(ob[i], cv2_chain.chain(bgr[i], "YCrCb", 2.0, 8, 5)) for i in range(n) if pb[i])
        assert all(np.array_equal(ob[i], bgr[i]) for i in range(n) if not pb[i])
        assert np.array_equal(ob, oy) and np.array_equal(pb, py) and (tb is None or np.array_equal(tb.view(np.uint16), ty.view(np.uint16)))
        dy = _torch(frames)                                            # device input, read in place
        torch.cuda.synchronize()
        od = np.zeros_like(bgr)
        td = np.zeros_like(tb) if tb is not None else None
        ctx.submit_io(dy, p, shape=(n, h, w), out=od, tensor=td, yuv=layout)
        ctx.wait()
        assert np.array_equal(od, ob) and (td is None or np.array_equal(td.view(np.uint16), tb.view(np.uint16))), kw
        ref = np.zeros_like(bgr)
        flag = np.zeros(n, np.int32)
        ctx._ck(ctx._lib.rv_chain_u8(ctx._h, bgr.ctypes.data, ref.ctypes.data, n, h, w, 3 * w, 3 * w, C.byref(p), N.MEM_HOST,
                                     flag.ctypes.data_as(C.POINTER(C.c_int32)), None))
        assert np.array_equal(ref, ob) and np.array_equal(flag, pb), kw
