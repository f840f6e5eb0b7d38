"""BGRA / BGRx and single-channel frames: CLAHEDehaze, MedianDerain and the gate as cv2 computes them on those arrays.

cv2 ignores the fourth channel in cvtColor (BGR2YCrCb / BGR2LAB / BGR2GRAY) and drops it from the CLAHE result, filters every channel
of medianBlur on its own, and has no colour conversion for one channel.  CPU tests pin those facts on the live cv2 and check that
what cv2 refuses raises ValueError before anything reaches the GPU; GPU tests require rv_chain_ex / rv_gray_span_ex and every Python
entry built on them to equal cv2 to the last bit.
"""
import ctypes as C
import itertools

import cv2
import numpy as np
import pytest

from oracle import cv2_chain

SHAPES = [(1080, 1920), (1080, 1923), (123, 457), (5, 300), (2, 2), (1, 1)]
GRIDS = [2, 7, 8, 16, 64]
CLIPS = [0.0, 0.001, 2.0, 40.0]
ALPHAS = ["random", "zero", "full"]


def bgra(h, w, alpha="random", seed=0, dtype=np.uint8):
    rng = np.random.default_rng(seed + 7919 * h + w)
    top = 256 if dtype == np.uint8 else 65536
    img = rng.integers(0, top, (h, w, 4), dtype=dtype)
    if h >= 4 and w >= 4:                                       # smooth content next to noise: CLAHE tiles differ
        yy, xx = np.mgrid[0:h, 0:w]
        smooth = ((yy * 3 + xx) * (top - 1) // max(1, 3 * (h - 1) + (w - 1))).astype(dtype)
        img[: h // 2, :, 0] = smooth[: h // 2]
        img[: h // 2, :, 1] = smooth[: h // 2] // 2
    if alpha == "zero":
        img[..., 3] = 0
    elif alpha == "full":
        img[..., 3] = top - 1
    return img


def gray(h, w, seed=0, dtype=np.uint8):
    rng = np.random.default_rng(seed + 31 * h + w)
    return rng.integers(0, 256 if dtype == np.uint8 else 65536, (h, w), dtype=dtype)


def _pipe(chain, gate=False, thresh=20.0):
    import rvb200
    return rvb200.PreprocessPipeline({"enabled": True, "chain": chain,
                                      "auto_gate": {"enable_low_contrast_gate": gate, "contrast_thresh": thresh}})


def _params(space="YCrCb", clip=2.0, grid=8, k=5, clahe=True, gate=False, thresh=20.0):
    import rvb200
    return rvb200.Params.make(space, clip, grid, k, clahe=clahe, gate=gate, gate_thresh=thresh)


STOCK = [{"name": "CLAHEDehaze", "params": {"clip_limit": 2.0, "tile_grid": 8}}, {"name": "MedianDerain", "params": {"ksize": 5}}]


# ---------------------------------------------------------------- CPU: what cv2 does with these arrays
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16])
def test_cv2_ignores_alpha_and_filters_channels_alone(dtype):
    img = bgra(37, 53, seed=1, dtype=dtype)
    other = img.copy()
    other[..., 3] = ~other[..., 3]
    codes = [cv2.COLOR_BGR2YCrCb, cv2.COLOR_BGR2GRAY] + ([cv2.COLOR_BGR2LAB] if dtype == np.uint8 else [])
    for code in codes:
        assert np.array_equal(cv2.cvtColor(img, code), cv2.cvtColor(other, code))
        assert np.array_equal(cv2.cvtColor(img, code), cv2.cvtColor(np.ascontiguousarray(img[..., :3]), code))
    for k in ((3, 5, 7, 9) if dtype == np.uint8 else (3, 5)):
        whole = cv2.medianBlur(img, k)
        assert whole.shape == img.shape
        for c in range(4):
            assert np.array_equal(whole[..., c], cv2.medianBlur(np.ascontiguousarray(img[..., c]), k))
    out = cv2_chain.clahe_dehaze(img, "YCrCb", 2.0, 8)
    assert out.shape == (37, 53, 3) and np.array_equal(out, cv2_chain.clahe_dehaze(np.ascontiguousarray(img[..., :3]), "YCrCb", 2.0, 8))


@pytest.mark.parametrize("dtype", [np.uint8, np.uint16])
def test_cv2_refuses_colour_on_one_channel(dtype):
    for g in (gray(9, 11, dtype=dtype), gray(9, 11, dtype=dtype)[..., None]):
        for code in (cv2.COLOR_BGR2YCrCb, cv2.COLOR_BGR2GRAY):
            with pytest.raises(cv2.error):
                cv2.cvtColor(g, code)
        assert cv2.medianBlur(g, 3).shape == (9, 11)


# ---------------------------------------------------------------- CPU: shapes and refusals before the GPU
def test_as_frame_shapes_and_the_validators_that_stay_strict():
    from rvb200.preprocess.base import as_bgr_frame, as_bgr_u8, as_frame
    base = np.arange(6 * 8 * 4, dtype=np.uint8).reshape(6, 8, 4)
    for view in (base, base[::2], base[:, ::-2]):
        f = as_frame(view)
        assert f.flags.c_contiguous and f.shape == view.shape and np.array_equal(f, view)
    g = np.arange(48, dtype=np.uint16).reshape(6, 8)
    assert as_frame(g).shape == (6, 8, 1) and as_frame(g[..., None]).shape == (6, 8, 1)
    for bad in (np.zeros((4, 4, 2), np.uint8), np.zeros((4, 4, 4), np.float32), np.zeros((0, 4, 4), np.uint8), np.zeros((4, 4, 5), np.uint8)):
        with pytest.raises(ValueError):
            as_frame(bad)
    for bad in (np.zeros((4, 4), np.uint8), np.zeros((4, 4, 4), np.uint8)):
        with pytest.raises(ValueError):
            as_bgr_u8(bad)
    with pytest.raises(ValueError):
        as_bgr_frame(np.zeros((4, 4, 4), np.uint16))


def test_refusals_raise_value_error_before_the_gpu():
    import rvb200
    g8 = gray(8, 8)
    for g in (g8, g8[..., None], g8.astype(np.uint16)):
        with pytest.raises(ValueError, match="single-channel"):
            rvb200.CLAHEDehaze()(g)
        with pytest.raises(ValueError, match="single-channel"):
            _pipe(STOCK)(g)
        with pytest.raises(ValueError, match="single-channel"):
            _pipe(STOCK[1:], gate=True)(g)                  # the gate's BGR2GRAY
    b16 = bgra(8, 8, dtype=np.uint16)
    with pytest.raises(ValueError, match="LAB"):
        rvb200.CLAHEDehaze(space="LAB")(b16)
    for k in (7, 9):
        with pytest.raises(ValueError, match="ksize"):
            rvb200.MedianDerain(ksize=k)(b16)
        with pytest.raises(ValueError, match="ksize"):
            rvb200.MedianDerain(ksize=k)(gray(8, 8, dtype=np.uint16))
    batch = np.stack([bgra(8, 8)] * 2)
    with pytest.raises(ValueError, match="mix"):
        _pipe(STOCK, gate=True).process_batch(batch)
    with pytest.raises(ValueError, match="mix"):
        _pipe(STOCK, gate=True).process_batch(batch, out="device")
    with pytest.raises(ValueError):
        _pipe(STOCK[1:]).process_batch(g8)                  # 3-D: never read as a batch of gray frames
    with pytest.raises(ValueError):
        _pipe(STOCK[1:]).process_batch(np.zeros((2, 8, 8, 2), np.uint8))
    with pytest.raises(ValueError, match="single-channel"):
        _pipe(STOCK).process_batch(g8[None, ..., None])
    with pytest.raises(ValueError, match="single-channel"):
        _pipe(STOCK[1:], gate=True).process_batch(g8[None, ..., None])
    with pytest.raises(ValueError):
        _pipe(STOCK).process_batch_to_tensor(batch)         # the detector tensor stays 3-channel


def test_c_abi_null_context():
    """rv_chain_ex / rv_gray_span_ex refuse a null context with RV_ERR_ARG (no GPU needed)."""
    from rvb200 import _native as N
    lib = N.load_library()
    buf = np.zeros(64, np.uint8)
    p = _params()
    assert lib.rv_chain_ex(None, buf.ctypes.data, buf.ctypes.data, 1, 2, 2, 8, 6, 8, 4, C.byref(p), N.MEM_HOST, None, None) == -1
    assert lib.rv_gray_span_ex(None, buf.ctypes.data, 1, 2, 2, 8, 8, 4, buf.ctypes.data, N.MEM_HOST) == -1


# ---------------------------------------------------------------- GPU
def _ctx():
    import rvb200
    return rvb200.default_context(0)


def _ex(ctx, frames, p, out_c, kind=None, processed=None):
    """rv_chain_ex on a contiguous host batch; returns the result and the return code."""
    from rvb200 import _native as N
    n, h, w, c = frames.shape
    sb = frames.dtype.itemsize
    out = np.zeros((n, h, w, out_c), frames.dtype)
    pp = processed.ctypes.data_as(C.POINTER(C.c_int32)) if processed is not None else None
    rc = ctx._lib.rv_chain_ex(ctx._h, frames.ctypes.data, out.ctypes.data, n, h, w, c * sb * w, out_c * sb * w, 8 * sb, c, C.byref(p),
                              N.MEM_HOST if kind is None else kind, pp, None)
    return out, rc


@pytest.mark.gpu
@pytest.mark.parametrize("h,w", SHAPES)
def test_gpu_bgra8_chain_matrix(h, w):
    """YCrCb and LAB x k 0/3/5/7/9 x grid x clip on BGRA uint8, alpha random / 0 / 255 in turn: 0 LSB against cv2."""
    ctx = _ctx()
    bad = []
    for i, (space, k, grid, clip) in enumerate(itertools.product(("YCrCb", "LAB"), (0, 3, 5, 7, 9), GRIDS, CLIPS)):
        if (h, w) == (1080, 1920) or i % 3 == 0 or h < 200:
            img = bgra(h, w, ALPHAS[i % 3], seed=i % 5)
            got = ctx.chain(img[None], _params(space, clip, grid, k))[0]
            if got.shape != (h, w, 3) or not np.array_equal(got, cv2_chain.chain(img, space, clip, grid, k)):
                bad.append((space, k, grid, clip))
    assert not bad, bad


@pytest.mark.gpu
def test_gpu_bgra8_4k_and_alpha_never_matters():
    ctx = _ctx()
    img = bgra(2160, 3840, seed=3)
    for space, k in (("YCrCb", 5), ("LAB", 3)):
        assert np.array_equal(ctx.chain(img[None], _params(space, 2.0, 16, k))[0], cv2_chain.chain(img, space, 2.0, 16, k))
    base = bgra(270, 481, seed=4)
    frames = np.stack([base] + [np.concatenate([base[..., :3], np.full_like(base[..., :1], a)], -1) for a in (0, 1, 128, 255)])
    frames[-1, ..., 3] = np.random.default_rng(5).integers(0, 256, frames.shape[1:3])
    for space, k, grid in (("YCrCb", 0, 8), ("LAB", 5, 7), ("YCrCb", 9, 64)):
        res = ctx.chain(frames, _params(space, 2.0, grid, k))
        for r in res[1:]:
            assert np.array_equal(r, res[0]), (space, k, grid)
        assert np.array_equal(res[0], cv2_chain.chain(base, space, 2.0, grid, k))


@pytest.mark.gpu
@pytest.mark.parametrize("h,w", SHAPES)
def test_gpu_bgra16_chain(h, w):
    ctx = _ctx()
    bad = []
    for i, (k, grid, clip) in enumerate(itertools.product((0, 3, 5), GRIDS, CLIPS)):
        if h < 200 or i % 3 == 0:
            img = bgra(h, w, ALPHAS[i % 3], seed=i % 5, dtype=np.uint16)
            got = ctx.chain(img[None], _params("YCrCb", clip, grid, k))[0]
            if got.dtype != np.uint16 or not np.array_equal(got, cv2_chain.chain(img, "YCrCb", clip, grid, k)):
                bad.append((k, grid, clip))
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16])
@pytest.mark.parametrize("h,w", SHAPES)
def test_gpu_median_gray_and_bgra(h, w, dtype):
    """Median on gray and on all four BGRA channels, every k cv2 has at this depth: the op, the pipeline and the batch."""
    import rvb200
    ctx = _ctx()
    for k in ((3, 5, 7, 9) if dtype == np.uint8 else (3, 5)):
        g = gray(h, w, seed=k, dtype=dtype)
        want = cv2.medianBlur(g, k)
        assert np.array_equal(rvb200.MedianDerain(ksize=k)(g), want), k
        got = rvb200.MedianDerain(ksize=k)(g[..., None])
        assert got.shape == (h, w) and np.array_equal(got, want), k
        assert np.array_equal(ctx.median(g[None, ..., None], k)[..., 0][0], want)
        b = bgra(h, w, ALPHAS[k % 3], seed=k, dtype=dtype)
        got = rvb200.MedianDerain(ksize=k)(b)
        assert got.shape == (h, w, 4) and np.array_equal(got, cv2.medianBlur(b, k)), k


@pytest.mark.gpu
@pytest.mark.parametrize("k", [3, 5, 7, 9])
def test_gpu_gray_median_two_level_frames(k):
    """0-1 principle on the single-plane kernel: two grey levels at densities around 1/2 put many windows exactly at the median
    threshold; the frame spans several tiles so every task, lane and tile edge is hit."""
    ctx = _ctx()
    h, w = 200, 380
    for dens, lo, hi, seed in [(0.5, 0, 255, 1), (0.47, 17, 18, 2), (0.53, 254, 255, 3), (0.5, 0, 1, 4)]:
        rng = np.random.RandomState(100 * k + seed)
        g = np.where(rng.rand(h, w) < dens, hi, lo).astype(np.uint8)
        assert np.array_equal(ctx.median(g[None, ..., None], k)[0, ..., 0], cv2.medianBlur(g, k)), (k, dens)
        b = np.where(rng.rand(h, w, 4) < dens, hi, lo).astype(np.uint8)
        assert np.array_equal(ctx.median(b[None], k)[0], cv2.medianBlur(b, k)), (k, dens)
        if k <= 5:
            g16 = g.astype(np.uint16) * 257 + 1
            assert np.array_equal(ctx.median(g16[None, ..., None], k)[0, ..., 0], cv2.medianBlur(g16, k)), (k, dens)


@pytest.mark.gpu
def test_gpu_c_abi_refuses_what_cv2_refuses():
    """The C entries apply cv2's refusals themselves (RV_ERR_ARG, nothing written), without the Python layer in front."""
    ctx = _ctx()
    g8 = gray(8, 8)[None, ..., None]
    b8 = bgra(8, 8)[None]
    b16 = bgra(8, 8, dtype=np.uint16)[None]
    cases = [(g8, _params(k=3), 3),                                   # CLAHE on one channel
             (g8, _params(k=3, clahe=False, gate=True), 1),           # the gate on one channel
             (b16, _params("LAB", k=3), 3),                           # LAB at 16 bits
             (b16, _params(k=7, clahe=False), 4), (b16, _params(k=9, clahe=False), 4),
             (b16, _params(gate=True, k=3), 3), (b8, _params(gate=True), 3),     # gate + CLAHE on 4 channels without `processed`
             (b8, _params(k=0, clahe=False), 4)]                      # nothing to do
    for frames, p, oc in cases:
        out, rc = _ex(ctx, frames, p, oc)
        assert rc == -1 and not out.any(), (frames.shape, frames.dtype, p.space, p.ksize, p.clahe, p.gate_enable)
    span = np.zeros(1, np.int32)
    assert ctx._lib.rv_gray_span_ex(ctx._h, g8.ctypes.data, 1, 8, 8, 8, 8, 1, span.ctypes.data, 0) == -1


@pytest.mark.gpu
def test_gpu_ex_channels3_equals_the_3_channel_entries():
    """rv_chain_ex(channels=3) is rv_chain_u8 / rv_chain_u16: same output, same launches."""
    from rvb200 import _native as N
    ctx = _ctx()
    for dtype in (np.uint8, np.uint16):
        frames = np.stack([bgra(135, 241, seed=i, dtype=dtype)[..., :3] for i in range(3)])
        n, h, w, _ = frames.shape
        fn = ctx._lib.rv_chain_u8 if dtype == np.uint8 else ctx._lib.rv_chain_u16
        sb = frames.dtype.itemsize
        for p in (_params(k=5), _params(k=3, clahe=False), _params(k=0, gate=True, thresh=1e9)):
            flag_a, flag_b = np.zeros(n, np.int32), np.zeros(n, np.int32)
            out_a = np.zeros_like(frames)
            l0 = ctx.launch_count
            ctx._ck(fn(ctx._h, frames.ctypes.data, out_a.ctypes.data, n, h, w, 3 * sb * w, 3 * sb * w, C.byref(p), N.MEM_HOST,
                       flag_a.ctypes.data_as(C.POINTER(C.c_int32)), None))
            l1 = ctx.launch_count
            out_b, rc = _ex(ctx, frames, p, 3, processed=flag_b)
            ctx._ck(rc)
            assert ctx.launch_count - l1 == l1 - l0 and np.array_equal(out_a, out_b) and np.array_equal(flag_a, flag_b), (dtype, p.ksize)


@pytest.mark.gpu
def test_gpu_memory_kinds_pitches_and_alignment():
    import rvb200
    from rvb200 import _native as N
    ctx = _ctx()
    frames = np.stack([bgra(135, 241, seed=i) for i in range(3)])
    n, h, w, _ = frames.shape
    p = _params("LAB", 2.0, 7, 5)
    want = np.stack([cv2_chain.chain(f, "LAB", 2.0, 7, 5) for f in frames])
    assert np.array_equal(ctx.chain(frames, p), want)                                      # pageable
    pin_in, pin_out = ctx.pinned_empty(frames.shape), ctx.pinned_empty((n, h, w, 3))
    pin_in[...] = frames
    assert ctx.chain(pin_in, p, out=pin_out) is pin_out and np.array_equal(pin_out, want)  # pinned
    # device: row pitches neither 4*w nor a multiple of 16, and an input that starts one byte into its allocation
    ip, op = 4 * w + 7, 3 * w + 5
    host_in = np.zeros((n, h, ip), np.uint8)
    host_in[:, :, :4 * w] = frames.reshape(n, h, 4 * w)
    din = rvb200.DeviceArray(ctx, (n * h * ip + 1,), np.uint8)
    dout = rvb200.DeviceArray(ctx, (n * h * op,), np.uint8)
    ctx._ck(ctx._lib.rv_memcpy(ctx._h, din.ptr + 1, host_in.ctypes.data, host_in.nbytes, 0))
    for pp, exp, oc in ((p, want, 3), (_params(k=7, clahe=False), np.stack([cv2.medianBlur(f, 7) for f in frames]), 4)):
        opp = op if oc == 3 else 4 * w + 9
        dout = rvb200.DeviceArray(ctx, (n * h * opp,), np.uint8)
        ctx._ck(ctx._lib.rv_chain_ex(ctx._h, C.c_void_p(din.ptr + 1), C.c_void_p(dout.ptr), n, h, w, ip, opp, 8, 4, C.byref(pp),
                                     N.MEM_DEVICE, None, None))
        got = dout.numpy().reshape(n, h, opp)[:, :, :oc * w].reshape(n, h, w, oc)
        assert np.array_equal(got, exp), oc
    # host memory with pitches
    out = np.zeros((n, h, op), np.uint8)
    ctx._ck(ctx._lib.rv_chain_ex(ctx._h, host_in.ctypes.data, out.ctypes.data, n, h, w, ip, op, 8, 4, C.byref(p), N.MEM_HOST, None, None))
    assert np.array_equal(out[:, :, :3 * w].reshape(n, h, w, 3), want)
    # 16-bit: odd pitch refused; short output pitch refused
    f16 = frames.astype(np.uint16)
    with pytest.raises(ValueError):
        ctx._ck(ctx._lib.rv_chain_ex(ctx._h, f16.ctypes.data, out.ctypes.data, n, h, w, 8 * w + 1, 6 * w, 16, 4, C.byref(_params()),
                                     N.MEM_HOST, None, None))
    with pytest.raises(ValueError):
        ctx._ck(ctx._lib.rv_chain_ex(ctx._h, frames.ctypes.data, out.ctypes.data, n, h, w, 4 * w, 3 * w - 1, 8, 4, C.byref(p),
                                     N.MEM_HOST, None, None))
    for bits, ch in ((8, 2), (12, 4)):
        with pytest.raises(ValueError):
            ctx._ck(ctx._lib.rv_chain_ex(ctx._h, frames.ctypes.data, out.ctypes.data, n, h, w, 4 * w, 4 * w, bits, ch, C.byref(p),
                                         N.MEM_HOST, None, None))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16])
def test_gpu_batches_numpy_device_and_torch(dtype):
    import torch
    ctx = _ctx()
    tdt = torch.uint8 if dtype == np.uint8 else torch.uint16
    b4 = np.stack([bgra(270, 481, ALPHAS[i % 3], seed=i, dtype=dtype) for i in range(4)])
    g1 = np.stack([gray(270, 481, seed=i, dtype=dtype)[..., None] for i in range(4)])
    cases = [(STOCK, b4, np.stack([cv2_chain.chain(f, "YCrCb", 2.0, 8, 5) for f in b4])),
             (STOCK[1:], b4, np.stack([cv2.medianBlur(f, 5) for f in b4])),
             (STOCK[1:], g1, np.stack([cv2.medianBlur(f, 5)[..., None] for f in g1])),
             # median first keeps 4 channels, then CLAHE gives 3
             (STOCK[::-1], b4, np.stack([cv2_chain.clahe_dehaze(cv2.medianBlur(f, 5), "YCrCb", 2.0, 8) for f in b4]))]
    for chain, frames, want in cases:
        pipe = _pipe(chain)
        got = pipe.process_batch(frames)
        assert got.shape == want.shape and np.array_equal(got, want)
        out = np.empty_like(want)
        assert pipe.process_batch(frames, out=out) is out and np.array_equal(out, want)
        pin = ctx.pinned_empty(frames.shape, dtype)
        pin[...] = frames
        assert np.array_equal(pipe.process_batch(pin), want)
        assert np.array_equal(pipe.process_batch(np.ascontiguousarray(frames[:, ::-1])[:, ::-1]), want)     # strided view of the same pixels
        dev = pipe.process_batch(frames, out="device")
        assert dev.shape == want.shape and np.array_equal(dev.numpy(), want)
        t = torch.from_numpy(frames.view(np.int8 if dtype == np.uint8 else np.int16)).view(tdt).cuda()
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            res = pipe.process_batch(t)
            tout = torch.empty(want.shape, dtype=tdt, device="cuda")
            res2 = pipe.process_batch(t, out=tout)
            host = res.view(torch.int8 if dtype == np.uint8 else torch.int16).cpu()
        side.synchronize()
        assert res.dtype == tdt and res2 is tout
        assert np.array_equal(host.numpy().view(dtype), want)
        assert np.array_equal(tout.view(torch.int8 if dtype == np.uint8 else torch.int16).cpu().numpy().view(dtype), want)
        for i in range(len(frames)):
            per = pipe(frames[i] if frames.shape[3] == 4 else frames[i, ..., 0])
            assert np.array_equal(per.reshape(want[i].shape), want[i]), i


@pytest.mark.gpu
def test_gpu_many_tiny_gray_frames():
    """40,000 gray 3x5 frames in one call: 157 frame groups of at most 256 frames, each checked against cv2."""
    ctx = _ctx()
    rng = np.random.default_rng(9)
    g = rng.integers(0, 256, (40000, 3, 5, 1), dtype=np.uint8)
    got = ctx.median(g, 3)
    for i in (0, 1, 32767, 32768, 39999):
        assert np.array_equal(got[i, ..., 0], cv2.medianBlur(g[i, ..., 0], 3)), i
    want = np.stack([cv2.medianBlur(f[..., 0], 3) for f in g])
    assert np.array_equal(got[..., 0], want)


@pytest.mark.gpu
def test_gpu_gate_on_bgra_at_the_threshold():
    """The gate's span ignores alpha; exactly at the threshold the frame is skipped (span < thresh runs).  Per frame, a skipped
    frame is the input object; in a median-only batch it is copied through with its alpha."""
    ctx = _ctx()
    img = bgra(64, 96, seed=11)
    img[..., 3] = 0
    img[0, 0, 3] = 255                                           # alpha spans the full range
    span = int(cv2.cvtColor(img, cv2.COLOR_BGR2GRAY).max()) - int(cv2.cvtColor(img, cv2.COLOR_BGR2GRAY).min())
    assert int(ctx.gray_span(img[None])[0]) == span
    img16 = img.astype(np.uint16) * 257
    span16 = int(cv2.cvtColor(img16, cv2.COLOR_BGR2GRAY).max()) - int(cv2.cvtColor(img16, cv2.COLOR_BGR2GRAY).min())
    assert int(ctx.gray_span(np.stack([img16, img16]))[1]) == span16
    for thresh, runs in ((span, False), (span + 0.5, True), (span + 1, True), (span - 0.5, False)):
        res = _pipe(STOCK, True, thresh)(img)
        assert (res is img) != runs, thresh
        if runs:
            assert np.array_equal(res, cv2_chain.chain(img, "YCrCb", 2.0, 8, 5))
        res = _pipe(STOCK[1:], True, thresh)(img)
        assert (res is img) != runs and np.array_equal(res, cv2.medianBlur(img, 5) if runs else img), thresh
        batch = _pipe(STOCK[1:], True, thresh).process_batch(np.stack([img, img]))
        assert np.array_equal(batch[1], cv2.medianBlur(img, 5) if runs else img), thresh
        # two passes: the gate decides up front, then both run on the selected frames
        batch = _pipe(STOCK[1:] * 2, True, thresh).process_batch(np.stack([img, img]))
        assert np.array_equal(batch[0], cv2.medianBlur(cv2.medianBlur(img, 5), 5) if runs else img), thresh
        # C ABI: gate + CLAHE on BGRA needs `processed`; skipped frames are left as they were
        flag = np.full(2, 7, np.int32)
        out, rc = _ex(ctx, np.stack([img, img]), _params(gate=True, thresh=thresh), 3, processed=flag)
        assert rc == 0 and list(flag) == [int(runs)] * 2
        assert np.array_equal(out[0], cv2_chain.chain(img, "YCrCb", 2.0, 8, 5) if runs else np.zeros_like(out[0])), thresh
        flag16 = np.zeros(1, np.int32)
        out16, rc = _ex(ctx, img16[None], _params(gate=True, thresh=span16 + (1 if runs else 0), k=3), 3, processed=flag16)
        assert rc == 0 and flag16[0] == int(runs)
        if runs:
            assert np.array_equal(out16[0], cv2_chain.chain(img16, "YCrCb", 2.0, 8, 3))
    _, rc = _ex(ctx, img[None], _params(gate=True), 3)
    assert rc == -1


@pytest.mark.gpu
def test_gpu_foreign_operator_between_passes_on_bgra():
    import rvb200

    class Flip(rvb200.PreprocessOp):
        def __call__(self, im):
            return np.ascontiguousarray(im[:, ::-1])
    img = bgra(120, 200, seed=13)
    pipe = _pipe(STOCK[::-1])
    pipe.ops.insert(1, Flip())
    want = cv2_chain.clahe_dehaze(np.ascontiguousarray(cv2.medianBlur(img, 5)[:, ::-1]), "YCrCb", 2.0, 8)
    assert np.array_equal(pipe(img), want)
    assert np.array_equal(pipe.process_batch(np.stack([img, img]))[1], want)
