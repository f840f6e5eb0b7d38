"""16-bit frames: the stock chain on (H,W,3) uint16 BGR, as cv2 computes it on CV_16U input.

CPU tests pin the restatement in oracle/rv_oracle16.py against the live cv2: the integer colour formulas, the
65,536-bin CLAHE over a shape / grid / clip / content matrix, the tile LUTs, the median and the whole chain; and they check that
what cv2 has no 16-bit path for (LAB, median k 7 / 9) raises ValueError before anything reaches the GPU.  GPU tests require the
CUDA path (rv_chain_u16) to equal cv2 to the last bit on the same matrix and through every memory kind and entry point.
"""
import itertools

import cv2
import numpy as np
import pytest

from oracle import cv2_chain
from oracle import rv_oracle16 as O

SHAPES = [(1080, 1920), (1080, 1923), (123, 457), (5, 300), (2, 2), (1, 1)]
GRIDS = [2, 7, 8, 16, 64]
CLIPS = [0.0, 0.001, 2.0, 40.0, 1000.0]
CONTENTS = ["uniform16", "12bit", "smooth", "constant", "twolevel"]
EDGE = np.array([0, 1, 2, 255, 256, 32767, 32768, 65534, 65535], np.int64)


def frame(kind, h, w, seed=0):
    rng = np.random.default_rng(seed + 7919 * h + w)
    if kind == "uniform16":
        return rng.integers(0, 65536, (h, w, 3), dtype=np.uint16)
    if kind == "12bit":
        return rng.integers(0, 4096, (h, w, 3), dtype=np.uint16)
    if kind == "smooth":
        yy, xx = np.mgrid[0:h, 0:w]
        v = ((yy * 3 + xx) * 255 // max(1, 3 * (h - 1) + (w - 1)))[..., None] + np.array([0, 20, 40])
        return ((np.clip(v, 0, 255) << 8) | rng.integers(0, 256, (h, w, 3))).astype(np.uint16)
    if kind == "constant":
        return np.full((h, w, 3), (40000, 41000, 39000), np.uint16)
    if kind == "twolevel":
        yy, xx = np.mgrid[0:h, 0:w]
        m = ((yy // 7 + xx // 11) % 2).astype(bool)[..., None]
        return np.where(m, np.array([1000, 1200, 900], np.uint16), np.array([60000, 58000, 61000], np.uint16))
    raise ValueError(kind)


def colours():
    rng = np.random.default_rng(1)
    rnd = rng.integers(0, 65536, (1 << 20, 3), dtype=np.uint16)
    grid = np.array(list(itertools.product(EDGE, repeat=3)), np.uint16)
    return np.concatenate([rnd, grid])[None]        # (1, N, 3) image


def _d(x):
    return (x + 8192) >> 14


# ---------------------------------------------------------------- CPU: the restated arithmetic against cv2
def test_ycrcb16_formulas_match_cv2_and_oracle():
    img = colours()
    B, G, R = (img[..., i].astype(np.int64) for i in range(3))
    Y = _d(1868 * B + 9617 * G + 4899 * R)
    delta = 32768 << 14
    Cr = np.clip(_d((R - Y) * 11682 + delta), 0, 65535)
    Cb = np.clip(_d((B - Y) * 9241 + delta), 0, 65535)
    want = np.stack([Y, Cr, Cb], -1)
    for x in (1868 * B + 9617 * G + 4899 * R, (R - Y) * 11682 + delta, (B - Y) * 9241 + delta):
        assert np.abs(x + 8192).max() < 1.08e9                  # int32 arithmetic is enough
    assert np.array_equal(cv2.cvtColor(img, cv2.COLOR_BGR2YCrCb), want)
    assert np.array_equal(O.bgr2ycrcb16(img), want)


def test_ycrcb16_inverse_matches_cv2_and_oracle():
    img = colours()
    Y, Cr, Cb = (img[..., i].astype(np.int64) for i in range(3))
    b = np.clip(Y + _d((Cb - 32768) * 29049), 0, 65535)
    g = np.clip(Y + _d((Cb - 32768) * -5636 + (Cr - 32768) * -11698), 0, 65535)
    r = np.clip(Y + _d((Cr - 32768) * 22987), 0, 65535)
    want = np.stack([b, g, r], -1)
    assert np.array_equal(cv2.cvtColor(img, cv2.COLOR_YCrCb2BGR), want)
    assert np.array_equal(O.ycrcb2bgr16(img), want)


def test_gray16_uses_the_8bit_coefficients():
    img = colours()
    B, G, R = (img[..., i].astype(np.int64) for i in range(3))
    want = (3735 * B + 19235 * G + 9798 * R + 16384) >> 15
    assert np.array_equal(cv2.cvtColor(img, cv2.COLOR_BGR2GRAY), want)
    assert np.array_equal(O.bgr2gray16(img), want)
    ycc_y = _d(1868 * B + 9617 * G + 4899 * R)
    assert np.mean(ycc_y != want) > 0.3           # the 14-bit Y formula is not the gray formula
    span = O.gray_span16(img)
    assert span == int(want.max()) - int(want.min())


def _clahe_cases():
    """The full 6 x 5 x 5 x 5 matrix is run on the GPU; on the CPU every shape x grid pair with a rotating clip and content,
    plus all clip x content pairs at 1080p grid 8 and the 1080p / 123x457 cases of the 16-bit CLAHE derivation."""
    cases = set()
    for si, (h, w) in enumerate(SHAPES):
        for gi, g in enumerate(GRIDS):
            cases.add((h, w, g, CLIPS[(si + gi) % 5], CONTENTS[(si + 2 * gi) % 5]))
    for c, k in itertools.product(CLIPS, CONTENTS):
        cases.add((1080, 1920, 8, c, k))
    for c in (0.0, 2.0, 40.0, 1000.0):
        for k in ("uniform16", "smooth", "12bit"):
            cases.add((1080, 1920, 8, c, k))
        cases.add((123, 457, 7, c, "uniform16"))
    return sorted(cases)


@pytest.mark.parametrize("h,w,grid,clip,content", _clahe_cases())
def test_clahe16_oracle_matches_cv2(h, w, grid, clip, content):
    plane = np.ascontiguousarray(frame(content, h, w)[..., 0])
    want = cv2.createCLAHE(clipLimit=clip, tileGridSize=(grid, grid)).apply(plane)
    assert np.array_equal(O.clahe16_plane(plane, clip, grid), want)


@pytest.mark.parametrize("clip", [0.0, 2.0, 40.0])
def test_clahe16_tile_lut_matches_cv2_on_tile_crops(clip):
    """cv2 never exposes its LUTs; a 1x1-grid CLAHE of one tile's crop reads that tile's LUT back at every value present."""
    plane = np.ascontiguousarray(frame("smooth", 240, 320)[..., 1])
    grid = 4
    th, tw = 240 // grid, 320 // grid
    for ty, tx in ((0, 0), (1, 2), (3, 3)):
        crop = np.ascontiguousarray(plane[ty * th:(ty + 1) * th, tx * tw:(tx + 1) * tw])
        lut = O.clahe16_tile_lut(plane, grid, clip, ty, tx)
        assert np.array_equal(lut[crop], cv2.createCLAHE(clipLimit=clip, tileGridSize=(1, 1)).apply(crop))


def test_clahe16_default_clip_redistributes_every_tile():
    """At clip 2.0 a 1080p grid-8 tile has clipInt = max(1, int(2 * 32400 / 65536)) = 1: every bin is cut, so the
    redistribution carries the whole LUT."""
    plane = np.ascontiguousarray(frame("uniform16", 1080, 1920)[..., 2])
    assert max(1, int(2.0 * 240 * 135 / 65536)) == 1
    want = cv2.createCLAHE(clipLimit=2.0, tileGridSize=(8, 8)).apply(plane)
    assert np.array_equal(O.clahe16_plane(plane, 2.0, 8), want)


@pytest.mark.parametrize("k", [3, 5])
@pytest.mark.parametrize("content", ["uniform16", "smooth", "twolevel"])
def test_median16_oracle_matches_cv2(k, content):
    img = frame(content, 97, 203)
    assert np.array_equal(O.median16(img, k), cv2.medianBlur(img, k))


def test_median16_k5_is_the_exact_median():
    img = frame("uniform16", 40, 60)
    pad = np.pad(img, ((2, 2), (2, 2), (0, 0)), mode="edge")
    win = np.lib.stride_tricks.sliding_window_view(pad, (5, 5), axis=(0, 1))
    assert np.array_equal(np.median(win.reshape(40, 60, 3, 25), -1).astype(np.uint16), cv2.medianBlur(img, 5))


@pytest.mark.parametrize("k", [0, 3, 5])
@pytest.mark.parametrize("shape,grid,clip", [((270, 480), 8, 2.0), ((123, 457), 7, 40.0), ((64, 64), 2, 0.0)])
def test_chain16_oracle_matches_cv2_chain(k, shape, grid, clip):
    img = frame("smooth", *shape)
    assert np.array_equal(O.chain16(img, clip, grid, k), cv2_chain.chain(img, "YCrCb", clip, grid, k))


def test_cv2_has_no_16bit_lab_or_large_median():
    """The scope of the 16-bit path follows cv2: these raise cv2.error in the reference."""
    img = frame("uniform16", 16, 16)
    with pytest.raises(cv2.error):
        cv2.cvtColor(img, cv2.COLOR_BGR2LAB)
    for k in (7, 9):
        with pytest.raises(cv2.error):
            cv2.medianBlur(img, k)


# ---------------------------------------------------------------- CPU: what is refused, refused before the GPU
def _pipe(chain, gate=False):
    import rvb200
    return rvb200.PreprocessPipeline({"enabled": True, "chain": chain,
                                      "auto_gate": {"enable_low_contrast_gate": gate, "contrast_thresh": 20.0}})


LAB_CHAIN = [{"name": "CLAHEDehaze", "params": {"space": "LAB"}}, {"name": "MedianDerain", "params": {"ksize": 3}}]
K7_CHAIN = [{"name": "CLAHEDehaze", "params": {}}, {"name": "MedianDerain", "params": {"ksize": 7}}]


def test_u16_lab_and_large_k_raise_value_error_before_the_gpu():
    import rvb200
    img = frame("uniform16", 8, 8)
    with pytest.raises(ValueError, match="LAB"):
        rvb200.CLAHEDehaze(space="LAB")(img)
    with pytest.raises(ValueError, match="tile_grid"):
        rvb200.CLAHEDehaze(tile_grid=65)(img)
    for k in (7, 9):
        with pytest.raises(ValueError, match="ksize"):
            rvb200.MedianDerain(ksize=k)(img)
    with pytest.raises(ValueError, match="LAB"):
        _pipe(LAB_CHAIN)(img)
    with pytest.raises(ValueError, match="ksize"):
        _pipe(K7_CHAIN, gate=True)(img)
    with pytest.raises(ValueError, match="ksize"):
        _pipe(K7_CHAIN).process_batch(img[None])
    with pytest.raises(ValueError, match="LAB"):
        _pipe(LAB_CHAIN).process_batch(img[None], out="device")
    with pytest.raises(ValueError, match="8-bit"):
        _pipe(K7_CHAIN[:1]).process_batch_to_tensor(img[None])


def test_u16_validator_and_u8_validator():
    from rvb200.preprocess.base import as_bgr_frame, as_bgr_u8
    img = frame("uniform16", 6, 5)[:, ::-1]
    out = as_bgr_frame(img)
    assert out.dtype == np.uint16 and out.flags.c_contiguous and np.array_equal(out, img)
    with pytest.raises(ValueError):
        as_bgr_u8(img)
    with pytest.raises(ValueError):
        as_bgr_frame(img[..., :2])
    with pytest.raises(ValueError):
        as_bgr_frame(img.astype(np.int32))


# ---------------------------------------------------------------- GPU: bit-exact against cv2
def _ctx():
    import rvb200
    return rvb200.default_context(0)


def _params(clip=2.0, grid=8, k=5, clahe=True, gate=False, thresh=20.0):
    import rvb200
    return rvb200.Params.make("YCrCb", clip, grid, k, clahe=clahe, gate=gate, gate_thresh=thresh)


@pytest.mark.gpu
@pytest.mark.parametrize("h,w", SHAPES)
def test_gpu_clahe16_matrix(h, w):
    """CLAHEDehaze alone on every grid x clip x content at each shape: 0 LSB against cv2."""
    ctx = _ctx()
    bad = []
    for content in CONTENTS:
        img = frame(content, h, w)
        for grid, clip in itertools.product(GRIDS, CLIPS):
            got = ctx.clahe_dehaze(img[None], "YCrCb", clip, grid)[0]
            want = cv2_chain.clahe_dehaze(img, "YCrCb", clip, grid)
            if not np.array_equal(got, want):
                bad.append((content, grid, clip, int(np.count_nonzero(got != want))))
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("k", [3, 5])
@pytest.mark.parametrize("h,w", SHAPES)
def test_gpu_chain16_and_median16(h, w, k):
    ctx = _ctx()
    bad = []
    for content in CONTENTS:
        img = frame(content, h, w, seed=k)
        if not np.array_equal(ctx.median(img[None], k)[0], cv2.medianBlur(img, k)):
            bad.append(("median", content))
        for grid, clip in ((8, 2.0), (7, 40.0), (64, 0.001), (2, 1000.0), (16, 0.0)):
            got = ctx.chain(img[None], _params(clip, grid, k))[0]
            if not np.array_equal(got, cv2_chain.chain(img, "YCrCb", clip, grid, k)):
                bad.append(("chain", content, grid, clip))
    assert not bad, bad


@pytest.mark.gpu
def test_gpu_chain16_4k():
    """4K at grid 16, and a constant 4K frame at grid 8: 129,600 pixels of one value per tile (more than a u16 counter holds)."""
    ctx = _ctx()
    img = frame("uniform16", 2160, 3840)
    for k in (0, 5):
        assert np.array_equal(ctx.chain(img[None], _params(2.0, 16, k))[0], cv2_chain.chain(img, "YCrCb", 2.0, 16, k))
    const = frame("constant", 2160, 3840)
    for clip in (0.0, 2.0, 40.0):
        assert np.array_equal(ctx.chain(const[None], _params(clip, 8, 3))[0], cv2_chain.chain(const, "YCrCb", clip, 8, 3))


@pytest.mark.gpu
def test_gpu_batch_equals_per_frame():
    ctx = _ctx()
    frames = np.stack([frame(c, 270, 480, seed=i) for i, c in enumerate(CONTENTS * 2)])
    for p in (_params(2.0, 8, 5), _params(40.0, 7, 0), _params(k=3, clahe=False)):
        batch = ctx.chain(frames, p)
        for i in range(len(frames)):
            assert np.array_equal(batch[i], ctx.chain(frames[i:i + 1], p)[0]), i
            want = cv2_chain.chain(frames[i], "YCrCb", p.clip_limit, p.grid, p.ksize) if p.clahe else cv2.medianBlur(frames[i], p.ksize)
            assert np.array_equal(batch[i], want), i


@pytest.mark.gpu
def test_gpu_memory_kinds_and_pitches():
    import ctypes as C
    import rvb200
    from rvb200 import _native as N
    ctx = _ctx()
    frames = np.stack([frame("smooth", 135, 241, seed=i) for i in range(3)])
    p = _params(2.0, 8, 5)
    want = np.stack([cv2_chain.chain(f, "YCrCb", 2.0, 8, 5) for f in frames])
    assert np.array_equal(ctx.chain(frames, p), want)                                  # pageable
    pin_in = ctx.pinned_empty(frames.shape, np.uint16)
    pin_out = ctx.pinned_empty(frames.shape, np.uint16)
    pin_in[...] = frames
    assert np.array_equal(ctx.chain(pin_in, p, out=pin_out), want)                     # pinned
    assert pin_out.ctypes.data == ctx.chain(pin_in, p, out=pin_out).ctypes.data
    # device buffers with row pitches that are neither 6*w nor a multiple of 16 (must stay even)
    n, h, w, _ = frames.shape
    ip, op = 6 * w + 10, 6 * w + 34
    din = rvb200.DeviceArray(ctx, (n * h * ip,), np.uint8)
    dout = rvb200.DeviceArray(ctx, (n * h * op,), np.uint8)
    host_in = np.zeros((n, h, ip), np.uint8)
    host_in[:, :, :6 * w] = frames.view(np.uint8).reshape(n, h, 6 * w)
    ctx._ck(ctx._lib.rv_memcpy(ctx._h, din.ptr, host_in.ctypes.data, host_in.nbytes, 0))
    ctx.chain_u16_device(din.ptr, dout.ptr, n, h, w, p, in_pitch=ip, out_pitch=op)
    got = dout.numpy().reshape(n, h, op)[:, :, :6 * w].copy().view(np.uint16).reshape(frames.shape)
    assert np.array_equal(got, want)
    # the same through rv_chain_u16 with host pitches
    out = np.zeros((n, h, op), np.uint8)
    ctx._ck(ctx._lib.rv_chain_u16(ctx._h, host_in.ctypes.data, out.ctypes.data, n, h, w, ip, op, C.byref(p), N.MEM_HOST, None, None))
    assert np.array_equal(out[:, :, :6 * w].copy().view(np.uint16).reshape(frames.shape), want)
    # odd pitch and LAB are refused by the C ABI itself
    with pytest.raises(ValueError):
        ctx._ck(ctx._lib.rv_chain_u16(ctx._h, host_in.ctypes.data, out.ctypes.data, n, h, w, ip - 1, op, C.byref(p), N.MEM_HOST, None,
                                      None))
    lab = rvb200.Params.make("LAB", 2.0, 8, 3)
    with pytest.raises(ValueError):
        ctx._ck(ctx._lib.rv_chain_u16(ctx._h, host_in.ctypes.data, out.ctypes.data, n, h, w, ip, op, C.byref(lab), N.MEM_HOST, None,
                                      None))


@pytest.mark.gpu
def test_gpu_torch_uint16_on_a_side_stream():
    import torch
    ctx_frames = np.stack([frame("uniform16", 270, 480, seed=i) for i in range(4)])
    pipe = _pipe([{"name": "CLAHEDehaze", "params": {"clip_limit": 2.0, "tile_grid": 8}},
                  {"name": "MedianDerain", "params": {"ksize": 5}}])
    want = np.stack([cv2_chain.chain(f, "YCrCb", 2.0, 8, 5) for f in ctx_frames])
    t = torch.from_numpy(ctx_frames.view(np.int16)).view(torch.uint16).cuda()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        res = pipe.process_batch(t)
        host = res.view(torch.int16).cpu()
    side.synchronize()
    assert res.dtype == torch.uint16
    assert np.array_equal(host.numpy().view(np.uint16), want)
    dev = pipe.process_batch(ctx_frames, out="device")
    assert dev.dtype == np.uint16 and np.array_equal(dev.numpy(), want)
    out = np.empty_like(ctx_frames)
    assert pipe.process_batch(ctx_frames, out=out) is out and np.array_equal(out, want)


@pytest.mark.gpu
def test_gpu_ops_and_pipeline_on_strided_u16():
    import rvb200
    base = frame("smooth", 300, 500)
    view = base[10:250:2, 480:20:-3]                    # row- and column-strided, negative stride
    cont = np.ascontiguousarray(view)
    got = rvb200.CLAHEDehaze(clip_limit=3.0, tile_grid=7)(view)
    assert got.dtype == np.uint16 and got.flags.c_contiguous and got.flags.writeable
    assert np.array_equal(got, cv2_chain.clahe_dehaze(cont, "YCrCb", 3.0, 7))
    got = rvb200.MedianDerain(ksize=4)(view)            # coerced to 5
    assert np.array_equal(got, cv2.medianBlur(cont, 5))
    # foreign operator between the fused pair's ops: three passes, the middle one is called as in the reference
    class Flip(rvb200.PreprocessOp):
        def __call__(self, im):
            return np.ascontiguousarray(im[:, ::-1])
    flip = Flip()
    pipe = _pipe([{"name": "CLAHEDehaze", "params": {}}, {"name": "MedianDerain", "params": {"ksize": 3}}])
    pipe.ops.insert(1, flip)
    want = cv2.medianBlur(np.ascontiguousarray(cv2_chain.clahe_dehaze(cont, "YCrCb", 2.0, 8)[:, ::-1]), 3)
    assert np.array_equal(pipe(view), want)
    assert np.array_equal(pipe.process_batch(np.stack([cont, cont]))[1], want)


@pytest.mark.gpu
def test_gpu_gate16_at_the_threshold():
    """The gate compares the 16-bit gray span (which exceeds 8-bit spans by far) with the threshold: span < thresh runs."""
    img = frame("twolevel", 64, 96)
    span = O.gray_span16(img)
    assert span > 1024
    ctx = _ctx()
    assert int(ctx.gray_span(img[None])[0]) == span
    chain = [{"name": "CLAHEDehaze", "params": {}}, {"name": "MedianDerain", "params": {"ksize": 3}}]
    want = cv2_chain.chain(img, "YCrCb", 2.0, 8, 3)
    for thresh, runs in ((span, False), (span + 0.5, True), (span + 1, True), (span - 0.5, False)):
        pipe = rvb200_pipe(chain, thresh)
        res = pipe(img)
        assert (res is img) != runs and np.array_equal(res, want if runs else img), thresh
        flag = np.zeros(2, np.int32)
        res = ctx.chain(np.stack([img, img]), _params(2.0, 8, 3, gate=True, thresh=thresh), processed=flag)
        assert list(flag) == [int(runs)] * 2 and np.array_equal(res[1], want if runs else img)
        # not one fused pass: the gate runs on its own, then the two ops
        pipe = rvb200_pipe(chain[:1] + [{"name": "MedianDerain", "params": {"ksize": 5}}, {"name": "MedianDerain", "params": {"ksize": 3}}],
                           thresh)
        batch = pipe.process_batch(np.stack([img, img]))
        want2 = cv2.medianBlur(cv2.medianBlur(want_clahe(img), 5), 3) if runs else img
        assert np.array_equal(batch[0], want2)


def rvb200_pipe(chain, thresh):
    import rvb200
    return rvb200.PreprocessPipeline({"enabled": True, "chain": chain,
                                      "auto_gate": {"enable_low_contrast_gate": True, "contrast_thresh": thresh}})


def want_clahe(img):
    return cv2_chain.clahe_dehaze(img, "YCrCb", 2.0, 8)
