#!/usr/bin/env python3
"""Packed YUV 4:2:2 camera frames (YUY2, UYVY) in the batch entries against what a user does without them, on the GPU, outputs checked
against cv2.

1080p x 64 frames, the stock chain (YCrCb clip 2 grid 8, median k5), for YUY2 and for UYVY.  Every comparison alternates its arms in
rounds (arm A, arm B, ...; >= --min-seconds of work per arm) and reports the median, min and max of the per-round times.
  device_resident  torch tensors on one stream, CUDA events:
    yuv_convert_then_chain   rv_yuv422_to_bgr into a BGR tensor + the BGR chain (rv_submit)
    bgr_chain_only           the BGR chain alone on the same pixels (already BGR)
    convert_only             rv_yuv422_to_bgr alone
    convert_only_scalar      the same frames read from one byte past an aligned address: the kernel's byte-wise path
  host_fed  pinned host frames in, host clock around calls that end synchronised, in the shapes of bench.py's legs:
            keep   = process_batch_to_tensor(frames, out="device")                  (e2e_keep: the tensor stays on the GPU)
            tensor = process_batch_to_tensor(frames, out=pinned, padding_present=True) (e2e_tensor: the tensor's image rows come back)
    yuv_in                   the pinned 4:2:2 frames with yuv=...: 2 bytes per pixel cross PCIe, converted on the GPU
    host_cv2_then_bgr        the user's workaround: cv2.cvtColor on the host into a pinned BGR batch, then the BGR call
    bgr_preconverted         the BGR call on frames converted beforehand (3 bytes per pixel cross PCIe)

Frames: the seeded road scenes of rvb200.synth (8 distinct 1080p frames, repeated to 64) through cv2's BGR -> YUY2 / UYVY, the chroma of
the last frame random.  One JSON object goes to stdout (and to --out).
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import ctypes as C  # noqa: E402

import cv2  # noqa: E402
import torch  # noqa: E402

import rvb200  # noqa: E402
from oracle import cv2_chain  # noqa: E402
from oracle import rv_oracle as O  # noqa: E402
from oracle import yuv422 as Y  # noqa: E402
from rvb200 import _native as N  # noqa: E402
from rvb200 import synth  # noqa: E402
from bench_yuv import gpu_info, rounds  # noqa: E402  (this directory: the same card query and alternating rounds)

H, W, N_FR, S = 1080, 1920, 64, 640
CODES = {"YUY2": cv2.COLOR_YUV2BGR_YUY2, "UYVY": cv2.COLOR_YUV2BGR_UYVY}
TO_422 = {"YUY2": cv2.COLOR_BGR2YUV_YUY2, "UYVY": cv2.COLOR_BGR2YUV_UYVY}
CHAIN = [{"name": "CLAHEDehaze", "params": {"space": "YCrCb", "clip_limit": 2.0, "tile_grid": 8}},
         {"name": "MedianDerain", "params": {"ksize": 5}}]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_yuv422 needs a GPU")
    ctx = rvb200.default_context(0)
    stream = torch.cuda.Stream()
    sp = stream.cuda_stream
    p = rvb200.Params.make("YCrCb", 2.0, 8, 5)
    res = {"info": gpu_info(), "shape": [H, W], "frames": N_FR, "chain": "YCrCb clip 2 grid 8, median k5",
           "input": "synth.frame_pool(1080, 1920, 8) x 8 through cv2 BGR2YUV_YUY2 / _UYVY, last frame's chroma random",
           "cv2_threads": cv2.getNumThreads(), "host_cpus": os.cpu_count()}
    pool = synth.frame_pool(H, W, 8, base_seed=1)
    rng = np.random.default_rng(0)
    chroma = rng.integers(0, 256, (2, H, W // 2), dtype=np.uint8)

    def timed_dev(fn, reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(reps):
                fn()
            e1.record(stream)
        stream.synchronize()
        return e0.elapsed_time(e1) / reps

    def timed_host(fn, reps):
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        return 1e3 * (time.perf_counter() - t0) / reps

    for layout in ("YUY2", "UYVY"):
        L = N.YUV422_LAYOUTS[layout]
        host = np.stack([cv2.cvtColor(pool[i % 8], TO_422[layout]) for i in range(N_FR)])
        host[-1] = Y.from_planes(Y.planes(host[-1], layout)[0], chroma[0], chroma[1], layout)
        bgr = np.stack([cv2.cvtColor(f, CODES[layout]) for f in host])
        want = {i: cv2_chain.chain(bgr[i], "YCrCb", 2.0, 8, 5) for i in (0, N_FR - 1)}
        want_t = {i: O.letterbox_f16(want[i], S) for i in want}
        cmp = {}

        # device-resident
        ty, tb = torch.from_numpy(host).cuda(), torch.from_numpy(bgr).cuda()
        tmp, o_y, o_b = torch.empty_like(tb), torch.empty_like(tb), torch.empty_like(tb)
        ty1 = torch.empty(host.size + 1, dtype=torch.uint8, device="cuda")
        ty1[1:] = ty.reshape(-1)
        tmp1 = torch.empty_like(tb)

        def convert_scalar():
            ctx._ck(ctx._lib.rv_yuv422_to_bgr(ctx._h, C.c_void_p(ty1.data_ptr() + 1), C.c_void_p(tmp1.data_ptr()), N_FR, H, W, 2 * W,
                                              3 * W, L, N.MEM_DEVICE, C.c_void_p(sp)))

        def convert():
            ctx._ck(ctx._lib.rv_yuv422_to_bgr(ctx._h, C.c_void_p(ty.data_ptr()), C.c_void_p(tmp.data_ptr()), N_FR, H, W, 2 * W, 3 * W, L,
                                              N.MEM_DEVICE, C.c_void_p(sp)))

        def yuv_chain():
            convert()
            ctx.submit_device(tmp.data_ptr(), o_y.data_ptr(), N_FR, H, W, p, stream=sp)
        d = rounds({"yuv_convert_then_chain": yuv_chain,
                    "bgr_chain_only": lambda: ctx.submit_device(tb.data_ptr(), o_b.data_ptr(), N_FR, H, W, p, stream=sp),
                    "convert_only": convert, "convert_only_scalar": convert_scalar}, timed_dev, args.min_seconds)
        d["bit_exact_vs_cv2"] = bool(torch.equal(tmp, tb) and torch.equal(tmp1, tb) and torch.equal(o_y, o_b) and
                                     all(np.array_equal(o_y[i].cpu().numpy(), want[i]) for i in want))
        d["bytes_per_batch"] = {"convert_read": host.nbytes, "convert_write": bgr.nbytes}
        cmp["device_resident"] = d
        del ty, tb, tmp, o_y, o_b, ty1, tmp1

        # host-fed from pinned memory
        pl = rvb200.PreprocessPipeline({"chain": CHAIN}, context=ctx)
        pin_y, pin_b, pin_w = ctx.pinned_empty(host.shape), ctx.pinned_empty(bgr.shape), ctx.pinned_empty(bgr.shape)
        pin_y[...] = host
        pin_b[...] = bgr
        pts = {k: ctx.pinned_empty((N_FR, 3, S, S), np.float16) for k in ("yuv_in", "host_cv2_then_bgr", "bgr_preconverted")}
        for t in pts.values():
            t[...] = 0
            ctx.fill_tensor_padding(t, H, W, S)

        def cv2_host():
            for i in range(N_FR):
                cv2.cvtColor(pin_y[i], CODES[layout], dst=pin_w[i])
        last = {}

        def keep(name, fn):
            def run():
                last[name] = fn()[0]
            return run
        arms = {"yuv_in": keep("yuv_in", lambda: pl.process_batch_to_tensor(pin_y, out="device", yuv=layout)),
                "host_cv2_then_bgr": keep("host_cv2_then_bgr", lambda: (cv2_host(), pl.process_batch_to_tensor(pin_w, out="device"))[1]),
                "bgr_preconverted": keep("bgr_preconverted", lambda: pl.process_batch_to_tensor(pin_b, out="device"))}
        h = rounds(arms, timed_host, args.min_seconds)
        h["bit_exact_vs_cv2"] = all(np.array_equal(last[k].numpy()[i].view(np.uint16), want_t[i].view(np.uint16)) for k in arms
                                    for i in want)
        h["h2d_bytes_per_batch"] = {"yuv_in": host.nbytes, "host_cv2_then_bgr": bgr.nbytes, "bgr_preconverted": bgr.nbytes}
        cmp["host_fed_keep"] = h
        arms = {"yuv_in": lambda: pl.process_batch_to_tensor(pin_y, out=pts["yuv_in"], padding_present=True, yuv=layout),
                "host_cv2_then_bgr": lambda: (cv2_host(), pl.process_batch_to_tensor(pin_w, out=pts["host_cv2_then_bgr"],
                                                                                     padding_present=True)),
                "bgr_preconverted": lambda: pl.process_batch_to_tensor(pin_b, out=pts["bgr_preconverted"], padding_present=True)}
        h = rounds(arms, timed_host, args.min_seconds)
        h["bit_exact_vs_cv2"] = all(np.array_equal(pts[k][i].view(np.uint16), want_t[i].view(np.uint16)) for k in arms for i in want)
        cmp["host_fed_tensor"] = h
        # the host conversion alone, as a user's CPU pays it per batch
        cv2_host()
        t0 = time.perf_counter()
        for _ in range(3):
            cv2_host()
        cmp["host_cv2_convert_ms_per_batch"] = round(1e3 * (time.perf_counter() - t0) / 3, 3)
        cmp["host_cv2_bit_exact"] = bool(np.array_equal(pin_w, bgr))
        res[layout] = cmp
        del pin_y, pin_b, pin_w, pts
    out = json.dumps(res)
    print(out)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(out + "\n")


if __name__ == "__main__":
    main()
