#!/usr/bin/env python3
"""YUV 4:2:0 (NV12, I420) frames in the batch entries against what a user does without them, on the GPU, outputs checked against cv2.

1080p x 64 frames, the stock chain (YCrCb clip 2 grid 8, median k5), for NV12 and for I420.  Every comparison alternates its arms in
rounds (arm A, arm B, ...; >= --min-seconds of work per arm) and reports the median, min and max of the per-round times.
  device_resident  torch tensors on one stream, CUDA events:
    yuv_convert_then_chain   rv_yuv420_to_bgr into a BGR tensor + the BGR chain (rv_submit)
    bgr_chain_only           the BGR chain alone on the same pixels (already BGR)
    convert_only             rv_yuv420_to_bgr alone
    convert_only_scalar      the same frames read from one byte past an aligned address: the kernel's scalar path, which also
                             converts I420 frames whose width is not a multiple of 8
  host_fed  pinned host frames in, host clock around calls that end synchronised, in the shapes of bench.py's legs:
            keep   = process_batch_to_tensor(frames, out="device")                  (e2e_keep: the tensor stays on the GPU)
            tensor = process_batch_to_tensor(frames, out=pinned, padding_present=True) (e2e_tensor: the tensor's image rows come back)
    yuv_in                   the pinned YUV frames with yuv=...: 1.5 bytes per pixel cross PCIe, converted on the GPU
    yuv_in_chunk8            the same on a context whose host pipeline cuts 8-frame chunks instead of the automatic 4 (keep only)
    host_cv2_then_bgr        the user's workaround: cv2.cvtColor on the host into a pinned BGR batch, then the BGR call
    bgr_preconverted         the BGR call on frames converted beforehand (3 bytes per pixel cross PCIe)

Frames: the seeded road scenes of rvb200.synth (8 distinct 1080p frames, repeated to 64) through cv2's BGR -> I420, the chroma of the
last frame random.  One JSON object goes to stdout (and to --out).
"""
import argparse
import json
import os
import subprocess
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
from oracle import yuv420 as Y  # noqa: E402
from rvb200 import _native as N  # noqa: E402
from rvb200 import synth  # noqa: E402

H, W, N_FR, S = 1080, 1920, 64, 640
CODES = {"NV12": cv2.COLOR_YUV2BGR_NV12, "I420": cv2.COLOR_YUV2BGR_I420}
CHAIN = [{"name": "CLAHEDehaze", "params": {"space": "YCrCb", "clip_limit": 2.0, "tile_grid": 8}},
         {"name": "MedianDerain", "params": {"ksize": 5}}]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:          # the numbers are still numbers; say that the card could not be read
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"not read ({e})"}


def stats(v, reps):
    v = sorted(v)
    med = v[len(v) // 2]
    return {"ms_per_batch": round(med, 4), "ms_min": round(v[0], 4), "ms_max": round(v[-1], 4),
            "spread_pct": round(100 * (v[-1] - v[0]) / med, 2), "fps": round(N_FR * 1e3 / med, 1), "rounds": len(v), "reps": reps}


def rounds(arms, timed, min_s, warmup=2):
    """arms: {name: fn}; timed(fn, reps) -> ms per call.  Rounds of (every arm `reps` times), alternating, until each arm has run
    >= min_s."""
    for fn in arms.values():
        timed(fn, warmup)
    probe = max(timed(fn, 2) for fn in arms.values())
    reps = max(1, int(100.0 / probe))                      # ~0.1 s per arm and round
    n = max(10, int(np.ceil(min_s * 1e3 / (reps * probe))))
    per = {k: [] for k in arms}
    for _ in range(n):
        for k, fn in arms.items():
            per[k].append(timed(fn, reps))
    return {k: stats(v, reps) for k, v in per.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_yuv needs a GPU")
    ctx = rvb200.default_context(0)
    ctx8 = rvb200.Context(0)
    ctx8.set_option("chunk_frames", 8)
    stream = torch.cuda.Stream()
    sp = stream.cuda_stream
    p = rvb200.Params.make("YCrCb", 2.0, 8, 5)
    res = {"info": gpu_info(), "shape": [H, W], "frames": N_FR, "chain": "YCrCb clip 2 grid 8, median k5",
           "input": "synth.frame_pool(1080, 1920, 8) x 8 through cv2 BGR2YUV_I420, last frame's chroma random",
           "cv2_threads": cv2.getNumThreads(), "host_cpus": os.cpu_count()}
    pool = synth.frame_pool(H, W, 8, base_seed=1)
    i420 = np.stack([cv2.cvtColor(pool[i % 8], cv2.COLOR_BGR2YUV_I420) for i in range(N_FR)])
    i420[-1, H:] = np.random.default_rng(0).integers(0, 256, i420[-1, H:].shape, dtype=np.uint8)

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

    for layout in ("NV12", "I420"):
        L = N.YUV_LAYOUTS[layout]
        host = i420 if layout == "I420" else np.stack([Y.from_planes(*Y.planes(f, "I420"), "NV12") for f in i420])
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
            ctx._ck(ctx._lib.rv_yuv420_to_bgr(ctx._h, C.c_void_p(ty1.data_ptr() + 1), C.c_void_p(tmp1.data_ptr()), N_FR, H, W, W, 3 * W, L,
                                              N.MEM_DEVICE, C.c_void_p(sp)))

        def convert():
            ctx._ck(ctx._lib.rv_yuv420_to_bgr(ctx._h, C.c_void_p(ty.data_ptr()), C.c_void_p(tmp.data_ptr()), N_FR, H, W, W, 3 * W, L,
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
        pl, pl8 = rvb200.PreprocessPipeline({"chain": CHAIN}, context=ctx), rvb200.PreprocessPipeline({"chain": CHAIN}, context=ctx8)
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
                "yuv_in_chunk8": keep("yuv_in_chunk8", lambda: pl8.process_batch_to_tensor(pin_y, out="device", yuv=layout)),
                "host_cv2_then_bgr": keep("host_cv2_then_bgr", lambda: (cv2_host(), pl.process_batch_to_tensor(pin_w, out="device"))[1]),
                "bgr_preconverted": keep("bgr_preconverted", lambda: pl.process_batch_to_tensor(pin_b, out="device"))}
        h = rounds(arms, timed_host, args.min_seconds)
        h["bit_exact_vs_cv2"] = all(np.array_equal(last[k].numpy()[i].view(np.uint16), want_t[i].view(np.uint16)) for k in arms
                                    for i in want)
        h["h2d_bytes_per_batch"] = {"yuv_in": host.nbytes, "yuv_in_chunk8": host.nbytes, "host_cv2_then_bgr": bgr.nbytes,
                                    "bgr_preconverted": bgr.nbytes}
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
    ctx8.close()
    out = json.dumps(res)
    print(out)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(out + "\n")


if __name__ == "__main__":
    main()
