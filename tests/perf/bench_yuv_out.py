#!/usr/bin/env python3
"""4:2:0 (NV12, I420) results from the batch entries against BGR results and against what a user does without them, on the GPU,
every arm's output checked against cv2.

1080p x 64 frames, the stock chain (YCrCb clip 2 grid 8, median k5).  Every comparison alternates its arms in rounds (arm A, arm B,
...; >= --min-seconds of work per arm) and reports the median, min and max of the per-round times.
  host_fed  pinned host frames in, pinned results out, host clock around calls that end synchronised (bench.py's e2e shape):
    bgr_in_bgr_out        process_batch(bgr, out=pinned): 3 bytes per pixel each way (the baseline)
    nv12_in_nv12_out      process_batch(nv12, out=pinned, yuv="NV12", out_yuv="NV12"): 1.5 bytes per pixel each way
    i420_in_i420_out      the same with I420
    bgr_in_nv12_out       process_batch(bgr, out=pinned, out_yuv="NV12"): 3 bytes per pixel in, 1.5 back
    nv12_in_bgr_out_cv2   the user's workaround: process_batch(nv12, yuv="NV12") to BGR, then cv2.cvtColor(COLOR_BGR2YUV_I420) on the
                          host for every frame and the U, V interleave into NV12
  device_resident  torch tensors on one stream, CUDA events:
    convert_only / convert_only_bytewise   rv_bgr_to_yuv420 on aligned buffers / one byte past them (the byte-wise path)
    chain_then_convert / chain_only        the BGR chain (rv_submit) with and without the conversion of its result

Frames: the seeded road scenes of rvb200.synth (8 distinct 1080p frames, repeated to 64), the last frame random.  One JSON object goes
to stdout (and to --out).
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
from oracle import yuv420 as Y  # noqa: E402
from rvb200 import _native as N  # noqa: E402
from rvb200 import synth  # noqa: E402

H, W, N_FR = 1080, 1920, 64
CHAIN = [{"name": "CLAHEDehaze", "params": {"space": "YCrCb", "clip_limit": 2.0, "tile_grid": 8}},
         {"name": "MedianDerain", "params": {"ksize": 5}}]
TO_BGR = {"NV12": cv2.COLOR_YUV2BGR_NV12, "I420": cv2.COLOR_YUV2BGR_I420}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:          # the numbers are still numbers; say that the card could not be read
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"not read ({e})"}


def to_yuv(bgr, layout):
    i420 = cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420)
    return i420 if layout == "I420" else Y.from_planes(*Y.planes(i420, "I420"), "NV12")


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
        raise SystemExit("bench_yuv_out needs a GPU")
    ctx = rvb200.default_context(0)
    stream = torch.cuda.Stream()
    sp = stream.cuda_stream
    p = rvb200.Params.make("YCrCb", 2.0, 8, 5)
    res = {"info": gpu_info(), "shape": [H, W], "frames": N_FR, "chain": "YCrCb clip 2 grid 8, median k5",
           "input": "synth.frame_pool(1080, 1920, 8) x 8, last frame random", "cv2_threads": cv2.getNumThreads(),
           "host_cpus": os.cpu_count()}
    pool = synth.frame_pool(H, W, 8, base_seed=1)
    bgr = np.stack([pool[i % 8] for i in range(N_FR)])
    bgr[-1] = np.random.default_rng(0).integers(0, 256, bgr[-1].shape, dtype=np.uint8)
    check = (0, N_FR - 1)
    proc = {i: cv2_chain.chain(bgr[i], "YCrCb", 2.0, 8, 5) for i in check}
    nv12 = np.stack([to_yuv(f, "NV12") for f in bgr])
    i420 = np.stack([to_yuv(f, "I420") for f in bgr])

    def timed_host(fn, reps):
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        return 1e3 * (time.perf_counter() - t0) / reps

    def timed_dev(fn, reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(reps):
                fn()
            e1.record(stream)
        stream.synchronize()
        return e0.elapsed_time(e1) / reps

    # host-fed from pinned memory.  The BGR each 4:2:0 input stands for is cv2's conversion of it.
    pl = rvb200.PreprocessPipeline({"chain": CHAIN}, context=ctx)
    src = {"bgr": bgr, "NV12": nv12, "I420": i420}
    stands_for = {"bgr": bgr, "NV12": np.stack([cv2.cvtColor(nv12[i], TO_BGR["NV12"]) for i in check]),
                  "I420": np.stack([cv2.cvtColor(i420[i], TO_BGR["I420"]) for i in check])}
    want = {("bgr", None): {i: proc[i] for i in check}}
    for k in ("NV12", "I420"):
        ref = {i: cv2_chain.chain(stands_for[k][j], "YCrCb", 2.0, 8, 5) for j, i in enumerate(check)}
        want[(k, None)] = ref
        want[(k, k)] = {i: to_yuv(ref[i], k) for i in check}
    want[("bgr", "NV12")] = {i: to_yuv(proc[i], "NV12") for i in check}
    pin_in = {k: ctx.pinned_empty(v.shape) for k, v in src.items()}
    for k, v in src.items():
        pin_in[k][...] = v
    pin_out = {"bgr": ctx.pinned_empty(bgr.shape), "NV12": ctx.pinned_empty(nv12.shape), "I420": ctx.pinned_empty(i420.shape),
               "bgr_nv12": ctx.pinned_empty(nv12.shape), "work_bgr": ctx.pinned_empty(bgr.shape), "work_nv12": ctx.pinned_empty(nv12.shape)}

    def workaround():
        pl.process_batch(pin_in["NV12"], out=pin_out["work_bgr"], yuv="NV12")
        o = pin_out["work_nv12"]
        for i in range(N_FR):
            yuv = cv2.cvtColor(pin_out["work_bgr"][i], cv2.COLOR_BGR2YUV_I420)
            o[i, :H] = yuv[:H]
            uv = o[i, H:].reshape(H // 2, W // 2, 2)
            uv[..., 0] = yuv[H:H + H // 4].reshape(H // 2, W // 2)
            uv[..., 1] = yuv[H + H // 4:].reshape(H // 2, W // 2)
    arms = {"bgr_in_bgr_out": lambda: pl.process_batch(pin_in["bgr"], out=pin_out["bgr"]),
            "nv12_in_nv12_out": lambda: pl.process_batch(pin_in["NV12"], out=pin_out["NV12"], yuv="NV12", out_yuv="NV12"),
            "i420_in_i420_out": lambda: pl.process_batch(pin_in["I420"], out=pin_out["I420"], yuv="I420", out_yuv="I420"),
            "bgr_in_nv12_out": lambda: pl.process_batch(pin_in["bgr"], out=pin_out["bgr_nv12"], out_yuv="NV12"),
            "nv12_in_bgr_out_cv2": workaround}
    h = rounds(arms, timed_host, args.min_seconds)
    got = {"bgr_in_bgr_out": (pin_out["bgr"], ("bgr", None)), "nv12_in_nv12_out": (pin_out["NV12"], ("NV12", "NV12")),
           "i420_in_i420_out": (pin_out["I420"], ("I420", "I420")), "bgr_in_nv12_out": (pin_out["bgr_nv12"], ("bgr", "NV12")),
           "nv12_in_bgr_out_cv2": (pin_out["work_nv12"], ("NV12", "NV12"))}
    h["bit_exact_vs_cv2"] = {k: all(np.array_equal(arr[i], want[key][i]) for i in check) for k, (arr, key) in got.items()}
    h["pcie_bytes_per_batch"] = {"bgr_in_bgr_out": [bgr.nbytes, bgr.nbytes], "nv12_in_nv12_out": [nv12.nbytes, nv12.nbytes],
                                 "i420_in_i420_out": [i420.nbytes, i420.nbytes], "bgr_in_nv12_out": [bgr.nbytes, nv12.nbytes],
                                 "nv12_in_bgr_out_cv2": [nv12.nbytes, bgr.nbytes], "order": "[H2D, D2H]"}
    base = h["bgr_in_bgr_out"]["ms_per_batch"]
    h["speedup_vs_bgr_in_bgr_out"] = {k: round(base / h[k]["ms_per_batch"], 3) for k in arms}
    res["host_fed"] = h
    del pin_in, pin_out

    # device-resident
    dev = {}
    tb = torch.from_numpy(bgr).cuda()
    tb1 = torch.empty(bgr.size + 1, dtype=torch.uint8, device="cuda")
    tb1[1:] = tb.reshape(-1)
    tproc = torch.empty_like(tb)
    for layout in ("NV12", "I420"):
        L = N.YUV_LAYOUTS[layout]
        ty = torch.empty(nv12.shape, dtype=torch.uint8, device="cuda")
        ty1 = torch.empty(nv12.size + 1, dtype=torch.uint8, device="cuda")
        tyc = torch.empty_like(ty)

        def convert(ty=ty, L=L):
            ctx._ck(ctx._lib.rv_bgr_to_yuv420(ctx._h, C.c_void_p(tb.data_ptr()), C.c_void_p(ty.data_ptr()), N_FR, H, W, 3 * W, W, L,
                                              N.MEM_DEVICE, C.c_void_p(sp)))

        def convert_bytewise(ty1=ty1, L=L):
            ctx._ck(ctx._lib.rv_bgr_to_yuv420(ctx._h, C.c_void_p(tb1.data_ptr() + 1), C.c_void_p(ty1.data_ptr() + 1), N_FR, H, W, 3 * W,
                                              W, L, N.MEM_DEVICE, C.c_void_p(sp)))

        def chain():
            ctx.submit_device(tb.data_ptr(), tproc.data_ptr(), N_FR, H, W, p, stream=sp)

        def chain_convert(tyc=tyc, L=L):
            chain()
            ctx._ck(ctx._lib.rv_bgr_to_yuv420(ctx._h, C.c_void_p(tproc.data_ptr()), C.c_void_p(tyc.data_ptr()), N_FR, H, W, 3 * W, W, L,
                                              N.MEM_DEVICE, C.c_void_p(sp)))
        d = rounds({"convert_only": convert, "convert_only_bytewise": convert_bytewise, "chain_then_convert": chain_convert,
                    "chain_only": chain}, timed_dev, args.min_seconds)
        torch.cuda.synchronize()
        yb = ty1[1:].reshape(ty.shape)
        d["bit_exact_vs_cv2"] = bool(all(np.array_equal(ty[i].cpu().numpy(), to_yuv(bgr[i], layout)) for i in check) and
                                     torch.equal(yb, ty) and
                                     all(np.array_equal(tyc[i].cpu().numpy(), to_yuv(proc[i], layout)) for i in check))
        d["bytes_per_batch"] = {"convert_read": bgr.nbytes, "convert_write": nv12.nbytes}
        d["convert_only_GBps"] = round((bgr.nbytes + nv12.nbytes) / (d["convert_only"]["ms_per_batch"] * 1e-3) / 1e9, 1)
        dev[layout] = d
        del ty, ty1, tyc
    res["device_resident"] = dev
    out = json.dumps(res)
    print(out)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(out + "\n")


if __name__ == "__main__":
    main()
