#!/usr/bin/env python3
"""BGRA and single-channel frames (rv_chain_ex) against what a user does without them, on the GPU, outputs checked against cv2.

  device-resident  1080p x 64 frames in torch tensors on one stream, CUDA events; each comparison alternates its arms in rounds
                   (arm A, arm B, ...; >= 1 s of work per arm) and reports the median, min and max of the per-round times
    bgra8_chain    YCrCb clip 2 grid 8 k5 on BGRA uint8: rv_chain_ex | x[..., :3].contiguous() + the 3-channel chain | the
                   3-channel chain alone on the same pixels (already BGR)
    gray8_median   median k3 / k5 on (H,W,1) uint8: rv_chain_ex | the plane replicated to 3 channels + the 3-channel median
    bgra16_chain, gray16_median   the same comparisons at 16 bits (YCrCb k5; median k3 / k5)
    bgra8_median   median k5 on all four BGRA uint8 channels (rv_chain_ex alone)
  latency          PreprocessPipeline(stock chain)(bgra_1080p) from pageable memory, p50 over 200 calls, beside the same call on
                   np.ascontiguousarray(bgra[..., :3])

Frames: the seeded road scenes of rvb200.synth (8 distinct 1080p frames, repeated to 64) with random alpha; gray = their G plane.
One JSON object goes to stdout (and to --out).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import cv2  # noqa: E402
import torch  # noqa: E402

import rvb200  # noqa: E402
from oracle import cv2_chain  # noqa: E402
from rvb200 import synth  # noqa: E402

H, W, N = 1080, 1920, 64


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:          # the numbers are still numbers; say that the card could not be read
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"not read ({e})"}


def timed(stream, fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
    stream.synchronize()
    return e0.elapsed_time(e1) / reps


def compare(stream, arms, min_s=1.0, warmup=3):
    """arms: {name: fn}.  Rounds of (every arm `reps` times), alternating, until each arm has run >= min_s."""
    for fn in arms.values():
        timed(stream, fn, warmup)
    probe = max(timed(stream, fn, 3) for fn in arms.values())
    reps = max(1, int(100.0 / probe))                      # ~0.1 s per arm and round
    rounds = max(10, int(np.ceil(min_s * 1e3 / (reps * probe))))
    per = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            per[k].append(timed(stream, fn, reps))
    out = {}
    for k, v in per.items():
        v = sorted(v)
        med = v[len(v) // 2]
        out[k] = {"ms_per_batch": round(med, 4), "ms_min": round(v[0], 4), "ms_max": round(v[-1], 4),
                  "spread_pct": round(100 * (v[-1] - v[0]) / med, 2), "fps": round(N * 1e3 / med, 1), "rounds": rounds, "reps": reps}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_channels needs a GPU")
    ctx = rvb200.default_context(0)
    stream = torch.cuda.Stream()
    sp = stream.cuda_stream
    P = rvb200.Params.make
    res = {"info": gpu_info(), "shape": [H, W], "frames": N, "input": "synth.frame_pool(1080, 1920, 8) x 8, random alpha"}

    pool = synth.frame_pool(H, W, 8, base_seed=1)
    rng = np.random.default_rng(0)
    host4 = np.concatenate([np.tile(pool, (N // 8, 1, 1, 1)), rng.integers(0, 256, (N, H, W, 1), dtype=np.uint8)], -1)
    x4 = torch.from_numpy(host4).cuda()
    x3 = x4[..., :3].contiguous()
    g1 = x4[..., 1:2].contiguous()
    host4_16 = host4.astype(np.uint16) * 257 + rng.integers(0, 257, host4.shape).astype(np.uint16)
    x4_16 = torch.from_numpy(host4_16.view(np.int16)).view(torch.uint16).cuda()
    x3_16 = x4_16[..., :3].contiguous()
    g1_16 = x4_16[..., 1:2].contiguous()

    def out_like(x, c):
        return torch.empty(x.shape[:3] + (c,), dtype=x.dtype, device=x.device)

    def np16(t):
        return t.view(torch.int16).cpu().numpy().view(np.uint16)

    def check(got, ref_fn, src):
        """frames 0 and N-1 against cv2"""
        got = got if isinstance(got, np.ndarray) else (np16(got) if got.dtype == torch.uint16 else got.cpu().numpy())
        return all(np.array_equal(got[i].reshape(ref_fn(src[i]).shape), ref_fn(src[i])) for i in (0, N - 1))

    cmp = {}
    # 1. BGRA uint8 chain
    p = P("YCrCb", 2.0, 8, 5)
    o_new, o_wa, o_3 = out_like(x4, 3), out_like(x4, 3), out_like(x4, 3)
    tmp = out_like(x4, 3)

    def wa8():
        tmp.copy_(x4[..., :3])
        ctx.submit_device(tmp.data_ptr(), o_wa.data_ptr(), N, H, W, p, stream=sp)
    arms = {"rv_chain_ex_bgra": lambda: ctx.chain_ex_device(x4.data_ptr(), o_new.data_ptr(), N, H, W, p, 8, 4, stream=sp),
            "strip_then_3ch": wa8,
            "3ch_chain_only": lambda: ctx.submit_device(x3.data_ptr(), o_3.data_ptr(), N, H, W, p, stream=sp)}
    cmp["bgra8_chain_ycrcb_k5"] = compare(stream, arms, args.min_seconds)
    ref = lambda f: cv2_chain.chain(f, "YCrCb", 2.0, 8, 5)                     # noqa: E731
    cmp["bgra8_chain_ycrcb_k5"]["bit_exact_vs_cv2"] = check(o_new, ref, host4) and check(o_wa, ref, host4) and torch.equal(o_new, o_3)

    # 2. gray uint8 median
    for k in (3, 5):
        pm = P(ksize=k, clahe=False)
        o_g, o_r = out_like(g1, 1), out_like(g1, 3)
        rep3 = out_like(g1, 3)

        def wa_g(pm=pm, o_r=o_r, rep3=rep3):
            rep3.copy_(g1.expand(-1, -1, -1, 3))
            ctx.submit_device(rep3.data_ptr(), o_r.data_ptr(), N, H, W, pm, stream=sp)
        arms = {"rv_chain_ex_gray": lambda pm=pm, o_g=o_g: ctx.chain_ex_device(g1.data_ptr(), o_g.data_ptr(), N, H, W, pm, 8, 1, stream=sp),
                "replicate_then_3ch_median": wa_g}
        name = f"gray8_median_k{k}"
        cmp[name] = compare(stream, arms, args.min_seconds)
        hg = g1.cpu().numpy()
        cmp[name]["bit_exact_vs_cv2"] = check(o_g, lambda f, k=k: cv2.medianBlur(f[..., 0], k), hg) and torch.equal(o_g[..., 0], o_r[..., 0])

    # 3. 16 bits, and median-only BGRA uint8
    o_new, o_wa, o_3 = out_like(x4_16, 3), out_like(x4_16, 3), out_like(x4_16, 3)
    tmp16 = out_like(x4_16, 3)

    def wa16():
        tmp16.copy_(x4_16[..., :3])
        ctx.chain_u16_device(tmp16.data_ptr(), o_wa.data_ptr(), N, H, W, p, stream=sp)
    arms = {"rv_chain_ex_bgra": lambda: ctx.chain_ex_device(x4_16.data_ptr(), o_new.data_ptr(), N, H, W, p, 16, 4, stream=sp),
            "strip_then_3ch": wa16,
            "3ch_chain_only": lambda: ctx.chain_u16_device(x3_16.data_ptr(), o_3.data_ptr(), N, H, W, p, stream=sp)}
    cmp["bgra16_chain_ycrcb_k5"] = compare(stream, arms, args.min_seconds)
    cmp["bgra16_chain_ycrcb_k5"]["bit_exact_vs_cv2"] = check(o_new, ref, host4_16) and torch.equal(o_new, o_wa) and torch.equal(o_new, o_3)
    hg16 = np16(g1_16)
    for k in (3, 5):
        pm = P(ksize=k, clahe=False)
        o_g, o_r = out_like(g1_16, 1), out_like(g1_16, 3)
        rep3 = out_like(g1_16, 3)

        def wa_g16(pm=pm, o_r=o_r, rep3=rep3):
            rep3.copy_(g1_16.expand(-1, -1, -1, 3))
            ctx.chain_u16_device(rep3.data_ptr(), o_r.data_ptr(), N, H, W, pm, stream=sp)
        arms = {"rv_chain_ex_gray": lambda pm=pm, o_g=o_g: ctx.chain_ex_device(g1_16.data_ptr(), o_g.data_ptr(), N, H, W, pm, 16, 1, stream=sp),
                "replicate_then_3ch_median": wa_g16}
        name = f"gray16_median_k{k}"
        cmp[name] = compare(stream, arms, args.min_seconds)
        cmp[name]["bit_exact_vs_cv2"] = check(o_g, lambda f, k=k: cv2.medianBlur(f[..., 0], k), hg16) and torch.equal(o_g[..., 0], o_r[..., 0])
    pm = P(ksize=5, clahe=False)
    o4 = out_like(x4, 4)
    cmp["bgra8_median_k5"] = compare(stream, {"rv_chain_ex_bgra": lambda: ctx.chain_ex_device(x4.data_ptr(), o4.data_ptr(), N, H, W, pm, 8, 4,
                                                                                             stream=sp)}, args.min_seconds)
    cmp["bgra8_median_k5"]["bit_exact_vs_cv2"] = check(o4, lambda f: cv2.medianBlur(f, 5), host4)
    res["device_resident"] = cmp

    # 4. per-frame latency from pageable memory
    pipe = rvb200.PreprocessPipeline({"enabled": True, "chain": [{"name": "CLAHEDehaze", "params": {}},
                                                                 {"name": "MedianDerain", "params": {"ksize": 5}}]})
    f4 = np.ascontiguousarray(host4[3])
    lat = {}
    for name, make in (("bgra", lambda: f4), ("bgr_after_ascontiguousarray", lambda: np.ascontiguousarray(f4[..., :3]))):
        for _ in range(10):
            got = pipe(make())
        ts = []
        for _ in range(200):
            t0 = time.perf_counter()
            pipe(make())
            ts.append(time.perf_counter() - t0)
        ts.sort()
        lat[name] = {"ms_p50": round(1e3 * ts[100], 3), "ms_min": round(1e3 * ts[0], 3),
                     "bit_exact_vs_cv2": bool(np.array_equal(got, cv2_chain.chain(f4, "YCrCb", 2.0, 8, 5)))}
    res["per_frame_pageable_1080p_stock_chain"] = lat
    out = json.dumps(res)
    print(out)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(out + "\n")


if __name__ == "__main__":
    main()
