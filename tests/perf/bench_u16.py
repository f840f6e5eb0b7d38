#!/usr/bin/env python3
"""Throughput and latency of the 16-bit chain (rv_chain_u16) on the GPU, every timed configuration checked bit-exact against cv2.

  device-resident  1080p x 64 frames: YCrCb k5, YCrCb k3, CLAHE only, median k3, median k5; 4K x 16 frames at grid 16 (k5)
                   CUDA events around `--reps` batches on one stream, torch uint16 tensors in and out
  latency          one 1080p frame per call from pageable memory (host clock, p50 / min), and a 64-frame batch end to end
                   from page-locked memory (host clock; H2D + kernels + D2H)
  kernel split     one torch.profiler run over a 1080p x 64 k5 batch (a run of its own: tracing slows the host)
  bytes            algorithmic frame traffic 2 * 6 * H * W per frame; LUT traffic reported apart: the LUT writes
                   (grid^2 * 128 KB per frame) and the four 2-byte gathers per pixel

Inputs are `(v << 8) | noise` frames (a smooth 8-bit image in the high byte, uniform noise in the low byte): every pixel's four LUT
gathers land in different cache sectors, as with real 16-bit sensor data.  One JSON object goes to stdout (and to --out).
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


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:          # the numbers are still numbers; say that the card could not be read
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"not read ({e})"}


def frames16(n, h, w, seed=0):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    base = ((yy * 3 + xx) * 255 // (3 * (h - 1) + (w - 1))).astype(np.int64)
    out = np.empty((n, h, w, 3), np.uint16)
    for i in range(n):
        v = (base[..., None] + np.array([0, 25, 50]) + 7 * i) % 256
        out[i] = (v << 8) | rng.integers(0, 256, (h, w, 3))
    return out


def reference(f, p):
    if not p.clahe:
        return cv2.medianBlur(f, p.ksize)
    return cv2_chain.chain(f, "YCrCb", p.clip_limit, p.grid, p.ksize)


def as_tensor(a):
    return torch.from_numpy(a.view(np.int16)).view(torch.uint16).cuda()


def to_numpy(t):
    return t.view(torch.int16).cpu().numpy().view(np.uint16)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--no-profile", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_u16 needs a GPU")
    ctx = rvb200.default_context(0)
    res = {"info": gpu_info(), "input": "(v << 8) | noise, 16-bit", "configs": []}
    P = rvb200.Params.make
    configs = [
        ("ycrcb_k5", 1080, 1920, 64, P("YCrCb", 2.0, 8, 5)),
        ("ycrcb_k3", 1080, 1920, 64, P("YCrCb", 2.0, 8, 3)),
        ("clahe_only", 1080, 1920, 64, P("YCrCb", 2.0, 8, 0)),
        ("median_k3", 1080, 1920, 64, P(ksize=3, clahe=False)),
        ("median_k5", 1080, 1920, 64, P(ksize=5, clahe=False)),
        ("4k_grid16_k5", 2160, 3840, 16, P("YCrCb", 2.0, 16, 5)),
    ]
    pools = {}
    stream = torch.cuda.Stream()
    for name, h, w, n, p in configs:
        if (h, w, n) not in pools:
            host = frames16(n, h, w)
            pools[(h, w, n)] = (host, as_tensor(host))
        host, din = pools[(h, w, n)]
        dout = torch.empty_like(din)
        with torch.cuda.stream(stream):
            for _ in range(args.warmup):
                ctx.chain_u16_device(din.data_ptr(), dout.data_ptr(), n, h, w, p, stream=stream.cuda_stream)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(args.reps):
                ctx.chain_u16_device(din.data_ptr(), dout.data_ptr(), n, h, w, p, stream=stream.cuda_stream)
            e1.record(stream)
        stream.synchronize()
        ms = e0.elapsed_time(e1) / args.reps
        got = to_numpy(dout)
        bad = [i for i in range(n) if not np.array_equal(got[i], reference(host[i], p))]
        frame_bytes = 2 * 6 * h * w
        row = {"name": name, "shape": [h, w], "frames": n, "ksize": p.ksize, "clahe": bool(p.clahe), "grid": p.grid if p.clahe else None,
               "ms_per_batch": round(ms, 4), "fps": round(n * 1e3 / ms, 1), "us_per_frame": round(1e3 * ms / n, 2),
               "frame_bytes": frame_bytes, "frame_GBps": round(n * frame_bytes / ms / 1e6, 1), "bit_exact_vs_cv2": not bad,
               "mismatching_frames": bad[:8]}
        if p.clahe:
            row["lut_write_bytes"] = p.grid * p.grid * 65536 * 2
            row["lut_gather_bytes"] = 4 * 2 * h * w
        res["configs"].append(row)
        print(json.dumps(row), flush=True, file=sys.stderr)
        del dout

    # per-frame latency (1080p, pageable in, fresh result out) and a pinned batch end to end
    p = P("YCrCb", 2.0, 8, 5)
    host = pools[(1080, 1920, 64)][0]
    one = np.ascontiguousarray(host[:1])
    want = reference(one[0], p)
    for _ in range(5):
        got = ctx.chain(one, p)
    assert np.array_equal(got[0], want)
    ts = []
    for _ in range(100):
        t0 = time.perf_counter(); ctx.chain(one, p); ts.append(time.perf_counter() - t0)
    ts.sort()
    tc = []
    for _ in range(5):
        t0 = time.perf_counter(); reference(one[0], p); tc.append(time.perf_counter() - t0)
    tc.sort()
    res["latency_1080p_k5"] = {"pageable_ms_p50": round(1e3 * ts[50], 3), "pageable_ms_min": round(1e3 * ts[0], 3),
                               "cv2_ms_p50_this_host": round(1e3 * tc[2], 2)}
    pin_in = ctx.pinned_empty(host.shape, np.uint16)
    pin_out = ctx.pinned_empty(host.shape, np.uint16)
    pin_in[...] = host
    for _ in range(2):
        ctx.chain(pin_in, p, out=pin_out)
    ts = []
    for _ in range(5):
        t0 = time.perf_counter(); ctx.chain(pin_in, p, out=pin_out); ts.append(time.perf_counter() - t0)
    ts.sort()
    bad = [i for i in range(0, 64, 9) if not np.array_equal(pin_out[i], reference(host[i], p))]
    res["e2e_pinned_1080p_x64_k5"] = {"ms_p50": round(1e3 * ts[2], 2), "fps": round(64 / ts[2], 1), "bit_exact_vs_cv2_sampled": not bad}

    if not args.no_profile:
        h, w, n = 1080, 1920, 64
        din = pools[(h, w, n)][1]
        dout = torch.empty_like(din)
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                ctx.chain_u16_device(din.data_ptr(), dout.data_ptr(), n, h, w, p)
            torch.cuda.synchronize()
        split = {}
        for ev in prof.key_averages():
            if ev.device_type is not None and "CUDA" in str(ev.device_type) and ev.count:
                t = getattr(ev, "self_device_time_total", None) or getattr(ev, "self_cuda_time_total", 0)
                name = ev.key.replace("(anonymous namespace)::", "").replace("void ", "").split("(")[0]
                split[name] = {"ms_per_batch": round(t / 1e3 / 3, 4), "launches_per_batch": ev.count / 3}
        tot = sum(v["ms_per_batch"] for v in split.values()) or 1.0
        for v in split.values():
            v["share"] = round(v["ms_per_batch"] / tot, 3)
        res["kernel_split_1080p_x64_k5"] = split
    out = json.dumps(res)
    print(out)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(out + "\n")


if __name__ == "__main__":
    main()
