#!/usr/bin/env python3
"""Headline benchmark: 1080p preprocessing-chain frames/s on N B200s (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A step is one pass of the hot path (CLAHEDehaze -> MedianDerain) over one batch of fogged + rained frames.  Workload at
every N: BASELINE.json configs[1] -- 1920x1080, batch 64 per GPU, YCrCb, clip 2.0, tile grid 8, median k5 (frames /
streams shard across GPUs with no inter-GPU traffic, so N GPUs process N such batches: weak scaling).  The frame pool
is eight frames made by the reference's own fog synthesiser (tests/golden/pool_1080p, tools/fog_batch.py parameters).

`value`      frames/s with inputs and outputs resident in HBM (CUDA events over exactly K steps, max over ranks).
`sustained`  the same loop repeated for >= 1 s (the K-step region is only ~19 ms at K = 20), clocks sampled over it.
`e2e`        same metric through the public plugin API (PreprocessPipeline.process_batch) from pinned host buffers,
             H2D and D2H of full frames inside the timed region.
`e2e_tensor` BASELINE configs[4] leg: pinned frames in, chain fused with the letterbox, only the (B,3,640,640) fp16
             detector tensor comes back (process_batch_to_tensor); `e2e_keep`: results stay on the GPU (no D2H).
`streams`    BASELINE configs[3] leg: one paced 1080p@30 camera stream per GPU (capture -> pinned ring -> chain ->
             pinned result), sustained fps and capture->result latency percentiles.
`roofline`   the dominant kernel (k_chain) against the measured HBM copy bandwidth; its time is measured live with CUDA
             events around every launch in a second pass of the same K steps; DRAM traffic and instruction counts come
             from the committed ncu capture profiles/final_k_chain.json, whose source hash must match the tree.
`cpu_baseline` / `--impl reference`: the reference's OWN PreprocessPipeline (oracle/_ref, installed by build()) on all
             host cores, one loop for both (64 frames per step, frame-parallel, one cv2 thread per process).
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

H, W, BATCH = 1080, 1920, 64
SPACE, CLIP, GRID, KSIZE = "YCrCb", 2.0, 8, 5
POOL = 8                                   # distinct frames, tiled to the batch
FRAME_BYTES = 3 * H * W
ALGO_BYTES_PER_FRAME = 2 * FRAME_BYTES     # read BGR once + write BGR once (SURVEY.md 8d)
TENSOR_SIZE = 640
TENSOR_BYTES = 3 * TENSOR_SIZE * TENSOR_SIZE * 2
METRIC, UNIT = "1080p preproc-chain frames/s", "frames/s"
CHAIN_CFG = {"enabled": True, "chain": [
    {"name": "CLAHEDehaze", "params": {"space": SPACE, "clip_limit": CLIP, "tile_grid": GRID}},
    {"name": "MedianDerain", "params": {"ksize": KSIZE}}]}
REF_ROOT = os.path.join(ROOT, "oracle", "_ref", "road-vision-system")


# ----------------------------------------------------------------------------- sharding / reductions
def shard_range(n, rank, world):
    """Contiguous slab [a, b) of n items for `rank` of `world` (sizes differ by at most one)."""
    base, rem = divmod(n, world)
    a = rank * base + min(rank, rem)
    return a, a + base + (1 if rank < rem else 0)


def _reduce(x, op, use_cuda):
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return float(x)
    t = torch.tensor([float(x)], dtype=torch.float64, device="cuda" if use_cuda else "cpu")
    dist.all_reduce(t, op=op)
    return float(t.item())


def max_over_ranks(x, use_cuda=True):
    import torch.distributed as dist
    return _reduce(x, dist.ReduceOp.MAX, use_cuda)


def min_over_ranks(x, use_cuda=True):
    import torch.distributed as dist
    return _reduce(x, dist.ReduceOp.MIN, use_cuda)


def sum_over_ranks(x, use_cuda=True):
    import torch.distributed as dist
    return _reduce(x, dist.ReduceOp.SUM, use_cuda)


def barrier():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        dist.barrier()


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ts, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7 or not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for nme, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nme)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------- frame pool
def load_pool():
    """The committed pool of reference-fogged 1080p frames (tests/golden/make_bench_pool.py), SHA-1 checked."""
    import cv2
    import numpy as np
    d = os.path.join(ROOT, "tests", "golden", "pool_1080p")
    frames = []
    for line in open(os.path.join(d, "index.txt")):
        if line.startswith("#") or not line.strip():
            continue
        name, _level, _seed, sha, _ref_sha = line.strip().split("|")[:5]
        img = cv2.imdecode(np.fromfile(os.path.join(d, name), np.uint8), cv2.IMREAD_COLOR)
        if img is None or img.shape != (H, W, 3) or hashlib.sha1(img.tobytes()).hexdigest() != sha:
            raise SystemExit(f"bench: {name} does not decode to the recorded frame")
        frames.append(img)
    if len(frames) != POOL:
        raise SystemExit("bench: frame pool incomplete")
    return np.stack(frames)


def pool_reference_shas():
    d = os.path.join(ROOT, "tests", "golden", "pool_1080p")
    return [ln.strip().split("|")[4] for ln in open(os.path.join(d, "index.txt")) if ln.strip() and not ln.startswith("#")]


DATA = ("synthetic: 8 distinct 1080p road scenes fogged by the reference's EnhancedFogSynthesizer (src/augment/fog.py, "
        "tools/fog_batch.py:19-27 parameters, seeded) + rain streaks, tiled to the batch (tests/golden/pool_1080p)")


# ----------------------------------------------------------------------------- CPU arm: the reference's own classes
_W = {}


def _cpu_init(frames, ref_root):
    """Pool initializer (spawned, never forked: a forked child inherits cv2's thread-pool state and can deadlock): every
    worker gets the frame pool once and builds the pipeline it will time, outside any timed region."""
    import cv2
    cv2.setNumThreads(1)
    _W["frames"] = frames
    _W["pipe"], _W["kind"] = _make_cpu_pipeline(ref_root)


def _make_cpu_pipeline(ref_root):
    """The reference's PreprocessPipeline from oracle/_ref when build() installed it (kind "reference"), else the restated
    six cv2 calls of oracle/cv2_chain.py (kind "port"; proven equal by tests/test_reference_equivalence.py)."""
    if ref_root and os.path.isfile(os.path.join(ref_root, "src", "preprocess", "pipeline.py")):
        saved = {k: sys.modules.pop(k) for k in [k for k in sys.modules if k == "src" or k.startswith("src.")]}
        sys.path.insert(0, ref_root)
        try:
            from src.preprocess import PreprocessPipeline as RefPipeline      # the reference, unmodified
            pipe = RefPipeline(CHAIN_CFG)
        finally:
            sys.path.remove(ref_root)
            for k in [k for k in sys.modules if k == "src" or k.startswith("src.")]:
                del sys.modules[k]
            sys.modules.update(saved)
        return pipe, "reference"
    from oracle import cv2_chain
    return (lambda img, ts=None: cv2_chain.chain(img, SPACE, CLIP, GRID, KSIZE)), "port"


def _cpu_worker(idx):
    t0 = time.perf_counter()
    fr = _W["frames"]
    for i in idx:
        _W["pipe"](fr[i % len(fr)])
    return time.perf_counter() - t0, _W["kind"]


def cpu_reference(pool, steps, warmup, budget_s=None):
    """ONE loop for `--impl reference` and for the `cpu_baseline` leg: every step is the whole 64-frame batch of the
    configured workload, frame-parallel over all host cores (one single-threaded cv2 per process), a barrier per step.
    steps: number of timed steps; with budget_s, as many steps as fit in that many seconds (at least 3)."""
    import multiprocessing as mp
    import cv2
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    chunks = [list(range(c, BATCH, cores)) for c in range(cores)]
    chunks = [c for c in chunks if c]
    with mp.get_context("spawn").Pool(len(chunks), initializer=_cpu_init, initargs=(list(pool), REF_ROOT)) as pp:
        kind = "port"
        for _ in range(max(warmup, 1)):
            kind = pp.map(_cpu_worker, chunks)[0][1]
        done, t0 = 0, time.perf_counter()
        while True:
            pp.map(_cpu_worker, chunks)
            done += 1
            if budget_s is None and done >= steps:
                break
            if budget_s is not None and done >= 3 and time.perf_counter() - t0 >= budget_s:
                break
        dt = time.perf_counter() - t0
    fps = BATCH * done / dt
    # as shipped: one process, cv2's own thread pool (what `python main_preview.py` does); reported, not the baseline
    pipe, _ = _make_cpu_pipeline(REF_ROOT)
    cv2.setNumThreads(-1)
    pipe(pool[0])
    n, t1 = 0, time.perf_counter()
    while n < 8 or time.perf_counter() - t1 < 1.5:
        pipe(pool[n % len(pool)])
        n += 1
    fps_shipped = n / (time.perf_counter() - t1)
    what = ("reference's own PreprocessPipeline (oracle/_ref/road-vision-system/src/preprocess)" if kind == "reference"
            else "reference's six cv2 calls restated (oracle/cv2_chain.py)")
    return {"value": fps, "unit": UNIT, "cores": len(chunks), "kind": kind,
            "sample": f"{done} steps x {BATCH} x 1080p frames ({dt:.1f} s), {what}, cv2 {cv2.__version__}, frame-parallel "
                      f"{len(chunks)} processes x 1 cv2 thread; as shipped (1 process, {cv2.getNumThreads()} cv2 threads): "
                      f"{fps_shipped:.1f} fps",
            "steps": done, "seconds": dt, "as_shipped_fps": fps_shipped}


def bind_near_gpu(index):
    """Pin this rank to the host cores next to its GPU (PCI device's local_cpulist) so that pinned staging buffers are
    first-touched on the GPU's NUMA node; with 8 ranks the end-to-end leg is host-memory bound.  Best effort."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(index)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        txt = open(f"/sys/bus/pci/devices/{bdf}/local_cpulist").read().strip()
        cpus = set()
        for part in txt.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        use = cpus & allowed
        if use and use != allowed:
            os.sched_setaffinity(0, use)
            return f"{len(use)} cores local to {bdf}"
        return "affinity unchanged (all allowed cores are local or none is)"
    except Exception as e:        # noqa: BLE001
        return f"affinity unchanged ({type(e).__name__})"


def base_line(n_gpus, steps, warmup):
    return {
        "metric": METRIC, "unit": UNIT, "n_gpus": n_gpus, "steps": steps, "warmup": warmup,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": DATA,
        "config": {"workload": "BASELINE configs[1]: 1920x1080 batch-64 chain, YCrCb, clip 2.0, tile_grid 8, MedianDerain k5",
                   "frames_per_gpu_per_step": BATCH, "global_batch": BATCH * n_gpus, "parallelism": f"frames sharded x{n_gpus}, no collective",
                   "l2": "per-step inputs+outputs (796 MB per GPU) exceed the 126 MB L2; no explicit flush"},
    }


def run_reference(args, rank, world):
    """The reference's CPU implementation of the path on all host cores; rank 0 only.  Same config and metric as the GPU arm,
    every step is the full 64-frame batch."""
    if rank != 0:
        return
    pool = load_pool()
    res = cpu_reference(pool, args.steps, args.warmup)
    line = base_line(args.gpus, args.steps, args.warmup)
    line.update({
        "impl": "reference", "value": res["value"], "ms_per_step": 1e3 * BATCH / res["value"],
        "cpu_baseline": res,
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- GPU arm
def timed_loop(fn, steps):
    """Wall-clock time of `steps` host-synchronous calls, max over ranks, barrier on both sides."""
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    dt = time.perf_counter() - t0
    return max_over_ranks(dt)


def stream_leg(rvb200, local_rank, pool, seconds, fps, skip_s=2.0):
    """One paced camera stream on this rank's GPU: SyntheticReader (paced) -> BatchFeeder (pinned ring, capture timestamps) ->
    PreprocessPipeline.process_batch (its own Context) -> pinned result; latency = result ready - capture timestamp."""
    import numpy as np
    from rvb200.io_video.capture import SyntheticReader
    ctx = rvb200.Context(local_rank)
    pipe = rvb200.PreprocessPipeline(CHAIN_CFG, context=ctx)
    nframes = int(seconds * fps)
    vs = rvb200.VideoSource(reader=SyntheticReader(list(pool[:4]), limit=nframes), pinned=None)   # the feeder's ring is the pinned memory
    feeder = rvb200.BatchFeeder(vs, batch=1, shape=(H, W, 3), alloc=ctx.pinned_empty, depth=3, fps=fps)
    out = ctx.pinned_empty((1, H, W, 3))
    warm = ctx.pinned_empty((1, H, W, 3))
    warm[:] = pool[:1]
    for _ in range(3):                                   # context warm-up (allocations, tables) before the camera starts
        pipe.process_batch(warm, out=out)
    lat, stamps = [], []
    for b in feeder:
        pipe.process_batch(b.frames, out=out[:b.count])
        done = time.time()
        lat.extend(done - b.ts)
        stamps.extend(b.ts)
        feeder.release(b)
    ctx.close()
    lat, stamps = np.array(lat), np.array(stamps)
    keep = stamps >= stamps[0] + skip_s
    lat_k, st_k = np.sort(lat[keep]), stamps[keep]
    span = float(st_k[-1] - st_k[0]) if len(st_k) > 1 else 0.0
    return {"frames": int(keep.sum()), "fps": (len(st_k) - 1) / span if span > 0 else 0.0,
            "p50_ms": 1e3 * float(lat_k[len(lat_k) // 2]), "p99_ms": 1e3 * float(lat_k[min(len(lat_k) - 1, int(len(lat_k) * 0.99))]),
            "max_ms": 1e3 * float(lat_k[-1])}


def load_ncu_constants(rvb200):
    """DRAM bytes and executed warp instructions of one k_chain launch from the committed ncu capture, tied to the source tree."""
    path = os.path.join(ROOT, "profiles", "final_k_chain.json")
    tree = rvb200.kernel_source_hash()
    try:
        j = json.load(open(path))
    except Exception:
        return None, {"traffic_source": None, "tree_hash": tree, "note": "profiles/final_k_chain.json missing"}
    # the capture is tied to the BINARY: the SASS of the measured kernel in the library loaded here must be the SASS the capture ran
    # on (a change elsewhere in csrc/ -- another instantiation's network, host code -- leaves it valid); the hash over the kernel
    # sources is reported next to it
    try:
        built = rvb200.kernel_sass_hash(j["kernel"])
    except Exception as e:                                   # cuobjdump missing: fall back to the source hash alone
        built = "unavailable: %s" % (str(e)[:80],)
    info = {"traffic_source": "profiles/final_k_chain.json", "capture": j.get("capture"), "kernel": j.get("kernel", "").split("(")[0],
            "capture_sass_hash": j.get("sass_hash"), "built_sass_hash": built,
            "capture_hash": j.get("source_hash"), "tree_hash": tree,
            "hash_match": (j.get("sass_hash") is not None and j.get("sass_hash") == built) or j.get("source_hash") == tree}
    return j, info


DUMP_ROWS, DUMP_SEED = 2048, 0


def sample_output_rows(d_out):
    """A fixed sample of an output batch (BATCH, H, W, 3) uint8 for comparing two builds: DUMP_ROWS whole rows, gathered on the
    device (so that later steps cannot overwrite them), and their (frame, row) index."""
    import numpy as np
    import torch
    pick = np.sort(np.random.default_rng(DUMP_SEED).choice(BATCH * H, DUMP_ROWS, replace=False))
    frame, row = pick // H, pick % H
    rows = d_out[torch.from_numpy(frame).to(d_out.device), torch.from_numpy(row).to(d_out.device)]
    return rows, np.stack([frame, row], axis=1)


def dump_outputs(out_dir, rows, index):
    """chain_out_rows.npy: the sampled rows as float32 (47 MB); chain_out_rows_index.npy: their (frame, row) as float64."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "chain_out_rows.npy"), rows.cpu().numpy().astype(np.float32))
    np.save(os.path.join(out_dir, "chain_out_rows_index.npy"), index.astype(np.float64))


def run_gpu(args, rank, world, local_rank):
    import numpy as np
    import torch
    import rvb200

    torch.cuda.set_device(local_rank)
    numa = bind_near_gpu(local_rank) if world > 1 else "single rank: not bound"
    ctx = rvb200.Context(local_rank)
    if args.group:
        ctx.set_option("group_frames", args.group)
    if args.chunk:
        ctx.set_option("chunk_frames", args.chunk)
    if args.overlap >= 0:
        ctx.set_option("overlap_groups", args.overlap)
    if args.prefetch >= 0:
        ctx.set_option("prefetch_ctas", args.prefetch)
    params = rvb200.Params.make(SPACE, CLIP, GRID, KSIZE)
    pool = load_pool()
    a, _ = shard_range(BATCH * world, rank, world)            # this rank's slab of the global frame index space
    host = np.stack([pool[(a + i) % POOL] for i in range(BATCH)])
    d_in = torch.from_numpy(host).cuda()
    d_out = torch.empty_like(d_in)
    tstream = torch.cuda.Stream()          # the stream every kernel of the step is launched on; events are recorded on it
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0

    def step():
        ctx.submit_device(d_in.data_ptr(), d_out.data_ptr(), BATCH, H, W, params, stream=stream)

    step(); torch.cuda.synchronize()
    # parity gate: the GPU output of every distinct pool frame must hash to what the REFERENCE's PreprocessPipeline produced
    # when the pool was generated (tests/golden/pool_1080p/index.txt) -- never report a wrong kernel's speed
    shas = pool_reference_shas()
    first = d_out[:POOL].cpu().numpy()
    for i in range(POOL):
        if hashlib.sha1(first[i].tobytes()).hexdigest() != shas[(a + i) % POOL]:
            raise SystemExit(f"bench: CUDA chain output of pool frame {(a + i) % POOL} differs from the reference's; refusing to report")
    gpu_first = first[0]

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize(); barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start(); time.sleep(0.25)
    l0 = ctx.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(); torch.cuda.synchronize()
    t0 = time.time()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize(); barrier()
    ms = e0.elapsed_time(e1)
    launches = ctx.launch_count - l0
    dump = sample_output_rows(d_out) if args.dump_outputs and rank == 0 else None
    ms_max = max_over_ranks(ms)
    frames_total = sum_over_ranks(BATCH * args.steps)
    value = frames_total / (ms_max * 1e-3)

    # sustained: the same step, back to back, for at least ~1.2 s of device time (same events, same stream)
    n_sus = max(args.steps, int(1.3e3 / max(ms / args.steps, 1e-3)))
    barrier(); torch.cuda.synchronize()
    e0.record()
    for _ in range(n_sus):
        step()
    e1.record()
    torch.cuda.synchronize(); barrier()
    ms_sus = max_over_ranks(e0.elapsed_time(e1))
    sustained = {"steps": n_sus, "seconds": ms_sus * 1e-3, "value": sum_over_ranks(BATCH * n_sus) / (ms_sus * 1e-3), "unit": UNIT}
    t1 = time.time()
    clocks = sampler.stop(t0, t1) if rank == 0 else None
    if dump is not None:                        # written outside the sampled clock window
        dump_outputs(args.dump_outputs, *dump)
        del dump
    if clocks is not None:
        clocks["window"] = "the K timed steps + the sustained loop (%d steps), %.2f s" % (n_sus, t1 - t0)

    # second pass: per-kernel device time with an event pair around every launch
    ctx.set_option("kernel_timing", 1)
    ctx.kernel_times(reset=True)
    for _ in range(args.steps):
        step()
    torch.cuda.synchronize()
    kt = ctx.kernel_times(reset=True)
    ctx.set_option("kernel_timing", 0)

    # ---- end to end through the plugin API from pinned host memory
    pl = rvb200.PreprocessPipeline(dict(CHAIN_CFG, device=local_rank), context=ctx)
    e2e = e2e_tensor = e2e_keep = None
    if not args.no_e2e:
        pin_in, pin_out = ctx.pinned_empty(host.shape), ctx.pinned_empty(host.shape)
        pin_in[:] = host
        e2e_steps = max(3, min(args.steps, 10))

        def full():
            pl.process_batch(pin_in, out=pin_out)
            return int(pin_out[-1, -1, -1, 0])                    # host read of the step's result

        for _ in range(2):
            full()
        e2e_s = timed_loop(full, e2e_steps)
        if not np.array_equal(pin_out[0], gpu_first):
            raise SystemExit("bench: end-to-end output differs from the device-resident output")
        e2e = {"value": sum_over_ranks(BATCH * e2e_steps) / e2e_s, "unit": UNIT, "h2d_bytes_per_step": BATCH * FRAME_BYTES,
               "d2h_bytes_per_step": BATCH * FRAME_BYTES, "steps": e2e_steps,
               "api": "PreprocessPipeline.process_batch(pinned in, pinned out)"}

        # configs[4]: chain fused with the letterbox, only the detector tensor returns
        pin_t = ctx.pinned_empty((BATCH, 3, TENSOR_SIZE, TENSOR_SIZE), np.float16)
        pin_t[:] = 0
        ctx.fill_tensor_padding(pin_t, H, W, TENSOR_SIZE)            # once per buffer: the constant padding rows never cross PCIe again
        _, lb_nh, _, _, _ = ctx.letterbox_geometry(H, W, TENSOR_SIZE)

        def tens():
            pl.process_batch_to_tensor(pin_in, size=TENSOR_SIZE, out=pin_t, padding_present=True)
            return float(pin_t[-1, -1, TENSOR_SIZE // 2, -1])         # host read of the step's result (an image row)

        for _ in range(2):
            tens()
        t_s = timed_loop(tens, e2e_steps)
        want_t, _ = pl.process_batch_to_tensor(host[:1], size=TENSOR_SIZE)
        if not np.array_equal(pin_t[0].view(np.uint16), want_t[0].view(np.uint16)):
            raise SystemExit("bench: pipelined tensor differs from the unpipelined one")
        e2e_tensor = {"value": sum_over_ranks(BATCH * e2e_steps) / t_s, "unit": UNIT, "h2d_bytes_per_step": BATCH * FRAME_BYTES,
                      "d2h_bytes_per_step": BATCH * 3 * lb_nh * TENSOR_SIZE * 2, "steps": e2e_steps,
                      "note": "the pinned tensor buffer holds its constant padding rows (written once); only the 360 image rows of each plane "
                              "come back per step; the complete tensor in host memory is checked against the unpipelined one",
                      "workload": "BASELINE configs[4]-style: headline chain fused with letterbox 640 + RGB fp16 NCHW; 64 frames per GPU per step",
                      "api": "PreprocessPipeline.process_batch_to_tensor(pinned frames, out=pinned (B,3,640,640) float16, padding_present=True)"}

        def keep():
            dev, _ = pl.process_batch_to_tensor(pin_in, size=TENSOR_SIZE, out="device")
            return dev

        for _ in range(2):
            keep()
        k_s = timed_loop(keep, e2e_steps)
        e2e_keep = {"value": sum_over_ranks(BATCH * e2e_steps) / k_s, "unit": UNIT, "h2d_bytes_per_step": BATCH * FRAME_BYTES,
                    "d2h_bytes_per_step": 0, "steps": e2e_steps,
                    "api": "PreprocessPipeline.process_batch_to_tensor(pinned frames, out='device'): the tensor stays on the GPU for the detector"}
        del pin_in, pin_out, pin_t

    # ---- configs[3]: one paced 1080p@30 stream per GPU
    streams = None
    if args.stream_seconds > 0:
        barrier()
        s = stream_leg(rvb200, local_rank, pool, args.stream_seconds, 30.0)
        streams = {"streams": world, "per_gpu": 1, "fps_requested": 30.0, "seconds": args.stream_seconds, "excluded_first_s": 2.0,
                   "fps_min": min_over_ranks(s["fps"]), "fps_mean": sum_over_ranks(s["fps"]) / world,
                   "latency_ms_p50_max_over_gpus": max_over_ranks(s["p50_ms"]), "latency_ms_p99_max_over_gpus": max_over_ranks(s["p99_ms"]),
                   "latency_ms_max": max_over_ranks(s["max_ms"]), "frames": sum_over_ranks(s["frames"]),
                   "path": "SyntheticReader paced at 30 fps -> BatchFeeder (pinned ring, time.time() at capture) -> "
                           "PreprocessPipeline(context=own Context).process_batch -> pinned result; latency = result - capture"}

    if rank != 0:
        return
    peaks, peak_src = None, "fallback (B200_PROFILING.md: 6650 GB/s)"
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        peak, peak_src = float(peaks["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        peak = 6650.0
    chain_ms, chain_n = kt["k_chain"]
    frames_per_launch = BATCH * args.steps / max(chain_n, 1)
    avg_launch_s = chain_ms * 1e-3 / max(chain_n, 1)
    achieved = ALGO_BYTES_PER_FRAME * frames_per_launch / avg_launch_s / 1e9 if chain_n else None
    total_k = sum(v[0] for v in kt.values())
    ncu, ncu_info = load_ncu_constants(rvb200)
    per64 = frames_per_launch / 64.0
    line = base_line(world, args.steps, args.warmup)
    line.update({
        "value": value, "ms_per_step": ms_max / args.steps, "gpu_launches": launches, "clocks": clocks,
        "sustained": sustained, "host_affinity": numa,
        "parity": "all 8 pool frames: SHA-1 of the CUDA output equals the SHA-1 of the reference PreprocessPipeline output recorded "
                  "with the pool (tests/golden/pool_1080p/index.txt)",
        "e2e": e2e, "e2e_tensor": e2e_tensor, "e2e_keep": e2e_keep, "streams": streams,
        "roofline": {"bound": "hbm", "kernel": "k_chain<YCrCb,5>", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": (achieved / peak) if achieved else None, "peak_source": peak_src,
                     "algorithmic_bytes_per_frame": ALGO_BYTES_PER_FRAME, "frames_per_launch": frames_per_launch,
                     "avg_launch_ms": avg_launch_s * 1e3,
                     "kernel_share_of_step": {k: (v[0] / total_k if total_k else None) for k, v in kt.items()},
                     "kernel_ms_per_step": {k: v[0] / args.steps for k, v in kt.items()},
                     "whole_chain_achieved_gbs": ALGO_BYTES_PER_FRAME * value / world / 1e9,
                     "traffic": (ncu["dram_bytes_read"] + ncu["dram_bytes_write"]) * per64 if ncu else None,
                     "traffic_info": ncu_info},
    })
    # why the HBM fraction is low: k_chain is bound by instruction issue, not by memory (DESIGN.md section 5).  Warp instructions
    # per launch come from the committed ncu capture (hash-tied to the tree), the launch time is the live measurement above.
    if ncu and chain_n:
        sm_clock = (clocks or {}).get("sm_mhz") or 1965.0
        sms = torch.cuda.get_device_properties(local_rank).multi_processor_count
        issue_peak = sms * 4 * sm_clock * 1e6                      # one warp instruction per scheduler per clock
        wi = ncu["warp_instructions"] * per64
        line["roofline"]["issue"] = {
            "warp_instr_per_launch": wi, "thread_instr_per_pixel": ncu["warp_instructions"] * 32 / (64.0 * H * W),
            "achieved_gwarp_instr_s": wi / avg_launch_s / 1e9, "peak_gwarp_instr_s": issue_peak / 1e9,
            "frac": wi / avg_launch_s / issue_peak,
            "source": "smsp__inst_executed.sum of one 64-frame k_chain launch (profiles/final_k_chain.json); peak = SMs x 4 schedulers x SM clock"}
    if world == 1 and not args.no_cpu:
        line["cpu_baseline"] = cpu_reference(pool, 0, 1, budget_s=args.cpu_seconds)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default 1200 for the GPU arm, sized so that the timed region spans > 1 s; 20 for the reference arm)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--group", type=int, default=0, help="frames per hist->lut->chain group (0 = library default)")
    ap.add_argument("--chunk", type=int, default=0, help="frames per host pipeline chunk (0 = library default)")
    ap.add_argument("--overlap", type=int, default=-1, help="groups per batch for the histogram/chain overlap (-1 = library default)")
    ap.add_argument("--prefetch", type=int, default=-1, help="k_chain L2 prefetch distance in CTAs per SM (-1 = library default, 0 = off)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true", help="skip the end-to-end legs (profiling runs)")
    ap.add_argument("--stream-seconds", type=float, default=32.0, help="length of the paced-stream leg (0 = skip)")
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="time budget of the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a seeded sample of the last step's output (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 20 if args.impl == "reference" else 1200
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the GPU arm's outputs")

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # plain `python bench.py --gpus N`: relaunch one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29577")] + sys.argv
        raise SystemExit(subprocess.call(cmd))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_gpu(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
