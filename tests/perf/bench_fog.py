#!/usr/bin/env python3
"""Fog synthesis throughput: this package on the GPU next to the reference's EnhancedFogSynthesizer on the host (where
oracle/install_ref.py has installed it under oracle/_ref), 1080p frames, fog_batch.py's parameters.  One JSON line."""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(1, os.path.join(ROOT, "tests"))
import rvb200  # noqa: E402
from rvb200 import synth  # noqa: E402
from rvb200.augment import EnhancedFogSynthesizer  # noqa: E402
from test_fog import KW  # noqa: E402
from oracle import install_ref  # noqa: E402


def reference_fog_class():
    """The reference's class from oracle/_ref, or None."""
    if not install_ref.available():
        return None
    sys.path.insert(0, install_ref.ref_root())
    try:
        sys.dont_write_bytecode = True
        from src.augment.fog import EnhancedFogSynthesizer as Ref
        return Ref
    finally:
        sys.path.remove(install_ref.ref_root())


clean = [synth.clean_scene(1080, 1920, 950 + i) for i in range(4)]
ctx = rvb200.default_context()
fog = EnhancedFogSynthesizer(level="medium", seed=5, context=ctx, **KW)
for i in range(3):
    fog.synthesize(clean[i % 4])
n, t0 = 0, time.perf_counter()
while time.perf_counter() - t0 < 3.0:
    fog.synthesize(clean[n % 4])
    n += 1
gpu = n / (time.perf_counter() - t0)
n, t0 = 0, time.perf_counter()
while time.perf_counter() - t0 < 3.0:
    fog.synthesize(clean[n % 4], meta=False)
    n += 1
gpu_nometa = n / (time.perf_counter() - t0)
row = {"what": "fog synthesis, 1080p, medium, fog_batch.py parameters", "gpu_frames_per_s": round(gpu, 1), "gpu_ms_per_frame": round(1e3 / gpu, 2),
       "gpu_frames_per_s_without_meta_maps": round(gpu_nometa, 1)}
Ref = reference_fog_class()
if Ref is not None:
    ref = Ref(level="medium", seed=5, **KW)
    ref.synthesize(clean[0])
    m, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < 5.0:
        ref.synthesize(clean[m % 4])
        m += 1
    cpu = m / (time.perf_counter() - t0)
    row.update({"reference_frames_per_s": round(cpu, 2), "speedup": round(gpu / cpu, 1)})
print(json.dumps(row), flush=True)
