#!/usr/bin/env python3
"""Install the UNMODIFIED reference (pure Python, no build system: 34 .py files + configs/default.yaml) under oracle/_ref/.

    python oracle/install_ref.py <checkout of road-vision-system>

BENCHMARK INFRASTRUCTURE ONLY.  __graft_entry__.build() runs it where a checkout of the reference is present; oracle/_ref/
is git-ignored (never part of the history).  Where it is installed,
`bench.py --impl reference` and the `cpu_baseline` leg time the reference's OWN `PreprocessPipeline`
(src/preprocess/pipeline.py:7-45 with ops/clahe_dehaze.py:13-32 and ops/median_derain.py:10-14); without it they time the
same cv2 calls restated in oracle/cv2_chain.py.

Nothing is edited: files are copied byte for byte.  Only bench.py's CPU legs read the result.
"""
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DEST = os.path.join(HERE, "_ref", "road-vision-system")
KEEP_EXT = (".py", ".yaml", ".yml", ".txt")


def ref_root():
    return DEST


def available():
    return os.path.isfile(os.path.join(DEST, "src", "preprocess", "pipeline.py"))


def install(src):
    """Copy the reference tree (source files only) into oracle/_ref/road-vision-system; returns the number of files."""
    if not os.path.isdir(os.path.join(src, "src", "preprocess")):
        return 0
    if os.path.isdir(DEST):
        shutil.rmtree(DEST)
    n = 0
    for dirpath, dirnames, files in os.walk(src):
        dirnames[:] = [d for d in dirnames if d not in ("__pycache__", ".idea", ".git")]
        rel = os.path.relpath(dirpath, src)
        for f in files:
            if f.endswith(KEEP_EXT):
                os.makedirs(os.path.join(DEST, rel), exist_ok=True)
                shutil.copyfile(os.path.join(dirpath, f), os.path.join(DEST, rel, f))
                n += 1
    return n


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    print(f"installed {install(sys.argv[1])} files under {DEST}")
