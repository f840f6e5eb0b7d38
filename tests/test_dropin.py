"""The drop-in claim: `from src.preprocess import PreprocessPipeline` (main_preview.py:6,58,94) and the `preprocess:` block of
the reference's configs/default.yaml drive the B200 ops unchanged when this package is mounted as `src/preprocess`
(INTEGRATION.md section 2); the GPU half also needs a B200."""
import os
import subprocess
import sys
import textwrap

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "road-vision-system_b200")

# what the reference's load_config() returns under "preprocess" for its stock configs/default.yaml:21-34
STOCK_PREPROCESS = {"enabled": True,
                    "chain": [{"name": "CLAHEDehaze", "params": {"space": "YCrCb", "clip_limit": 2.0, "tile_grid": 8}},
                              {"name": "MedianDerain", "params": {"ksize": 3}}],
                    "auto_gate": {"enable_low_contrast_gate": False, "contrast_thresh": 20.0}}


def make_tree(tmp_path):
    """<tmp>/src/{preprocess,io_video,_native.py,csrc,synth.py} -> this package."""
    src = tmp_path / "src"
    src.mkdir()
    (src / "__init__.py").write_text("")
    for name in ("preprocess", "io_video", "_native.py", "csrc", "synth.py"):
        os.symlink(os.path.join(PKG, name), src / name)
    return tmp_path


def run(tmp, body):
    code = "import sys; sys.dont_write_bytecode = True; sys.path.insert(0, %r); sys.path.insert(1, %r)\n" % (str(tmp), ROOT)
    code += textwrap.dedent(body)
    return subprocess.run([sys.executable, "-c", code], cwd=str(tmp), capture_output=True, text=True, timeout=600)


def test_stock_yaml_builds_the_pipeline(tmp_path):
    tmp = make_tree(tmp_path)
    r = run(tmp, """
        from src.preprocess import PreprocessPipeline         # main_preview.py:6
        from src.preprocess.registry import REGISTRY
        pp = %r
        pipe = PreprocessPipeline(pp)                         # main_preview.py:58
        assert pipe.enabled and [type(o).__name__ for o in pipe.ops] == ["CLAHEDehaze", "MedianDerain"], pipe.ops
        seg = pipe._segments()
        assert len(seg) == 1 and (seg[0].space, seg[0].grid, seg[0].ksize, seg[0].clip_limit) == (0, 8, 3, 2.0)
        assert set(REGISTRY) >= {"CLAHEDehaze", "MedianDerain", "CUDACLAHEDehaze", "CUDAMedianDerain"}
        import numpy as np
        img = np.zeros((4, 4, 3), np.uint8)
        assert PreprocessPipeline({"enabled": False})(img) is img
        print("ok")
    """ % (STOCK_PREPROCESS,))
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]


@pytest.mark.gpu
def test_stock_chain_runs_on_gpu_as_src_preprocess(tmp_path):
    """GPU half: the same mount as `src/preprocess` and the same stock `preprocess:` block, one camera-sized frame."""
    tmp = make_tree(tmp_path)
    r = run(tmp, """
        import numpy as np
        from src.preprocess import PreprocessPipeline         # main_preview.py:6
        from src import synth
        from oracle import rv_oracle as O
        pipe = PreprocessPipeline(%r)                         # main_preview.py:58
        raw = synth.road_frame(480, 640, 1)                   # default.yaml:3-4 camera size
        keep = raw.copy()
        proc = pipe(raw, ts=0.0)                              # main_preview.py:94
        assert proc is not raw and proc.flags.writeable and proc.flags.c_contiguous
        assert np.array_equal(raw, keep)
        assert np.array_equal(proc, O.chain(raw, O.SPACE_YCRCB, 2.0, 8, 3))
        proc[:] = 0                                           # draw_detections writes into it (main_preview.py:114)
        print("ok")
    """ % (STOCK_PREPROCESS,))
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]
