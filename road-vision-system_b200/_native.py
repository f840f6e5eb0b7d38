"""ctypes binding of librv_b200.so (include/rv_b200.h).  Plumbing only -- no arithmetic here."""
import ctypes as C
import os
import shutil
import subprocess
import threading
import weakref

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "csrc")
_SO = os.path.join(_CSRC, "librv_b200.so")

SPACE_YCRCB, SPACE_LAB = 0, 1
MEM_HOST, MEM_PINNED, MEM_DEVICE = 0, 1, 2
YUV_LAYOUTS = {"NV12": 1, "I420": 2}        # enum rv_yuv
YUV422_LAYOUTS = {"YUY2": 16, "UYVY": 17}   # enum rv_yuv422


class RvError(RuntimeError):
    """A call into the CUDA library failed (no silent CPU fallback exists)."""


class Params(C.Structure):
    """rv_params: parameters *after* the reference's coercions."""
    _fields_ = [
        ("space", C.c_int32), ("grid", C.c_int32), ("ksize", C.c_int32), ("clahe", C.c_int32),
        ("clip_limit", C.c_double), ("gate_enable", C.c_int32), ("reserved", C.c_int32),
        ("gate_thresh", C.c_double),
    ]

    @classmethod
    def make(cls, space="YCrCb", clip_limit=2.0, grid=8, ksize=3, clahe=True, gate=False, gate_thresh=20.0):
        return cls(SPACE_LAB if space == "LAB" else SPACE_YCRCB, int(grid), int(ksize), 1 if clahe else 0,
                   float(clip_limit), 1 if gate else 0, 0, float(gate_thresh))


class IO(C.Structure):
    """rv_io: one job of rv_submit_io -- every end (frames in, frames out, detector tensor out) has its own memory kind."""
    _fields_ = [
        ("in_", C.c_void_p), ("in_pitch", C.c_size_t), ("out", C.c_void_p), ("out_pitch", C.c_size_t),
        ("tensor", C.c_void_p), ("processed", C.c_void_p),
        ("in_kind", C.c_int32), ("out_kind", C.c_int32), ("tensor_kind", C.c_int32),
        ("tensor_size", C.c_int32), ("pad_value", C.c_int32), ("tensor_flags", C.c_int32),
    ]


class DeviceArray:
    """A result that stayed on the GPU (process_batch(..., out="device")): device memory owned by the context, freed when
    this object is garbage-collected.  Exposes `__cuda_array_interface__` (version 3), so `torch.as_tensor(x, device="cuda")`
    and `cupy.asarray(x)` wrap it without a copy; `numpy()` downloads it."""

    def __init__(self, ctx, shape, dtype=np.uint8):
        self.shape, self.dtype = tuple(int(v) for v in shape), np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        self.ptr, self.ctx = ctx._device_block(max(self.nbytes, 1)), ctx
        self._finalizer = weakref.finalize(self, ctx._device_block_done, self.ptr, max(self.nbytes, 1))

    @property
    def __cuda_array_interface__(self):
        return {"shape": self.shape, "typestr": self.dtype.str, "data": (self.ptr, False), "version": 3, "strides": None}

    def numpy(self):
        out = np.empty(self.shape, self.dtype)
        self.ctx._ck(self.ctx._lib.rv_memcpy(self.ctx._h, out.ctypes.data, C.c_void_p(self.ptr), self.nbytes, 1))
        return out


def chunk_schedule(n, chunk_frames, taper=True):
    """Chunk sizes the host pipeline cuts a job of n frames into (rv_chunk_schedule; needs the library, not a GPU)."""
    lib = load_library()
    cnt = lib.rv_chunk_schedule(n, chunk_frames, 1 if taper else 0, None, 0)
    if cnt < 0:
        raise ValueError("bad arguments")
    out = (C.c_int * max(cnt, 1))()
    lib.rv_chunk_schedule(n, chunk_frames, 1 if taper else 0, out, cnt)
    return [int(out[i]) for i in range(cnt)]


def library_path():
    return _SO


def build_library(force=False, verbose=False):
    """Compile csrc/ for sm_100a with nvcc (works without a GPU)."""
    srcs = [os.path.join(_CSRC, f) for f in sorted(os.listdir(_CSRC)) if f.endswith((".cu", ".cuh", ".h")) or f == "Makefile"]
    srcs.append(os.path.join(os.path.dirname(_HERE), "include", "rv_b200.h"))
    srcs = [s for s in srcs if os.path.exists(s)]
    stale = (not os.path.exists(_SO)) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs)
    if force or stale:
        cmd = ["make", "-C", _CSRC, "librv_b200.so"] + (["-B"] if force else [])
        subprocess.check_call(cmd, stdout=None if verbose else subprocess.DEVNULL)
    return _SO


KERNEL_SOURCES = ("Makefile", "rv_common.cuh", "rv_colour.cuh", "rv_hist_lut.cuh", "rv_chain.cuh", "rv_median_net.h", "rv_lab_tables.h",
                  "rv_ycc_g.h")


def kernel_source_hash():
    """SHA-256 (first 16 hex digits) over the files that determine the device code of the chain's kernels (not the host-side
    C ABI), with comments and white space removed -- so that editing a comment does not orphan a profile, while any change a
    compiler could see does.  profiles/final_*.json records it with every ncu capture; bench.py and the CPU test suite compare it
    with the tree, so profile-derived constants can never silently outlive the code they were measured on."""
    import hashlib
    import re
    h = hashlib.sha256()
    for name in KERNEL_SOURCES:
        with open(os.path.join(_CSRC, name), "r") as fh:
            text = fh.read()
        if name != "Makefile":
            text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)           # block comments
            text = re.sub(r"//[^\n]*", " ", text)                        # line comments (no string in these files contains //)
        else:
            text = re.sub(r"#[^\n]*", " ", text)
        text = " ".join(text.split())
        h.update(name.encode() + b"\0" + text.encode() + b"\0")
    return h.hexdigest()[:16]


_sass_cache = {}


def kernel_sass_hashes(so=None):
    """{demangled kernel name: SHA-256 (first 16 hex digits) of its SASS listing} for every kernel in the built library
    (`cuobjdump -sass`, names through `cu++filt`).  This is the tie between a profile and the BINARY: an ncu capture stays valid
    for as long as the machine code of the kernel it measured is unchanged, whatever else is edited in csrc/ (another
    instantiation's network, a comment, host code); profiles/final_*.json record it as `sass_hash` next to `source_hash`."""
    import hashlib
    import re
    so = so or _SO
    key = (so, os.path.getmtime(so))
    if key in _sass_cache:
        return _sass_cache[key]
    cuda_bin = os.path.dirname(shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump")
    text = subprocess.run([os.path.join(cuda_bin, "cuobjdump"), "-sass", so], capture_output=True, text=True, check=True).stdout
    parts = re.split(r"^\s*Function : (\S+)\s*$", text, flags=re.M)
    names, bodies = parts[1::2], parts[2::2]
    dem = subprocess.run([os.path.join(cuda_bin, "cu++filt")] + names, capture_output=True, text=True, check=True).stdout.splitlines()
    out = {}
    for n, body in zip(dem, bodies):
        body = body.split("Fatbin elf code:")[0]
        body = "\n".join(ln.strip() for ln in body.splitlines() if ln.strip() and not ln.strip().startswith(("=", ".")))
        n = re.sub(r"\((?:int|bool)\)", "", n).replace("rv::", "")
        out[n] = hashlib.sha256(body.encode()).hexdigest()[:16]
    _sass_cache[key] = out
    return out


def kernel_sass_hash(kernel, so=None):
    """SASS hash of one kernel, named the way ncu prints it (e.g. 'k_chain<0, 5>'; a prefix of the full signature is enough)."""
    import re
    want = re.sub(r"^void\s+", "", kernel).replace("rv::", "")
    want = want.split("(")[0].replace(" ", "")
    hits = [h for n, h in kernel_sass_hashes(so).items() if re.sub(r"^void\s+", "", n).split("(")[0].replace(" ", "") == want]
    if len(hits) != 1:
        raise KeyError(f"kernel {kernel!r} not found (or ambiguous) in {so or _SO}")
    return hits[0]


_lib = None
_lib_lock = threading.Lock()

_u8p = C.POINTER(C.c_uint8)
_i32p = C.POINTER(C.c_int32)

EXPORTS = {
    # name: (restype, argtypes)
    "rv_version": (C.c_char_p, []),
    "rv_device_count": (C.c_int, []),
    "rv_ycc_table": (C.c_int, [C.POINTER(C.c_uint32)]),
    "rv_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "rv_destroy": (None, [C.c_void_p]),
    "rv_last_error": (C.c_char_p, [C.c_void_p]),
    "rv_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_long]),
    "rv_launch_count": (C.c_long, [C.c_void_p]),
    "rv_chunk_schedule": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.c_int]),
    "rv_alloc_pinned": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "rv_free_pinned": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rv_host_register": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "rv_host_unregister": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rv_alloc_device": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "rv_free_device": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rv_memcpy": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]),
    "rv_sync": (C.c_int, [C.c_void_p]),
    "rv_chain_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t,
                              C.POINTER(Params), C.c_int, _i32p, C.c_void_p]),
    "rv_submit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t,
                            C.POINTER(Params), C.c_int, C.c_void_p]),
    "rv_submit_io": (C.c_int, [C.c_void_p, C.POINTER(IO), C.c_int, C.c_int, C.c_int, C.POINTER(Params)]),
    "rv_kernel_time": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_long)]),
    "rv_kernel_time_reset": (C.c_int, [C.c_void_p]),
    "rv_wait": (C.c_int, [C.c_void_p]),
    "rv_luma_hist": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_int, C.c_int,
                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "rv_build_lut": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_int]),
    "rv_clahe_dehaze": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t,
                                  C.c_int, C.c_double, C.c_int, C.c_int]),
    "rv_median": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t,
                            C.c_int, C.c_int]),
    "rv_letterbox_geometry": (C.c_int, [C.c_int, C.c_int, C.c_int, _i32p, _i32p, _i32p, _i32p, _i32p]),
    "rv_letterbox_f16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "rv_chain_letterbox_f16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.POINTER(Params),
                                         C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "rv_fog_set_geometry": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float),
                                      C.POINTER(C.c_float)]),
    "rv_fog_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float),
                            C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "rv_gray_span": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_int]),
    "rv_chain_u16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t,
                               C.POINTER(Params), C.c_int, _i32p, C.c_void_p]),
    "rv_gray_span_u16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_int]),
    "rv_chain_ex": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_int, C.c_int,
                              C.POINTER(Params), C.c_int, _i32p, C.c_void_p]),
    "rv_gray_span_ex": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_int]),
    "rv_yuv420_to_bgr": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_int, C.c_int,
                                   C.c_void_p]),
    "rv_submit_io_yuv": (C.c_int, [C.c_void_p, C.POINTER(IO), C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(Params)]),
    "rv_bgr_to_yuv420": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_int, C.c_int,
                                   C.c_void_p]),
    "rv_submit_io_fmt": (C.c_int, [C.c_void_p, C.POINTER(IO), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(Params)]),
    "rv_yuv422_to_bgr": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_int, C.c_int,
                                   C.c_void_p]),
}


def load_library():
    """dlopen the in-tree library and declare every symbol of include/rv_b200.h. Raises if it is missing."""
    global _lib, _SO
    with _lib_lock:
        if _lib is None:
            if os.environ.get("RV_B200_LIB"):        # tuning builds of the same source (tools/gpu_variants.sh)
                _SO = os.path.join(_CSRC, os.environ["RV_B200_LIB"])
            if not os.path.exists(_SO):
                raise RvError(f"{_SO} is not built; run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU fallback)")
            lib = C.CDLL(_SO)
            for name, (res, args) in EXPORTS.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _torch_stream(device):
    """torch's current stream on `device` as a cudaStream_t int for the C entries, or None on the legacy default stream: torch's
    queued work is then waited for, and the call runs on the context's stream, synchronously."""
    import torch
    stream = torch.cuda.current_stream(device)
    if stream.cuda_stream == 0:
        stream.synchronize()
    return stream.cuda_stream or None


def _check_torch_out(out, shape, dtype, device, msg):
    """A caller's `out` tensor (None: none given) must be contiguous, of `shape` and `dtype`, on `device`; ValueError(msg) if not."""
    if out is not None and not (_is_torch(out) and out.dtype == dtype and tuple(out.shape) == tuple(shape) and out.device == device
                                and out.is_contiguous()):
        raise ValueError(msg)


_U8 = (np.dtype(np.uint8),)
_U8_U16 = (np.dtype(np.uint8), np.dtype(np.uint16))
CHANNELS = (1, 3, 4)        # gray, BGR, BGRA / BGRx


def _check_frames(frames, dtypes=_U8, channels=(3,)):
    """(N,H,W,C) frames of one of `dtypes`, C in `channels` (BGR only by default)."""
    if not isinstance(frames, np.ndarray):
        raise TypeError("frames must be a numpy.ndarray")
    if frames.dtype not in dtypes:
        raise ValueError(f"{' or '.join(d.name for d in dtypes)} BGR frames expected, got dtype {frames.dtype}")
    if frames.ndim != 4 or frames.shape[3] not in channels:
        want = "3" if channels == (3,) else "C" + f" with C in {channels}"
        raise ValueError(f"(N,H,W,{want}) {frames.dtype} expected, got shape {frames.shape}")
    if frames.shape[1] < 1 or frames.shape[2] < 1:
        raise ValueError("empty frame")


def check_yuv_frames(shape, is_uint8, yuv):
    """A batch of YUV 4:2:0 frames in cv2's single-array form, (B, 3H/2, W) uint8, as cv2.cvtColor(COLOR_YUV2BGR_NV12 / _I420) takes
    them: returns (layout, B, H, W) of the BGR frames they convert to.  Raises ValueError for an unknown `yuv`, a wrong shape or dtype,
    rows not divisible by 3 (H must be even), an odd W (cv2 raises for it) and empty frames.  A 4:2:2 `yuv` ("YUY2", "UYVY") takes
    the rule of check_yuv422_frames instead, so that every entry with a `yuv=` argument checks its frames here."""
    if yuv in YUV422_LAYOUTS:
        return check_yuv422_frames(shape, is_uint8, yuv)
    if yuv not in YUV_LAYOUTS:
        raise ValueError(f"yuv must be None, 'NV12', 'I420', 'YUY2' or 'UYVY', got {yuv!r}")
    shape = tuple(int(v) for v in shape)
    if len(shape) == 4:
        raise ValueError(f"yuv={yuv!r} takes (B,3H/2,W) frames, not (B,H,W,C) ones (got shape {shape})")
    if len(shape) != 3:
        raise ValueError(f"yuv={yuv!r} takes (B,3H/2,W) uint8 frames, got shape {shape}")
    if not is_uint8:
        raise ValueError(f"yuv={yuv!r} takes uint8 frames")
    b, rows, w = shape
    if rows == 0 or w == 0:
        raise ValueError(f"empty {yuv} frames (shape {shape})")
    if rows % 3:
        raise ValueError(f"{yuv} frames have 3H/2 rows with an even H: {rows} rows is not a multiple of 3")
    if w % 2:
        raise ValueError(f"{yuv} frames need an even width, got {w}")
    return YUV_LAYOUTS[yuv], b, rows // 3 * 2, w


def check_yuv422_frames(shape, is_uint8, yuv):
    """A batch of packed YUV 4:2:2 camera frames, (B, H, W, 2) uint8, as cv2.cvtColor(COLOR_YUV2BGR_YUY2 / _UYVY) takes them (each row
    holds W/2 groups of 4 bytes, one per pixel pair: YUY2 Y0 U Y1 V, UYVY U Y0 V Y1): returns (layout, B, H, W) of the BGR frames they
    convert to.  Raises ValueError for a wrong shape, channel count or dtype, an odd W (cv2 raises for it) and empty frames."""
    shape = tuple(int(v) for v in shape)
    if len(shape) != 4 or shape[3] != 2:
        raise ValueError(f"yuv={yuv!r} takes (B,H,W,2) uint8 frames, got shape {shape}")
    if not is_uint8:
        raise ValueError(f"yuv={yuv!r} takes uint8 frames")
    b, h, w, _ = shape
    if h == 0 or w == 0:
        raise ValueError(f"empty {yuv} frames (shape {shape})")
    if w % 2:
        raise ValueError(f"{yuv} frames need an even width (one (U, V) pair per pixel pair), got {w}")
    return YUV422_LAYOUTS[yuv], b, h, w


def yuv_pitch(layout, w):
    """Row pitch in bytes of contiguous YUV frames of `layout` (enum rv_yuv / rv_yuv422) and width w."""
    return 2 * w if layout in YUV422_LAYOUTS.values() else w


def check_out_yuv(out_yuv):
    """The enum rv_yuv value of a 4:2:0 output layout; ValueError for an unknown one."""
    if out_yuv not in YUV_LAYOUTS:
        raise ValueError(f"out_yuv must be None, 'NV12' or 'I420', got {out_yuv!r}")
    return YUV_LAYOUTS[out_yuv]


def check_bgr_for_yuv(shape, is_uint8, out_yuv):
    """A (B,H,W,3) uint8 BGR batch to be returned as 4:2:0 frames (cv2.cvtColor(COLOR_BGR2YUV_I420) takes 8-bit BGR only): returns
    (layout, B, H, W).  Raises ValueError for an unknown `out_yuv`, another rank, channel count or dtype, empty frames, and an odd H
    or W (cv2 raises for both)."""
    layout = check_out_yuv(out_yuv)
    shape = tuple(int(v) for v in shape)
    if len(shape) != 4 or shape[3] != 3:
        raise ValueError(f"out_yuv={out_yuv!r} takes (B,H,W,3) BGR frames (no gray or BGRA ones), got shape {shape}")
    if not is_uint8:
        raise ValueError(f"out_yuv={out_yuv!r} takes uint8 frames (no 4:2:0 output of 16-bit frames)")
    b, h, w, _ = shape
    if h == 0 or w == 0:
        raise ValueError(f"empty frames (shape {shape})")
    if h % 2 or w % 2:
        raise ValueError(f"4:2:0 output needs an even height and width, got {h}x{w}")
    return layout, b, h, w


U16_MAX_GRID = 64


def check_u16_params(params):
    """The chain's parameters on 16-bit frames: what cv2 has no CV_16U path for (LAB, median k 7 / 9) and the tile grid limit of
    this build raise ValueError here, before anything reaches the GPU."""
    if params.space == SPACE_LAB:
        raise ValueError("LAB is not supported on uint16 frames (cv2.cvtColor BGR2LAB has no 16-bit path); use space YCrCb")
    if params.ksize not in (0, 3, 5):
        raise ValueError(f"median ksize {params.ksize} is not supported on uint16 frames (cv2.medianBlur: k = 3 or 5 at 16 bits)")
    if params.clahe and not 2 <= params.grid <= U16_MAX_GRID:
        raise ValueError(f"tile_grid {params.grid} is not supported on uint16 frames (limit {U16_MAX_GRID}: each tile has a "
                         "65,536-entry LUT)")
    if not params.clahe and params.ksize == 0:
        raise ValueError("nothing to do (no CLAHE, no median)")


def check_frame_params(params, dtype, channels):
    """What cv2 rejects for a pass over (..., channels) frames of `dtype` raises ValueError here, before the GPU: the 16-bit limits
    (check_u16_params), CLAHE and the low-contrast gate on a single channel (cv2.cvtColor has no BGR2YCrCb / BGR2LAB / BGR2GRAY for
    one channel).  Returns the channel count of the result: 3 after CLAHE (which drops alpha, as cv2.cvtColor does), else `channels`."""
    if np.dtype(dtype) == np.uint16:
        check_u16_params(params)
    if channels not in CHANNELS:
        raise ValueError(f"frames with {channels} channels are not supported (1, 3 or 4)")
    if channels == 1 and params.clahe:
        raise ValueError("CLAHEDehaze needs BGR or BGRA frames: cv2.cvtColor BGR2YCrCb / BGR2LAB reject single-channel input")
    if channels == 1 and params.gate_enable:
        raise ValueError("the low-contrast gate needs BGR or BGRA frames: cv2.cvtColor BGR2GRAY rejects single-channel input")
    return 3 if params.clahe else channels


class _Lease(np.ndarray):
    """Owner of one hand-out of a pooled page-locked block (see Context._pooled_pinned); users only ever see plain ndarray
    views whose `.base` is this object."""
    _home = None

    def __del__(self):
        home = self._home
        if home is not None:
            ctx, free, blk, keep = home
            if len(free) < keep:
                free.append(blk)
            else:
                ctx._pinned.pop(blk[0], None)
                try:
                    ctx._lib.rv_free_pinned(ctx._h, C.c_void_p(blk[0]))
                except Exception:          # interpreter shutdown
                    pass


class Context:
    """One rv_ctx: a CUDA device, its streams and workspaces. Not thread-safe."""

    def __init__(self, device=0):
        self._lib = load_library()
        h = C.c_void_p()
        rc = self._lib.rv_create(int(device), C.byref(h))
        if rc != 0:
            raise RvError(f"rv_create(device={device}) failed with {rc}: no usable sm_100 GPU (no CPU fallback)")
        self._h = h
        self.device = int(device)
        self._pinned = {}          # base address -> nbytes
        self._pin_pool = {}        # nbytes -> [free page-locked blocks] (results of per-frame calls)
        self._dev_pool = {}        # nbytes -> [free device blocks] (results that stay on the GPU)
        self._finalizer = weakref.finalize(self, self._lib.rv_destroy, h)

    # -- plumbing ------------------------------------------------------------------------
    def _ck(self, rc):
        if rc != 0:
            msg = self._lib.rv_last_error(self._h)
            raise (ValueError if rc == -1 else RvError)(f"rv_b200 error {rc}: {msg.decode() if msg else ''}")

    def close(self):
        self._finalizer()

    def set_option(self, name, value):
        self._ck(self._lib.rv_set_option(self._h, name.encode(), int(value)))

    @property
    def launch_count(self):
        return int(self._lib.rv_launch_count(self._h))

    def sync(self):
        self._ck(self._lib.rv_sync(self._h))

    def pinned_empty(self, shape, dtype=np.uint8):
        """A numpy array in page-locked host memory (freed when the array is garbage-collected)."""
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        self._ck(self._lib.rv_alloc_pinned(self._h, nbytes, C.byref(p)))
        buf = (C.c_uint8 * max(nbytes, 1)).from_address(p.value)
        arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
        self._pinned[p.value] = nbytes
        owner = self                # keeps the context alive until its pinned buffers are gone

        def _free(addr=p.value):
            owner._pinned.pop(addr, None)
            owner._lib.rv_free_pinned(owner._h, C.c_void_p(addr))
        weakref.finalize(buf, _free)
        return arr

    def _pooled_pinned(self, shape, dtype=np.uint8, keep=4):
        """Like pinned_empty, but the page-locked block goes back to a small per-size pool when the array dies, so a
        per-frame loop (`proc = pipeline(raw)`, main_preview.py:94) gets DMA-able result arrays without paying
        cudaHostAlloc per call.  The array is the caller's: fresh, writable, never aliased while it is alive.

        Cheap by construction (about a microsecond): every block carries one persistent memoryview; a hand-out is an
        `_Lease` (an ndarray subclass over that memoryview whose destructor returns the block) viewed as a plain ndarray,
        so the block is recycled exactly when the last view of the array is gone."""
        dt = np.dtype(dtype)
        count = 1
        for v in shape:
            count *= int(v)
        nbytes = max(count * dt.itemsize, 1)
        free = self._pin_pool.get(nbytes)
        if free is None:
            free = self._pin_pool[nbytes] = []
        if free:
            blk = free.pop()
        else:
            p = C.c_void_p()
            self._ck(self._lib.rv_alloc_pinned(self._h, nbytes, C.byref(p)))
            self._pinned[p.value] = nbytes
            blk = (p.value, memoryview((C.c_uint8 * nbytes).from_address(p.value)).cast("B"))
        lease = np.ndarray.__new__(_Lease, shape, dt, blk[1])
        lease._home = (self, free, blk, keep)
        self._last_lease_addr = blk[0]
        return lease.view(np.ndarray)

    def _host_result(self, shape):
        """A new uint8 host array for a result: pooled page-locked memory (the D2H copy is a plain DMA) up to 64 MB, pageable above."""
        return self._pooled_pinned(shape) if int(np.prod(shape)) <= (64 << 20) else np.empty(shape, np.uint8)

    def _device_block(self, nbytes):
        """Device memory for a DeviceArray; blocks are recycled per size (cudaMalloc / cudaFree cost milliseconds and
        synchronise the device, which a per-batch allocation must not pay)."""
        free = self._dev_pool.setdefault(nbytes, [])
        if free:
            return free.pop()
        p = C.c_void_p()
        self._ck(self._lib.rv_alloc_device(self._h, nbytes, C.byref(p)))
        return p.value

    def _device_block_done(self, ptr, nbytes, keep=3):
        free = self._dev_pool.setdefault(nbytes, [])
        if len(free) < keep:
            free.append(ptr)
        else:
            self._lib.rv_free_device(self._h, C.c_void_p(ptr))

    def mem_kind(self, arr):
        a = arr.ctypes.data
        for base, n in self._pinned.items():
            if base <= a < base + max(n, 1):
                return MEM_PINNED
        return MEM_HOST

    # -- the chain -----------------------------------------------------------------------
    def chain(self, frames, params, out=None, processed=None):
        """rv_chain_u8 over host frames (N,H,W,3) uint8, rv_chain_u16 over uint16 ones, rv_chain_ex over (N,H,W,1) gray and
        (N,H,W,4) BGRA frames of either dtype; returns a new (or `out`) array, with 3 channels after CLAHE (cv2 drops alpha)."""
        _check_frames(frames, _U8_U16, CHANNELS)
        n, h, w, c = frames.shape
        bits = 8 * frames.dtype.itemsize
        if c == 3 and bits == 8:
            fn = self._lib.rv_chain_u8
        elif c == 3:
            check_u16_params(params)
            fn = self._lib.rv_chain_u16
        else:
            check_frame_params(params, frames.dtype, c)
            fn = None
        oc = 3 if params.clahe else c
        shape = (n, h, w, oc)
        if not frames.flags.c_contiguous:
            frames = np.ascontiguousarray(frames)
        out_addr = None
        if out is None:
            # small results (the per-frame contract) land in recycled page-locked memory: the D2H copy is a plain DMA
            if frames.nbytes <= (64 << 20):
                out = self._pooled_pinned(shape, frames.dtype)
                out_addr = self._last_lease_addr
            else:
                out = np.empty(shape, frames.dtype)
        elif out.shape != shape or out.dtype != frames.dtype or not out.flags.c_contiguous:
            raise ValueError(f"out must be a C-contiguous {frames.dtype} array of shape {shape}")
        if out_addr is None:
            out_addr = out.ctypes.data
        if n == 1:
            kind = MEM_HOST
        else:
            kind = MEM_PINNED if (self.mem_kind(frames) == MEM_PINNED and self.mem_kind(out) == MEM_PINNED) else MEM_HOST
        pp = processed.ctypes.data_as(_i32p) if processed is not None else None
        sb = frames.dtype.itemsize
        if fn is None:
            rc = self._lib.rv_chain_ex(self._h, frames.ctypes.data, out_addr, n, h, w, c * sb * w, oc * sb * w, bits, c, C.byref(params),
                                       kind, pp, None)
        else:
            rc = fn(self._h, frames.ctypes.data, out_addr, n, h, w, 3 * sb * w, 3 * sb * w, C.byref(params), kind, pp, None)
        if rc != 0:
            self._ck(rc)
        return out

    def chain_ex_device(self, in_ptr, out_ptr, n, h, w, params, bits, channels, stream=None):
        """rv_chain_ex over contiguous device frames (ints) of `channels` channels and `bits` bits: asynchronous on `stream` (a
        cudaStream_t int) when given, else synchronous on the context's stream."""
        oc = check_frame_params(params, np.uint8 if bits == 8 else np.uint16, channels)
        sb = bits // 8
        self._ck(self._lib.rv_chain_ex(self._h, C.c_void_p(in_ptr), C.c_void_p(out_ptr), n, h, w, channels * sb * w, oc * sb * w, bits,
                                       channels, C.byref(params), MEM_DEVICE, None, C.c_void_p(stream) if stream else None))

    def chain_u16_device(self, in_ptr, out_ptr, n, h, w, params, in_pitch=None, out_pitch=None, stream=None):
        """rv_chain_u16 over device pointers (ints, pitches in bytes): asynchronous on `stream` (a cudaStream_t int) when given,
        else synchronous on the context's stream."""
        check_u16_params(params)
        self._ck(self._lib.rv_chain_u16(self._h, C.c_void_p(in_ptr), C.c_void_p(out_ptr), n, h, w, in_pitch or 6 * w,
                                        out_pitch or 6 * w, C.byref(params), MEM_DEVICE, None, C.c_void_p(stream) if stream else None))

    def chain_device(self, in_ptr, out_ptr, n, h, w, params, in_pitch=None, out_pitch=None, stream=None):
        """rv_chain_u8 over device pointers (ints); synchronises the stream before returning."""
        self._ck(self._lib.rv_chain_u8(self._h, C.c_void_p(in_ptr), C.c_void_p(out_ptr), n, h, w,
                                       in_pitch or 3 * w, out_pitch or 3 * w, C.byref(params), MEM_DEVICE, None,
                                       C.c_void_p(stream) if stream else None))

    def submit_device(self, in_ptr, out_ptr, n, h, w, params, in_pitch=None, out_pitch=None, stream=None):
        """Enqueue the chain over device pointers without synchronising (on `stream`, a cudaStream_t int, if given)."""
        self._ck(self._lib.rv_submit(self._h, C.c_void_p(in_ptr), C.c_void_p(out_ptr), n, h, w,
                                     in_pitch or 3 * w, out_pitch or 3 * w, C.byref(params), MEM_DEVICE,
                                     C.c_void_p(stream) if stream else None))

    def yuv420_to_bgr(self, frames, yuv, out=None):
        """cv2.cvtColor(COLOR_YUV2BGR_NV12 / _I420) of every frame of a (B,3H/2,W) uint8 batch -> (B,H,W,3) BGR, on the GPU.
        `frames`: a numpy array (pageable or pinned; synchronous) or a contiguous torch CUDA tensor (asynchronous on torch's current
        stream; the result is a tensor).  `out` (optional): an array / tensor of the result's shape to write into."""
        if yuv in YUV422_LAYOUTS:
            raise ValueError(f"yuv420_to_bgr takes 'NV12' or 'I420' frames; {yuv!r} frames go to yuv422_to_bgr")
        return self._convert(frames, yuv, None, out)

    def yuv422_to_bgr(self, frames, yuv, out=None):
        """cv2.cvtColor(COLOR_YUV2BGR_YUY2 / _UYVY) of every frame of a (B,H,W,2) uint8 batch of packed 4:2:2 camera frames ->
        (B,H,W,3) BGR, on the GPU.  `frames`: a numpy array (pageable or pinned; synchronous) or a contiguous torch CUDA tensor
        (asynchronous on torch's current stream; the result is a tensor).  `out` (optional): an array / tensor of the result's shape to
        write into."""
        if yuv not in YUV422_LAYOUTS:
            raise ValueError(f"yuv422_to_bgr takes 'YUY2' or 'UYVY' frames, got {yuv!r}")
        return self._convert(frames, yuv, None, out)

    def bgr_to_yuv420(self, frames, yuv, out=None):
        """cv2.cvtColor(COLOR_BGR2YUV_I420) of every frame of a (B,H,W,3) uint8 batch -> (B,3H/2,W) 4:2:0 frames, on the GPU; with
        yuv="NV12" the U and V planes come interleaved (U first) in H/2 rows, the layout video encoders take.  `frames`: a numpy array
        (pageable or pinned; synchronous), a contiguous torch CUDA tensor (asynchronous on torch's current stream; the result is a
        tensor) or a DeviceArray (synchronous; the result is a DeviceArray).  `out` (optional): an array / tensor / DeviceArray of the
        result's shape to write into."""
        return self._convert(frames, None, yuv, out)

    def _convert(self, frames, in_layout, out_layout, out=None):
        """The conversion of every frame of a batch from `in_layout` ("NV12", "I420", "YUY2", "UYVY") to BGR, or from BGR to
        `out_layout` ("NV12", "I420"); the other layout is None.  `frames`: a numpy array (synchronous), a contiguous torch CUDA tensor
        (asynchronous on torch's current stream) or a DeviceArray (synchronous); the result is of the same kind, `out` if given."""
        torch_in = _is_torch(frames)
        if torch_in:
            import torch
            u8 = frames.dtype == torch.uint8
        elif isinstance(frames, (np.ndarray, DeviceArray)):
            u8 = frames.dtype == np.uint8
        else:
            raise ValueError("frames must be a numpy array or a torch CUDA tensor")
        if in_layout is not None:
            layout, b, h, w = check_yuv_frames(frames.shape, u8, in_layout)
            shape, pitches = (b, h, w, 3), (yuv_pitch(layout, w), 3 * w)
            fn = self._lib.rv_yuv422_to_bgr if in_layout in YUV422_LAYOUTS else self._lib.rv_yuv420_to_bgr
        else:
            layout, b, h, w = check_bgr_for_yuv(frames.shape, u8, out_layout)
            shape, pitches, fn = (b, h * 3 // 2, w), (3 * w, w), self._lib.rv_bgr_to_yuv420
        if torch_in:
            if not (frames.is_cuda and frames.is_contiguous()):
                raise ValueError("device frames must be a contiguous CUDA tensor")
            _check_torch_out(out, shape, torch.uint8, frames.device,
                             f"out must be a contiguous uint8 CUDA tensor of shape {shape} on the input's device")
            out = torch.empty(shape, dtype=torch.uint8, device=frames.device) if out is None else out
            self._ck(fn(self._h, C.c_void_p(frames.data_ptr()), C.c_void_p(out.data_ptr()), b, h, w, *pitches, layout, MEM_DEVICE,
                        _torch_stream(frames.device)))
            return out
        dev = isinstance(frames, DeviceArray)
        frames = frames if dev else np.ascontiguousarray(frames)
        if out is None:
            out = DeviceArray(self, shape) if dev else np.empty(shape, np.uint8)
        elif not (isinstance(out, DeviceArray if dev else np.ndarray) and out.shape == shape and out.dtype == np.uint8
                  and (dev or out.flags.c_contiguous)):
            raise ValueError(f"out must be a C-contiguous uint8 array of shape {shape}")
        (src, kind), (dst, out_kind) = self._end(frames), self._end(out)
        self._ck(fn(self._h, src, dst, b, h, w, *pitches, layout, kind if kind == out_kind else MEM_HOST, None))
        return out

    def kernel_times(self, reset=False):
        """{name: (total_ms, launches)} for the hot-path kernels (needs set_option('kernel_timing', 1))."""
        res = {}
        for which, name in enumerate(("k_luma_hist", "k_build_lut", "k_chain")):
            ms, cnt = C.c_double(), C.c_long()
            self._ck(self._lib.rv_kernel_time(self._h, which, C.byref(ms), C.byref(cnt)))
            res[name] = (ms.value, cnt.value)
        if reset:
            self._ck(self._lib.rv_kernel_time_reset(self._h))
        return res

    def submit(self, frames, out, params):
        """Asynchronous rv_submit over pinned host arrays; call wait() before reading `out`."""
        _check_frames(frames)
        n, h, w, _ = frames.shape
        if self.mem_kind(frames) != MEM_PINNED or self.mem_kind(out) != MEM_PINNED:
            raise ValueError("submit() needs arrays from Context.pinned_empty()")
        self._ck(self._lib.rv_submit(self._h, frames.ctypes.data, out.ctypes.data, n, h, w, 3 * w, 3 * w,
                                     C.byref(params), MEM_PINNED, None))

    def wait(self):
        self._ck(self._lib.rv_wait(self._h))

    def _end(self, x):
        """(pointer, rv_mem kind) of one end of a job: numpy array (pinned or pageable), DeviceArray, or a raw device pointer."""
        if x is None:
            return None, MEM_HOST
        if isinstance(x, np.ndarray):
            if not x.flags.c_contiguous:
                raise ValueError("arrays handed to submit_io must be C-contiguous")
            return x.ctypes.data, self.mem_kind(x)
        if isinstance(x, DeviceArray):
            return x.ptr, MEM_DEVICE
        if hasattr(x, "__cuda_array_interface__"):
            return int(x.__cuda_array_interface__["data"][0]), MEM_DEVICE
        return int(x), MEM_DEVICE

    def fill_tensor_padding(self, tensor, h, w, size=640, pad_value=114):
        """Write the letterbox padding (pad_value / 255 as a half) into the rows above and below the image of a host
        (B,3,size,size) float16 array for (h, w) frames.  A buffer prepared like this once (a ring of pinned tensors) can be
        handed to process_batch_to_tensor(..., padding_present=True): only the image rows then cross PCIe on the way back."""
        nw, nh, top, left, _ = self.letterbox_geometry(h, w, size)
        v = np.float16(np.float32(pad_value) / np.float32(255))
        tensor[:, :, :top, :] = v
        tensor[:, :, top + nh:, :] = v
        return tensor

    def submit_io(self, frames, params, shape=None, out=None, tensor=None, size=640, pad_value=114, processed=None, padding_present=False,
                  yuv=None, out_yuv=None):
        """rv_submit_io: asynchronous job whose ends live independently on the host or on the GPU; call wait() afterwards.

        frames: (N,H,W,3) uint8 numpy array (pinned or pageable) or a device object / pointer (then pass shape=(N,H,W)).
        out:    frames result, numpy or device (DeviceArray / anything with __cuda_array_interface__ / int pointer), or None.
        tensor: (N,3,size,size) float16 detector input, numpy or device, or None.
        yuv:    "NV12" / "I420": `frames` are (N,3H/2,W) 4:2:0 frames (rv_submit_io_yuv; `shape` is still (N,H,W)), converted to BGR on
                the GPU, so only their 1.5 bytes per pixel cross PCIe.  "YUY2" / "UYVY": `frames` are (N,H,W,2) packed 4:2:2 frames
                (rv_submit_io_fmt), so only their 2 bytes per pixel cross PCIe.
        out_yuv: "NV12" / "I420": `out` receives (N,3H/2,W) 4:2:0 frames (rv_submit_io_fmt), converted from the BGR result on the GPU,
                so only their 1.5 bytes per pixel cross PCIe on the way back."""
        layout = 0
        out_layout = check_out_yuv(out_yuv) if out_yuv is not None else 0
        if out_layout and yuv is None and isinstance(frames, np.ndarray):
            check_bgr_for_yuv(frames.shape, frames.dtype == np.uint8, out_yuv)
        if yuv is not None:
            if isinstance(frames, np.ndarray):
                layout, n, h, w = check_yuv_frames(frames.shape, frames.dtype == np.uint8, yuv)
            else:
                n, h, w = shape
                layout = check_yuv_frames((n, h, w, 2) if yuv in YUV422_LAYOUTS else (n, h * 3 // 2, w), True, yuv)[0]
        elif isinstance(frames, np.ndarray):
            _check_frames(frames)
            n, h, w, _ = frames.shape
        else:
            n, h, w = shape
        io = IO()
        io.in_, io.in_kind = self._end(frames)
        io.in_pitch = yuv_pitch(layout, w) if layout else 3 * w
        io.out, io.out_kind = self._end(out)
        io.out_pitch = w if out_layout else 3 * w
        io.tensor, io.tensor_kind = self._end(tensor)
        io.tensor_size, io.pad_value = int(size), int(pad_value)
        io.tensor_flags = 1 if padding_present else 0
        io.processed = processed.ctypes.data if processed is not None else None
        self._ck(self._lib.rv_submit_io_fmt(self._h, C.byref(io), layout, out_layout, n, h, w, C.byref(params)))

    # -- stage-level entry points (parity tests) ---------------------------------------------
    def luma_hist(self, frames, space, grid, want_luma=True, want_gray=False):
        _check_frames(frames)
        frames = np.ascontiguousarray(frames)
        n, h, w, _ = frames.shape
        hist = np.empty((n, grid * grid, 256), np.int32)
        luma = np.empty((n, h, w), np.uint8) if want_luma else None
        mm = np.empty((n, 2), np.int32) if want_gray else None
        self._ck(self._lib.rv_luma_hist(self._h, frames.ctypes.data, n, h, w, 3 * w,
                                        SPACE_LAB if space == "LAB" else SPACE_YCRCB, grid, hist.ctypes.data,
                                        luma.ctypes.data if want_luma else None, mm.ctypes.data if want_gray else None,
                                        MEM_HOST))
        return hist, luma, mm

    def build_lut(self, hist, h, w, grid, clip_limit):
        hist = np.ascontiguousarray(hist, np.int32)
        n = hist.shape[0]
        lut = np.empty((n, grid * grid, 256), np.uint8)
        self._ck(self._lib.rv_build_lut(self._h, hist.ctypes.data, n, h, w, grid, float(clip_limit), lut.ctypes.data, MEM_HOST))
        return lut

    def clahe_dehaze(self, frames, space, clip_limit, grid):
        return self.chain(frames, Params.make(space, clip_limit, grid, 0, clahe=True))

    def median(self, frames, ksize):
        return self.chain(frames, Params.make(ksize=ksize, clahe=False))

    # -- detector-input stage (letterbox + RGB + CHW + /255 + fp16) ---------------------------
    @staticmethod
    def letterbox_geometry(h, w, size=640):
        """(new_w, new_h, top, left, fused_scale) of the square letterbox; fused_scale > 0 = exact integer down-scale."""
        v = [C.c_int32() for _ in range(5)]
        rc = load_library().rv_letterbox_geometry(h, w, size, *[C.byref(x) for x in v])
        if rc != 0:
            raise ValueError("bad letterbox geometry arguments")
        return tuple(x.value for x in v)

    def letterbox_f16(self, frames, size=640, pad_value=114):
        """BGR frames (N,H,W,3) uint8 -> (N,3,size,size) float16 network input (no chain)."""
        _check_frames(frames)
        frames = np.ascontiguousarray(frames)
        n, h, w, _ = frames.shape
        out = np.empty((n, 3, size, size), np.float16)
        self._ck(self._lib.rv_letterbox_f16(self._h, frames.ctypes.data, n, h, w, 3 * w, out.ctypes.data, size, pad_value, MEM_HOST))
        return out

    def chain_letterbox(self, frames, params, size=640, pad_value=114, want_full=False, out=None, padding_present=False):
        """Chain + detector input in one call: returns (tensor (N,3,size,size) float16, full-res result or None)."""
        if padding_present:
            if out is None:
                raise ValueError("padding_present needs an `out` buffer prepared with fill_tensor_padding")
            _check_frames(frames)
            frames = np.ascontiguousarray(frames)
            full = None
            if want_full:
                full = self._host_result(frames.shape)
            self.submit_io(frames, params, out=full, tensor=out, size=size, pad_value=pad_value, padding_present=True)
            self.wait()
            return out, full
        _check_frames(frames)
        frames = np.ascontiguousarray(frames)
        n, h, w, _ = frames.shape
        if out is None:
            out = np.empty((n, 3, size, size), np.float16)
        full = None
        if want_full:
            full = self._host_result(frames.shape)
        kind = MEM_PINNED if (self.mem_kind(frames) == MEM_PINNED and self.mem_kind(out) == MEM_PINNED and
                              (full is None or self.mem_kind(full) == MEM_PINNED)) else MEM_HOST
        self._ck(self._lib.rv_chain_letterbox_f16(self._h, frames.ctypes.data, n, h, w, 3 * w, C.byref(params), out.ctypes.data,
                                                  size, pad_value, full.ctypes.data if want_full else None, 3 * w, kind, None))
        return out, full

    def chain_letterbox_device(self, in_ptr, out_ptr, n, h, w, params, size=640, pad_value=114, full_ptr=None, stream=None):
        """Device pointers; asynchronous on `stream` when given."""
        self._ck(self._lib.rv_chain_letterbox_f16(self._h, C.c_void_p(in_ptr), n, h, w, 3 * w, C.byref(params), C.c_void_p(out_ptr),
                                                  size, pad_value, C.c_void_p(full_ptr) if full_ptr else None, 3 * w, MEM_DEVICE,
                                                  C.c_void_p(stream) if stream else None))

    def gray_span(self, frames):
        """Gray span (max - min of cv2's BGR2GRAY) of every (N,H,W,3) BGR or (N,H,W,4) BGRA frame (alpha ignored)."""
        _check_frames(frames, _U8_U16, (3, 4))
        frames = np.ascontiguousarray(frames)
        n, h, w, c = frames.shape
        span = np.empty(n, np.int32)
        sb = frames.dtype.itemsize
        if c == 4:
            self._ck(self._lib.rv_gray_span_ex(self._h, frames.ctypes.data, n, h, w, 4 * sb * w, 8 * sb, 4, span.ctypes.data, MEM_HOST))
            return span
        fn = self._lib.rv_gray_span if sb == 1 else self._lib.rv_gray_span_u16
        self._ck(fn(self._h, frames.ctypes.data, n, h, w, 3 * sb * w, span.ctypes.data, MEM_HOST))
        return span


_default = {}
_default_lock = threading.Lock()


def default_context(device=None):
    """Process-wide context per device, created on first use (RV_DEVICE or LOCAL_RANK picks the default GPU)."""
    if device is None:
        device = int(os.environ.get("RV_DEVICE", os.environ.get("LOCAL_RANK", "0")))
    with _default_lock:
        if device not in _default:
            _default[device] = Context(device)
        return _default[device]
