"""Raw-frame ingest (SURVEY.md section 8f row 3): the on-disk formats either side of the hot path.

Host side of ``libt3d_ingest.so`` (C ABI: include/t3d_ingest.h, C++ + zlib, no CUDA).  Mirrors what
data/dataset_loader.py does per sample in its DataLoader workers -- ``cv2.imread(path, cv2.IMREAD_ANYDEPTH)``
of the 16-bit thermal PNGs (:237-239) and ``np.load(path)`` + ``.float()`` of the pseudo-GT arrays
(:159-201) -- but per BATCH: a small native thread pool decodes straight into one pinned host buffer, which
goes to the device in a single asynchronous copy and from there into ``preprocess_thermal_batch`` (the
resize and the percentile normalisation the workers did on the CPU now run on the GPU).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import threading
from typing import Optional, Sequence

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libt3d_ingest.so")
CSRC_DIR = os.path.join(_HERE, "csrc_host")

_lock = threading.Lock()
_lib = None

_SIGNATURES = {
    "t3d_ingest_version": (C.c_int, []),
    "t3d_ingest_last_error": (C.c_char_p, []),
    "t3d_png_info": (C.c_int, [C.c_void_p, C.c_size_t] + [C.POINTER(C.c_int)] * 5),
    "t3d_png_decode_gray16": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_int]),
    "t3d_png_decode_files_gray16": (C.c_int, [C.POINTER(C.c_char_p), C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                              C.POINTER(C.c_int)]),
    "t3d_npy_header": (C.c_int, [C.c_void_p, C.c_size_t, C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                 C.POINTER(C.c_int64), C.POINTER(C.c_size_t)]),
    "t3d_npy_read_files_f32": (C.c_int, [C.POINTER(C.c_char_p), C.c_int, C.c_void_p, C.c_size_t, C.c_int,
                                         C.POINTER(C.c_int)]),
}


class IngestError(RuntimeError):
    pass


def build(verbose: bool = False) -> str:
    out = subprocess.run(["make", "-C", CSRC_DIR], capture_output=True, text=True)
    if verbose or out.returncode != 0:
        print(out.stdout[-2000:], out.stderr[-2000:])
    if out.returncode != 0:
        raise IngestError("building libt3d_ingest.so failed")
    return LIB_PATH


def declared_symbols():
    return sorted(_SIGNATURES)


def lib():
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.isfile(LIB_PATH):
                raise IngestError(f"{LIB_PATH} not found: run `python -c 'import __graft_entry__ as g; g.build()'`")
            h = C.CDLL(LIB_PATH)
            for name, (res, args) in _SIGNATURES.items():
                fn = getattr(h, name)
                fn.restype, fn.argtypes = res, args
            if h.t3d_ingest_version() != 1:
                raise IngestError("libt3d_ingest.so ABI version mismatch")
            _lib = h
    return _lib


def _check(rc: int, what: str):
    if rc != 0:
        raise IngestError(f"{what} failed (status {rc}): {lib().t3d_ingest_last_error().decode(errors='replace')}")


def _paths(paths: Sequence[str]):
    arr = (C.c_char_p * len(paths))(*[os.fsencode(p) for p in paths])
    return arr


def _host_buffer(shape, dtype, pin: bool) -> torch.Tensor:
    t = torch.empty(shape, dtype=dtype)
    if pin and torch.cuda.is_available():
        t = t.pin_memory()
    return t


def png_info(path: str):
    """(width, height, bit_depth, color_type, interlace) of a PNG file."""
    with open(path, "rb") as f:
        head = f.read(64)
    v = [C.c_int(0) for _ in range(5)]
    buf = C.create_string_buffer(head, len(head))
    _check(lib().t3d_png_info(C.cast(buf, C.c_void_p), len(head), *[C.byref(x) for x in v]), "t3d_png_info")
    return tuple(x.value for x in v)


def read_thermal_png_batch(paths: Sequence[str], threads: int = 8, pin: bool = True,
                           out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Decode 16-bit (or 8-bit) grayscale PNG frames of identical size into one host tensor [B,H,W] uint16
    -- ``cv2.imread(p, cv2.IMREAD_ANYDEPTH)`` for every path (data/dataset_loader.py:237-239), raw counts kept."""
    if len(paths) == 0:
        raise ValueError("no paths")
    w, h, depth, color, interlace = png_info(paths[0])
    if out is None:
        out = _host_buffer((len(paths), h, w), torch.uint16, pin)
    if out.dtype != torch.uint16 or tuple(out.shape) != (len(paths), h, w) or not out.is_contiguous() or out.is_cuda:
        raise ValueError(f"out must be a contiguous host uint16 tensor of shape {(len(paths), h, w)}")
    status = (C.c_int * len(paths))()
    rc = lib().t3d_png_decode_files_gray16(_paths(paths), len(paths), out.data_ptr(), w, h, int(threads), status)
    _check(rc, "t3d_png_decode_files_gray16")
    return out


def read_npy_batch_f32(paths: Sequence[str], shape: Sequence[int], threads: int = 8, pin: bool = True,
                       out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``torch.from_numpy(np.load(p)).float()`` for every path (data/dataset_loader.py:159-201), each array of
    `shape` (float32 / float64 / float16 on disk), into one host tensor [B, *shape] float32."""
    if len(paths) == 0:
        raise ValueError("no paths")
    shape = tuple(int(s) for s in shape)
    elems = 1
    for s in shape:
        elems *= s
    if out is None:
        out = _host_buffer((len(paths),) + shape, torch.float32, pin)
    if out.dtype != torch.float32 or tuple(out.shape) != (len(paths),) + shape or not out.is_contiguous() or out.is_cuda:
        raise ValueError(f"out must be a contiguous host float32 tensor of shape {(len(paths),) + shape}")
    status = (C.c_int * len(paths))()
    rc = lib().t3d_npy_read_files_f32(_paths(paths), len(paths), out.data_ptr(), elems, int(threads), status)
    _check(rc, "t3d_npy_read_files_f32")
    return out


def npy_header(path: str):
    """(descr, fortran_order, shape, data_offset) of a .npy file (for np.memmap-style access)."""
    with open(path, "rb") as f:
        head = f.read(4096)
    descr = C.create_string_buffer(16)
    fortran, ndim, off = C.c_int(0), C.c_int(0), C.c_size_t(0)
    shape = (C.c_int64 * 8)()
    buf = C.create_string_buffer(head, len(head))
    _check(lib().t3d_npy_header(C.cast(buf, C.c_void_p), len(head), descr, C.byref(fortran), C.byref(ndim), shape,
                                C.byref(off)), "t3d_npy_header")
    return descr.value.decode(), bool(fortran.value), tuple(int(shape[i]) for i in range(ndim.value)), int(off.value)


def load_thermal_batch(paths: Sequence[str], img_size=(224, 224), device=None, threads: int = 8, **kw):
    """paths -> ThermalBatch on the GPU: native PNG decode into pinned memory, one H2D copy, then
    ``preprocess_thermal_batch`` (= FreiburgDataset._load_thermal_image + enhance_thermal_contrast per frame; with
    ``normalization="fixed_range"`` + enhance_thermal_fixed_range, the loader's alternative at
    data/dataset_loader.py:111,119).  Keyword arguments go to ``preprocess_thermal_batch``."""
    from . import preprocessing as _pre
    raw = read_thermal_png_batch(paths, threads=threads, pin=True)
    dev = torch.device(device if device is not None else "cuda")
    return _pre.preprocess_thermal_batch(raw.to(dev, non_blocking=True), img_size, path="train", **kw)
