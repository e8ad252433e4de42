"""ctypes binding of libt3d_sm100.so (C ABI declared in include/t3d.h).

The library is built in-tree (``thermal3d_vision_b200/libt3d_sm100.so``) by
``__graft_entry__.build()`` / ``csrc/Makefile``.  There is no CPU or PyTorch
fallback: if the library is missing or a call fails, this module raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libt3d_sm100.so")
CSRC_DIR = os.path.join(_HERE, "csrc")

ABI_VERSION = 3    # T3D_ABI_VERSION of include/t3d.h
_lock = threading.Lock()
_lib = None

c_f32p = C.c_void_p   # device pointers travel as plain integers
c_ptr = C.c_void_p

# name -> (restype, argtypes); must list every symbol include/t3d.h declares
_SIGNATURES = {
    "t3d_version": (C.c_int, []),
    "t3d_last_error": (C.c_char_p, []),
    "t3d_device_info": (C.c_int, [C.POINTER(C.c_int)] * 3),
    "t3d_launch_count": (C.c_uint64, []),
    "t3d_profile_begin": (C.c_int, [C.c_char_p, C.c_int]),
    "t3d_profile_end": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "t3d_profile_stride": (C.c_int, [C.c_int]),
    "t3d_profile_timeline": (C.c_int, [C.c_char_p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_int,
                                       C.POINTER(C.c_int)]),
    "t3d_loss_workspace_bytes": (C.c_size_t, [C.c_int] * 4),
    "t3d_loss_fwd_bwd": (C.c_int, [c_ptr] * 4 + [C.c_int] * 2 + [c_ptr] * 2 + [C.c_int] * 2 + [c_ptr] * 2 + [C.c_int]
                         + [c_ptr, c_ptr, C.c_int] + [c_ptr] * 4 + [C.c_int] * 4 + [C.c_float] * 5 + [c_ptr] * 4
                         + [c_ptr, C.c_size_t, c_ptr]),
    "t3d_loss_v1_workspace_bytes": (C.c_size_t, [C.c_int] * 3),
    "t3d_loss_v1_fwd_bwd": (C.c_int, [c_ptr] * 8 + [C.c_int] + [c_ptr] * 4 + [C.c_int] * 3 + [C.c_float] * 4
                            + [c_ptr] * 3 + [c_ptr, C.c_size_t, c_ptr]),
    "t3d_loss_rescale_invalid": (C.c_int, [c_ptr] * 6 + [C.c_int] * 3 + [c_ptr]),
    "t3d_scale_grads": (C.c_int, [c_ptr] * 5 + [C.c_int] * 3 + [c_ptr]),
    "t3d_resize_bilinear": (C.c_int, [c_ptr, c_ptr] + [C.c_int] * 6 + [c_ptr]),
    "t3d_resize_nearest_f32": (C.c_int, [c_ptr, c_ptr] + [C.c_int] * 5 + [c_ptr]),
    "t3d_interp_bilinear_f32": (C.c_int, [c_ptr, c_ptr] + [C.c_int] * 6 + [c_ptr]),
    "t3d_preprocess_workspace_bytes": (C.c_size_t, [C.c_int] * 3),
    "t3d_preprocess_train_u16": (C.c_int, [c_ptr] + [C.c_int] * 5 + [c_ptr, C.c_int, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int,
                                                                    c_ptr, C.c_size_t, C.c_int, c_ptr]),
    "t3d_preprocess_stats_tiles": (C.c_int, [C.c_int, C.c_int]),
    "t3d_preprocess_stats_scales": (C.c_int, [C.c_int, C.c_int]),
    "t3d_preprocess_fallback_count": (C.c_int, [c_ptr, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_uint), c_ptr]),
    "t3d_contrast_normalize_workspace_bytes": (C.c_size_t, [C.c_int]),
    "t3d_contrast_normalize_f32": (C.c_int, [c_ptr, C.c_int, C.c_int, C.c_int, c_ptr, C.c_int,
                                             c_ptr, c_ptr, c_ptr, C.c_size_t, c_ptr]),
    "t3d_channels_close": (C.c_int, [c_ptr, C.c_int, C.c_int, c_ptr, c_ptr]),
    "t3d_fixed_range_normalize": (C.c_int, [c_ptr, c_ptr, C.c_size_t, C.c_size_t, c_ptr, C.c_int, c_ptr]),
    "t3d_depth_metrics_workspace_bytes": (C.c_size_t, [C.c_int] * 3),
    "t3d_depth_metrics": (C.c_int, [c_ptr, C.c_int, C.c_int, c_ptr, C.c_int, C.c_int, c_ptr]
                          + [C.c_int] * 4 + [c_ptr] * 3 + [c_ptr, C.c_size_t, c_ptr, C.c_int, c_ptr]),
    "t3d_depth_metrics_state_bytes": (C.c_size_t, [C.c_int]),
    "t3d_metrics_accumulate": (C.c_int, [c_ptr, C.c_int, c_ptr, c_ptr]),
    "t3d_pointmap_to_depth": (C.c_int, [c_ptr, c_ptr, C.c_size_t, c_ptr]),
    "t3d_estimate_focal": (C.c_int, [c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr]),
    "t3d_sobel_workspace_bytes": (C.c_size_t, [C.c_int] * 4),
    "t3d_sobel_enhance_fwd": (C.c_int, [c_ptr, c_ptr] + [C.c_int] * 5 + [c_ptr, c_ptr, C.c_size_t, c_ptr]),
    "t3d_sobel_enhance_bwd_params": (C.c_int, [c_ptr, c_ptr, c_ptr] + [C.c_int] * 5 + [c_ptr, c_ptr, C.c_size_t, c_ptr]),
    "t3d_percentiles_f32": (C.c_int, [c_ptr, C.c_int, C.c_int, C.c_double, C.c_double, c_ptr, c_ptr, C.c_size_t, c_ptr]),
    "t3d_clahe_workspace_bytes": (C.c_size_t, [C.c_int] * 3),
    "t3d_clahe_u8": (C.c_int, [c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, c_ptr, C.c_size_t, c_ptr]),
    "t3d_canny_workspace_bytes": (C.c_size_t, [C.c_int] * 2),
    "t3d_canny_u8": (C.c_int, [c_ptr, c_ptr, C.c_int, C.c_int, C.c_double, C.c_double, c_ptr, C.c_size_t, c_ptr]),
    "t3d_sobel3_f32": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, c_ptr]),
    "t3d_histogram100": (C.c_int, [c_ptr, C.c_size_t, c_ptr, c_ptr]),
    "t3d_bilateral_f32": (C.c_int, [c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, c_ptr, c_ptr]),
    "t3d_depth_outlier_median": (C.c_int, [c_ptr, c_ptr, C.c_int, C.c_int, c_ptr, c_ptr, c_ptr]),
    "t3d_fire_gray": (C.c_int, [c_ptr, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr]),
    "t3d_fire_norm_u8": (C.c_int, [c_ptr, C.c_int, C.c_int, c_ptr, c_ptr, c_ptr, c_ptr]),
    "t3d_fire_compose": (C.c_int, [c_ptr, C.c_int, C.c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "t3d_fire_adv_u8": (C.c_int, [c_ptr, C.c_int, C.c_int, c_ptr, c_ptr, c_ptr]),
    "t3d_fire_adv_compose": (C.c_int, [c_ptr, C.c_int, C.c_int, C.c_double, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "t3d_hwc_to_chw_clip01": (C.c_int, [c_ptr, C.c_int, C.c_int, c_ptr, c_ptr]),
    "t3d_step_epilogue": (C.c_int, [c_ptr] * 7 + [C.c_int] * 5 + [c_ptr, C.c_int] + [c_ptr, c_ptr]),
    "t3d_rescale_global": (C.c_int, [c_ptr] * 6 + [C.c_int] * 3 + [c_ptr]),
    "t3d_mailbox_bytes": (C.c_size_t, []),
    "t3d_step_epilogue_peers": (C.c_int, [c_ptr] * 7 + [C.c_int] * 4 + [c_ptr, C.c_int] + [c_ptr, c_ptr, C.c_int, C.c_int, C.c_uint64, c_ptr]),
    "t3d_mailbox_reduce": (C.c_int, [c_ptr, C.c_int, C.c_uint64, c_ptr] + [c_ptr] * 5 + [C.c_int] * 3 + [c_ptr]),
    "t3d_project_points": (C.c_int, [c_ptr] + [C.c_float] * 4 + [c_ptr, C.c_size_t, c_ptr]),
}


class T3DError(RuntimeError):
    pass


def source_hash() -> str:
    """SHA-256 over every source the library is built from (kernels, headers, Makefile)."""
    import glob
    import hashlib
    h = hashlib.sha256()
    files = sorted(glob.glob(os.path.join(CSRC_DIR, "*.cu")) + glob.glob(os.path.join(CSRC_DIR, "*.cuh")) +
                   glob.glob(os.path.join(_HERE, "..", "include", "*.h")) + [os.path.join(CSRC_DIR, "Makefile")])
    for f in files:
        h.update(os.path.basename(f).encode())
        with open(f, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def build(verbose: bool = False, force: bool = False) -> str:
    """Compile libt3d_sm100.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    Incremental by default (make); `force=True` recompiles every object (`make -B`).  The hash of the sources the
    library was built from is kept next to it: a library whose recorded hash differs from the tree's sources (objects
    shipped from elsewhere, clock skew) is rebuilt from scratch as well."""
    stamp = LIB_PATH + ".srchash"
    want = source_hash()
    have = open(stamp).read().strip() if os.path.isfile(stamp) else ""
    if os.path.isfile(LIB_PATH) and have != want:
        force = True
    cmd = ["make", "-C", CSRC_DIR, "-j8"] + (["-B"] if force else [])
    out = subprocess.run(cmd, capture_output=True, text=True)
    if out.returncode == 0:
        with open(stamp, "w") as fh:
            fh.write(want + "\n")
    if verbose or out.returncode != 0:
        print(out.stdout[-4000:])
        print(out.stderr[-4000:])
    if out.returncode != 0:
        raise T3DError("building libt3d_sm100.so failed")
    return LIB_PATH


def declared_symbols():
    return sorted(_SIGNATURES)


def lib():
    """Load (once) and return the ctypes handle.  Raises if the .so is absent."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.isfile(LIB_PATH):
                raise T3DError(
                    f"{LIB_PATH} not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
                    "(there is no CPU fallback)")
            handle = C.CDLL(LIB_PATH)
            for name, (res, args) in _SIGNATURES.items():
                fn = getattr(handle, name)      # AttributeError if a symbol is missing
                fn.restype = res
                fn.argtypes = args
            if handle.t3d_version() != ABI_VERSION:
                raise T3DError("libt3d_sm100.so ABI version mismatch")
            _lib = handle
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().t3d_last_error().decode(errors="replace")
        raise T3DError(f"{what or 't3d call'} failed (status {rc}): {msg}")


def launch_count() -> int:
    return int(lib().t3d_launch_count())


def profile_begin(kernel_substr: str, max_launches: int = 4096, every_nth: int = 1) -> None:
    check(lib().t3d_profile_begin(kernel_substr.encode(), int(max_launches)), "t3d_profile_begin")
    if every_nth > 1:
        check(lib().t3d_profile_stride(int(every_nth)), "t3d_profile_stride")


def profile_end():
    """-> (total kernel ms, launches timed) for the kernel named in profile_begin."""
    ms, n = C.c_double(0.0), C.c_int(0)
    check(lib().t3d_profile_end(C.byref(ms), C.byref(n)), "t3d_profile_end")
    return ms.value, n.value


def profile_timeline(cap: int = 4096):
    """-> [(kernel name, start ms, stop ms)] of the launches timed since profile_begin (then call profile_end)."""
    stride = 64
    names = C.create_string_buffer(cap * stride)
    t0, t1, n = (C.c_double * cap)(), (C.c_double * cap)(), C.c_int(0)
    check(lib().t3d_profile_timeline(names, stride, t0, t1, cap, C.byref(n)), "t3d_profile_timeline")
    raw = names.raw
    return [(raw[i * stride:(i + 1) * stride].split(b"\0", 1)[0].decode(), t0[i], t1[i]) for i in range(n.value)]


def ptr(t):
    """Device pointer of a tensor (or None -> NULL)."""
    return None if t is None else t.data_ptr()


def current_stream_ptr(device=None):
    """cudaStream_t of torch's current stream on `device` (default: the current device; inside `on_tensor_device`
    / `device_guard` that is the device the tensors live on)."""
    import torch
    return torch.cuda.current_stream(device).cuda_stream


def _first_cuda_device(objs):
    import torch
    for o in objs:
        if isinstance(o, torch.Tensor):
            if o.is_cuda:
                return o.device
        elif isinstance(o, dict):
            d = _first_cuda_device(o.values())
            if d is not None:
                return d
        elif isinstance(o, (list, tuple)):
            d = _first_cuda_device(o)
            if d is not None:
                return d
    return None


def device_guard(device):
    """Context manager making `device` the current CUDA device: the library launches on the CURRENT device (it never
    calls cudaSetDevice) and takes the stream from torch's current stream, so every entry point runs under the guard
    of the device its tensors live on -- tensors on cuda:1 while cuda:0 is current would otherwise get kernels
    launched on device 0 with device-1 pointers."""
    import contextlib
    import torch
    if device is None:
        return contextlib.nullcontext()
    device = torch.device(device)
    if device.type != "cuda" or device.index is None or device.index == torch.cuda.current_device():
        return contextlib.nullcontext()
    return torch.cuda.device(device)


def on_tensor_device(fn):
    """Decorator: run `fn` with the device of its first CUDA tensor argument as the current device."""
    import functools

    @functools.wraps(fn)
    def wrapped(*args, **kwargs):
        dev = _first_cuda_device(args) or _first_cuda_device(kwargs.values())
        if dev is None:
            return fn(*args, **kwargs)
        with device_guard(dev):
            return fn(*args, **kwargs)
    return wrapped


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise T3DError("expected CUDA tensors (the library has no CPU path)")
