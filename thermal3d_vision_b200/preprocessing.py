"""Thermal preprocessing -- host side of the sm_100a kernels in csrc/t3d_preprocess.cu.

Mirrors /root/reference/utils/preprocessing.py (same names, arguments, return
conventions; SURVEY.md section 8b) plus the image loaders around it
(data/dataset_loader.py:237-249, thermal_dustr_inference.py:25-60).  Device rule:
CUDA tensor in -> CUDA tensor out; CPU tensor in -> uploaded, processed on the
GPU, returned on the CPU (the reference always returns CPU tensors).  There is
no CPU implementation.
"""
from __future__ import annotations

import os
from typing import NamedTuple, Optional

import ctypes as C

import numpy as np
import torch

from . import _lib


def _cuda_device():
    if not torch.cuda.is_available():
        raise _lib.T3DError("no CUDA device: thermal3d_vision_b200 has no CPU path")
    return torch.device("cuda", torch.cuda.current_device())


def _to_cuda(t: torch.Tensor):
    return t if t.is_cuda else t.to(_cuda_device())


# ----------------------------------------------------------------------------- resize
@_lib.on_tensor_device
def resize_bilinear(src: torch.Tensor, size_hw, mode: Optional[str] = None) -> torch.Tensor:
    """cv2.resize(src, (w, h)) INTER_LINEAR (IPP-off recipe), bit-exact.

    src [B,H,W] or [H,W]; uint16 -> uint16 (mode 'u16'), uint16 -> float32 after /65535
    (mode 'u16_to_unit_f32'), float32 -> float32 (mode 'f32')."""
    squeeze = src.dim() == 2
    x = _to_cuda(src.unsqueeze(0) if squeeze else src).contiguous()
    if mode is None:
        mode = "u16" if x.dtype == torch.uint16 else "f32"
    code = {"u16": 0, "u16_to_unit_f32": 1, "f32": 2}[mode]
    if code in (0, 1) and x.dtype != torch.uint16:
        raise ValueError("uint16 input expected")
    if code == 2 and x.dtype != torch.float32:
        x = x.float()
    B, sh, sw = x.shape
    dh, dw = int(size_hw[0]), int(size_hw[1])
    out = torch.empty(B, dh, dw, dtype=torch.uint16 if code == 0 else torch.float32, device=x.device)
    rc = _lib.lib().t3d_resize_bilinear(_lib.ptr(x), _lib.ptr(out), code, B, sh, sw, dh, dw,
                                        _lib.current_stream_ptr())
    _lib.check(rc, "t3d_resize_bilinear")
    out = out[0] if squeeze else out
    return out if src.is_cuda else out.cpu()


@_lib.on_tensor_device
def resize_nearest(src: torch.Tensor, size_hw) -> torch.Tensor:
    """cv2.resize(..., INTER_NEAREST) of float32 maps (utils/evaluate_depth_metrics.py:320-323)."""
    squeeze = src.dim() == 2
    x = _to_cuda(src.unsqueeze(0) if squeeze else src).float().contiguous()
    B, sh, sw = x.shape
    dh, dw = int(size_hw[0]), int(size_hw[1])
    out = torch.empty(B, dh, dw, dtype=torch.float32, device=x.device)
    rc = _lib.lib().t3d_resize_nearest_f32(_lib.ptr(x), _lib.ptr(out), B, sh, sw, dh, dw, _lib.current_stream_ptr())
    _lib.check(rc, "t3d_resize_nearest_f32")
    out = out[0] if squeeze else out
    return out if src.is_cuda else out.cpu()


# ----------------------------------------------------------------------------- batched train / inference paths
class ThermalBatch(NamedTuple):
    thermal: torch.Tensor                      # [B, C, h, w] float32 in [0, 1]
    percentiles: torch.Tensor                  # [B, 2] float64 (p2, p98)
    histogram: Optional[torch.Tensor] = None   # [B, 65536] int32 view of the uint32 counts (train path)
    grad_stats: Optional[torch.Tensor] = None  # [B, tiles, 4] partial sums of |Dx gray|, |Dy gray| (train path)
    stats_scales: int = 1                      # 2: grad_stats[..., 2:4] hold the half-resolution sums (multi-scale loss)


@_lib.on_tensor_device
def preprocess_thermal_batch(raw_u16: torch.Tensor, img_size=(224, 224), path: str = "train",
                             out_channels: int = 3, out: Optional[dict] = None,
                             histogram: bool = True, half_res_stats: bool = False, phase: int = 0,
                             shared: bool = False, grad_stats: bool = True) -> ThermalBatch:
    """16-bit radiometric frames [B,Hs,Ws] -> normalised thermal [B,3,h,w].

    img_size is (W, H) in cv2 order like the reference's --img_size.  path='train':
    data/dataset_loader.py:237-249 + enhance_thermal_contrast (u16 resize, raw counts);
    path='inference': thermal_dustr_inference.py:25-60 (/65535, float resize).
    histogram=True also returns the exact 65 536-bin histogram of every resized frame (the percentiles are
    read off it); histogram=False computes the same percentiles, bit for bit, from sampled value windows
    without a per-pixel histogram atomic (about twice as fast; the reference itself never builds a histogram).
    half_res_stats=True (train path): grad_stats also carries the thermal-gradient sums of the 2x2 average-pooled image
    the multi-scale loss needs (utils/loss.py:133-174), where the shape allows (ThermalBatch.stats_scales == 2).
    phase (train path, histogram=False; pipeline.HotPathStep): 1 = launch only the window-sampling kernel for these frames
    (outputs stay in out["workspace"]), 2 = everything after it, on the same `out`; 0 = the whole call.
    shared=True (train path) is a scheduling hint: other kernels run concurrently on another stream (the metric chain
    of pipeline.HotPathStep / EvalStep), so the resize kernel leaves them room on every SM.  Same results.
    grad_stats=False (train path): no thermal-gradient sums (ThermalBatch.grad_stats is None), for a loss that does not
    use the thermal images; the thermal planes are the same."""
    x = _to_cuda(raw_u16).contiguous()
    if x.dtype != torch.uint16:
        raise ValueError(f"raw frames must be uint16, got {x.dtype}")
    if x.dim() == 2:
        x = x.unsqueeze(0)
    B, sh, sw = x.shape
    dw, dh = int(img_size[0]), int(img_size[1])
    lib = _lib.lib()
    dev = x.device
    out = out or {}
    stream = _lib.current_stream_ptr()
    thermal = out.get("thermal")
    if thermal is None:
        thermal = torch.empty(B, out_channels, dh, dw, dtype=torch.float32, device=dev)
    pct = out.get("percentiles")
    if pct is None:
        pct = torch.empty(B, 2, dtype=torch.float64, device=dev)
    if path == "train":
        hist = None
        if histogram:
            hist = out.get("histogram")
            if hist is None:
                hist = torch.empty(B, 65536, dtype=torch.int32, device=dev)
        ws_bytes = lib.t3d_preprocess_workspace_bytes(B, dh, dw)
        ws = out.get("workspace")
        if ws is None or ws.numel() < ws_bytes:
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        tiles = lib.t3d_preprocess_stats_tiles(dh, dw) if grad_stats else 0
        stats = None
        if tiles > 0:
            stats = out.get("grad_stats")
            if stats is None:
                stats = torch.empty(B, tiles, 4, dtype=torch.float32, device=dev)
        scales = 1
        if half_res_stats and stats is not None and lib.t3d_preprocess_stats_scales(dh, dw) == 2:
            scales = 2
        rc = lib.t3d_preprocess_train_u16(_lib.ptr(x), B, sh, sw, dh, dw, _lib.ptr(thermal), out_channels,
                                          _lib.ptr(hist), _lib.ptr(pct), _lib.ptr(stats), scales, int(bool(shared)),
                                          _lib.ptr(ws), ws.numel(), int(phase), stream)
        _lib.check(rc, "t3d_preprocess_train_u16")
        return ThermalBatch(thermal, pct, hist, stats, scales)
    if path == "inference":
        resized = torch.empty(B, dh, dw, dtype=torch.float32, device=dev)
        rc = lib.t3d_resize_bilinear(_lib.ptr(x), _lib.ptr(resized), 1, B, sh, sw, dh, dw, stream)
        _lib.check(rc, "t3d_resize_bilinear")
        flags = torch.empty(B, dtype=torch.int32, device=dev)
        fws = torch.empty(lib.t3d_contrast_normalize_workspace_bytes(B), dtype=torch.uint8, device=dev)
        rc = lib.t3d_contrast_normalize_f32(_lib.ptr(resized), B, 1, dh * dw, _lib.ptr(thermal), out_channels,
                                            _lib.ptr(pct), _lib.ptr(flags), _lib.ptr(fws), fws.numel(), stream)
        _lib.check(rc, "t3d_contrast_normalize_f32")
        return ThermalBatch(thermal, pct, None)
    raise ValueError("path must be 'train' or 'inference'")


@_lib.on_tensor_device
def bracket_fallback_count(workspace: torch.Tensor, B: int, img_size) -> int:
    """Diagnostics: frames of the last preprocess_thermal_batch(..., histogram=False, out={'workspace': ws}) call
    whose percentiles needed the exact per-frame select (same result, slower).  Synchronises."""
    n = C.c_uint(0)
    rc = _lib.lib().t3d_preprocess_fallback_count(_lib.ptr(workspace), int(B), int(img_size[1]), int(img_size[0]),
                                                  C.byref(n), _lib.current_stream_ptr())
    _lib.check(rc, "t3d_preprocess_fallback_count")
    return int(n.value)


# ----------------------------------------------------------------------------- reference signatures
@_lib.on_tensor_device
def enhance_thermal_contrast(thermal_tensor):
    """Drop-in for utils/preprocessing.py:6-30 (percentile clip-normalise, 3-channel output)."""
    if thermal_tensor is None:
        print("Warning: Received None instead of a thermal image tensor")
        return None
    src_cuda = thermal_tensor.is_cuda
    x = _to_cuda(thermal_tensor)
    if x.dtype != torch.float32:
        x = x.float()       # the reference would compute in that dtype; thermal tensors are float32
    x = x.contiguous()
    if x.dim() == 0:
        raise ValueError("thermal tensor must have at least one dimension")
    shape = tuple(x.shape)
    three = shape[0] == 3
    if three:
        channels, n = 3, int(np.prod(shape[1:])) if len(shape) > 1 else 1
        plane_shape = shape[1:]
    else:
        channels, n = 1, int(np.prod(shape))
        plane_shape = shape
    rep = 3 if len(plane_shape) == 2 else 1                 # :27-28 only 2-D results are replicated
    out = torch.empty((rep,) + tuple(plane_shape) if rep == 3 else tuple(plane_shape),
                      dtype=torch.float32, device=x.device)
    pct = torch.empty(1, 2, dtype=torch.float64, device=x.device)
    flags = torch.empty(1, dtype=torch.int32, device=x.device)
    fws = torch.empty(_lib.lib().t3d_contrast_normalize_workspace_bytes(1), dtype=torch.uint8, device=x.device)
    rc = _lib.lib().t3d_contrast_normalize_f32(_lib.ptr(x), 1, channels, n, _lib.ptr(out), rep,
                                               _lib.ptr(pct), _lib.ptr(flags), _lib.ptr(fws), fws.numel(),
                                               _lib.current_stream_ptr())
    _lib.check(rc, "t3d_contrast_normalize_f32")
    return out if src_cuda else out.cpu()


@_lib.on_tensor_device
def enhance_thermal_fixed_range(thermal_tensor, normalized=True):
    """Drop-in for utils/preprocessing.py:32-73 (Freiburg fixed window 21800..25000).

    Output has the input's shape.  For a 3-channel input whose channels are np.allclose the
    reference normalises channel 0 and replicates it (:39-41,67-71); that decision is taken on
    the device (no host sync)."""
    if thermal_tensor is None:
        return None
    src_cuda = thermal_tensor.is_cuda
    x = _to_cuda(thermal_tensor)
    if x.dtype != torch.float32:
        x = x.float()
    x = x.contiguous()
    lib = _lib.lib()
    stream = _lib.current_stream_ptr()
    flag = None
    plane = max(x.numel(), 1)
    if x.dim() == 3 and x.shape[0] == 3:
        plane = x.shape[1] * x.shape[2]
        flag = torch.empty(1, dtype=torch.int32, device=x.device)
        _lib.check(lib.t3d_channels_close(_lib.ptr(x), 1, plane, _lib.ptr(flag), stream), "t3d_channels_close")
    y = torch.empty_like(x)
    rc = lib.t3d_fixed_range_normalize(_lib.ptr(x), _lib.ptr(y), x.numel(), plane, _lib.ptr(flag),
                                       1 if normalized else 0, stream)
    _lib.check(rc, "t3d_fixed_range_normalize")
    return y if src_cuda else y.cpu()


def load_thermal_image_train(path: str, img_size=(224, 224)):
    """Drop-in for FreiburgDataset._load_thermal_image (data/dataset_loader.py:237-249):
    raw uint16 -> cv2.resize (uint16) -> float32 raw counts, 3 channels, CHW.  Decode on the host
    (file I/O is out of scope), everything else on the GPU.  Returns a CPU tensor like the reference."""
    import cv2
    img = cv2.imread(path, cv2.IMREAD_ANYDEPTH)
    if img is None:
        return None
    if img.dtype == np.uint16 and img.ndim == 2:
        r = resize_bilinear(torch.from_numpy(img), (img_size[1], img_size[0]), mode="u16")
        t = r.to(torch.float32)
    else:
        t = resize_bilinear(torch.from_numpy(img.astype(np.float32)), (img_size[1], img_size[0]), mode="f32")
    return t.unsqueeze(0).repeat(3, 1, 1)


def load_and_preprocess_thermal_image(path, img_size=(224, 224)):
    """Drop-in for thermal_dustr_inference.py:25-60 == utils/evaluate_depth_metrics.py:162-197."""
    import cv2
    if not os.path.exists(path):
        print(f"Error: Image file {path} does not exist")
        return None
    img = cv2.imread(path, cv2.IMREAD_ANYDEPTH)
    if img is None:
        img = cv2.imread(path)
        if img is None:
            print(f"Error: Could not read image {path}")
            return None
        img = cv2.cvtColor(img, cv2.COLOR_BGR2RGB)
    dw, dh = int(img_size[0]), int(img_size[1])
    if img.dtype == np.uint16 and img.ndim == 2:
        tb = preprocess_thermal_batch(torch.from_numpy(img), (dw, dh), path="inference")
        return tb.thermal[0].cpu()
    x = torch.from_numpy(img.astype(np.float32) / (65535.0 if img.dtype == np.uint16 else 255.0))
    if x.dim() == 2:
        x = x.unsqueeze(-1).repeat(1, 1, 3)
    planes = resize_bilinear(x.permute(2, 0, 1).contiguous(), (dh, dw), mode="f32")   # per-channel == 3-ch resize
    return enhance_thermal_contrast(planes)
