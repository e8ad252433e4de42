"""Depth metrics -- host side of csrc/t3d_metrics.cu.

Mirrors /root/reference/utils/metrics.py (compute_depth_metrics,
evaluate_thermal_depth) and the 3-metric variant of
utils/evaluate_depth_metrics.py:20-80.  Tensors or ndarrays in; numpy scalars in
a dict out, exactly the reference's keys and dtypes (SURVEY.md Appendix C).
``compute_depth_metrics_batch`` is the batched, sync-free extension.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from . import _lib

KEYS7 = ("abs_rel", "sq_rel", "rmse", "rmse_log", "acc_1", "acc_2", "acc_3")


def _as_cuda(x, dtype=None):
    if isinstance(x, np.ndarray):
        x = torch.from_numpy(np.ascontiguousarray(x))
    if not isinstance(x, torch.Tensor):
        x = torch.as_tensor(x)
    if not x.is_cuda:
        if not torch.cuda.is_available():
            raise _lib.T3DError("no CUDA device: thermal3d_vision_b200 has no CPU path")
        x = x.cuda()
    if dtype is not None and x.dtype != dtype:
        x = x.to(dtype)
    return x.detach()


PHASE_ALL, PHASE_SAMPLE, PHASE_REST = 0, 1, 2      # T3D_PHASE_* (include/t3d.h)


@_lib.on_tensor_device
def compute_depth_metrics_batch(pred, gt_depth, mask=None, median_scaling=True, out: Optional[dict] = None,
                                phase: int = PHASE_ALL):
    """Batched metrics on the device, no host sync.

    phase (pipeline.HotPathStep): PHASE_SAMPLE launches only the bracket-sampling kernel for these inputs (its outputs go
    to out["state"], t3d_depth_metrics_state_bytes(B) bytes, or into the workspace) and returns None; PHASE_REST the
    remaining passes of the same inputs on the same workspace / state.

    pred: depth maps [B,H,W] or AoS pointmaps [B,H,W,3] (the Z channel is read in place --
    depth is never materialised); gt_depth [B,gh,gw] (nearest-resampled when the size differs);
    mask optional bool/uint8 [B,H,W].  Returns dict(metrics [B,8] float32: abs_rel, sq_rel, rmse,
    rmse_log, acc_1, acc_2, acc_3, n_valid; metrics_f64 [B,8]; medians [B,2])."""
    pred = _as_cuda(pred, torch.float32)
    gt = _as_cuda(gt_depth, torch.float32).contiguous()
    if pred.dim() == 4:
        if pred.shape[-1] != 3:
            raise ValueError("pointmaps must be [B,H,W,3]")
        pred = pred.contiguous()
        B, H, W, _ = pred.shape
        stride, offset = 3, 2
    elif pred.dim() == 3:
        B, H, W = pred.shape
        st = pred.stride()
        if st[2] == 3 and st[1] == 3 * W and (B == 1 or st[0] == 3 * W * H):
            stride, offset = 3, 0          # a pointmap[..., 2] view: read through its stride
        else:
            pred = pred.contiguous()
            stride, offset = 1, 0
    else:
        raise ValueError(f"pred must be [B,H,W] or [B,H,W,3], got {tuple(pred.shape)}")
    if gt.dim() != 3 or gt.shape[0] != B:
        raise ValueError(f"gt must be [B,h,w] with B={B}, got {tuple(gt.shape)}")
    m = None
    if mask is not None:
        m = _as_cuda(mask)
        if tuple(m.shape) != (B, H, W):
            raise ValueError("mask must be [B,H,W]")
        m = (m != 0).to(torch.uint8).contiguous()
    lib = _lib.lib()
    dev = pred.device
    out = out or {}
    ws_bytes = lib.t3d_depth_metrics_workspace_bytes(B, H, W)
    ws = out.get("workspace")
    if ws is None or ws.numel() < ws_bytes:
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    res = out.get("metrics")
    if res is None:
        res = torch.empty(B, 8, dtype=torch.float32, device=dev)
    res64 = out.get("metrics_f64")
    if res64 is None:
        res64 = torch.empty(B, 8, dtype=torch.float64, device=dev)
    med = out.get("medians")
    if med is None:
        med = torch.empty(B, 2, dtype=torch.float32, device=dev)
    state = out.get("state")
    rc = lib.t3d_depth_metrics(_lib.ptr(pred), stride, offset, _lib.ptr(gt), gt.shape[1], gt.shape[2], _lib.ptr(m),
                               B, H, W, 1 if median_scaling else 0, _lib.ptr(res), _lib.ptr(res64), _lib.ptr(med),
                               _lib.ptr(ws), ws.numel(), _lib.ptr(state), int(phase), _lib.current_stream_ptr())
    _lib.check(rc, "t3d_depth_metrics")
    if phase == PHASE_SAMPLE:
        return None
    return {"metrics": res, "metrics_f64": res64, "medians": med}


def _single(pred_depth, gt_depth, mask, median_scaling):
    pred = _as_cuda(pred_depth, torch.float32)
    gt = _as_cuda(gt_depth, torch.float32)
    if pred.dim() != 2 or gt.dim() != 2:
        raise ValueError(f"expected [H,W] depth maps, got {tuple(pred.shape)} and {tuple(gt.shape)}")
    if pred.shape != gt.shape:
        # numpy boolean indexing would raise IndexError in the reference
        raise IndexError(f"boolean index did not match: pred {tuple(pred.shape)} vs gt {tuple(gt.shape)}")
    m = None if mask is None else _as_cuda(mask).unsqueeze(0)
    r = compute_depth_metrics_batch(pred.unsqueeze(0), gt.unsqueeze(0), m, bool(median_scaling))
    return r["metrics_f64"][0].cpu().numpy()       # one 64-byte D2H


def compute_depth_metrics(pred_depth, gt_depth, mask=None, median_scaling=True):
    """Drop-in for utils/metrics.py:4-69: 4 np.float32 + 3 np.float64 values; empty mask ->
    NaNs and the keys a1/a2/a3 (the reference's key mismatch, SURVEY.md Appendix D.11)."""
    v = _single(pred_depth, gt_depth, mask, median_scaling)
    if v[7] == 0:
        return {"abs_rel": np.nan, "sq_rel": np.nan, "rmse": np.nan, "rmse_log": np.nan,
                "a1": 0.0, "a2": 0.0, "a3": 0.0}
    return {"abs_rel": np.float32(v[0]), "sq_rel": np.float32(v[1]), "rmse": np.float32(v[2]),
            "rmse_log": np.float32(v[3]), "acc_1": np.float64(v[4]), "acc_2": np.float64(v[5]),
            "acc_3": np.float64(v[6])}


def compute_depth_metrics_eval(pred_depth, gt_depth, mask=None, median_scaling=True):
    """Drop-in for utils/evaluate_depth_metrics.py:20-80 (rmse, acc_1.25, acc_1.25^2)."""
    v = _single(pred_depth, gt_depth, mask, median_scaling)
    if v[7] == 0:
        return {"rmse": np.nan, "acc_1.25": 0.0, "acc_1.25^2": 0.0}
    return {"rmse": np.float32(v[2]), "acc_1.25": np.float64(v[4]), "acc_1.25^2": np.float64(v[5])}


class MetricAccumulator:
    """Accumulator with the semantics of utils/metrics.py:86-136: per-image metrics are summed when
    finite and divided by the count of ALL images.  Lives on the device; `all_reduce` makes it the
    data-parallel accumulator (one packed NCCL all-reduce of 8 doubles)."""

    def __init__(self, device):
        self.state = torch.zeros(8, dtype=torch.float64, device=device)   # 7 sums + image count

    @_lib.on_tensor_device
    def update(self, metrics_f64: torch.Tensor):
        if metrics_f64.dtype != torch.float64 or not metrics_f64.is_contiguous() or metrics_f64.shape[1] != 8:
            raise ValueError("metrics_f64 must be a contiguous float64 [B, 8] tensor (compute_depth_metrics_batch)")
        rc = _lib.lib().t3d_metrics_accumulate(_lib.ptr(metrics_f64), int(metrics_f64.shape[0]), _lib.ptr(self.state),
                                               _lib.current_stream_ptr())
        _lib.check(rc, "t3d_metrics_accumulate")

    def all_reduce(self):
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dist.all_reduce(self.state, op=dist.ReduceOp.SUM)
        return self

    def result(self):
        s = self.state.cpu().numpy()
        n = s[7]
        return {k: (s[i] / n if n > 0 else np.nan) for i, k in enumerate(KEYS7)}


def evaluate_thermal_depth(model, dataloader, device):
    """Drop-in for utils/metrics.py:72-138.  The model forward is the caller's (out of scope); the loop, the
    output conventions it accepts (:105-117) and the accumulator semantics (:128-136: non-finite metrics are
    skipped, the sample still counts) are the reference's; z-extraction + metrics run on the GPU and the per-sample
    metrics stay on the device until the single read at the end (the reference syncs once per sample)."""
    model.eval()
    dev = torch.device(device)
    if dev.type != "cuda":
        dev = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else dev
    acc = None
    with torch.no_grad():
        for batch in dataloader:
            thermal1 = batch["thermal1"].to(device)
            if "depth1" in batch and batch["depth1"] is not None:
                gt_depth = batch["depth1"].to(device)
                for i in range(thermal1.size(0)):
                    view = {"img": thermal1[i:i + 1], "instance": []}        # monocular mode (:103-104)
                    output = model(view, view)
                    pred = output[0] if isinstance(output, tuple) else output.get("pred1", {})
                    pred_pointmap = pred.get("pts3d") if isinstance(pred, dict) else pred
                    if len(pred_pointmap.shape) == 4:                        # [B,H,W,3] -> first element (:116-117)
                        pred_pointmap = pred_pointmap[0]
                    if acc is None:
                        acc = MetricAccumulator(dev)
                    # pointmap -> depth happens inside the metric kernels (Z read in place, stride 3)
                    r = compute_depth_metrics_batch(pred_pointmap.unsqueeze(0), gt_depth[i:i + 1])
                    acc.update(r["metrics_f64"])
    if acc is None:                                                          # sample_count == 0 (:134-135)
        return {k: np.nan for k in KEYS7}
    return acc.result()
