"""Thermal-aware training loss -- host side of the fused sm_100a kernels.

Mirrors /root/reference/utils/loss.py: same function names, positional order,
keyword names, defaults and return types (SURVEY.md section 8b), so
``train_thermal_dustr.py`` can import this module as ``utils.loss``.  All
arithmetic happens in libt3d_sm100.so (``t3d_loss_fwd_bwd``): one fused pass
produces the loss partial sums AND d/dpred, d/dconf; autograd only hands the
precomputed gradients back (scaled on the device by ``grad_output``).

Extension over the reference: the batched entry points
``fused_thermal_loss`` / ``fused_thermal_loss_fwd_bwd`` take ``[B,H,W,3]``
tensors and reproduce the training loop's "mean over valid samples"
(train_thermal_dustr.py:182-360) without any host synchronisation.
"""
from __future__ import annotations

import os
from typing import NamedTuple, Optional

import torch

from . import _lib

OUT_STRIDE = 8  # T3D_LOSS_OUT_STRIDE
THERMAL_REPLICATED = 0x100  # T3D_THERMAL_REPLICATED
LOSS_MULTI_SCALE, LOSS_CONF_MIN_ONLY, LOSS_STATS_TWO_SCALES = 0x1, 0x2, 0x4   # T3D_LOSS_* flags
# Debug / test mode (T3D_DEBUG_CHECKS=1, set by tests/conftest.py): caller promises are verified on the device --
# today `thermal_replicated` (a wrong flag would silently change the results).  Costs a pass + a host sync per call.
DEBUG_CHECKS = os.environ.get("T3D_DEBUG_CHECKS", "0") not in ("", "0")


class FusedLossResult(NamedTuple):
    loss: torch.Tensor          # 0-d: mean over valid samples (or the sample's loss when B == 1)
    per_sample: torch.Tensor    # [B, 8] total, basic, edge, smooth, detail, valid, -, -
    batch: torch.Tensor         # [8]   mean total, mean components, n_valid, B, -


def _prep(t: Optional[torch.Tensor], device) -> Optional[torch.Tensor]:
    if t is None:
        return None
    if t.dtype != torch.float32:
        t = t.float()
    if t.device != device:
        t = t.to(device)
    return t.contiguous()


@_lib.on_tensor_device
def _launch(bwd, p1, p2, g1, g2, c1, c2, t1, t2, need_dconf, alpha, ew, sw, dw, multi, grad_scale,
            rescale_invalid, out=None, thermal_stats=None, thermal_replicated=False, conf_min_only=False,
            thermal_stats_scales=1):
    """Raw call into the C ABI on already-prepared [B,H,W,3] CUDA tensors."""
    lib = _lib.lib()
    B, H, W, _ = p1.shape
    dev = p1.device
    tch = 0 if t1 is None or t2 is None else int(t1.shape[1])
    if thermal_replicated and tch == 3:
        tch |= THERMAL_REPLICATED          # include/t3d.h: the kernel reads plane 0 only
    flags = (LOSS_MULTI_SCALE if multi else 0) | (LOSS_CONF_MIN_ONLY if conf_min_only else 0)
    ws_bytes = lib.t3d_loss_workspace_bytes(B, H, W, flags)
    if out is None:
        out = {}
    ws = out.get("workspace")
    if ws is None or ws.numel() < ws_bytes:
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    per_sample = out.get("per_sample")
    if per_sample is None:
        per_sample = torch.empty(B, OUT_STRIDE, dtype=torch.float32, device=dev)
    batch = out.get("batch")
    if batch is None:
        batch = torch.empty(OUT_STRIDE, dtype=torch.float32, device=dev)
    f64 = out.get("per_sample_f64")
    stream = _lib.current_stream_ptr()
    st1 = st2 = None
    st_tiles = 0
    if thermal_stats is not None and tch and (not multi or thermal_stats_scales == 2):
        st1, st2 = thermal_stats
        if st1 is not None and st2 is not None:
            if st1.shape != st2.shape or st1.dim() != 3 or st1.shape[0] != B or st1.shape[2] != 4 \
                    or st1.dtype != torch.float32 or not st1.is_contiguous() or not st2.is_contiguous():
                raise ValueError("thermal_stats must be two contiguous float32 [B, tiles, 4] tensors")
            st_tiles = int(st1.shape[1])
        else:
            st1 = st2 = None
    if multi and st1 is not None:
        flags |= LOSS_STATS_TWO_SCALES     # the statistics carry the half-resolution sums (thermal_stats_scales == 2)
    resampled = tuple(g1.shape[1:3]) != (H, W) or (c1 is not None and tuple(c1.shape[1:3]) != (H, W))
    dp1 = dp2 = dc1 = dc2 = None
    if resampled:
        # pseudo-GT (and its confidence) at another resolution: bilinear taps inside the loss kernel's loads
        # (train_thermal_dustr.py:234-271); a confidence at the GT's size never takes a gradient.  The thermal
        # statistics of the preprocessing are honoured as on the same-size path.
        gh, gw = int(g1.shape[1]), int(g1.shape[2])
        ch, cw = (int(c1.shape[1]), int(c1.shape[2])) if c1 is not None else (H, W)
        if bwd:
            dp1 = out.get("dpred1"); dp2 = out.get("dpred2")
            dp1 = torch.empty_like(p1) if dp1 is None else dp1
            dp2 = torch.empty_like(p2) if dp2 is None else dp2
            if need_dconf[0] and (ch, cw) == (H, W):
                dc1 = out.get("dconf1")
                dc1 = torch.empty(B, H, W, dtype=torch.float32, device=dev) if dc1 is None else dc1
            if need_dconf[1] and (ch, cw) == (H, W):
                dc2 = out.get("dconf2")
                dc2 = torch.empty(B, H, W, dtype=torch.float32, device=dev) if dc2 is None else dc2
        rc = lib.t3d_loss_fwd_bwd_resampled_stats(
            _lib.ptr(p1), _lib.ptr(p2), _lib.ptr(g1), _lib.ptr(g2), gh, gw, _lib.ptr(c1), _lib.ptr(c2), ch, cw,
            _lib.ptr(t1), _lib.ptr(t2), tch, _lib.ptr(st1), _lib.ptr(st2), st_tiles,
            _lib.ptr(dp1), _lib.ptr(dp2), _lib.ptr(dc1), _lib.ptr(dc2),
            B, H, W, flags, alpha, ew, sw, dw, grad_scale,
            _lib.ptr(per_sample), _lib.ptr(batch), _lib.ptr(f64), _lib.ptr(ws), ws.numel(), stream)
        _lib.check(rc, "t3d_loss_fwd_bwd_resampled_stats")
        if bwd and rescale_invalid:
            rc = lib.t3d_loss_rescale_invalid(_lib.ptr(dp1), _lib.ptr(dp2), _lib.ptr(dc1), _lib.ptr(dc2),
                                              _lib.ptr(per_sample), _lib.ptr(batch), B, H, W, stream)
            _lib.check(rc, "t3d_loss_rescale_invalid")
        return per_sample, batch, dp1, dp2, dc1, dc2
    if bwd:
        dp1 = out.get("dpred1"); dp2 = out.get("dpred2")
        if dp1 is None:
            dp1 = torch.empty_like(p1)
        if dp2 is None:
            dp2 = torch.empty_like(p2)
        if need_dconf[0]:
            dc1 = out.get("dconf1")
            if dc1 is None:
                dc1 = torch.empty(B, H, W, dtype=torch.float32, device=dev)
        if need_dconf[1]:
            dc2 = out.get("dconf2")
            if dc2 is None:
                dc2 = torch.empty(B, H, W, dtype=torch.float32, device=dev)
        rc = lib.t3d_loss_fwd_bwd(
            _lib.ptr(p1), _lib.ptr(p2), _lib.ptr(g1), _lib.ptr(g2), _lib.ptr(c1), _lib.ptr(c2),
            _lib.ptr(t1), _lib.ptr(t2), tch, _lib.ptr(st1), _lib.ptr(st2), st_tiles,
            _lib.ptr(dp1), _lib.ptr(dp2), _lib.ptr(dc1), _lib.ptr(dc2),
            B, H, W, flags, alpha, ew, sw, dw, grad_scale,
            _lib.ptr(per_sample), _lib.ptr(batch), _lib.ptr(f64), _lib.ptr(ws), ws.numel(), stream)
        _lib.check(rc, "t3d_loss_fwd_bwd")
        if rescale_invalid:
            rc = lib.t3d_loss_rescale_invalid(_lib.ptr(dp1), _lib.ptr(dp2), _lib.ptr(dc1), _lib.ptr(dc2),
                                              _lib.ptr(per_sample), _lib.ptr(batch), B, H, W, stream)
            _lib.check(rc, "t3d_loss_rescale_invalid")
    else:
        rc = lib.t3d_loss_fwd(
            _lib.ptr(p1), _lib.ptr(p2), _lib.ptr(g1), _lib.ptr(g2), _lib.ptr(c1), _lib.ptr(c2),
            _lib.ptr(t1), _lib.ptr(t2), tch, _lib.ptr(st1), _lib.ptr(st2), st_tiles,
            B, H, W, flags, alpha, ew, sw, dw,
            _lib.ptr(per_sample), _lib.ptr(batch), _lib.ptr(f64), _lib.ptr(ws), ws.numel(), stream)
        _lib.check(rc, "t3d_loss_fwd")
    return per_sample, batch, dp1, dp2, dc1, dc2


def _hand_back_grads(ctx, g_loss):
    """backward of the fused losses: the forward kernel already produced d(loss)/d(inputs); scale them by
    grad_output on the device (a no-op kernel when it is 1) and hand them to autograd.  The buffers are scaled in
    place, so they can be consumed once: a second backward through the same node (retain_graph=True, two losses
    sharing the graph) raises instead of silently contributing zeros."""
    if ctx.grads == "none":             # forward ran without any input requiring grad
        return (None,) * 9
    if ctx.grads is None:
        raise RuntimeError("thermal3d_vision_b200: the fused loss gradients of this node were already consumed by a "
                           "previous backward (they are scaled in place); call the loss again instead of "
                           "backpropagating twice through it")
    dp1, dp2, dc1, dc2 = ctx.grads
    ctx.grads = None
    B, H, W, _ = ctx.shape
    with _lib.device_guard(dp1.device):
        go = g_loss.detach().to(dtype=torch.float32, device=dp1.device).reshape(1).contiguous()
        rc = _lib.lib().t3d_scale_grads(_lib.ptr(dp1), _lib.ptr(dp2), _lib.ptr(dc1), _lib.ptr(dc2),
                                       _lib.ptr(go), B, H, W, _lib.current_stream_ptr())
        _lib.check(rc, "t3d_scale_grads")
    need = ctx.needs_input_grad
    return (dp1 if need[0] else None, dp2 if need[1] else None,
            dc1 if need[2] else None, dc2 if need[3] else None, None, None, None, None, None)


class _FusedLoss(torch.autograd.Function):
    """forward = fused fwd+bwd kernel; backward = device-side scale by grad_output."""

    @staticmethod
    def forward(ctx, p1, p2, c1, c2, g1, g2, t1, t2, cfg):
        alpha, ew, sw, dw, multi, batch_mean, conf_min_only = cfg
        need = ctx.needs_input_grad
        bwd = bool(need[0] or need[1] or need[2] or need[3])
        need_dconf = (bool(need[2]) and c1 is not None, bool(need[3]) and c2 is not None)
        B = p1.shape[0]
        per_sample, batch, dp1, dp2, dc1, dc2 = _launch(
            bwd, p1, p2, g1, g2, c1, c2, t1, t2, need_dconf, alpha, ew, sw, dw, multi,
            (1.0 / B) if batch_mean else 1.0, rescale_invalid=batch_mean, conf_min_only=conf_min_only)
        ctx.shape = tuple(p1.shape)
        ctx.grads = (dp1, dp2, dc1, dc2) if bwd else "none"
        ctx.mark_non_differentiable(per_sample, batch)
        # B == 1 per-sample call: the loss itself (no validity filter, as utils/loss.py:295)
        loss = batch[0] if batch_mean else per_sample[0, 0]
        return loss.clone(), per_sample, batch

    @staticmethod
    def backward(ctx, g_loss, _g_ps, _g_b):
        return _hand_back_grads(ctx, g_loss)


def _device_of(*ts):
    for t in ts:
        if t is not None and t.is_cuda:
            return t.device
    if not torch.cuda.is_available():
        raise _lib.T3DError("no CUDA device: thermal3d_vision_b200 has no CPU path")
    return torch.device("cuda", torch.cuda.current_device())


def fused_thermal_loss(pred_pts1, pred_pts2, gt_pts1, gt_pts2, confidences1=None, confidences2=None,
                       thermal_img1=None, thermal_img2=None, *, alpha=0.2, edge_weight=0.5,
                       smoothness_weight=0.3, detail_weight=0.3, multi_scale=True,
                       batch_mean=True, conf_min_only=False) -> FusedLossResult:
    """Batched fused loss: tensors are [B,H,W,3] / [B,H,W] / [B,C,H,W].

    ``loss`` = mean over VALID samples (finite and > 0) of the per-sample
    enhanced_thermal_aware_loss; gradients w.r.t. pred and confidences flow
    through autograd.  No host synchronisation.  ``conf_min_only``: clamp the confidence from below only
    (train_thermal_dustr.py:278-279,305-318, the plain confidence-weighted L1 without utils/loss.py's upper clamp at 10).
    """
    dev = _device_of(pred_pts1, pred_pts2, gt_pts1, gt_pts2)
    p1, p2, g1, g2 = (_prep(t, dev) for t in (pred_pts1, pred_pts2, gt_pts1, gt_pts2))
    c1, c2, t1, t2 = (_prep(t, dev) for t in (confidences1, confidences2, thermal_img1, thermal_img2))
    if p1.dim() != 4 or p1.shape[-1] != 3:
        raise ValueError(f"pointmaps must be [B,H,W,3], got {tuple(p1.shape)}")
    if p2.shape != p1.shape:
        raise ValueError(f"pred_pts2 shape {tuple(p2.shape)} != pred_pts1 shape {tuple(p1.shape)}")
    B, H, W, _ = p1.shape
    # the pseudo-GT may come at another resolution (train_thermal_dustr.py:234-271 resamples it to the prediction's
    # size; here the taps are fused into the kernel's loads): [B,gh,gw,3], both views alike
    if g1.dim() != 4 or g1.shape[-1] != 3 or g1.shape[0] != B or g2.shape != g1.shape:
        raise ValueError(f"gt pointmaps must be two [B,h,w,3] tensors with B={B}, got {tuple(g1.shape)} / {tuple(g2.shape)}")
    for name, t in (("confidences1", c1), ("confidences2", c2)):
        if t is not None and tuple(t.shape) not in ((B, H, W), (B,) + tuple(g1.shape[1:3])):
            raise ValueError(f"{name} must be [B,H,W]={B, H, W} (or the GT's size), got {tuple(t.shape)}")
    if c1 is not None and c2 is not None and c1.shape != c2.shape:
        raise ValueError("confidences1 / confidences2 must have the same size")
    if (t1 is None) != (t2 is None):
        t1 = t2 = None                                     # utils/loss.py:116: both or nothing
    if t1 is not None:
        if t1.dim() != 4 or t1.shape[1] not in (1, 3) or t1.shape != t2.shape or \
                tuple(t1.shape[2:]) != (H, W) or t1.shape[0] != B:
            raise ValueError(f"thermal images must be [B,1|3,H,W], got {tuple(t1.shape)} / {tuple(t2.shape)}")
        if multi_scale and (H < 4 or W < 4):
            raise ValueError("multi_scale needs H, W >= 4 (the reference breaks on squeezed dims; SURVEY.md D.7)")
    cfg = (float(alpha), float(edge_weight), float(smoothness_weight), float(detail_weight),
           bool(multi_scale), bool(batch_mean), bool(conf_min_only))
    loss, per_sample, batch = _FusedLoss.apply(p1, p2, c1, c2, g1, g2, t1, t2, cfg)
    return FusedLossResult(loss, per_sample, batch)


def fused_thermal_loss_fwd_bwd(pred_pts1, pred_pts2, gt_pts1, gt_pts2, confidences1=None, confidences2=None,
                               thermal_img1=None, thermal_img2=None, *, alpha=0.2, edge_weight=0.5,
                               smoothness_weight=0.3, detail_weight=0.3, multi_scale=True,
                               conf_grad=True, out=None, thermal_stats=None, grad_scale=None,
                               thermal_replicated=False, rescale_invalid=True, thermal_stats_scales=1):
    """Functional (no autograd) fused step on prepared contiguous fp32 CUDA tensors.

    Returns dict(per_sample, batch, dpred1, dpred2, dconf1, dconf2); gradients are those of the
    mean over valid samples.  ``out`` may hold preallocated buffers of the same names (+ 'workspace').
    ``thermal_stats`` = (ThermalBatch.grad_stats of view 1, of view 2): the thermal-gradient sums the
    preprocessing kernel already produced; the loss then skips its own pass over the thermal images
    (``multi_scale``: only if they carry the half-resolution sums too, ``thermal_stats_scales=2`` =
    ThermalBatch.stats_scales of a batch preprocessed with ``half_res_stats=True``).
    ``grad_scale`` (default 1/B) is the a-priori upstream gradient, e.g. 1/(B * world_size) for the mean
    over a data-parallel global batch.  ``thermal_replicated``: promise that the 3 planes of every thermal
    image are bit-identical (ThermalBatch.replicated; what enhance_thermal_contrast always returns): the
    kernel then reads one plane instead of three, same results.  ``rescale_invalid=False`` leaves the
    validity fix-up of the gradients to the caller (pipeline.HotPathStep: t3d_step_epilogue does it together
    with the result packing in one launch).
    """
    _lib.require_cuda(pred_pts1, pred_pts2, gt_pts1, gt_pts2, confidences1, confidences2, thermal_img1, thermal_img2)
    if thermal_replicated and DEBUG_CHECKS and not torch.cuda.is_current_stream_capturing():
        check_thermal_replicated(thermal_img1, thermal_img2)
    B = pred_pts1.shape[0]
    need_dconf = (conf_grad and confidences1 is not None, conf_grad and confidences2 is not None)
    ps, bt, dp1, dp2, dc1, dc2 = _launch(
        True, pred_pts1, pred_pts2, gt_pts1, gt_pts2, confidences1, confidences2, thermal_img1, thermal_img2,
        need_dconf, float(alpha), float(edge_weight), float(smoothness_weight), float(detail_weight),
        bool(multi_scale), (1.0 / B) if grad_scale is None else float(grad_scale), rescale_invalid=bool(rescale_invalid), out=out,
        thermal_stats=thermal_stats, thermal_replicated=thermal_replicated, thermal_stats_scales=int(thermal_stats_scales))
    return {"per_sample": ps, "batch": bt, "dpred1": dp1, "dpred2": dp2, "dconf1": dc1, "dconf2": dc2}


def check_thermal_replicated(*thermal):
    """Raise unless the 3 planes of every image are bit-identical (the promise behind thermal_replicated=True)."""
    for t in thermal:
        if t is None or t.shape[1] != 3:
            continue
        with _lib.device_guard(t.device):
            bits = t.view(torch.int32)
            if not (torch.equal(bits[:, 0], bits[:, 1]) and torch.equal(bits[:, 0], bits[:, 2])):
                raise ValueError("thermal_replicated=True but the three thermal planes are not bit-identical")


# ----------------------------------------------------------------------------- reference signatures
def _unbatched(pred_pts1, pred_pts2, gt_pts1, gt_pts2, c1, c2, t1, t2, alpha, ew, sw, dw, multi):
    src_device = pred_pts1.device
    if pred_pts1.dim() != 3 or pred_pts1.shape[-1] != 3:
        raise ValueError(f"expected [H,W,3] pointmaps, got {tuple(pred_pts1.shape)}")
    if t1 is not None and t2 is not None:
        if not (isinstance(t1, torch.Tensor) and t1.dim() == 3):
            # the reference leaves thermal_gray1 unbound here (utils/loss.py:118-140, NameError)
            raise ValueError("thermal images must be 3-D [C,H,W] tensors")
        if t1.shape[0] not in (1, 3):
            t1, t2 = t1[:1], t2[:1]                         # utils/loss.py:123: channel 0
        t1, t2 = t1.unsqueeze(0), t2.unsqueeze(0)
    else:
        t1 = t2 = None
    ub = lambda t: None if t is None else t.unsqueeze(0)
    res = fused_thermal_loss(ub(pred_pts1), ub(pred_pts2), ub(gt_pts1), ub(gt_pts2), ub(c1), ub(c2), t1, t2,
                             alpha=alpha, edge_weight=ew, smoothness_weight=sw, detail_weight=dw,
                             multi_scale=multi, batch_mean=False)
    loss = res.loss if res.loss.device == src_device else res.loss.to(src_device)
    return loss, res.per_sample


def confidence_weighted_regression_loss(pred_pts1, pred_pts2, gt_pts1, gt_pts2,
                                        confidences1=None, confidences2=None, alpha=0.2):
    """Drop-in for utils/loss.py:75-98."""
    loss, _ = _unbatched(pred_pts1, pred_pts2, gt_pts1, gt_pts2, confidences1, confidences2,
                         None, None, alpha, 0.0, 0.0, 0.0, False)
    return loss


def enhanced_thermal_aware_loss(pred_pts1, pred_pts2, gt_pts1, gt_pts2,
                                confidences1=None, confidences2=None,
                                thermal_img1=None, thermal_img2=None,
                                alpha=0.2, edge_weight=0.5, smoothness_weight=0.3,
                                detail_weight=0.3, multi_scale=True):
    """Drop-in for utils/loss.py:100-305: returns (total_loss, dict of python floats)."""
    loss, per_sample = _unbatched(pred_pts1, pred_pts2, gt_pts1, gt_pts2, confidences1, confidences2,
                                  thermal_img1, thermal_img2, alpha, edge_weight, smoothness_weight,
                                  detail_weight, multi_scale)
    vals = per_sample[0, :5].tolist()                       # one 20-byte D2H (the reference does 4 .item())
    thermal_on = thermal_img1 is not None and thermal_img2 is not None
    comps = {
        "basic_loss": vals[1],
        "edge_loss": vals[2] if thermal_on else 0,
        "smoothness_loss": vals[3] if thermal_on else 0,
        "detail_loss": vals[4] if thermal_on else 0,
    }
    return loss, comps


class _LossV1(torch.autograd.Function):
    @staticmethod
    @_lib.on_tensor_device
    def forward(ctx, p1, p2, c1, c2, g1, g2, t1, t2, cfg):
        alpha, ew, sw = cfg
        lib = _lib.lib()
        B, H, W, _ = p1.shape
        dev = p1.device
        need = ctx.needs_input_grad
        bwd = bool(need[0] or need[1] or need[2] or need[3])
        tch = 0 if t1 is None else int(t1.shape[1])
        ws = torch.empty(lib.t3d_loss_v1_workspace_bytes(B, H, W), dtype=torch.uint8, device=dev)
        per_sample = torch.empty(B, OUT_STRIDE, dtype=torch.float32, device=dev)
        batch = torch.empty(OUT_STRIDE, dtype=torch.float32, device=dev)
        dp1 = torch.empty_like(p1) if bwd else None
        dp2 = torch.empty_like(p2) if bwd else None
        dc1 = torch.empty(B, H, W, dtype=torch.float32, device=dev) if (bwd and need[2] and c1 is not None) else None
        dc2 = torch.empty(B, H, W, dtype=torch.float32, device=dev) if (bwd and need[3] and c2 is not None) else None
        rc = lib.t3d_loss_v1_fwd_bwd(_lib.ptr(p1), _lib.ptr(p2), _lib.ptr(g1), _lib.ptr(g2), _lib.ptr(c1), _lib.ptr(c2),
                                     _lib.ptr(t1), _lib.ptr(t2), tch, _lib.ptr(dp1), _lib.ptr(dp2), _lib.ptr(dc1),
                                     _lib.ptr(dc2), B, H, W, alpha, ew, sw, 1.0, _lib.ptr(per_sample), _lib.ptr(batch),
                                     None, _lib.ptr(ws), ws.numel(), _lib.current_stream_ptr())
        _lib.check(rc, "t3d_loss_v1_fwd_bwd")
        ctx.shape = tuple(p1.shape)
        ctx.grads = (dp1, dp2, dc1, dc2) if bwd else "none"
        ctx.mark_non_differentiable(per_sample)
        return per_sample[0, 0].clone(), per_sample

    @staticmethod
    def backward(ctx, g_loss, _g_ps):
        return _hand_back_grads(ctx, g_loss)


def thermal_aware_loss(pred_pts1, pred_pts2, gt_pts1, gt_pts2,
                       confidences1=None, confidences2=None,
                       thermal_img1=None, thermal_img2=None,
                       alpha=0.2, edge_weight=0.5, smoothness_weight=0.3):
    """Drop-in for utils/loss.py:4-72 (v1 loss; the reference imports it but never calls it)."""
    src_device = pred_pts1.device
    dev = _device_of(pred_pts1, pred_pts2, gt_pts1, gt_pts2)
    if pred_pts1.dim() != 3 or pred_pts1.shape[-1] != 3:
        raise ValueError(f"expected [H,W,3] pointmaps, got {tuple(pred_pts1.shape)}")
    t1 = t2 = None
    thermal_on = thermal_img1 is not None and thermal_img2 is not None
    if thermal_on and isinstance(thermal_img1, torch.Tensor) and thermal_img1.dim() == 3:   # :19
        t1, t2 = thermal_img1, thermal_img2
        if t1.shape[0] != 3:
            t1, t2 = t1[:1], t2[:1]
        t1, t2 = _prep(t1.unsqueeze(0), dev), _prep(t2.unsqueeze(0), dev)
    elif thermal_on:
        # reference: edge stays 0 but the smoothness branch hits unbound gradients -> NameError (:54-58)
        raise ValueError("thermal images must be 3-D [C,H,W] tensors")
    ub = lambda t: None if t is None else _prep(t.unsqueeze(0), dev)
    loss, ps = _LossV1.apply(ub(pred_pts1), ub(pred_pts2), ub(confidences1), ub(confidences2),
                             ub(gt_pts1), ub(gt_pts2), t1, t2,
                             (float(alpha), float(edge_weight), float(smoothness_weight)))
    vals = ps[0, :4].tolist()
    comps = {"basic_loss": vals[1], "edge_loss": vals[2] if t1 is not None else 0,
             "smoothness_loss": vals[3] if t1 is not None else 0}
    return (loss if loss.device == src_device else loss.to(src_device)), comps
