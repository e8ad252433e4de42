"""Data-parallel plumbing for the hot path (torch.distributed; NCCL on GPUs, gloo in CPU tests).

The path shards by image: rank r owns a contiguous slice of the batch / dataset and runs the
kernels on it with no data-path collective.  The only exchange per step is ONE all-reduce (SUM)
of the packed result vector (RESULT_SIZE doubles) that ``t3d_step_epilogue`` produces on the device
(SURVEY.md section 8e): sums of valid losses / components / counts and sums of finite metrics /
image count, i.e. exactly the accumulators of train_thermal_dustr.py:320,359 and
utils/metrics.py:128-136.  Gradients w.r.t. pointmaps stay local to the rank.
"""
from __future__ import annotations

from typing import Dict, Tuple

import torch
import torch.distributed as dist

RESULT_SIZE = 24
METRIC_KEYS = ("abs_rel", "sq_rel", "rmse", "rmse_log", "acc_1", "acc_2", "acc_3")


def world() -> Tuple[int, int]:
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_range(n: int, rank: int, world_size: int) -> Tuple[int, int]:
    """Contiguous, balanced [lo, hi) slice of n images for `rank` (first n % world ranks get one more)."""
    base, rem = divmod(n, world_size)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def all_reduce_result(vec: torch.Tensor, async_op: bool = False):
    """In-place SUM all-reduce of the packed result vector (no-op for a single process).
    async_op=True returns the work handle (None for a single process): the collective then runs on the backend's
    own stream and overlaps whatever the caller enqueues next; `handle.wait()` orders the current stream after it."""
    if vec.numel() != RESULT_SIZE:
        raise ValueError(f"packed result must have {RESULT_SIZE} elements")
    _, w = world()
    if w > 1:
        h = dist.all_reduce(vec, op=dist.ReduceOp.SUM, async_op=async_op)
        return h if async_op else vec
    return None if async_op else vec


def bind_to_gpu_numa_node(device_index: int) -> bool:
    """Pin the calling process to the CPUs closest to its GPU (NVML's ideal CPU affinity) so that pinned host
    buffers allocated afterwards live on the GPU's NUMA node: with 8 ranks staging 0.8 GB per step each, remote-node
    pinned memory halves the aggregate H2D rate.  Returns False when NVML is unavailable."""
    try:
        import os
        import pynvml
        pynvml.nvmlInit()
        phys = device_index
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if device_index < len(ids) and ids[device_index].isdigit():
                phys = int(ids[device_index])
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(phys))
        return True
    except Exception:
        return False


def global_grad_scale(local_batch: int) -> float:
    """A-priori scale of the local loss gradients so that they are those of the GLOBAL batch mean
    (all ranks hold `local_batch` samples; invalid samples are fixed up on the device afterwards)."""
    _, w = world()
    return 1.0 / (local_batch * w)


def summarize(vec) -> Dict[str, float]:
    """Packed (all-reduced) vector -> the numbers the reference logs: mean loss over valid samples and
    dataset-mean metrics (finite values summed, divided by the count of ALL images)."""
    r = [float(v) for v in vec]
    nv, n_img = max(r[5], 1.0), max(r[14], 1.0)
    out = {"loss": r[0] / nv, "basic_loss": r[1] / nv, "edge_loss": r[2] / nv, "smoothness_loss": r[3] / nv,
           "detail_loss": r[4] / nv, "n_valid": r[5], "n_pairs": r[6], "n_images": r[14]}
    for i, k in enumerate(METRIC_KEYS):
        out[k] = r[7 + i] / n_img
    # parameter gradients summed over the ranks (slots 16..): with the a-priori 1 / (B * world) scale of the loss
    # gradients upstream, the sum IS the gradient of the global batch mean (what DDP's all-reduce produces)
    out["param_grads"] = r[16:RESULT_SIZE]
    return out
