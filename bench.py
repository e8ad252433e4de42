#!/usr/bin/env python
"""bench.py -- throughput of the Thermal3D-Vision per-pixel hot path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W]                 # our sm_100a path
  python bench.py --impl reference [--gpus N] [--steps K] [--warmup W]  # CPU oracle port of the reference
  python bench.py --dump-outputs DIR ...    # also store the last timed step's outputs as DIR/<name>.npy

A "step" is one pass of the hot path over one batch of synthetic input:
thermal preprocessing of 2B raw 16-bit frames -> fused thermal-aware loss
fwd+bwd over B pointmap pairs -> pointmap->depth + depth metrics of B frames
(thermal3d_vision_b200.pipeline.HotPathStep).  Workload = BASELINE.json
configs[2] ("DUSt3R-512 shape: batch=64 512x384 pointmap pairs"), the
configuration the metric's 70 %-of-HBM target is quoted on; per-rank batch is
fixed as N grows (weak scaling, sharded by image; the 16 packed doubles of a step
are exchanged over NVLink peer memory by the step's own epilogue kernel).  One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (no __pycache__)
sys.path.insert(0, ROOT)

METRIC = "frames/sec of fused loss fwd+bwd+preproc"
UNIT = "pairs/s"
EDGE_W, SMOOTH_W, DETAIL_W, ALPHA = 0.5, 0.3, 0.4, 0.2


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="pairs per rank")
    ap.add_argument("--height", type=int, default=384)
    ap.add_argument("--width", type=int, default=512)
    ap.add_argument("--multi-scale", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample-pairs", type=int, default=4)
    ap.add_argument("--no-extras", action="store_true", help="skip the extra blocks (multi-scale, configs[1], eval shard)")
    ap.add_argument("--workload", default="train", choices=["train", "eval"],
                    help="train: BASELINE configs[2] (the metric's configuration, default); eval: configs[4] "
                         "(640x512 u16 preprocessing + pointmap->depth + metrics over a dataset shard; extra line)")
    ap.add_argument("--eval-frames", type=int, default=2560, help="frames per rank for --workload eval (8 ranks: 20 480)")
    ap.add_argument("--eval-batch", type=int, default=256, help="frames per evaluation step (the dataset shard is cut into batches of this size)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned to its caller as DIR/<name>.npy "
                         "(float32 / float64; arrays above %d elements as a fixed seeded sample, see dump_outputs)" % DUMP_SAMPLE)
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "b200" or a.workload != "train"):
        ap.error("--dump-outputs applies to the timed step of --impl b200 --workload train")
    return a


def workload_name(a):
    return f"dust3r512_batch{a.batch}_{a.width}x{a.height}_pairs_loss_fwd_bwd+preproc_640x512_u16+depth_metrics"


EXCHANGE_TEXT = {
    None: "single process, no exchange",
    "peer": "per step one 192-byte exchange of the packed scalars over NVLink peer memory (symmetric-memory mailboxes written by "
            "the step's epilogue kernel), no NCCL call in the step",
    "nccl": "per step one asynchronous NCCL all-reduce of the packed scalars (24 doubles)",
    "cpu": "host cores only",
}


def config_dict(a, world, exchange=None):
    return {"workload": workload_name(a), "per_rank_batch": a.batch, "global_batch": a.batch * world,
            "pointmap_hw": [a.height, a.width], "raw_frame_hw": [512, 640], "multi_scale": bool(a.multi_scale),
            "edge_weight": EDGE_W, "smoothness_weight": SMOOTH_W, "detail_weight": DETAIL_W, "alpha": ALPHA,
            "parallelism": f"dp{world} (sharded by image; {EXCHANGE_TEXT[exchange]})",
            "l2_policy": "inputs_exceed_l2 (1.2 GB of inputs per step vs 126 MB L2; no flush needed)"}


# --------------------------------------------------------------------------- synthetic inputs (SURVEY.md 8d)
def make_inputs_torch(B, H, W, seed, device, raw_hw=(512, 640)):
    import torch
    RH, RW = raw_hw
    g = torch.Generator(device=device).manual_seed(seed)
    r = lambda *s: torch.randn(*s, device=device, generator=g)
    gt1, gt2 = r(B, H, W, 3), r(B, H, W, 3)
    gt1[..., 2] = 1.5 + 3 * gt1[..., 2].abs()
    gt2[..., 2] = 1.5 + 3 * gt2[..., 2].abs()
    pred1 = gt1 + 0.1 * r(B, H, W, 3)
    pred2 = gt2 + 0.1 * r(B, H, W, 3)
    conf1 = 1 + 4 * torch.rand(B, H, W, device=device, generator=g)
    conf2 = 1 + 4 * torch.rand(B, H, W, device=device, generator=g)
    raws = []
    for _ in range(2):          # day: N(22800, 400); night: N(22300, 250) + hot blobs -- inside the Freiburg window
        night = torch.rand(B, 1, 1, device=device, generator=g) < 0.4
        f = torch.where(night, 22300 + 250 * r(B, RH, RW), 22800 + 400 * r(B, RH, RW))
        blobs = (torch.rand(B, (RH + 31) // 32, (RW + 31) // 32, device=device, generator=g) < 0.01).float()
        blobs = blobs.repeat_interleave(32, 1).repeat_interleave(32, 2)[:, :RH, :RW] * 1500.0
        f = f + torch.where(night, blobs, torch.zeros_like(blobs))
        raws.append(f.clamp(0, 65535).to(torch.int32).to(torch.uint16))
    gt_depth = gt1[..., 2].contiguous()
    both = torch.cat(raws)            # the two views as halves of one tensor: preprocessed by one call
    raws = [both[:B], both[B:]]
    return {"raw1": raws[0], "raw2": raws[1], "pred1": pred1, "pred2": pred2, "gt1": gt1, "gt2": gt2,
            "conf1": conf1, "conf2": conf2, "gt_depth": gt_depth}


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region.  In-process NVML (a sample every ~2 ms from a
    thread; the timed region of a default run is only ~0.1 s, too short for an nvidia-smi subprocess to start);
    falls back to `nvidia-smi -lms` when pynvml is missing."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.nvml, self.handle, self.stop_flag, self.t = None, None, threading.Event(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if vis:
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if index < len(ids) and ids[index].isdigit():
                    phys = int(ids[index])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _nvml_loop(self):
        nv = self.nvml
        bits = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self.stop_flag.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
                r = int(get_reasons(self.handle))
                for name, bit in bits.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nvml is not None:
            self.t = threading.Thread(target=self._nvml_loop, daemon=True)
            self.t.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def mark(self):
        """Drop what was sampled so far (called right before the timed region starts)."""
        self.samples.clear(); self.reasons.clear(); self.lines.clear()

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag.set()
            self.t.join(timeout=1)
            sm = sorted(self.samples)
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
                    "reasons": sorted(self.reasons), "samples": len(sm), "source": "nvml, ~2 ms period, timed region only"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 6:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 20"}


# --------------------------------------------------------------------------- CPU arm (oracle port of the reference)
def cpu_step_fn(a, n, H=None, W=None):
    """Returns (fn() -> None, description): one CPU step over n pairs.  The unmodified reference cannot travel to the
    GPU box, so this is the oracle port (oracle/): same per-sample loop as train_thermal_dustr.py:182-360 (loss per
    sample -> mean over valid -> one backward), cv2.resize + percentile normalisation per frame as
    data/dataset_loader.py:237-249 / utils/preprocessing.py:6-30, compute_depth_metrics per frame."""
    import numpy as np
    import torch
    from oracle import ref_loss, ref_metrics, ref_preprocess
    try:
        import cv2
        resize = lambda f, hw: cv2.resize(f, (hw[1], hw[0]))      # what the reference actually calls
    except Exception:
        resize = ref_preprocess.resize_bilinear
    torch.set_num_threads(os.cpu_count() or 1)
    H, W = H or a.height, W or a.width
    P1, P2, G1, G2, C1, C2, _, _ = ref_loss.make_batch_inputs(n, H, W, seed=0, smooth=False)
    raw = ref_preprocess.make_raw_frames(2 * n, seed=0)
    kw = dict(alpha=ALPHA, edge_weight=EDGE_W, smoothness_weight=SMOOTH_W, detail_weight=DETAIL_W,
              multi_scale=bool(a.multi_scale))

    def step():
        th = []
        for f in raw:
            r = resize(f, (H, W)).astype(np.float32)
            t = torch.from_numpy(np.repeat(r[None], 3, 0))
            th.append(torch.from_numpy(ref_preprocess.enhance_thermal_contrast(t.numpy())[0]))
        p1, p2 = P1.clone().requires_grad_(), P2.clone().requires_grad_()
        c1, c2 = C1.clone().requires_grad_(), C2.clone().requires_grad_()
        tot, nv = 0.0, 0
        for i in range(n):
            loss, _ = ref_loss.enhanced_thermal_aware_loss_torch(p1[i], p2[i], G1[i], G2[i], c1[i], c2[i],
                                                                 th[2 * i], th[2 * i + 1], **kw)
            if torch.isfinite(loss) and loss > 0:
                tot = tot + loss
                nv += 1
        (tot / max(nv, 1)).backward()
        for i in range(n):
            ref_metrics.compute_depth_metrics(p1[i, ..., 2].detach().numpy(), G1[i, ..., 2].numpy())

    return step, f"{n} pairs ({W}x{H}) per step: per-sample loss loop + backward, 2 frames/pair preprocessed (640x512 u16), metrics per pair"


def time_cpu(a, n, H=None, W=None, min_seconds=10.0, max_iters=2000, warmup=1):
    step, desc = cpu_step_fn(a, n, H, W)
    for _ in range(warmup):
        step()
    t0, it = time.perf_counter(), 0
    while True:
        step(); it += 1
        el = time.perf_counter() - t0
        if el >= min_seconds or it >= max_iters:
            break
    return {"value": n * it / el, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port",
            "sample": desc + f"; {it} iterations in {el:.1f} s"}


def run_reference(a):
    """The reference arm: the oracle port of the reference's CPU path on the host cores, EXACTLY --warmup + --steps
    steps; every step processes `sample_pairs` pairs of the workload -- the whole batch when warmup + steps full
    batches fit the time budget on this host, otherwise the largest sample (>= 8 pairs) that does."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    # size the per-step sample from a 2-pair probe of this host (untimed): the whole batch when warmup + steps full
    # batches fit in ~150 s at half the probed rate (a batch-64 graph runs slower per pair than a 2-pair one:
    # its saved activations no longer fit the caches), never fewer than 8 pairs
    probe, _ = cpu_step_fn(a, 2)
    probe()
    t0 = time.perf_counter()
    probe()
    rate = 2.0 / max(time.perf_counter() - t0, 1e-3)
    n = int(max(min(a.batch, 8), min(a.batch, (150.0 * 0.5 * rate) // max(a.steps + a.warmup, 1))))
    step, desc = cpu_step_fn(a, n)
    for _ in range(a.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        step()
    el = time.perf_counter() - t0
    v = n * a.steps / el
    cfg = config_dict(a, world, "cpu")
    cfg["sample_pairs"] = n
    cfg["sample_note"] = (f"each timed step runs {n} of the {a.batch} pairs of the batch" if n < a.batch
                          else "each timed step runs the whole batch")
    out = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
           "warmup": a.warmup, "ms_per_step": 1e3 * el / a.steps, "ms_per_full_batch_extrapolated": 1e3 * el / a.steps * a.batch / n,
           "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
           "cpu_baseline": {"value": v, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port", "sample": desc},
           "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0, "note": "oracle port of the reference's CPU path on the host cores; the python reference "
                                      "itself is not on the GPU box (no /root/reference there)"}
    print(json.dumps(out), flush=True)


# --------------------------------------------------------------------------- our arm
KEYS = ("raw1", "raw2", "pred1", "pred2", "gt1", "gt2", "conf1", "conf2", "gt_depth")


def load_peak():
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    src = "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    return peak, src


DUMP_SAMPLE = 1 << 20      # elements kept of each large output: 5 sampled arrays x 4 MB stay well under 64 MB


def dump_outputs(step, out_dir):
    """Write the outputs of the step's latest call as out_dir/<name>.npy: the packed result vector, the per-sample
    loss rows, the per-image metrics, the percentiles, the four gradients and the preprocessed thermal batch.  An
    array with more than DUMP_SAMPLE elements is stored as the elements at DUMP_SAMPLE flat indices drawn without
    replacement (sorted) by a generator seeded with 0, so that two runs with the same arguments store the same
    positions.  Call after the step's results are ordered on the current stream (finish() / wait_result())."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"result": step.result, "per_sample": step.loss_out["per_sample"], "batch": step.loss_out["batch"],
              "metrics": step.met_out["metrics_f64"], "percentiles": step.pre_both["percentiles"],
              "thermal": step.pre_both["thermal"]}
    arrays.update({k: step.loss_out[k] for k in ("dpred1", "dpred2", "dconf1", "dconf2")})
    for name, t in arrays.items():
        if t.numel() > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_SAMPLE, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        a = t.cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64 if a.dtype == np.float64 else np.float32))


def time_steps(fn, steps, warmup, finish=None):
    """CUDA-event time of `steps` calls of fn() after `warmup` untimed ones (ms per call)."""
    import torch
    for _ in range(warmup):
        fn()
    if finish:
        finish()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    if finish:
        finish()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def extra_multi_scale(a, dev, d, peak):
    """multi_scale=True (the reference function's default, utils/loss.py:104): the same step, device-timed, plus the
    summed duration of the loss call's kernels (thermal statistics + one-pass marching kernel + second stage) per step."""
    from thermal3d_vision_b200 import _lib
    from thermal3d_vision_b200.pipeline import HotPathStep
    B, H, W = a.batch, a.height, a.width
    step = HotPathStep(B, H, W, device=dev, multi_scale=True, alpha=ALPHA, edge_weight=EDGE_W, smoothness_weight=SMOOTH_W,
                       detail_weight=DETAIL_W)
    args = [d[k] for k in KEYS]
    ms = time_steps(lambda: step.run_device(*args), 20, 3, step.finish)
    _lib.profile_begin("loss_|thermal_stats", 256)
    for _ in range(10):
        step.run_device(*args)
    step.finish()
    tl = _lib.profile_timeline()
    _lib.profile_end()
    per = {}
    for name, t0, t1 in tl:
        per[name] = per.get(name, 0.0) + (t1 - t0) / 10.0
    loss_ms = sum(per.values())
    ab = step.algorithmic_bytes()
    s = HotPathStep.summarize(step.wait_result().cpu())
    return {"ms_per_step": ms, "pairs_per_s": B / (ms * 1e-3), "loss_kernels_ms": loss_ms, "loss_kernels": per,
            "loss_frac_of_peak": ab["loss"] / (loss_ms * 1e-3) / 1e9 / peak if loss_ms > 0 else None,
            "step_frac_of_peak": sum(ab.values()) / (ms * 1e-3) / 1e9 / peak,
            "check": {"loss": s["loss"], "n_valid": s["n_valid"]},
            "note": "same workload with multi_scale=True; loss_kernels_ms = CUDA-event time of every kernel of the loss call per step "
                    "(thermal gradient statistics at both scales + the one-pass marching kernel + second stage) "
                    "(bracketing events serialise the streams, so the step itself is timed separately without them)"}


def extra_cfg2(a, dev, peak):
    """BASELINE configs[1] (batch 8, 224x224) replayed as one CUDA graph, and configs[0]: the same step on the host
    cores (oracle port)."""
    import torch
    from thermal3d_vision_b200.pipeline import HotPathStep
    B, H, W = 8, 224, 224
    d = make_inputs_torch(B, H, W, seed=2, device=dev)
    step = HotPathStep(B, H, W, device=dev, alpha=ALPHA, edge_weight=EDGE_W, smoothness_weight=SMOOTH_W, detail_weight=DETAIL_W)
    replay = step.capture_graph(*[d[k] for k in KEYS])
    # 45 MB of inputs + 13 MB of outputs per step fit the 126 MB L2: flush it between replays (write 256 MB) and
    # time only the replays
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(30)]
    for _ in range(5):
        replay()
    for e0, e1 in ev:
        flush.fill_(1.0)
        e0.record(); replay(); e1.record()
    torch.cuda.synchronize()
    ms_cold = sorted(e0.elapsed_time(e1) for e0, e1 in ev)[len(ev) // 2]
    ms_warm = time_steps(replay, 200, 5)
    ab = sum(step.algorithmic_bytes().values())
    s = HotPathStep.summarize(replay().cpu())
    eager = HotPathStep(B, H, W, device=dev, alpha=ALPHA, edge_weight=EDGE_W, smoothness_weight=SMOOTH_W, detail_weight=DETAIL_W)
    ms_eager = time_steps(lambda: eager.run_device(*[d[k] for k in KEYS]), 200, 5, eager.finish)
    out = {"workload": "batch8_224x224_pairs_loss_fwd_bwd+preproc_640x512_u16+depth_metrics (BASELINE configs[1], CUDA-graph replay)",
           "ms_per_step": ms_cold, "pairs_per_s": B / (ms_cold * 1e-3), "ms_per_step_l2_warm": ms_warm,
           "ms_per_step_stream_launches": ms_eager,
           "l2_policy": "flushed between replays (256 MB fill), median of 30; l2_warm = 200 back-to-back replays",
           "roofline": {"bound": "hbm", "achieved": ab / (ms_cold * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": ab / (ms_cold * 1e-3) / 1e9 / peak, "step_algorithmic_bytes": ab,
                        "note": "launch-/latency-bound shape: 58 MB of traffic is ~9 us of HBM time"},
           "check": {"loss": s["loss"], "abs_rel": s["abs_rel"], "n_valid": s["n_valid"]}}
    if not a.no_cpu_baseline:
        out["cpu_baseline_cfg0"] = time_cpu(a, B, H, W, min_seconds=6.0)
    return out


def run_b200(a):
    import torch
    import torch.distributed as dist
    from thermal3d_vision_b200 import _lib
    from thermal3d_vision_b200.pipeline import HotPathStep

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from thermal3d_vision_b200.distributed import bind_to_gpu_numa_node
    all_cpus = os.sched_getaffinity(0)
    numa_bound = bind_to_gpu_numa_node(local)          # before any pinned allocation (matters for the e2e leg at N > 1)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    if world != a.gpus and rank == 0:
        print(f"[bench] note: --gpus {a.gpus} but WORLD_SIZE={world}; using {world}", file=sys.stderr)
    _lib.lib()

    B, H, W = a.batch, a.height, a.width
    # pipelined: the next step's side chains (preprocessing, metrics) start when this step's loss kernel has left the
    # machine, i.e. beside its second-stage reduction, epilogue and exchange instead of behind them; every step does all
    # of its own work on its own output set (T3D_PIPELINED=0: plain stream semantics, a few microseconds slower per
    # step).  The timed region ends with finish(), i.e. after the last step's last kernel and exchange.
    pipelined = os.environ.get("T3D_PIPELINED", "1") not in ("", "0")
    step = HotPathStep(B, H, W, device=dev, multi_scale=bool(a.multi_scale), alpha=ALPHA, edge_weight=EDGE_W,
                       smoothness_weight=SMOOTH_W, detail_weight=DETAIL_W, distributed=world > 1, pipelined=pipelined)
    d = make_inputs_torch(B, H, W, seed=rank, device=dev)
    args = tuple(d[k] for k in KEYS)
    host = {k: v.cpu().pin_memory() for k, v in d.items()}
    os.sched_setaffinity(0, all_cpus)                  # the pinned pages are placed; the CPU baseline leg uses every core

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return t.item()
        return ms

    # ---------------- device-resident timing ("value")
    for _ in range(max(a.warmup, 3)):
        step.run_device(*args)
    step.finish()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.15)
    dominant = "loss_tile_kernel" if a.multi_scale else "loss_march_kernel"
    # the dominant kernel is bracketed by CUDA events in every 4th step of the timed region (the event records cost
    # stream time: ~5 us per bracketed launch); launches_timed says how many
    _lib.profile_begin(dominant, a.steps + 4, every_nth=4 if a.steps >= 16 else 1)
    n0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if rank == 0:
        sampler.mark()
    e0.record()
    for _ in range(a.steps):
        step.run_device(*args)
    step.finish()                        # every step's last kernel and outstanding exchange belong to the timed region
    e1.record()
    barrier()
    launches = _lib.launch_count() - n0
    kern_ms, kern_n = _lib.profile_end()
    ms_dev = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if rank == 0 else None
    result_vec = step.wait_result().clone()
    step_result_size = result_vec.numel()
    if a.dump_outputs and rank == 0:
        dump_outputs(step, a.dump_outputs)
    summary = HotPathStep.summarize(result_vec.cpu())

    # ---------------- data parallel: the exchanged vector against an independent all-gather of the local vectors
    check_exchange = {"exchange": step.exchange or "none"}
    if world > 1:
        last = (step.calls - 1) & 1
        gathered = [torch.zeros_like(step.local[last]) for _ in range(world)]
        dist.all_gather(gathered, step.local[last].contiguous())
        total = torch.zeros_like(gathered[0])
        for g in gathered:                  # rank order, the order the exchange adds in
            total = total + g
        check_exchange["exchange_bitwise_ok"] = bool(torch.equal(total, result_vec))
        check_exchange["ranks_seen"] = int(round(total[6].item() / B))
        if step.exchange_fallback:
            check_exchange["peer_unavailable"] = step.exchange_fallback

    # ---------------- end to end through the public API with HOST buffers ("e2e")
    for _ in range(2):
        step.run_host(host)
    barrier()
    e0.record()
    for _ in range(a.steps):
        step.run_host(host)
    e1.record()
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))

    if rank == 0:
        peak, peak_src = load_peak()
        ab = step.algorithmic_bytes()
        kern_bytes = ab["loss"]
        kern_avg_ms = kern_ms / max(kern_n, 1)
        achieved = kern_bytes / (kern_avg_ms * 1e-3) / 1e9 if kern_n else None
        step_bytes = sum(ab.values())
        # DRAM bytes of one launch of the dominant kernel from the committed ncu capture (profiles/traffic.json);
        # only valid for the exact configuration it was taken on
        traffic, traffic_src = None, None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(dominant)
            c = tj["config"]
            if (c["batch"], c["height"], c["width"], bool(c["multi_scale"])) == (B, H, W, bool(a.multi_scale)):
                traffic = int(tj["dram_read_bytes"]) + int(tj["dram_write_bytes"])
                traffic_src = tj["source"] + " (dram__bytes_read.sum + dram__bytes_write.sum, 1 launch)"
        except Exception:
            pass
        cfg = config_dict(a, world, step.exchange)
        cfg["step_overlap"] = ("the next step's preprocessing / metric chains start when this step's loss kernel ends, beside its "
                               "second-stage reduction, epilogue and exchange (internal streams, two alternating output sets)" if pipelined else
                               "none across steps; inside a step the preprocessing and metric chains run on two streams beside each other")
        out = {
            "metric": METRIC, "value": world * B * a.steps / (ms_dev * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms_dev / a.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg,
            "roofline": {"bound": "hbm", "kernel": dominant + " (fused loss fwd+bwd, both views)",
                         "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                         "traffic_source": traffic_src,
                         "algorithmic_bytes_per_launch": kern_bytes,
                         "algorithmic_bytes_note": "96 B per pixel-pair: 2x12 pred + 2x12 gt + 2x4 conf + 2x4 thermal read, "
                                                   "2x12 dpred + 2x4 dconf written; the three thermal planes are replicas by "
                                                   "construction, so one is read (SURVEY.md 8d: 96 B with 1-channel thermal, "
                                                   "112 B when all three planes are read)",
                         "avg_launch_ms": kern_avg_ms,
                         "launches_timed": kern_n, "peak_source": peak_src,
                         "step_algorithmic_bytes": step_bytes,
                         "step_frac_of_peak": step_bytes / (ms_dev / a.steps * 1e-3) / 1e9 / peak},
            "e2e": {"value": world * B * a.steps / (ms_e2e * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": HotPathStep.h2d_bytes(host), "d2h_bytes_per_step": 8 * int(step_result_size),
                    "ms_per_step": ms_e2e / a.steps,
                    "h2d_gbs_aggregate": world * HotPathStep.h2d_bytes(host) / (ms_e2e / a.steps * 1e-3) / 1e9},
            "gpu_launches": int(launches),
            "host_numa_bound": bool(numa_bound),
            "clocks": clocks,
            "check": dict({k: summary[k] for k in ("loss", "abs_rel", "acc_1", "n_valid")}, **check_exchange),
        }
        if world == 1 and not a.no_cpu_baseline:
            n_cpu = max(1, min(a.cpu_sample_pairs, B))
            out["cpu_baseline"] = time_cpu(a, n_cpu)
        else:
            out["cpu_baseline"] = None
    del step, host
    torch.cuda.empty_cache()
    # ---------------- extra blocks: the other BASELINE configs, device-timed in the same run
    extra = {}
    if not a.no_extras and not a.multi_scale:
        if world == 1:
            peak, _ = load_peak()
            extra["multi_scale"] = extra_multi_scale(a, dev, d, peak)
            extra["cfg2"] = extra_cfg2(a, dev, peak)
        if world in (1, 8):
            del d
            torch.cuda.empty_cache()
            ev = eval_shard(a, dev, rank, world, local)
            if rank == 0:
                extra["eval"] = ev
    if rank == 0:
        if extra:
            out["extra"] = extra
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


# --------------------------------------------------------------------------- configs[4]: evaluation shard
def eval_shard(a, dev, rank, world, local):
    """frames/s of the evaluation path (BASELINE.json configs[4]): every step = one batch of `--batch` full-res
    640x512 16-bit frames -> preprocessing to the model size + pointmap -> depth -> depth metrics vs 512x512 GT
    depth (nearest resample), accumulated on the device; ONE all-reduce of the accumulator at the end.  The shard
    (`--eval-frames` per rank; 8 ranks x 2 560 = the 20 480 frames of configs[4]) is processed once, timed on the
    device, max over ranks.  Returns the JSON block (rank 0) or None."""
    import torch
    import torch.distributed as dist
    from thermal3d_vision_b200 import _lib
    from thermal3d_vision_b200.pipeline import EvalStep

    B, H, W = a.eval_batch, a.height, a.width
    nb = max(1, a.eval_frames // B)
    step = EvalStep(B, H, W, gt_hw=(512, 512), device=dev)
    g = torch.Generator(device=dev).manual_seed(100 + rank)
    # a pool of distinct synthetic batches (> 1 GB) cycled over the shard: larger than L2, no flush needed
    pool = []
    npool = 4 if B <= 64 else 2
    for k in range(npool):
        d = make_inputs_torch(B, H, W, seed=1000 * rank + k, device=dev)
        gt = 1.5 + 3 * torch.randn(B, 512, 512, device=dev, generator=g).abs()
        pm = d["pred1"].clone()
        pm[..., 2] = torch.nn.functional.interpolate(gt[:, None], size=(H, W), mode="nearest")[:, 0] * \
            (1 + 0.05 * torch.randn(B, H, W, device=dev, generator=g)) * 0.7
        pool.append((d["raw1"], pm, gt))
        del d
    # the sampling kernels of batch k+1 are launched ahead of batch k (EvalStep.prefetch): both inputs of the synthetic
    # shard are known in advance; in a real loop only the raw frames are (see EvalStep.prefetch)
    ahead = os.environ.get("T3D_EVAL_PREFETCH", "1") != "0"

    def run(k, last):
        if ahead:       # also for the last batch: the timed region then holds exactly `nb` samplings and `nb` batches
            step.prefetch(*pool[(k + 1) % npool])
        step.run_batch(*pool[k % npool])

    nw = max(a.warmup, 3)
    if ahead:
        step.prefetch(*pool[0])
    for k in range(nw):
        run(k, False)
    torch.cuda.synchronize()
    step.acc.state.zero_()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(nb):
        run(nw + k, k == nb - 1)
    e1.record()
    res = step.finish()                      # the one all-reduce + host read
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    if rank != 0:
        return None
    peak, _ = load_peak()
    frames = world * nb * B
    ab = step.algorithmic_bytes() * nb
    return {
        "metric": "frames/sec of 640x512 u16 preprocessing + pointmap->depth + metrics (BASELINE configs[4])",
        "value": frames / (ms * 1e-3), "unit": "frames/s", "n_gpus": world, "steps": nb, "warmup": max(a.warmup, 3),
        "ms_per_step": ms / nb, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": f"eval_shard_{nb * B}_frames_per_rank_640x512_u16_to_{W}x{H}+depth_metrics_gt512x512",
                                        "per_rank_frames": nb * B, "global_frames": frames, "batch": B,
                                        "l2_policy": f"inputs_exceed_l2 (pool of {npool} batches of {B} frames, > 1 GB)"},
        "roofline": {"bound": "hbm", "achieved": world * ab / (ms * 1e-3) / 1e9 / world, "peak": peak, "unit": "GB/s",
                     "frac": ab / (ms * 1e-3) / 1e9 / peak, "traffic": None,
                     "note": "per GPU: whole evaluation step (algorithmic bytes of preprocessing + metrics / step time)"},
        "gpu_launches": int(_lib.launch_count() - n0), "check": {k: res[k] for k in ("abs_rel", "rmse", "acc_1")},
    }


def run_eval(a):
    """`--workload eval`: only the evaluation shard (see eval_shard), printed as its own JSON line."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    out = eval_shard(a, dev, rank, world, local)
    if rank == 0:
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    elif a.workload == "eval":
        run_eval(a)
    else:
        run_b200(a)


if __name__ == "__main__":
    main()
