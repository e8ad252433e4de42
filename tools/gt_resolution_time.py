"""Loss call and step time with the pseudo-GT at its stored resolution (512x512) against predictions at 224x224 and
384x512, on one GPU.

Loss call (fused_thermal_loss_fwd_bwd: statistics pass, main kernel, second stage), three variants alternated
iteration by iteration in the same process:
  rs      this library, GT at 512x512 (where the dispatch takes it, the marching kernel resamples the GT while
          staging it: loss_march_rs_kernel; "kernels" lists what ran)
  parent  a build of the parent commit (--baseline-lib), same call: the tile kernel with fused taps
  same    this library on GT resampled beforehand to the prediction's size (reference: loss_march_kernel)
Each iteration is bracketed by CUDA events; a 256 MB buffer is overwritten between iterations, so no input is
served from the 126 MB L2.  HotPathStep step time: B = 64 at 384x512 with gt_hw=(512, 512) against same-size GT
(alternating blocks of 10 steps), and B = 8 at 224x224 from capture_graph replay as bench.py's second config.

  python tools/gt_resolution_time.py --baseline-lib _ab/libt3d_parent.so --out profiles/gt_resolution_time.json
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import bench  # noqa: E402
from thermal3d_vision_b200 import _lib, loss as tl  # noqa: E402
from thermal3d_vision_b200.pipeline import HotPathStep, rows_touched  # noqa: E402
from thermal3d_vision_b200.training import resample_bilinear  # noqa: E402

PEAK = 6.53e12           # measured HBM read+write peak of this project's B200 (BASELINE.md)
KW = dict(alpha=0.2, edge_weight=0.5, smoothness_weight=0.3, detail_weight=0.4)
GT_HW = (512, 512)


def loss_bytes(B, H, W, gt_hw):
    n = H * W
    gt = 24 * n if gt_hw is None else 24 * rows_touched(gt_hw[0], H) * gt_hw[1]
    return B * (72 * n + gt)


def parent_handle(path):
    h = C.CDLL(os.path.abspath(path))
    res, args = _lib._SIGNATURES["t3d_loss_fwd_bwd"]     # the parent's C ABI is the same (version 3)
    h.t3d_loss_fwd_bwd.restype, h.t3d_loss_fwd_bwd.argtypes = res, args
    h.t3d_last_error.restype = C.c_char_p
    h.t3d_version.restype = C.c_int
    assert h.t3d_version() == _lib.ABI_VERSION
    return h


def loss_case(B, H, W, dev, parent, iters):
    d = bench.make_inputs_torch(B, H, W, 0, dev)
    g = torch.Generator(device=dev).manual_seed(1)
    gt = []
    for _ in range(2):
        x = torch.randn(B, *GT_HW, 3, device=dev, generator=g)
        x[..., 2] = 1.5 + 3 * x[..., 2].abs()
        gt.append(x)
    gs = [resample_bilinear(x, (H, W)) for x in gt]
    th = [torch.rand(B, 1, H, W, device=dev, generator=g).expand(B, 3, H, W).contiguous() for _ in range(2)]
    f32 = dict(dtype=torch.float32, device=dev)
    out = {"workspace": torch.empty(_lib.lib().t3d_loss_workspace_bytes(B, H, W, 0), dtype=torch.uint8, device=dev),
           "per_sample": torch.empty(B, 8, **f32), "batch": torch.empty(8, **f32),
           "dpred1": torch.empty(B, H, W, 3, **f32), "dpred2": torch.empty(B, H, W, 3, **f32),
           "dconf1": torch.empty(B, H, W, **f32), "dconf2": torch.empty(B, H, W, **f32)}
    args = lambda g1, g2: (d["pred1"], d["pred2"], g1, g2, d["conf1"], d["conf2"], th[0], th[1])
    call = lambda g1, g2: tl.fused_thermal_loss_fwd_bwd(*args(g1, g2), out=out, thermal_replicated=True,
                                                        rescale_invalid=False, **KW, multi_scale=False)
    # the parent's library, same call through its C ABI (the same buffers)
    ws = out["workspace"]
    P = _lib.ptr

    def call_parent():
        rc = parent.t3d_loss_fwd_bwd(
            P(d["pred1"]), P(d["pred2"]), P(gt[0]), P(gt[1]), GT_HW[0], GT_HW[1], P(d["conf1"]), P(d["conf2"]), H, W,
            P(th[0]), P(th[1]), 3 | tl.THERMAL_REPLICATED, None, None, 0, P(out["dpred1"]), P(out["dpred2"]),
            P(out["dconf1"]), P(out["dconf2"]), B, H, W, 0, KW["alpha"], KW["edge_weight"], KW["smoothness_weight"],
            KW["detail_weight"], 1.0 / B, P(out["per_sample"]), P(out["batch"]), None, None, P(ws), ws.numel(),
            _lib.current_stream_ptr())
        assert rc == 0, parent.t3d_last_error()

    variants = {"rs": lambda: call(gt[0], gt[1]), "parent": call_parent, "same": lambda: call(gs[0], gs[1])}
    # which kernel each variant runs
    kernels = {}
    for k, fn in variants.items():
        torch.cuda.synchronize()
        _lib.profile_begin("loss_", 64)
        fn()
        torch.cuda.synchronize()
        kernels[k] = sorted({n for n, _, _ in _lib.profile_timeline(64)})
        _lib.profile_end()
    # the three compute the same loss: the tile kernel to rounding, the marching kernel bit for bit with resample-first
    res = {}
    for k, fn in variants.items():
        fn()
        res[k] = (out["per_sample"].clone(), out["dpred1"].clone())
    if "loss_march_rs_kernel" in kernels["rs"]:
        assert torch.equal(res["rs"][0], res["same"][0]) and torch.equal(res["rs"][1], res["same"][1])
    torch.testing.assert_close(res["rs"][0], res["same"][0], rtol=2e-6, atol=1e-7)
    torch.testing.assert_close(res["rs"][0], res["parent"][0], rtol=2e-6, atol=1e-7)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ev = {k: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
          for k in variants}
    for _ in range(5):
        for fn in variants.values():
            fn()
    for it in range(iters):
        order = list(variants)[it % 3:] + list(variants)[:it % 3]
        for k in order:
            flush.fill_(it & 255)
            e0, e1 = ev[k][it]
            e0.record(); variants[k](); e1.record()
    torch.cuda.synchronize()
    rows = {}
    for k in variants:
        t = [a.elapsed_time(b) * 1e3 for a, b in ev[k]]
        nbytes = loss_bytes(B, H, W, None if k == "same" else GT_HW)
        med = statistics.median(t)
        rows[k] = {"median_us": round(med, 1), "mean_us": round(statistics.mean(t), 1), "min_us": round(min(t), 1),
                   "algorithmic_bytes": nbytes, "achieved_TBps": round(nbytes / med * 1e-6, 3),
                   "share_of_peak": round(nbytes / med * 1e-6 / (PEAK * 1e-12), 3)}
        if k != "parent":           # (the parent library's own launches are not visible to this library's profiler)
            rows[k]["kernels"] = kernels[k]
    return rows


def step_times(dev, blocks):
    out = {}
    # B = 64 at 384x512: run_device, gt_hw=(512, 512) against same-size GT
    B, H, W = 64, 384, 512
    d = bench.make_inputs_torch(B, H, W, 0, dev)
    g = torch.Generator(device=dev).manual_seed(2)
    big = dict(d, gt1=torch.randn(B, *GT_HW, 3, device=dev, generator=g), gt2=torch.randn(B, *GT_HW, 3, device=dev, generator=g))
    keys = ("raw1", "raw2", "pred1", "pred2", "gt1", "gt2", "conf1", "conf2", "gt_depth")
    steps = {"gt_hw": (HotPathStep(B, H, W, device=dev, gt_hw=GT_HW), big), "same": (HotPathStep(B, H, W, device=dev), d)}
    out["b64_384x512"] = _time_alternating({k: (lambda s=s, a=a: s.run_device(*[a[x] for x in keys])) for k, (s, a) in steps.items()},
                                           blocks, 10)
    for k, (s, _) in steps.items():
        out["b64_384x512"][k]["loss_algorithmic_bytes"] = s.algorithmic_bytes()["loss"]
    # B = 8 at 224x224: CUDA-graph replay (bench.py configs[1])
    B, H, W = 8, 224, 224
    d = bench.make_inputs_torch(B, H, W, 0, dev)
    big = dict(d, gt1=torch.randn(B, *GT_HW, 3, device=dev, generator=g), gt2=torch.randn(B, *GT_HW, 3, device=dev, generator=g))
    reps = {"gt_hw": HotPathStep(B, H, W, device=dev, gt_hw=GT_HW).capture_graph(*[big[x] for x in keys]),
            "same": HotPathStep(B, H, W, device=dev).capture_graph(*[d[x] for x in keys])}
    out["b8_224x224_graph"] = _time_alternating(reps, blocks, 50)
    return out


def _time_alternating(fns, blocks, per_block):
    t = {k: [] for k in fns}
    for fn in fns.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    for b in range(blocks):
        for k in (list(fns) if b % 2 == 0 else list(fns)[::-1]):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(per_block):
                fns[k]()
            e1.record()
            torch.cuda.synchronize()
            t[k].append(e0.elapsed_time(e1) * 1e3 / per_block)
    return {k: {"median_us": round(statistics.median(v), 1), "min_us": round(min(v), 1)} for k, v in t.items()}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--baseline-lib", required=True, help="libt3d_sm100.so built from the parent commit")
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--blocks", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    parent = parent_handle(a.baseline_lib)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True).stdout.strip()
    except OSError:
        power = "unknown"
    res = {"device": torch.cuda.get_device_name(dev), "power_limit": power, "peak_Bps": PEAK,
           "l2": "256 MB buffer overwritten between timed loss calls", "iters": a.iters,
           "loss_call": {f"b{B}_{H}x{W}_from_512x512": loss_case(B, H, W, dev, parent, a.iters)
                         for B, H, W in ((8, 224, 224), (64, 384, 512))},
           "step": step_times(dev, a.blocks)}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
