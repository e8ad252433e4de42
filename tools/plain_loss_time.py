"""The plain confidence-weighted loss (no thermal images) on loss_basic_kernel against the tile kernel that ran it
before, and HotPathStep(use_thermal_aware_loss=False) against the thermal-aware step, on one GPU.

Loss call: this library (`new`) against a build of the parent commit (`parent`, --baseline-lib: the tile kernel's
vector variant), the same t3d_loss_fwd_bwd call on the same buffers, alternated call by call.  A 256 MB buffer is
overwritten before every timed call, so no input is served from the 126 MB L2; each call is bracketed by CUDA events
and the median of --iters calls is reported, with the algorithmic bytes (what the loss must read and write) over that
time and its share of the 6.53 TB/s read+write peak measured on this project's B200 (BASELINE.md).  Cases:
  b64_384x512_same        batch 64, GT at the prediction's size, predicted confidence, forward + backward
  b64_384x512_from_512    the same with the GT at 512x512
  b8_224x224_from_512     batch 8, 224x224 <- 512x512
  validation_b64_384x512  no confidence, alpha 0, forward only (validation_batch_loss)
(`kernels_new` names what this library ran: where the dispatch keeps the tile kernel, both builds run it)
Step: B = 64 at 384x512, pipelined, blocks of 10 steps alternated between the two losses.

  python tools/plain_loss_time.py --baseline-lib _ab/libt3d_parent.so --out profiles/plain_loss_time.json
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

PEAK = 6.53e12           # measured HBM read+write peak of this project's B200 (BASELINE.md)
ALPHA = 0.2


def parent_handle(path):
    h = C.CDLL(os.path.abspath(path))
    res, args = _lib._SIGNATURES["t3d_loss_fwd_bwd"]     # the parent's C ABI is the same (version 3)
    h.t3d_loss_fwd_bwd.restype, h.t3d_loss_fwd_bwd.argtypes = res, args
    h.t3d_last_error.restype = C.c_char_p
    h.t3d_version.restype = C.c_int
    assert h.t3d_version() == _lib.ABI_VERSION
    return h


def loss_bytes(B, H, W, gt_hw, conf, bwd):
    """Bytes the loss must move: pred (and d/dpred) 2 x 12 per pixel, the GT source rows the taps touch, the predicted
    confidence (and d/dconf)."""
    n = H * W
    gt = 24 * n if gt_hw is None else 24 * rows_touched(gt_hw[0], H) * gt_hw[1]
    c = 8 * n * (2 if bwd else 1) if conf == "pred" else 0
    return B * (24 * n * (2 if bwd else 1) + gt + c)


def loss_case(name, B, H, W, gt_hw, conf, bwd, dev, parent, iters, flush):
    g = torch.Generator(device=dev).manual_seed(1)
    d = bench.make_inputs_torch(B, H, W, 0, dev)
    gh, gw = gt_hw if gt_hw is not None else (H, W)
    gt = []
    for _ in range(2):
        x = torch.randn(B, gh, gw, 3, device=dev, generator=g)
        x[..., 2] = 1.5 + 3 * x[..., 2].abs()
        gt.append(x)
    cf = [d["conf1"], d["conf2"]] if conf == "pred" else [None, None]
    alpha = ALPHA if conf is not None else 0.0
    f32 = dict(dtype=torch.float32, device=dev)
    flags = tl.LOSS_CONF_MIN_ONLY
    ws = torch.empty(_lib.lib().t3d_loss_workspace_bytes(B, H, W, flags), dtype=torch.uint8, device=dev)
    out = {"per_sample": torch.empty(B, 8, **f32), "batch": torch.empty(8, **f32)}
    if bwd:
        out["dpred1"], out["dpred2"] = torch.empty(B, H, W, 3, **f32), torch.empty(B, H, W, 3, **f32)
        if conf == "pred":
            out["dconf1"], out["dconf2"] = torch.empty(B, H, W, **f32), torch.empty(B, H, W, **f32)
    P = _lib.ptr

    def call(lib):
        rc = lib.t3d_loss_fwd_bwd(
            P(d["pred1"]), P(d["pred2"]), P(gt[0]), P(gt[1]), gh, gw, P(cf[0]), P(cf[1]), H, W, None, None, 0, None, None, 0,
            P(out.get("dpred1")), P(out.get("dpred2")), P(out.get("dconf1")), P(out.get("dconf2")),
            B, H, W, flags, alpha, 0.0, 0.0, 0.0, 1.0 / B, P(out["per_sample"]), P(out["batch"]), None, None,
            P(ws), ws.numel(), _lib.current_stream_ptr())
        assert rc == 0, lib.t3d_last_error()

    variants = {"new": lambda: call(_lib.lib()), "parent": lambda: call(parent)}
    torch.cuda.synchronize()
    _lib.profile_begin("loss_", 64)
    variants["new"]()
    torch.cuda.synchronize()
    kernels = sorted({n for n, _, _ in _lib.profile_timeline(64)})
    _lib.profile_end()
    # the two compute the same loss: the same gradient bits, the per-sample sums to rounding (grouped differently)
    res = {}
    for k, fn in variants.items():
        fn()
        res[k] = {n: t.clone() for n, t in out.items()}
    torch.testing.assert_close(res["new"]["per_sample"], res["parent"]["per_sample"], rtol=2e-6, atol=0)
    grads_equal = all(torch.equal(res["new"][n], res["parent"][n]) for n in out if n.startswith("d"))
    ev = {k: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
          for k in variants}
    for _ in range(5):
        for fn in variants.values():
            fn()
    for it in range(iters):
        for k in (list(variants) if it % 2 == 0 else list(variants)[::-1]):
            flush.fill_(it & 255)
            e0, e1 = ev[k][it]
            e0.record(); variants[k](); e1.record()
    torch.cuda.synchronize()
    nbytes = loss_bytes(B, H, W, gt_hw, conf, bwd)
    rows = {"algorithmic_bytes": nbytes, "peak_us": round(nbytes / PEAK * 1e6, 1), "kernels_new": kernels,
            "gradients_bit_identical": grads_equal}
    for k in variants:
        t = [a.elapsed_time(b) * 1e3 for a, b in ev[k]]
        med = statistics.median(t)
        rows[k] = {"median_us": round(med, 1), "min_us": round(min(t), 1),
                   "achieved_TBps": round(nbytes / med * 1e-6, 3), "share_of_peak": round(nbytes / med * 1e-6 / (PEAK * 1e-12), 3)}
    rows["speedup"] = round(rows["parent"]["median_us"] / rows["new"]["median_us"], 3)
    print(name, json.dumps(rows), flush=True)
    return rows


def step_times(dev, blocks, per_block=10):
    B, H, W = 64, 384, 512
    d = bench.make_inputs_torch(B, H, W, 0, dev)
    keys = ("raw1", "raw2", "pred1", "pred2", "gt1", "gt2", "conf1", "conf2", "gt_depth")
    steps = {"plain": HotPathStep(B, H, W, device=dev, pipelined=True, use_thermal_aware_loss=False),
             "thermal_aware": HotPathStep(B, H, W, device=dev, pipelined=True)}
    t = {k: [] for k in steps}
    for s in steps.values():
        for _ in range(3):
            s.run_device(*[d[x] for x in keys])
        s.finish()
    torch.cuda.synchronize()
    for b in range(blocks):
        for k in (list(steps) if b % 2 == 0 else list(steps)[::-1]):
            s = steps[k]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(per_block):
                s.run_device(*[d[x] for x in keys])
            s.finish()
            e1.record()
            torch.cuda.synchronize()
            t[k].append(e0.elapsed_time(e1) * 1e3 / per_block)
    out = {k: {"median_us": round(statistics.median(v), 1), "min_us": round(min(v), 1),
               "loss_algorithmic_bytes": steps[k].algorithmic_bytes()["loss"]} for k, v in t.items()}
    out["config"] = f"B={B} {W}x{H} pipelined, blocks of {per_block} steps alternated, {blocks} blocks"
    return out


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
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    cases = [("b64_384x512_same", 64, 384, 512, None, "pred", True),
             ("b64_384x512_from_512", 64, 384, 512, (512, 512), "pred", True),
             ("b8_224x224_from_512", 8, 224, 224, (512, 512), "pred", True),
             ("validation_b64_384x512", 64, 384, 512, None, None, False)]
    res = {"device": torch.cuda.get_device_name(dev), "power_limit": power, "peak_Bps": PEAK,
           "l2": "256 MB buffer overwritten before every timed loss call", "iters": a.iters,
           "loss_call": {c[0]: loss_case(*c, dev=dev, parent=parent, iters=a.iters, flush=flush) for c in cases},
           "step": step_times(dev, a.blocks)}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
