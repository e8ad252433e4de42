"""The fixed-window preprocessing (t3d_preprocess_fixed_range_u16, one kernel) against the percentile chain
(t3d_preprocess_train_u16 with hist=NULL), and HotPathStep with each normalisation, on one GPU.

Preprocessing call: 128 frames 640x512 -> 512x384, 3 planes, thermal-gradient statistics on, alternated call by call.
A 256 MB buffer is overwritten before every timed call, so no input is served from the 126 MB L2; each call is bracketed
by CUDA events and the median of --iters calls is reported, with the algorithmic bytes (u16 frame in, 3 fp32 planes
out: 3 014 656 B per frame) over that time and its share of the 6.53 TB/s read+write peak measured on this project's
B200 (BASELINE.md).  Step: B = 64 at 384x512 from 512x640, pipelined, blocks of 10 steps alternated between the two
normalisations, --rounds rounds.

  python tools/fixed_range_time.py --out profiles/fixed_range_time.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import bench  # noqa: E402
from oracle import ref_preprocess  # noqa: E402
from thermal3d_vision_b200 import _lib  # noqa: E402
from thermal3d_vision_b200.pipeline import HotPathStep  # noqa: E402

PEAK = 6.53e12           # measured HBM read+write peak of this project's B200 (BASELINE.md)


def preprocess_calls(dev, iters, flush, B=128, src=(512, 640), dst=(384, 512)):
    lib = _lib.lib()
    (sh, sw), (dh, dw) = src, dst
    raw = torch.from_numpy(ref_preprocess.make_raw_frames(B, seed=0, hw=src)).to(dev)
    f32 = dict(dtype=torch.float32, device=dev)
    out = {k: torch.empty(B, 3, dh, dw, **f32) for k in ("fixed_range", "percentile")}
    stats = {k: torch.empty(B, lib.t3d_preprocess_stats_tiles(dh, dw), 4, **f32) for k in out}
    pct = torch.empty(B, 2, dtype=torch.float64, device=dev)
    ws = torch.empty(lib.t3d_preprocess_workspace_bytes(B, dh, dw), dtype=torch.uint8, device=dev)
    P = _lib.ptr

    def fixed():
        _lib.check(lib.t3d_preprocess_fixed_range_u16(P(raw), B, sh, sw, dh, dw, 0, P(out["fixed_range"]), 3,
                                                      P(stats["fixed_range"]), 1, _lib.current_stream_ptr()))

    def percentile():
        _lib.check(lib.t3d_preprocess_train_u16(P(raw), B, sh, sw, dh, dw, P(out["percentile"]), 3, None, P(pct),
                                                P(stats["percentile"]), 1, 0, P(ws), ws.numel(), 0, _lib.current_stream_ptr()))
    variants = {"fixed_range": fixed, "percentile": percentile}
    torch.cuda.synchronize()
    kernels = {}
    for k, fn in variants.items():
        _lib.profile_begin("", 64)
        fn()
        torch.cuda.synchronize()
        kernels[k] = [n for n, _, _ in _lib.profile_timeline(64)]
        _lib.profile_end()
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
    nbytes = B * (2 * sh * sw + 3 * 4 * dh * dw)
    rows = {"config": f"B={B} {sw}x{sh} -> {dw}x{dh}, 3 planes, grad_stats", "algorithmic_bytes": nbytes,
            "floor_us": round(nbytes / PEAK * 1e6, 1), "kernels": kernels}
    for k in variants:
        t = [a.elapsed_time(b) * 1e3 for a, b in ev[k]]
        med = statistics.median(t)
        rows[k] = {"median_us": round(med, 1), "min_us": round(min(t), 1),
                   "achieved_TBps": round(nbytes / med * 1e-6, 3), "share_of_peak": round(nbytes / med * 1e-6 / (PEAK * 1e-12), 3)}
    print("preprocess", json.dumps(rows), flush=True)
    return rows


def step_times(dev, rounds, blocks, per_block=10):
    B, H, W = 64, 384, 512
    d = bench.make_inputs_torch(B, H, W, 0, dev)
    steps = {k: HotPathStep(B, H, W, device=dev, pipelined=True, normalization=k) for k in ("fixed_range", "percentile")}
    for s in steps.values():
        for _ in range(3):
            s.run_device(*[d[x] for x in bench.KEYS])
        s.finish()
    torch.cuda.synchronize()
    res = []
    for _ in range(rounds):
        t = {k: [] for k in steps}
        for b in range(blocks):
            for k in (list(steps) if b % 2 == 0 else list(steps)[::-1]):
                s = steps[k]
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(per_block):
                    s.run_device(*[d[x] for x in bench.KEYS])
                s.finish()
                e1.record()
                torch.cuda.synchronize()
                t[k].append(e0.elapsed_time(e1) * 1e3 / per_block)
        res.append({k: {"median_us": round(statistics.median(v), 1), "min_us": round(min(v), 1)} for k, v in t.items()})
        print("step", json.dumps(res[-1]), flush=True)
    return {"config": f"B={B} {W}x{H} from 640x512, pipelined, blocks of {per_block} steps alternated, {blocks} blocks per round",
            "rounds": res}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--blocks", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True).stdout.strip()
    except OSError:
        power = "unknown"
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    res = {"device": torch.cuda.get_device_name(dev), "power_limit": power, "peak_Bps": PEAK,
           "l2": "256 MB buffer overwritten before every timed preprocessing call", "iters": a.iters,
           "preprocess_call": preprocess_calls(dev, a.iters, flush),
           "step": step_times(dev, a.rounds, a.blocks)}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
