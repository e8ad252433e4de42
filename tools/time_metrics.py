"""Developer tool: depth-metric chain alone (batch 64, 512x384) -- time per call and its kernels."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import bench
from thermal3d_vision_b200 import metrics as tm, _lib
dev = torch.device("cuda:0")
B, H, W = 64, 384, 512
d = bench.make_inputs_torch(B, H, W, 0, dev)
out = {}
r = tm.compute_depth_metrics_batch(d["pred1"], d["gt_depth"], out=out)
out.update(r)
def run(): tm.compute_depth_metrics_batch(d["pred1"], d["gt_depth"], out=out)
flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)
for _ in range(5): run()
torch.cuda.synchronize()
ts = []
for _ in range(20):
    flush.fill_(1.0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); run(); e1.record(); torch.cuda.synchronize()
    ts.append(e0.elapsed_time(e1) * 1e3)
ts.sort()
print(f"metric chain, L2 flushed before each call: median {ts[len(ts)//2]:.1f} us  min {ts[0]:.1f} us")
_lib.profile_begin("", 64)
flush.fill_(1.0)
run(); torch.cuda.synchronize()
for nm, a, b in _lib.profile_timeline(): print(f"  {nm:28s} {(b - a) * 1e3:7.1f} us")
_lib.profile_end()
print(r["metrics_f64"][0].tolist())
