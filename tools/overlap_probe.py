"""Developer tool: loss kernel alone, preprocessing alone, metric chain alone, plain step and pipelined step."""
import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import bench
from thermal3d_vision_b200.pipeline import HotPathStep
from thermal3d_vision_b200 import preprocessing as pp, loss as tl, metrics as tm
dev = torch.device("cuda:0")
B, H, W = 64, 384, 512
d = bench.make_inputs_torch(B, H, W, 0, dev)
args = tuple(d[k] for k in bench.KEYS)
kw = dict(alpha=0.2, edge_weight=0.5, smoothness_weight=0.3, detail_weight=0.4, multi_scale=False)
res = {}
raw2 = torch.cat([d["raw1"], d["raw2"]])
tb = pp.preprocess_thermal_batch(raw2, (W, H), histogram=False)
out = {}
def loss_only():
    r = tl.fused_thermal_loss_fwd_bwd(d["pred1"], d["pred2"], d["gt1"], d["gt2"], d["conf1"], d["conf2"], tb.thermal[:B], tb.thermal[B:],
                                      out=out, thermal_stats=(tb.grad_stats[:B], tb.grad_stats[B:]), thermal_replicated=True, **kw)
    out.update(r)
res["loss_only_us"] = bench.time_steps(loss_only, 50, 5) * 1e3
pre_out = {}
def pre_only():
    t = pp.preprocess_thermal_batch(raw2, (W, H), histogram=False, out=pre_out)
    pre_out.update({"thermal": t.thermal, "percentiles": t.percentiles, "grad_stats": t.grad_stats})
res["pre_only_us"] = bench.time_steps(pre_only, 50, 5) * 1e3
met_out = {}
def met_only():
    met_out.update(tm.compute_depth_metrics_batch(d["pred1"], d["gt_depth"], out=met_out))
res["metrics_only_us"] = bench.time_steps(met_only, 50, 5) * 1e3
for pl in (False, True):
    step = HotPathStep(B, H, W, device=dev, pipelined=pl)
    res[f"step_pipelined={pl}_us"] = bench.time_steps(lambda: step.run_device(*args), 100, 5, step.finish) * 1e3
print(json.dumps(res))
