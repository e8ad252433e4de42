"""preprocess_thermal_batch(normalization="fixed_range") -- t3d_preprocess_fixed_range_u16, one kernel that resizes and
applies the Freiburg fixed window -- bit-exact against the reference's recorded outputs and the oracle, its
thermal-gradient statistics against float64 and the loss, and HotPathStep / EvalStep on the fixed window."""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import ref_loss, ref_metrics, ref_preprocess
from test_fixed_range_cpu import SIZES, golden_frames, inference_path_fixed_range, sha, train_path_fixed_range

pytestmark = pytest.mark.gpu

ORACLE = {"train": train_path_fixed_range, "inference": inference_path_fixed_range}
KW = dict(alpha=0.2, edge_weight=0.5, smoothness_weight=0.3, detail_weight=0.4)
PERCENTILE_KERNELS = ("bracket_sample", "resize_march", "percentile_from_brackets", "normalize_stats")


def _pool():
    return ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1))


def fixed(raw, wh, path, **kw):
    from thermal3d_vision_b200 import preprocessing as pp
    return pp.preprocess_thermal_batch(raw, wh, path=path, normalization="fixed_range", **kw)


def oracle_frames(raw, hw, path, channels=3):
    with _pool() as ex:
        return np.stack(list(ex.map(lambda f: ORACLE[path](f, hw)[:channels], raw)))


def assert_frames(got, raw, hw, path, what, channels=3):
    want = oracle_frames(raw, hw, path, channels)
    got = got.cpu().numpy()
    for i in range(len(raw)):
        assert np.array_equal(got[i], want[i]), f"{what}: frame {i}"


def _launched(fn):
    """(fn(), names of every library kernel it launched)."""
    from thermal3d_vision_b200 import _lib
    torch.cuda.synchronize()
    _lib.profile_begin("", 4096)
    out = fn()
    torch.cuda.synchronize()
    names = {n for n, _, _ in _lib.profile_timeline()}
    _lib.profile_end()
    return out, names


@pytest.mark.parametrize("path", ["train", "inference"])
def test_golden_hashes(cuda_device, path):
    """All 12 <tag>_fixed hashes of the live reference, one batch of the four frames per size."""
    g, frames = golden_frames()
    raw = torch.from_numpy(np.stack(list(frames.values()))).to(cuda_device)
    for (w, h) in SIZES:
        tb = fixed(raw, (w, h), path)
        assert tb.percentiles is None and tb.histogram is None
        th = tb.thermal.cpu().numpy()
        for i, name in enumerate(frames):
            assert sha(th[i]) == g[f"{name}_{w}x{h}_fixed"][0 if path == "inference" else 1], f"{name} {w}x{h} {path}"


SHAPES = {   # (src h, w), dst (w, h)
    "h54": ((512, 640), (512, 384)),          # the dataset's geometry: compile-time 5:4 x taps
    "same": ((96, 160), (160, 96)),
    "up": ((50, 60), (100, 84)),
    "small": ((64, 80), (36, 28)),
    "w_mod4": ((512, 640), (333, 217)),       # dst_w % 4 != 0: the scalar kernel
    "w_mod8_4": ((120, 150), (100, 60)),      # dst_w % 8 == 4: half a lane
    "unstaged": ((240, 1500), (24, 20)),      # a band's source rows do not fit shared memory
}


@pytest.mark.parametrize("path", ["train", "inference"])
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("channels", [1, 3])
def test_shapes_bit_equal_oracle(cuda_device, path, shape, channels):
    src, (w, h) = SHAPES[shape]
    raw = ref_preprocess.make_raw_frames(3, seed=11, hw=src)
    tb = fixed(torch.from_numpy(raw).to(cuda_device), (w, h), path, out_channels=channels)
    assert tuple(tb.thermal.shape) == (3, channels, h, w)
    assert_frames(tb.thermal, raw, (h, w), path, f"{shape} {path} c{channels}", channels)


def _adversarial():
    rng = np.random.default_rng(3)
    alt = np.zeros((512, 640), np.uint16)
    alt[:, 1::2] = 65535
    return np.stack([np.zeros((512, 640), np.uint16), np.full((512, 640), 65535, np.uint16),
                     rng.choice(np.array([21799, 21800, 25000, 25001], np.uint16), (512, 640)), alt])


@pytest.mark.parametrize("path", ["train", "inference"])
@pytest.mark.parametrize("wh", [(512, 384), (333, 217), (640, 512)])
def test_adversarial_frames(cuda_device, path, wh):
    raw = _adversarial()
    tb = fixed(torch.from_numpy(raw).to(cuda_device), wh, path)
    assert_frames(tb.thermal, raw, (wh[1], wh[0]), path, f"adversarial {wh} {path}")


@pytest.mark.parametrize("path", ["train", "inference"])
def test_equals_resize_then_drop_in(cuda_device, path):
    """Bit-equal to t3d_resize_bilinear followed by the drop-in enhance_thermal_fixed_range, frame by frame."""
    from thermal3d_vision_b200 import preprocessing as pp
    raw = torch.from_numpy(ref_preprocess.make_raw_frames(3, seed=21)).to(cuda_device)
    for (w, h) in SIZES:
        tb = fixed(raw, (w, h), path)
        for i in range(raw.shape[0]):
            if path == "train":
                r = pp.resize_bilinear(raw[i], (h, w), mode="u16").to(torch.float32)
                want = pp.enhance_thermal_fixed_range(r.unsqueeze(0).repeat(3, 1, 1), normalized=False)
            else:
                r = pp.resize_bilinear(raw[i], (h, w), mode="u16_to_unit_f32")
                want = pp.enhance_thermal_fixed_range(r.unsqueeze(0).repeat(3, 1, 1), normalized=True)
            assert torch.equal(tb.thermal[i], want), f"{w}x{h} {path} frame {i}"


@pytest.mark.parametrize("path", ["train", "inference"])
def test_persistent_grid_past_two_items(cuda_device, path):
    """128 frames of 640x512 -> 512x384: 24 (frame, band) items per frame, at least 2 per CTA of any grid the SMs can
    hold (at most 2048 / 256 CTAs of 256 threads per SM).  Every frame bit-exact, equal to its own B = 1 call, and a
    rerun is bit-identical."""
    B = 128
    sms = torch.cuda.get_device_properties(cuda_device).multi_processor_count
    assert B * 24 >= 2 * sms * (2048 // 256), "the batch no longer gives every CTA two items"
    raw_np = ref_preprocess.make_raw_frames(B, seed=31)
    raw = torch.from_numpy(raw_np).to(cuda_device)
    stats = path == "train"
    a = fixed(raw, (512, 384), path, half_res_stats=True)
    b = fixed(raw, (512, 384), path, half_res_stats=True)
    assert torch.equal(a.thermal, b.thermal)
    if stats:
        assert a.stats_scales == 2 and torch.equal(a.grad_stats, b.grad_stats)
    assert_frames(a.thermal, raw_np, (384, 512), path, f"B=128 {path}")
    for i in range(0, B, 7):
        one = fixed(raw[i:i + 1].clone(), (512, 384), path, half_res_stats=True)
        assert torch.equal(one.thermal[0], a.thermal[i]), f"frame {i}"
        if stats:
            assert torch.equal(one.grad_stats[0], a.grad_stats[i]), f"grad_stats of frame {i}"


def _np_sums(th):
    g = (np.float32(0.299) * th[:, 0] + np.float32(0.587) * th[:, 1]) + np.float32(0.114) * th[:, 2]
    B, h, w = g.shape
    h2, w2 = h // 2, w // 2
    q = g[:, :2 * h2, :2 * w2].reshape(B, h2, 2, w2, 2)
    pooled = (((q[:, :, 0, :, 0] + q[:, :, 0, :, 1]) + q[:, :, 1, :, 0]) + q[:, :, 1, :, 1]) * np.float32(0.25)
    d = lambda a, ax: np.abs(np.diff(a.astype(np.float64), axis=ax)).sum(axis=(1, 2))
    return np.stack([d(g, 2), d(g, 1), d(pooled, 2), d(pooled, 1)], 1)


@pytest.mark.parametrize("wh", [(160, 96), (512, 384)])
@pytest.mark.parametrize("multi", [False, True])
def test_grad_stats_feed_the_loss(cuda_device, wh, multi):
    """The kernel's thermal-gradient sums equal float64 numpy on the produced image (both scales); a loss fed with them
    equals the loss computing its own statistics, and matches the oracle."""
    from thermal3d_vision_b200 import loss as t3d
    (W, H), B = wh, 3
    raw = torch.from_numpy(ref_preprocess.make_raw_frames(2 * B, seed=5)).to(cuda_device)
    tb1 = fixed(raw[:B], wh, "train", half_res_stats=multi)
    tb2 = fixed(raw[B:], wh, "train", half_res_stats=multi)
    scales = min(tb1.stats_scales, tb2.stats_scales)
    assert scales == (2 if multi else 1)
    got = tb1.grad_stats.double().sum(1).cpu().numpy()
    want = _np_sums(tb1.thermal.cpu().numpy())
    np.testing.assert_allclose(got[:, :2], want[:, :2], rtol=1e-5)
    if multi:
        np.testing.assert_allclose(got[:, 2:], want[:, 2:], rtol=1e-5)
    else:
        assert float(tb1.grad_stats[..., 2:].abs().sum()) == 0.0
    P1, P2, G1, G2, C1, C2, _, _ = ref_loss.make_batch_inputs(B, H, W, seed=9)
    d = [x.to(cuda_device) for x in (P1, P2, G1, G2, C1, C2)]
    kw = dict(KW, multi_scale=multi)
    a = t3d.fused_thermal_loss_fwd_bwd(*d, tb1.thermal, tb2.thermal, **kw)
    b = t3d.fused_thermal_loss_fwd_bwd(*d, tb1.thermal, tb2.thermal, thermal_stats=(tb1.grad_stats, tb2.grad_stats),
                                       thermal_stats_scales=scales, thermal_replicated=True, **kw)
    torch.testing.assert_close(a["per_sample"], b["per_sample"], rtol=2e-6, atol=0)
    for k in ("dpred1", "dpred2"):
        torch.testing.assert_close(a[k], b[k], rtol=1e-5, atol=1e-10)
    _, rows, _ = ref_loss.batched_loss_torch(P1, P2, G1, G2, C1, C2, tb1.thermal.cpu(), tb2.thermal.cpu(), **kw)
    np.testing.assert_allclose(b["per_sample"][:, :5].cpu().numpy(), rows, rtol=1e-5)


def test_rejects_bad_arguments(cuda_device):
    from thermal3d_vision_b200 import _lib
    from thermal3d_vision_b200 import preprocessing as pp
    from thermal3d_vision_b200.pipeline import EvalStep, HotPathStep
    raw = torch.from_numpy(ref_preprocess.make_raw_frames(1, seed=1, hw=(64, 80))).to(cuda_device)
    with pytest.raises(ValueError):
        pp.preprocess_thermal_batch(raw, (32, 24), normalization="minmax")
    with pytest.raises(ValueError):
        HotPathStep(2, 64, 96, raw_hw=(128, 160), device=cuda_device, normalization="minmax")
    with pytest.raises(ValueError):
        EvalStep(2, 64, 96, raw_hw=(128, 160), device=cuda_device, normalization="minmax")
    # phase 1 (sampling ahead) has nothing to do on the fixed window
    out = {"thermal": torch.full((1, 3, 24, 32), -1.0, device=cuda_device)}
    tb = fixed(raw, (32, 24), "train", out=out, phase=1)
    assert tb.percentiles is None and bool((tb.thermal == -1.0).all())
    # statistics need the vector path
    th = torch.empty(1, 3, 217, 333, device=cuda_device)
    st = torch.empty(1, 24, 4, device=cuda_device)
    rc = _lib.lib().t3d_preprocess_fixed_range_u16(_lib.ptr(raw), 1, 64, 80, 217, 333, 0, _lib.ptr(th), 3, _lib.ptr(st), 1,
                                                   _lib.current_stream_ptr())
    assert rc != 0


# ---------------------------------------------------------------------------------------------- HotPathStep
STEP_VARIANTS = {      # name -> (HotPathStep options, loss work-item queue of test_persistent_scale_gpu)
    "default": ({}, "march"),
    "multi_scale": (dict(multi_scale=True), "ms"),
    "gt_hw": (dict(gt_hw=(512, 512)), "march"),
    "plain": (dict(use_thermal_aware_loss=False), "basic"),
}


def _run_steps(step, inputs):
    import bench
    for d in inputs:
        step.run_device(*[d[k] for k in bench.KEYS])
    step.finish()


@pytest.mark.parametrize("variant", list(STEP_VARIANTS))
def test_hot_path_step_matches_f64(cuda_device, variant):
    """HotPathStep(normalization="fixed_range") as bench.py runs it (batch 64, 384x512 from 512x640, pipelined), two
    steps: all 128 frames of each bit-exact, rows and gradients against float64 (the bounds of
    test_persistent_scale_gpu), depth metrics bit-equal to the percentile step's on the same inputs, and no kernel of
    the percentile chain launched."""
    import bench
    import test_persistent_scale_gpu as ps
    from thermal3d_vision_b200.pipeline import HotPathStep
    opts, queue = STEP_VARIANTS[variant]
    weights = dict(alpha=bench.ALPHA, edge_weight=bench.EDGE_W, smoothness_weight=bench.SMOOTH_W, detail_weight=bench.DETAIL_W)
    step = HotPathStep(64, 384, 512, device=cuda_device, pipelined=True, normalization="fixed_range", **weights, **opts)
    base = HotPathStep(64, 384, 512, device=cuda_device, pipelined=True, **weights, **opts)
    inputs = [ps._step_inputs(seed, cuda_device, opts.get("gt_hw")) for seed in (0, 1)]
    _, names = _launched(lambda: _run_steps(step, inputs))
    assert "fixed_range_march_kernel" in names, names
    assert not any(k in n for n in names for k in PERCENTILE_KERNELS), names
    _run_steps(base, inputs)
    torch.cuda.synchronize()
    B, H, W = 64, 384, 512
    for i, d in enumerate(inputs):
        what = f"{variant} step {i + 1}"
        lo, res = step.loss_sets[i], step.results[i].cpu().numpy()
        c = {k: v.cpu() for k, v in d.items()}
        raw = torch.cat([c["raw1"], c["raw2"]]).numpy()
        T = oracle_frames(raw, (H, W), "train")
        th = step.pre_sets[i]["thermal"].cpu().numpy()
        for j in range(2 * B):
            assert np.array_equal(th[j], T[j]), f"{what}: thermal frame {j}"
        T = torch.from_numpy(T)
        thermal = opts.get("use_thermal_aware_loss", True)
        G1, G2 = c["gt1"], c["gt2"]
        if "gt_hw" in opts:
            up = lambda G: F.interpolate(G.permute(0, 3, 1, 2), size=(H, W), mode="bilinear",
                                         align_corners=False).permute(0, 2, 3, 1).contiguous()
            G1, G2 = up(G1), up(G2)
        kw = {} if thermal else dict(edge_weight=0.0, smoothness_weight=0.0, detail_weight=0.0)
        refs = ps.f64_refs(c["pred1"], c["pred2"], G1, G2, c["conf1"], c["conf2"], T[:B] if thermal else None,
                           T[B:] if thermal else None, multi_scale=opts.get("multi_scale", False), **kw)
        waves = ps.Waves(lo["workspace"], B, H, W, queue)
        np.testing.assert_allclose(res[0:5], [sum(r[k] for r in refs) for k in ps.ROWS], rtol=1e-5, err_msg=what)
        ps.check_rows(what, lo["per_sample"], refs, range(B))
        ps.check_grads(what, lo, refs, B, waves, range(B))
        assert torch.equal(step.met_sets[i]["metrics_f64"], base.met_sets[i]["metrics_f64"]), f"{what}: metrics"
        assert torch.equal(step.results[i][7:15], base.results[i][7:15]), f"{what}: packed metrics"


def test_hot_path_step_sobel_and_graph(cuda_device):
    """sobel=True: the enhancer reads the fixed-window thermal batch and the loss is unchanged; a captured graph
    replays the step bit for bit."""
    import bench
    import test_persistent_scale_gpu as ps
    from thermal3d_vision_b200 import sobel
    from thermal3d_vision_b200.pipeline import HotPathStep
    d = ps._step_inputs(0, cuda_device, None)
    args = [d[k] for k in bench.KEYS]
    plain = HotPathStep(64, 384, 512, device=cuda_device, normalization="fixed_range")
    r0 = plain.run_device(*args).clone()
    s = HotPathStep(64, 384, 512, device=cuda_device, normalization="fixed_range", sobel=True)
    r1 = s.run_device(*args).clone()
    torch.cuda.synchronize()
    assert torch.equal(r0[:16], r1[:16])
    assert torch.equal(s.pre_both["thermal"], plain.pre_both["thermal"])
    want = sobel.sobel_enhance(s.pre_both["thermal"], 0.5, 1.0)
    torch.testing.assert_close(s.sobel_out["enhanced"], want, rtol=0, atol=0)
    g = HotPathStep(64, 384, 512, device=cuda_device, normalization="fixed_range")
    replay = g.capture_graph(*args)
    g.pre_sets[0]["thermal"].zero_()
    r2 = replay().clone()
    torch.cuda.synchronize()
    assert torch.equal(r2, r0)
    assert torch.equal(g.pre_sets[0]["thermal"], plain.pre_both["thermal"])


def test_hot_path_step_rejects_histogram(cuda_device):
    import bench
    import test_persistent_scale_gpu as ps
    from thermal3d_vision_b200.pipeline import HotPathStep
    d = ps._step_inputs(0, cuda_device, None)
    step = HotPathStep(64, 384, 512, device=cuda_device, normalization="fixed_range")
    step.histogram = True
    with pytest.raises(ValueError):
        step.run_device(*[d[k] for k in bench.KEYS])


# ---------------------------------------------------------------------------------------------- EvalStep
@pytest.mark.parametrize("path", ["train", "inference"])
@pytest.mark.parametrize("prefetch", [False, True])
def test_eval_step(cuda_device, path, prefetch):
    """EvalStep(normalization="fixed_range"): every thermal batch bit-exact, the accumulator bit-equal to the
    percentile EvalStep's on the same batches (the metrics do not depend on the normalisation)."""
    from thermal3d_vision_b200.pipeline import EvalStep
    B, H, W, n = 4, 224, 224, 3
    rng = np.random.default_rng(8)
    raws = [ref_preprocess.make_raw_frames(B, seed=40 + k) for k in range(n)]
    pms = [rng.normal(size=(B, H, W, 3)).astype(np.float32) for _ in range(n)]
    gts = [(1.5 + 3 * np.abs(rng.normal(size=(B, H, W)))).astype(np.float32) for _ in range(n)]
    for p, g in zip(pms, gts):
        p[..., 2] = g * (1 + 0.2 * rng.normal(size=g.shape)).astype(np.float32)
    dev = lambda a: torch.from_numpy(a).to(cuda_device)
    batches = [(dev(r), dev(p), dev(g)) for r, p, g in zip(raws, pms, gts)]

    def run(step):
        outs = []
        for k, (r, p, g) in enumerate(batches):
            if prefetch and k + 1 < n:
                step.prefetch(batches[k + 1][0], batches[k + 1][1], batches[k + 1][2])
            outs.append(step.run_batch(r, p, g).clone())
        torch.cuda.synchronize()
        return outs
    fx = EvalStep(B, H, W, device=cuda_device, path=path, normalization="fixed_range")
    pc = EvalStep(B, H, W, device=cuda_device, path=path)
    outs = run(fx)
    run(pc)
    for k, o in enumerate(outs):
        assert_frames(o, raws[k], (H, W), path, f"eval {path} batch {k}")
    assert torch.equal(fx.acc.state, pc.acc.state)
    per = [ref_metrics.compute_depth_metrics(pms[k][b, ..., 2], gts[k][b]) for k in range(n) for b in range(B)]
    assert fx.acc.state[7].item() == n * B and len(per) == n * B
