"""GPU parity: pointmap->depth + depth metrics through the C ABI vs oracle / golden vectors.
Bar: rtol 1e-5 on the float metrics; the delta-accuracies are exact counts / n."""
import os

import numpy as np
import pytest
import torch

from oracle import ref_depth, ref_metrics

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
K7 = ref_metrics.KEYS7


@pytest.fixture(scope="module")
def kat():
    return np.load(os.path.join(G, "metrics_kat.npz"))


def _vec(m):
    return np.array([m[k] for k in K7], np.float64)


def _close(got, ref):
    np.testing.assert_allclose(got[:4], ref[:4], rtol=1e-5)
    np.testing.assert_array_equal(got[4:7], ref[4:7])


@pytest.mark.parametrize("split", ["day", "night"])
def test_reference_golden_real_depth_maps(cuda_device, kat, split):
    from thermal3d_vision_b200 import metrics as tm
    gt, pred = kat[f"{split}_gt"], kat[f"{split}_pred"]
    for ms in (True, False):
        m = tm.compute_depth_metrics(torch.from_numpy(pred).to(cuda_device), gt, median_scaling=ms)
        assert [type(m[k]).__name__ for k in K7] == ["float32"] * 4 + ["float64"] * 3
        _close(_vec(m), kat[f"{split}_crop_ms{int(ms)}"])
        e = tm.compute_depth_metrics_eval(pred, gt, median_scaling=ms)
        ref = kat[f"{split}_crop_eval_ms{int(ms)}"]
        assert e["rmse"] == pytest.approx(ref[0], rel=1e-5) and e["acc_1.25"] == ref[1] and e["acc_1.25^2"] == ref[2]
    m = tm.compute_depth_metrics(pred, gt, mask=kat[f"{split}_mask"])
    _close(_vec(m), kat[f"{split}_crop_masked"])
    # GT at another resolution: fused nearest resample (utils/evaluate_depth_metrics.py:320-323)
    r = tm.compute_depth_metrics_batch(torch.from_numpy(pred)[None], torch.from_numpy(kat[f"{split}_gt_big"])[None])
    _close(r["metrics_f64"][0, :7].cpu().numpy(), kat[f"{split}_crop_resampled"])


def test_empty_mask_and_key_quirk(cuda_device, kat):
    from thermal3d_vision_b200 import metrics as tm
    m = tm.compute_depth_metrics(kat["day_pred"], np.zeros_like(kat["day_gt"]))
    assert set(m) == {"abs_rel", "sq_rel", "rmse", "rmse_log", "a1", "a2", "a3"}
    assert np.isnan(m["abs_rel"]) and m["a1"] == 0.0
    e = tm.compute_depth_metrics_eval(kat["day_pred"], np.zeros_like(kat["day_gt"]))
    assert np.isnan(e["rmse"]) and e["acc_1.25"] == 0.0


@pytest.mark.parametrize("H,W", [(224, 224), (384, 512), (37, 53), (1, 9)])
def test_pointmap_z_in_place_batched(cuda_device, H, W):
    """pointmap -> depth fused into the metric pass (utils/metrics.py:121), odd sizes, B > 1."""
    from thermal3d_vision_b200 import metrics as tm
    rng = np.random.default_rng(H * W)
    B = 3
    gt = (1.5 + 3 * np.abs(rng.normal(size=(B, H, W)))).astype(np.float32)
    pm = rng.normal(size=(B, H, W, 3)).astype(np.float32)
    pm[..., 2] = gt * (1 + 0.3 * rng.normal(size=gt.shape)).astype(np.float32)
    pm[..., 2] = np.abs(pm[..., 2]) + 0.05
    gt[1, : H // 4] = 0
    gt[1, 0, : W // 3] = 0
    gt[2].flat[0] = np.nan
    d = torch.from_numpy(pm).to(cuda_device)
    r = tm.compute_depth_metrics_batch(d, torch.from_numpy(gt))
    got = r["metrics_f64"].cpu().numpy()
    for b in range(B):
        ref = ref_metrics.compute_depth_metrics(ref_depth.pointmap_to_depth(pm[b]), gt[b])
        _close(got[b, :7], _vec(ref))
        exact = ref_metrics.compute_depth_metrics(pm[b, ..., 2], gt[b], dtype=np.float64)
        np.testing.assert_allclose(got[b, :4], _vec(exact)[:4], rtol=2e-5)
    # a strided pointmap[..., 2] view goes through the same in-place path
    m = tm.compute_depth_metrics(d[0][..., 2], gt[0])
    _close(_vec(m), _vec(ref_metrics.compute_depth_metrics(pm[0, ..., 2], gt[0])))
    # medians are exact order statistics
    med = r["medians"].cpu().numpy()
    for b in range(B):
        mk = (gt[b] > 0) & np.isfinite(gt[b])
        assert med[b, 0] == np.median(gt[b][mk]) and med[b, 1] == np.median(pm[b, ..., 2][mk])


def _check_batch(tm, pm_or_depth, gt, cuda_device, **kw):
    d = torch.from_numpy(pm_or_depth).to(cuda_device)
    r = tm.compute_depth_metrics_batch(d, torch.from_numpy(gt).to(cuda_device), **kw)
    got, med = r["metrics_f64"].cpu().numpy(), r["medians"].cpu().numpy()
    z = pm_or_depth[..., 2] if pm_or_depth.ndim == 4 else pm_or_depth
    for b in range(gt.shape[0]):
        ref = ref_metrics.compute_depth_metrics(z[b], gt[b], median_scaling=kw.get("median_scaling", True))
        _close(got[b, :7], _vec(ref))
        mk = (gt[b] > 0) & np.isfinite(gt[b])
        if kw.get("median_scaling", True) and mk.any():
            assert med[b, 0] == np.median(gt[b][mk]) and med[b, 1] == np.median(z[b][mk]), b


@pytest.mark.parametrize("kind", ["walls", "ties", "constant", "two_values", "ramp", "tiny_spread"])
def test_median_candidates_on_clustered_depth(cuda_device, kind):
    """The sampled median brackets and the candidates the extraction kernels collect inside them, on distributions
    that stress them: spatially coherent depth (whole chunks inside the bracket: the CTA stage spills to the image's
    list), heavy ties (every candidate the same key), constant images (the bracket holds everything -> candidate
    overflow -> exact fallback), an even split between two values (the two middle order statistics differ), a ramp,
    a spread of a few ulps.  AoS and planar predictions, with and without median scaling."""
    from thermal3d_vision_b200 import metrics as tm
    rng = np.random.default_rng(11)
    B, H, W = 11, 96, 128                      # B not a multiple of the wave size
    gt = np.empty((B, H, W), np.float32)
    for b in range(B):
        if kind == "walls":                    # piecewise-constant planes + tiny noise, sorted spatially
            levels = np.sort(rng.uniform(1.0, 9.0, 6)).astype(np.float32)
            gt[b] = np.repeat(levels, H * W // 6 + 1)[:H * W].reshape(H, W) + 1e-4 * rng.standard_normal((H, W)).astype(np.float32)
        elif kind == "ties":
            gt[b] = rng.integers(2, 5, (H, W)).astype(np.float32)
        elif kind == "constant":
            gt[b] = 3.25
        elif kind == "two_values":
            gt[b] = np.where(np.arange(H * W).reshape(H, W) % 2 == 0, 2.0, 5.0)
        elif kind == "ramp":
            gt[b] = np.linspace(0.5, 20.0, H * W, dtype=np.float32).reshape(H, W)
        else:
            gt[b] = np.float32(4.0) + np.float32(4.7683716e-07) * rng.integers(0, 6, (H, W)).astype(np.float32)
    gt[1, :5] = 0.0
    gt[2, 3, 7] = np.inf
    pm = rng.standard_normal((B, H, W, 3)).astype(np.float32)
    noise = 0.15          # a noiseless prediction makes every term pure rounding noise, in the reference too
    pm[..., 2] = np.abs(gt * (1.0 + noise * rng.standard_normal(gt.shape)).astype(np.float32)) * np.float32(0.8) + np.float32(0.01)
    pm[..., 2][~np.isfinite(pm[..., 2])] = 1.0
    _check_batch(tm, pm, gt, cuda_device)
    _check_batch(tm, np.ascontiguousarray(pm[..., 2]), gt, cuda_device)                 # planar prediction
    _check_batch(tm, pm, gt, cuda_device, median_scaling=False)


def test_resampled_gt_many_images(cuda_device):
    """GT at another size (nearest resample through the fast kernels' index tables), 19 images, one of them with an
    empty mask; two runs give the same bits."""
    from oracle import ref_preprocess
    from thermal3d_vision_b200 import metrics as tm
    rng = np.random.default_rng(5)
    B, H, W, gh, gw = 19, 48, 64, 80, 72
    big = (1.5 + 3 * np.abs(rng.standard_normal((B, gh, gw)))).astype(np.float32)
    big[3, :9] = 0.0
    big[7] = 0.0                                   # empty mask
    small = np.stack([ref_preprocess.resize_nearest(g, (H, W)) for g in big])
    pm = rng.standard_normal((B, H, W, 3)).astype(np.float32)
    pm[..., 2] = np.abs(small * (1 + 0.2 * rng.standard_normal(small.shape)).astype(np.float32)) + 0.02
    r = tm.compute_depth_metrics_batch(torch.from_numpy(pm).to(cuda_device), torch.from_numpy(big).to(cuda_device))
    got = r["metrics_f64"].cpu().numpy()
    for b in range(B):
        if b == 7:
            assert np.isnan(got[b, :4]).all() and (got[b, 4:8] == 0).all()
            continue
        _close(got[b, :7], _vec(ref_metrics.compute_depth_metrics(pm[b, ..., 2], small[b])))
    # two runs: bit-identical (fixed-order sums, exact selection)
    r2 = tm.compute_depth_metrics_batch(torch.from_numpy(pm).to(cuda_device), torch.from_numpy(big).to(cuda_device))
    assert torch.equal(torch.nan_to_num(r["metrics_f64"]), torch.nan_to_num(r2["metrics_f64"]))


def _misaligned(t):
    """A contiguous copy at element offset 1 of its storage: not 16-byte aligned."""
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    return v


@pytest.mark.parametrize("case", ["aos", "planar", "aos_gt_other_size", "masked", "w_not_mult_4",
                                  "misaligned", "z_view", "w_not_mult_4_gt_other_size"])
def test_extraction_and_sum_kernels_per_input_class(cuda_device, case):
    """choose_metrics_path: which extraction and sum kernels each input class runs (the library's launch names), and
    that the metrics equal the oracle's on each of them."""
    from oracle import ref_preprocess
    from thermal3d_vision_b200 import _lib
    from thermal3d_vision_b200 import metrics as tm
    rng = np.random.default_rng(21)
    B, H, W = 2, 48, 53 if case.startswith("w_not_mult_4") else 64
    gh, gw = (80, 72) if case.endswith("gt_other_size") else (H, W)
    gt = (1.5 + 3 * np.abs(rng.standard_normal((B, gh, gw)))).astype(np.float32)
    gt[0, :5] = 0.0
    gt_small = np.stack([ref_preprocess.resize_nearest(g, (H, W)) for g in gt]) if (gh, gw) != (H, W) else gt
    pm = rng.standard_normal((B, H, W, 3)).astype(np.float32)
    pm[..., 2] = np.abs(gt_small * (1 + 0.2 * rng.standard_normal(gt_small.shape)).astype(np.float32)) + 0.02
    z = np.ascontiguousarray(pm[..., 2])
    mask = ((rng.random((B, H, W)) < 0.7) & (gt_small > 0)) if case == "masked" else None
    d = torch.from_numpy(pm).to(cuda_device)
    pred = {"planar": torch.from_numpy(z).to(cuda_device), "misaligned": _misaligned(torch.from_numpy(z).to(cuda_device)),
            "z_view": d[..., 2]}.get(case, d)
    fast = case in ("aos", "planar", "aos_gt_other_size")
    torch.cuda.synchronize()
    _lib.profile_begin("depth_extract|metrics_sum", 64)
    r = tm.compute_depth_metrics_batch(pred, torch.from_numpy(gt).to(cuda_device),
                                       None if mask is None else torch.from_numpy(mask).to(cuda_device))
    torch.cuda.synchronize()
    names = [n for n, _, _ in _lib.profile_timeline(64)]
    _lib.profile_end()
    assert names == (["depth_extract_fast_kernel", "metrics_sum_fast_kernel"] if fast else
                     ["depth_extract_kernel", "metrics_sum_kernel"]), names
    got = r["metrics_f64"].cpu().numpy()
    for b in range(B):
        _close(got[b, :7], _vec(ref_metrics.compute_depth_metrics(z[b], gt_small[b], mask=None if mask is None else mask[b])))


def test_nan_and_degenerate_predictions(cuda_device):
    from thermal3d_vision_b200 import metrics as tm
    rng = np.random.default_rng(3)
    gt = (1 + rng.random((16, 20))).astype(np.float32)
    pred = gt.copy(); pred[3, 4] = np.nan
    ref = ref_metrics.compute_depth_metrics(pred, gt)
    got = tm.compute_depth_metrics(pred, gt)
    for k in K7:
        assert (np.isnan(ref[k]) and np.isnan(got[k])) or ref[k] == pytest.approx(got[k], rel=1e-5), k
    pred = np.zeros_like(gt)                     # median 0 -> scale inf
    ref = ref_metrics.compute_depth_metrics(pred, gt)
    got = tm.compute_depth_metrics(pred, gt)
    for k in K7:
        assert (np.isnan(ref[k]) and np.isnan(got[k])) or ref[k] == got[k] or ref[k] == pytest.approx(got[k], rel=1e-5), k


def test_depth_and_intrinsics_helpers(cuda_device, kat):
    from thermal3d_vision_b200 import depth as td
    pm = kat["focal_pointmap"]
    z = td.pointmap_to_depth(pm)
    assert isinstance(z, np.ndarray) and (z == pm[..., 2]).all()
    zt = td.pointmap_to_depth(torch.from_numpy(pm).to(cuda_device))
    assert zt.is_cuda and (zt.cpu().numpy() == pm[..., 2]).all()
    K = td.estimate_camera_intrinsics(pm, pm[..., 2])
    np.testing.assert_array_equal(K, kat["focal_K"])
    uv = td.project_points(pm, kat["calib_json_K"]).cpu().numpy()
    u, v = ref_depth.project_points(pm, kat["calib_json_K"])
    np.testing.assert_array_equal(uv[..., 0], u); np.testing.assert_array_equal(uv[..., 1], v)
    with pytest.raises(ValueError):
        td.load_thermal_calibration("calib.txt")


def test_accumulator_matches_reference_semantics(cuda_device, kat):
    from thermal3d_vision_b200 import metrics as tm
    preds = np.stack([kat["day_pred"], kat["night_pred"], kat["day_pred"]])
    gts = np.stack([kat["day_gt"], kat["night_gt"], np.zeros_like(kat["day_gt"])])   # last image: empty mask
    r = tm.compute_depth_metrics_batch(preds, gts)
    acc = tm.MetricAccumulator(cuda_device)
    acc.update(r["metrics_f64"])
    got = acc.result()
    per = [ref_metrics.compute_depth_metrics(preds[i], gts[i]) for i in range(2)]
    per.append({k: np.nan for k in K7})      # what a KeyError-free reference would accumulate (Appendix D.11/12)
    ref = ref_metrics.accumulate_dataset(per)
    for k in K7[:4]:
        assert got[k] == pytest.approx(ref[k], rel=1e-5)


def test_eval_step_config5_shape(cuda_device):
    """BASELINE configs[4] at a reduced frame count: 640x512 u16 frames -> 512x384 model input, pointmap -> depth
    -> metrics against GT depth of another size (nearest resample), dataset accumulator vs the oracle loop."""
    from oracle import ref_preprocess
    from thermal3d_vision_b200.pipeline import EvalStep
    B, H, W, gh, gw = 3, 384, 512, 512, 512
    rng = np.random.default_rng(3)
    raw = ref_preprocess.make_raw_frames(2 * B, seed=31)
    gts = (1.5 + 3 * np.abs(rng.standard_normal((2 * B, gh, gw)))).astype(np.float32)
    gts[1, :40] = 0.0                                     # invalid region
    gts[4] = 0.0                                          # an image with an empty mask (counted, contributes nothing)
    pms = rng.standard_normal((2 * B, H, W, 3)).astype(np.float32)
    step = EvalStep(B, H, W, gt_hw=(gh, gw), device=cuda_device)
    per = []
    for k in range(2):                                    # two batches
        sl = slice(k * B, (k + 1) * B)
        gt_small = np.stack([ref_preprocess.resize_nearest(g, (H, W)) for g in gts[sl]])
        pms[sl, ..., 2] = gt_small * (1.0 + 0.05 * rng.standard_normal((B, H, W))).astype(np.float32) * 0.7
        th = step.run_batch(torch.from_numpy(raw[sl]).to(cuda_device), torch.from_numpy(pms[sl]).to(cuda_device),
                            torch.from_numpy(gts[sl]).to(cuda_device))
        for i in range(B):
            o, _, _, _ = ref_preprocess.train_path(raw[k * B + i], (H, W))
            assert (th[i].cpu().numpy() == o).all()       # the model input is bit-exact
            if (gt_small[i] > 0).any():
                per.append(ref_metrics.compute_depth_metrics(pms[k * B + i, ..., 2], gt_small[i]))
            else:
                per.append({k7: np.nan for k7 in K7})
    got = step.finish()
    ref = ref_metrics.accumulate_dataset(per)
    for k7 in K7:
        assert got[k7] == pytest.approx(ref[k7], rel=1e-5), k7


@pytest.mark.parametrize("what", ["both", "raw_only", "mismatch"])
def test_eval_step_prefetch_gives_the_same_bits(cuda_device, what):
    """EvalStep.prefetch (sampling kernels of batch k+1 launched while batch k is in flight) changes when the kernels
    run, not what they compute: thermal batches and the accumulated metrics equal the plain loop's, also when only the
    raw frames are sampled ahead and when a prefetch is followed by a different batch."""
    from oracle import ref_preprocess
    from thermal3d_vision_b200.pipeline import EvalStep
    B, H, W, gh, gw, nb = 4, 96, 160, 128, 160, 4
    rng = np.random.default_rng(9)
    raws = [torch.from_numpy(ref_preprocess.make_raw_frames(B, seed=40 + k, hw=(120, 200))).to(cuda_device) for k in range(nb)]
    gts = [torch.from_numpy((1.0 + 2 * np.abs(rng.standard_normal((B, gh, gw)))).astype(np.float32)).to(cuda_device) for _ in range(nb)]
    pms = [torch.from_numpy((rng.standard_normal((B, H, W, 3)) + 3).astype(np.float32)).to(cuda_device) for _ in range(nb)]
    plain = EvalStep(B, H, W, raw_hw=(120, 200), gt_hw=(gh, gw), device=cuda_device)
    want_th = [plain.run_batch(raws[k], pms[k], gts[k]).clone() for k in range(nb)]
    want = plain.finish()
    step = EvalStep(B, H, W, raw_hw=(120, 200), gt_hw=(gh, gw), device=cuda_device)
    order = list(range(nb))
    def pf(k):
        if what == "both": step.prefetch(raws[k], pms[k], gts[k])
        elif what == "raw_only": step.prefetch(raws[k])
        else: step.prefetch(raws[(k + 2) % nb], pms[(k + 2) % nb], gts[(k + 2) % nb])     # not the batch that follows
    pf(0)
    for k in order:
        if k + 1 < nb:
            pf(k + 1)
        th = step.run_batch(raws[k], pms[k], gts[k])
        assert torch.equal(th, want_th[k]), k
    got = step.finish()
    for k7 in K7:
        assert got[k7] == want[k7] or (np.isnan(got[k7]) and np.isnan(want[k7])), k7


@pytest.mark.parametrize("conv", ["tuple_dict_batched", "dict_pred1", "tuple_tensor"])
def test_evaluate_thermal_depth_matches_reference_run(cuda_device, conv):
    """evaluate_thermal_depth(model, dataloader, device) (utils/metrics.py:72-138) with a fake model and loader
    (oracle/fake_eval.py) against what the LIVE reference function returned for the same model and data in the build
    container (tests/golden/evaluate_kat.npz, written by oracle/gen_golden.py): every output convention of the
    model the loop accepts, batches without depth skipped, a sample with non-finite metrics skipped but counted."""
    from oracle import fake_eval
    from thermal3d_vision_b200 import metrics as tm
    gold = np.load(os.path.join(G, "evaluate_kat.npz"))
    model = fake_eval.FakeModel(conv).to(cuda_device)
    model.train()
    got = tm.evaluate_thermal_depth(model, fake_eval.make_loader(seed=7), cuda_device)
    assert not model.training and model.calls == int(gold[conv + "_calls"])
    assert list(got) == list(fake_eval.KEYS)
    np.testing.assert_allclose(fake_eval.as_vector(got), gold[conv], rtol=1e-5)
    # nothing to evaluate -> NaNs (sample_count == 0, :134-135)
    empty = tm.evaluate_thermal_depth(model, [{"thermal1": torch.rand(1, 3, 8, 8)}], cuda_device)
    assert all(np.isnan(v) for v in empty.values())
