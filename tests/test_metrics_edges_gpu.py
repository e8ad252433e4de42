"""The depth metrics where their kernels can go wrong without random depths ever noticing, against numpy
(oracle.ref_metrics): pairs whose ratio lies within a few ulps of a delta-threshold, in every exponent band of fp32,
on every sum-kernel class of choose_metrics_path; signs (negative predictions, a negative or zero median prediction);
and EvalStep at the evaluation shard's own batch of 256 frames on both preprocessing paths.

The delta-counts are exact counts: they must equal numpy's.  The four float metrics are compared with the float64
evaluation of the same formulas (rtol 2e-5) where numpy's float32 result is finite and non-zero; where it is not, the
kernels follow numpy's float32 semantics: the same NaN / inf, and 0 where every (gt - pred)^2 underflows."""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

from oracle import ref_metrics, ref_preprocess
from test_metrics_nodiv_cpu import THRESHOLDS, near_threshold_pairs, random_in_band

pytestmark = pytest.mark.gpu
K7 = ref_metrics.KEYS7
F32 = np.float32
FLT_MAX = np.finfo(F32).max

# exponent range [lo, hi) of the smaller value of each pair; the larger is below 2^128 for hi <= 127
BANDS = {"2^-126..2^-120": (-126, -120), "2^-120..2^-100": (-120, -100), "2^-4..2^8": (-4, 8),
         "2^100..2^126": (100, 126), "2^126..FLT_MAX": (126, 127)}
ORDINARY = "2^-4..2^8"

FAST = ["depth_extract_fast_kernel", "metrics_sum_fast_kernel"]
GENERAL = ["depth_extract_kernel", "metrics_sum_kernel"]
# class -> (H, W, GT scale, prediction layout, caller mask, kernels launched)
CLASSES = {
    "fast_aos": (384, 512, 1, "aos", False, FAST),
    "fast_planar": (384, 512, 1, "planar", False, FAST),
    "fast_aos_gt_2x": (384, 512, 2, "aos", False, FAST),            # GT at 2H x 2W, nearest-resampled
    "masked": (384, 512, 1, "aos", True, GENERAL),
    "resampled": (384, 510, 2, "aos", False, GENERAL),              # W % 4 != 0, GT of another size
    "plain": (384, 510, 1, "aos", False, GENERAL),                  # W % 4 != 0: metrics_sum_kernel's 128-bit loop
    "plain_odd_n": (383, 509, 1, "planar", False, GENERAL),         # H * W odd: its scalar loop
    "plain_misaligned": (384, 512, 1, "misaligned", False, GENERAL),
}


def _pool():
    return ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1))


def band_image(rng, lo, hi, n, anchored):
    """(gt, pred), n fp32 pixels in a random order.  Near-threshold pairs of every T in both orientations (gt = a,
    pred = b and gt = b, pred = a), the rest pairs of ordinary ratio in the same band.  anchored: more than half of
    the pixels are (c, c), so that both medians are c and median scaling multiplies by exactly 1 -- also under a mask
    that keeps 90 % of them: 60 % are anchors."""
    n_anchor = 3 * n // 5 if anchored else 0
    m = (n - n_anchor) * 3 // 4 // (2 * 10 * len(THRESHOLDS))          # 10 pairs per b (near_threshold_pairs)
    gt, pred = [], []
    for T in THRESHOLDS:
        a, b = near_threshold_pairs(rng, lo, hi, m, T)
        gt += [a, b]
        pred += [b, a]
    gt, pred = np.concatenate(gt), np.concatenate(pred)
    k = n - n_anchor - gt.size
    fb = random_in_band(rng, lo, hi, k)
    fr = (fb.astype(np.float64) * rng.uniform(0.55, 1.9, k)).astype(F32)
    if hi == 127:                                                      # the largest finite depths
        fb[:2], fr[:2] = (FLT_MAX, F32(0.6) * FLT_MAX), (F32(0.75) * FLT_MAX, FLT_MAX)
    c = random_in_band(rng, lo, hi, 1)
    gt = np.concatenate([gt, fb, np.full(n_anchor, c[0], F32)])
    pred = np.concatenate([pred, fr, np.full(n_anchor, c[0], F32)])
    perm = rng.permutation(n)
    assert np.isfinite(gt).all() and np.isfinite(pred).all() and (gt > 0).all() and (pred > 0).all()
    return gt[perm], pred[perm]


def mixed_groups(gt, pred):
    """A copy with one prediction in every 4-pixel quad -- so in every 8-pixel group of a sum kernel -- replaced by a
    zero, a negative or a subnormal value: those groups take the literal formula."""
    pred = pred.copy()
    q = np.arange(pred.size // 4)
    i = 4 * q + q % 4
    v = pred[i]
    pred[i] = np.where(q % 3 == 0, F32(0), np.where(q % 3 == 1, -v, F32(1e-40)))
    return gt, pred


def threshold_batch(n, anchored, seed):
    """One image per band, and the ordinary band's image with mixed groups: [6, n] gt and pred, and the names."""
    rng = np.random.default_rng(seed)
    imgs = {name: band_image(rng, lo, hi, n, anchored) for name, (lo, hi) in BANDS.items()}
    imgs["mixed groups"] = mixed_groups(*imgs[ORDINARY])
    names = list(imgs)
    return np.stack([imgs[k][0] for k in names]), np.stack([imgs[k][1] for k in names]), names


def _misaligned(t):
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    return v


def run_class(cls, gt, pred, median_scaling, dev):
    """compute_depth_metrics_batch on the input class `cls` for gt, pred [B, H, W] at the prediction's size; asserts
    the kernels choose_metrics_path picked.  -> (metrics_f64 [B, 8], the mask or None)."""
    from thermal3d_vision_b200 import _lib
    from thermal3d_vision_b200 import metrics as tm
    H, W, scale, layout, masked, kernels = CLASSES[cls]
    B = gt.shape[0]
    g = gt
    if scale == 2:                     # each value over a 2x2 block: cv2's nearest rule maps back to gt
        g = np.repeat(np.repeat(gt, 2, axis=1), 2, axis=2)
        assert all(np.array_equal(ref_preprocess.resize_nearest(g[b], (H, W)), gt[b]) for b in range(B))
    if layout == "aos":
        p = np.random.default_rng(1).standard_normal((B, H, W, 3)).astype(F32)
        p[..., 2] = pred
        p = torch.from_numpy(p).to(dev)
    else:
        p = torch.from_numpy(np.ascontiguousarray(pred)).to(dev)
        if layout == "misaligned":
            p = _misaligned(p)
    mask = (np.random.default_rng(2).random(gt.shape) < 0.9) if masked else None
    torch.cuda.synchronize()
    _lib.profile_begin("depth_extract|metrics_sum", 64)
    r = tm.compute_depth_metrics_batch(p, torch.from_numpy(g).to(dev), None if mask is None else torch.from_numpy(mask).to(dev),
                                       median_scaling=median_scaling)
    torch.cuda.synchronize()
    names = [n for n, _, _ in _lib.profile_timeline(64)]
    _lib.profile_end()
    assert names == kernels, (cls, names)
    return r["metrics_f64"].cpu().numpy(), mask


def _same_nonfinite(g, r):
    return (np.isnan(g) and np.isnan(r)) or g == r


def check_image(what, got, gt, pred, mask, median_scaling):
    """-> the ways image `what`'s metrics differ from numpy's (empty when they agree)."""
    ref32 = ref_metrics.compute_depth_metrics(pred, gt, mask=mask, median_scaling=median_scaling)
    ref64 = ref_metrics.compute_depth_metrics(pred, gt, mask=mask, median_scaling=median_scaling, dtype=np.float64)
    bad = []
    if got[4:7].tolist() != [ref32[k] for k in K7[4:]]:
        bad.append(f"{what}: delta-counts {got[4:7].tolist()} vs numpy {[float(ref32[k]) for k in K7[4:]]}")
    for i, k in enumerate(K7[:4]):
        r32, r64, g = float(ref32[k]), float(ref64[k]), float(got[i])
        if not np.isfinite(r32):
            ok = _same_nonfinite(g, r32)
        elif r32 == 0.0:                             # every (gt - pred)^2 underflowed
            ok = g == 0.0
        else:
            ok = abs(g - r64) <= 2e-5 * abs(r64)
        if not ok:
            bad.append(f"{what}: {k} = {g!r}, float64 {r64!r}, numpy float32 {r32!r}")
    return bad


@pytest.mark.parametrize("median_scaling", [False, True])
@pytest.mark.parametrize("cls", list(CLASSES))
def test_threshold_pairs_every_band(cuda_device, cls, median_scaling):
    """Pairs within 3 ulp of fl32(T b), and the pairs closest to a tie, for T = 1.25, 1.5625, 1.953125, in five
    exponent bands from the bottom of the normal range to FLT_MAX; one more image puts a zero, negative or subnormal
    prediction in every 8-pixel group.  median_scaling=True: anchored images, the scale is exactly 1."""
    H, W = CLASSES[cls][:2]
    gt, pred, names = threshold_batch(H * W, median_scaling, seed=7)
    gt, pred = gt.reshape(-1, H, W), pred.reshape(-1, H, W)
    got, mask = run_class(cls, gt, pred, median_scaling, cuda_device)
    with _pool() as ex:
        bad = sum(ex.map(lambda b: check_image(f"{cls}, {names[b]}", got[b], gt[b], pred[b], None if mask is None else mask[b],
                                               median_scaling), range(len(names))), [])
    assert not bad, "\n".join(bad)


def signs_batch(H, W):
    """Ordinary depths; image 0: negative Z in a region, image 1: a negative median prediction (scale < 0), image 2:
    a median prediction of 0 (scale inf), image 3: no sign change."""
    rng = np.random.default_rng(5)
    gt = (1.5 + 3 * np.abs(rng.standard_normal((4, H, W)))).astype(F32)
    pred = (gt * (1 + 0.2 * rng.standard_normal(gt.shape))).astype(F32)
    pred[0, H // 4:H // 2, W // 4:W // 2] *= -1
    pred[1][rng.random((H, W)) < 0.7] *= -1
    pred[2][rng.random((H, W)) < 0.6] = 0
    return gt, pred


@pytest.mark.parametrize("cls", ["fast_aos", "fast_planar", "plain_misaligned"])
def test_signs(cuda_device, cls):
    """numpy counts a negative ratio as inside every threshold and makes rmse_log NaN; a negative scale flips every
    prediction; an infinite one makes 0 * inf = NaN.  Exact counts, numpy's NaN / inf, float32 values to rtol 1e-5."""
    H, W = CLASSES[cls][:2]
    gt, pred = signs_batch(H, W)
    got, _ = run_class(cls, gt, pred, True, cuda_device)
    for b in range(gt.shape[0]):
        ref = ref_metrics.compute_depth_metrics(pred[b], gt[b])
        assert got[b, 4:7].tolist() == [ref[k] for k in K7[4:]], (cls, b, got[b, 4:7])
        for i, k in enumerate(K7[:4]):
            r, g = float(ref[k]), float(got[b, i])
            assert _same_nonfinite(g, r) if not np.isfinite(r) else abs(g - r) <= 1e-5 * abs(r), (cls, b, k, g, r)
    assert np.isnan(got[0, 3]) and np.isnan(got[1, :4]).sum() == 1 and np.isnan(got[2, :4]).all()


# ---------------------------------------------------------------------------------------------- the evaluation shard
def eval_batches(dev, B, H, W, n):
    """n batches built the way bench.eval_shard builds its pool (bench.make_inputs_torch for the raw frames and the
    pointmaps, GT depth at 512 x 512, the pointmaps' Z a noisy 0.7 x nearest-resampled GT); image 5 of every batch
    has an empty mask."""
    import bench
    g = torch.Generator(device=dev).manual_seed(100)
    out = []
    for k in range(n):
        d = bench.make_inputs_torch(B, H, W, seed=k, device=dev)
        gt = 1.5 + 3 * torch.randn(B, 512, 512, device=dev, generator=g).abs()
        pm = d["pred1"].clone()
        pm[..., 2] = torch.nn.functional.interpolate(gt[:, None], size=(H, W), mode="nearest")[:, 0] * \
            (1 + 0.05 * torch.randn(B, H, W, device=dev, generator=g)) * 0.7
        gt[5] = 0.0
        out.append((d["raw1"], pm, gt))
        del d
    return out


@pytest.mark.parametrize("path", ["train", "inference"])
def test_eval_step_at_shard_batch(cuda_device, path):
    """EvalStep(256, 384, 512, gt_hw=(512, 512)) for two batches: path="train" sampling ahead (prefetch) as bench.py
    does, path="inference" with the percentile normalisation.  Every thermal frame bit-exact, every image's metrics
    against numpy on the nearest-resampled GT, finish() against the reference's accumulator."""
    from thermal3d_vision_b200.pipeline import EvalStep
    B, H, W = 256, 384, 512
    batches = eval_batches(cuda_device, B, H, W, 2)
    step = EvalStep(B, H, W, gt_hw=(512, 512), device=cuda_device, path=path)
    outs = []
    if path == "train":
        step.prefetch(*batches[0])
    for k, bt in enumerate(batches):
        if path == "train" and k + 1 < len(batches):
            step.prefetch(*batches[k + 1])
        th = step.run_batch(*bt)
        outs.append((th.clone(), step.met_out["metrics_f64"].clone()))
    got = step.finish()
    oracle = ref_preprocess.train_path if path == "train" else ref_preprocess.inference_path
    per = []
    for k, ((raw, pm, gt), (th, m)) in enumerate(zip(batches, outs)):
        raw, z, gt, th, m = raw.cpu().numpy(), pm[..., 2].cpu().numpy(), gt.cpu().numpy(), th.cpu().numpy(), m.cpu().numpy()
        with _pool() as ex:
            frames = ex.map(lambda i: oracle(raw[i], (H, W))[0], range(B))
            for i, f in enumerate(frames):
                assert np.array_equal(th[i], f), f"{path} batch {k}: thermal frame {i}"
            refs = list(ex.map(lambda i: ref_metrics.compute_depth_metrics(z[i], ref_preprocess.resize_nearest(gt[i], (H, W))),
                               range(B)))
        for i, ref in enumerate(refs):
            if i == 5:
                assert np.isnan(m[i, :4]).all() and (m[i, 4:8] == 0).all(), f"{path} batch {k}: empty image {m[i]}"
                per.append({k7: np.nan for k7 in K7})
                continue
            np.testing.assert_allclose(m[i, :4], [ref[k7] for k7 in K7[:4]], rtol=1e-5, err_msg=f"{path} batch {k}: image {i}")
            assert m[i, 4:7].tolist() == [ref[k7] for k7 in K7[4:]], f"{path} batch {k}: delta-counts of image {i}"
            per.append(ref)
    want = ref_metrics.accumulate_dataset(per)
    assert len(per) == 2 * B and step.acc.state[7].item() == 2 * B
    for k7 in K7:
        assert got[k7] == pytest.approx(want[k7], rel=1e-5), k7
