"""CPU: the oracle restatements equal the LIVE, unmodified reference on fresh random inputs, and the stock
libraries the reference calls (cv2, numpy, scipy).  The reference tree is not part of this repository
(oracle/reference_bridge.py): where it is not mounted, the comparisons with the live reference functions skip and the
golden vectors it wrote (tests/golden/, test_oracle_golden.py) carry the pin; the comparisons with the stock
libraries and with those golden vectors run everywhere."""
import numpy as np
import pytest
import torch

from oracle import ref_loss, ref_metrics, ref_preprocess, ref_sobel, reference_bridge


@pytest.fixture(scope="module")
def ref():
    if not reference_bridge.available():
        pytest.skip("reference tree not mounted")
    return reference_bridge.load()


@pytest.fixture(scope="module")
def live_ref():
    """The loaded reference, or None where it is not mounted."""
    return reference_bridge.load() if reference_bridge.available() else None


@pytest.fixture(scope="module")
def cv2():
    cv2 = pytest.importorskip("cv2")
    cv2.ipp.setUseIPP(False)        # the deterministic C++ paths, as reference_bridge.load() sets them
    return cv2


@pytest.mark.parametrize("H,W,multi", [(33, 47, True), (64, 64, False), (224, 224, True)])
def test_loss_equals_live_reference(ref, H, W, multi):
    kw = dict(alpha=0.2, edge_weight=0.5, smoothness_weight=0.3, detail_weight=0.4, multi_scale=multi)
    ins = ref_loss.make_kat_inputs(H, W, seed=H + W)

    def run(fn):
        a = [x.clone() for x in ins]
        a[4] = a[4] * 3 - 1
        for k in (0, 1, 4, 5):
            a[k].requires_grad_()
        loss, comp = fn(*a, **kw)
        loss.backward()
        return loss.item(), comp, [a[k].grad for k in (0, 1, 4, 5)]

    r, o = run(ref.loss.enhanced_thermal_aware_loss), run(ref_loss.enhanced_thermal_aware_loss_torch)
    # same fp32 op sequence per term; only the order in which the per-view terms are added differs
    assert r[0] == pytest.approx(o[0], rel=2e-6)
    for k in r[1]:
        assert r[1][k] == pytest.approx(o[1][k], rel=2e-6)
    for x, y in zip(r[2], o[2]):
        assert (x - y).abs().max().item() <= 2e-9


def test_preprocess_equals_live_reference(live_ref, cv2):
    raw = ref_preprocess.make_raw_frames(2, seed=11)
    for frame in raw:
        for (w, h) in ((224, 224), (512, 384), (301, 199)):
            assert (cv2.resize(frame, (w, h)) == ref_preprocess.resize_bilinear(frame, (h, w))).all()
            x = frame.astype(np.float32) / 65535.0
            assert (cv2.resize(x, (w, h)) == ref_preprocess.resize_bilinear(x, (h, w))).all()
            if live_ref is not None:
                t = torch.from_numpy(np.repeat(cv2.resize(frame, (w, h)).astype(np.float32)[None], 3, 0))
                assert (live_ref.preprocessing.enhance_thermal_contrast(t).numpy() ==
                        ref_preprocess.train_path(frame, (h, w))[0]).all()


def test_metrics_equal_live_reference(ref):
    rng = np.random.default_rng(0)
    gt = (1.5 + 3 * np.abs(rng.normal(size=(96, 128)))).astype(np.float32)
    pred = (gt * (1 + 0.2 * rng.normal(size=gt.shape))).astype(np.float32)
    gt[:5] = 0
    for ms in (True, False):
        a = ref.metrics.compute_depth_metrics(pred.copy(), gt.copy(), median_scaling=ms)
        b = ref_metrics.compute_depth_metrics(pred, gt, median_scaling=ms)
        assert all(a[k] == b[k] for k in a)


def test_sobel_equals_live_reference(ref):
    m = ref.model.ThermalDUSt3R(torch.nn.Identity())
    x = torch.rand(1, 1, 31, 45)
    assert torch.equal(m.preprocess_thermal(x), ref_sobel.preprocess_thermal_torch(x, m.edge_weight, m.temp_scale))


def test_evaluate_golden_is_the_live_reference(live_ref):
    """tests/golden/evaluate_kat.npz (what the GPU test of evaluate_thermal_depth compares with) is what the live
    reference function returns for the fake model / loader of oracle/fake_eval.py, and equals the oracle's
    accumulate_dataset over per-sample oracle metrics."""
    import os
    from oracle import fake_eval
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "evaluate_kat.npz"))
    for conv in (fake_eval.CONVENTIONS if live_ref is not None else ()):
        model = fake_eval.FakeModel(conv)
        res = live_ref.metrics.evaluate_thermal_depth(model, fake_eval.make_loader(seed=7), torch.device("cpu"))
        np.testing.assert_array_equal(fake_eval.as_vector(res), gold[conv])
    per = []
    model = fake_eval.FakeModel("tuple_tensor")
    for batch in fake_eval.make_loader(seed=7):
        if batch.get("depth1") is None:
            continue
        for i in range(batch["thermal1"].shape[0]):
            view = {"img": batch["thermal1"][i:i + 1], "instance": []}
            pm = model(view, view)[0][0]
            per.append(ref_metrics.compute_depth_metrics(pm[..., 2].numpy(), batch["depth1"][i].numpy()))
    acc = ref_metrics.accumulate_dataset(per)
    np.testing.assert_allclose([acc[k] for k in fake_eval.KEYS], gold["tuple_tensor"], rtol=1e-6)


def test_fire_restatements_equal_live_libraries(live_ref, cv2):
    """oracle/ref_fire.py: the NumPy restatements of cv2 CLAHE / Canny / np.histogram / scipy find_peaks are identical
    to the live libraries, Sobel / bilateral agree to rounding; the three reference functions restated on the stock
    libraries equal the live reference (np.random seeded); tests/golden/fire_kat.npz is what the live reference gives."""
    import importlib, os, sys
    from scipy.signal import find_peaks
    from oracle import ref_fire
    rng = np.random.default_rng(0)
    for (h, w) in ((96, 128), (75, 100), (224, 224)):
        f = ref_fire.make_fire_frame(h, w, seed=h)
        u8 = np.clip(f[0] * 255 + rng.integers(-6, 6, (h, w)), 0, 255).astype(np.uint8)
        for clip in (2.5, 3.0):
            assert np.array_equal(cv2.createCLAHE(clipLimit=clip, tileGridSize=(8, 8)).apply(u8), ref_fire.clahe_u8(u8, clip))
        for lo in (30, 50):
            assert np.array_equal(cv2.Canny(u8, lo, 150), ref_fire.canny_u8(u8, lo, 150))
        assert np.array_equal(np.histogram(f[0].flatten(), bins=100, range=(0, 1))[0], ref_fire.histogram100(f[0]))
        dx, dy = ref_fire.sobel3(f[0])
        assert np.abs(dx - cv2.Sobel(f[0], cv2.CV_32F, 1, 0, ksize=3)).max() < 1e-6
        assert np.abs(dy - cv2.Sobel(f[0], cv2.CV_32F, 0, 1, ksize=3)).max() < 1e-6
        d = (3 + rng.standard_normal((h, w))).astype(np.float32)
        np.testing.assert_allclose(ref_fire.bilateral(d, 5, 50, 50), cv2.bilateralFilter(d, 5, 50, 50), rtol=2e-6, atol=2e-6)
    for _ in range(300):
        hh = rng.integers(0, rng.integers(3, 60), 100)
        assert list(find_peaks(hh, height=hh.max() * 0.3, distance=10)[0]) == list(ref_fire.find_peaks_height_distance(hh, hh.max() * 0.3, 10))
    m = None
    if live_ref is not None:
        sys.path.insert(0, live_ref.root)
        try:
            m = importlib.import_module("thermal_dustr_inference_for_experiment")
        finally:
            sys.path.remove(live_ref.root)
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fire_kat.npz"))
    for (h, w) in ((96, 128), (75, 100)):
        tag = f"{h}x{w}"
        f = ref_fire.make_fire_frame(h, w, seed=h)
        np.random.seed(11); nz = np.random.rand(h, w)
        assert np.array_equal(ref_fire.preprocess_fire_scene_thermal(f, nz), gold["pre_" + tag])
        np.random.seed(12); nz = np.random.rand(h, w)
        assert np.array_equal(ref_fire.advanced_fire_scene_processing(f, nz), gold["adv_" + tag])
        if m is not None:
            np.random.seed(11); live = m.preprocess_fire_scene_thermal(torch.from_numpy(f)).numpy()
            assert np.array_equal(live, gold["pre_" + tag])
            np.random.seed(12); live = m.advanced_fire_scene_processing(torch.from_numpy(f)).numpy()
            assert np.array_equal(live, gold["adv_" + tag])
        assert np.array_equal(ref_fire.depth_refinement(gold["depth_" + tag]), gold["refined_" + tag])
