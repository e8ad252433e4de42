"""The plain confidence-weighted loss (no thermal images: train_thermal_dustr.py:305-318, the validation loss,
confidence_weighted_regression_loss) on its streaming kernel, loss_basic_kernel: the same gradient bits as the tile
kernel, reference parity, downsampled GT (bit-identical to resampling first), edge values, determinism and batch
independence, and HotPathStep(use_thermal_aware_loss=False)."""
import pytest
import torch
import torch.nn.functional as F

from oracle import ref_loss

pytestmark = pytest.mark.gpu
OUTS = ("per_sample", "batch", "dpred1", "dpred2", "dconf1", "dconf2")
GRADS = ("dpred1", "dpred2", "dconf1", "dconf2")
SHAPES = [(384, 512), (40, 132), (97, 260), (3, 8), (1, 4)]


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _gt(B, GH, GW, g):
    G = torch.randn(B, GH, GW, 3, generator=g)
    G[..., 2] = 1.5 + 3 * G[..., 2].abs()
    return G


def _case(B, H, W, seed, dev, GH=None, GW=None):
    """pred / conf at (H, W), gt at (GH, GW) (default: the prediction's size); confidences between 0.5 and 20, so both
    clamps of the reference's confidence act."""
    GH, GW = GH or H, GW or W
    g = torch.Generator().manual_seed(seed)
    G1, G2 = _gt(B, GH, GW, g), _gt(B, GH, GW, g)
    up = lambda G: F.interpolate(G.permute(0, 3, 1, 2), size=(H, W), mode="bilinear", align_corners=False).permute(0, 2, 3, 1)
    P1 = up(G1) + 0.1 * torch.randn(B, H, W, 3, generator=g)
    P2 = up(G2) + 0.1 * torch.randn(B, H, W, 3, generator=g)
    C1, C2 = 0.5 + 19.5 * torch.rand(B, H, W, generator=g), 0.5 + 19.5 * torch.rand(B, H, W, generator=g)
    return [t.contiguous().to(dev) for t in (P1, P2, G1, G2, C1, C2)]


def _misaligned(t):
    """A contiguous copy at element offset 1 of its storage: not 16-byte aligned, so the call takes the tile kernel."""
    if t is None:
        return None
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    return v


def _fb(P1, P2, G1, G2, C1, C2, **kw):
    from thermal3d_vision_b200 import loss as t3d
    return t3d.fused_thermal_loss_fwd_bwd(P1, P2, G1, G2, C1, C2, None, None, multi_scale=False, **kw)


def _fwd(P1, P2, G1, G2, C1, C2, conf_min_only=False, alpha=0.2):
    """Forward only (detached inputs: no gradient buffers)."""
    from thermal3d_vision_b200 import loss as t3d
    r = t3d.fused_thermal_loss(P1, P2, G1, G2, C1, C2, None, None, alpha=alpha, multi_scale=False,
                               conf_min_only=conf_min_only)
    return {"per_sample": r.per_sample, "batch": r.batch, "dpred1": None, "dpred2": None, "dconf1": None, "dconf2": None}


def _launched(fn):
    """(fn(), names of the library's loss kernels it launched)."""
    from thermal3d_vision_b200 import _lib
    torch.cuda.synchronize()
    _lib.profile_begin("loss_", 512)
    out = fn()
    torch.cuda.synchronize()
    names = {n for n, _, _ in _lib.profile_timeline(512)}
    _lib.profile_end()
    return out, names


def _basic_ran(names):
    assert "loss_basic_kernel" in names and "loss_tile_kernel" not in names, names


def _assert_same(a, b, nan=False):
    for k in OUTS:
        if a[k] is None or b[k] is None:
            assert a[k] is None and b[k] is None, k
        elif nan:
            torch.testing.assert_close(a[k], b[k], rtol=0, atol=0, equal_nan=True, msg=k)
        else:
            assert torch.equal(a[k], b[k]), k


# ---------------------------------------------------------------------------------------- against the tile kernel
@pytest.mark.parametrize("bwd", [True, False], ids=["fwd_bwd", "fwd"])
@pytest.mark.parametrize("conf_min_only", [True, False], ids=["min_only", "clamp10"])
@pytest.mark.parametrize("conf", ["pred", "none"])
@pytest.mark.parametrize("H,W", SHAPES)
def test_same_gradients_as_tile_kernel(dev, H, W, conf, conf_min_only, bwd):
    B = 2
    args = _case(B, H, W, seed=H * 7 + W, dev=dev)
    if conf == "none":
        args[4] = args[5] = None
    call = (lambda *a: _fb(*a, conf_min_only=conf_min_only)) if bwd else (lambda *a: _fwd(*a, conf_min_only=conf_min_only))
    got, names = _launched(lambda: call(*args))
    _basic_ran(names)
    ref, names = _launched(lambda: call(*[_misaligned(t) for t in args]))
    assert "loss_tile_kernel" in names and "loss_basic_kernel" not in names, names
    for k in GRADS:
        if got[k] is None or ref[k] is None:
            assert got[k] is None and ref[k] is None, k
        else:
            assert torch.equal(got[k], ref[k]), k
    torch.testing.assert_close(got["per_sample"][:, :2], ref["per_sample"][:, :2], rtol=2e-6, atol=0)
    assert torch.equal(got["per_sample"][:, 2:], ref["per_sample"][:, 2:])


# ---------------------------------------------------------------------------------------- reference parity
@pytest.mark.parametrize("H,W", [(40, 132), (97, 260)])
def test_matches_oracle(dev, H, W):
    """ref_loss.plain_confidence_loss_torch per sample, mean over the (valid) samples, autograd for the gradients:
    loss rtol 1e-5, gradients rtol 1e-4 / atol 1e-6 and, against the float64 closed form, within 1e-5 of the largest
    gradient magnitude (DESIGN §2)."""
    B, alpha = 3, 0.2
    args = _case(B, H, W, seed=H, dev=dev)
    res, names = _launched(lambda: _fb(*args, conf_min_only=True, alpha=alpha))
    _basic_ran(names)
    for dtype in (torch.float32, torch.float64):
        leaves = [t.cpu().to(dtype).requires_grad_() for t in (args[0], args[1], args[4], args[5])]
        p1, p2, c1, c2 = leaves
        g1, g2 = args[2].cpu().to(dtype), args[3].cpu().to(dtype)
        tot = 0.0
        for i in range(B):
            loss = ref_loss.plain_confidence_loss_torch(p1[i], p2[i], g1[i], g2[i], c1[i], c2[i], alpha=alpha)
            if dtype == torch.float32:
                assert res["per_sample"][i, 0].item() == pytest.approx(loss.item(), rel=1e-5)
                assert res["per_sample"][i, 1].item() == res["per_sample"][i, 0].item()
            tot = tot + loss
        (tot / B).backward()
        for got, leaf in zip((res["dpred1"], res["dpred2"], res["dconf1"], res["dconf2"]), leaves):
            got = got.cpu()
            if dtype == torch.float32:
                torch.testing.assert_close(got, leaf.grad, rtol=1e-4, atol=1e-6)
            else:
                err = (got.double() - leaf.grad).abs().max().item()
                assert err <= 1e-5 * leaf.grad.abs().max().item(), err
    assert torch.equal(res["per_sample"][:, 2:5], torch.zeros_like(res["per_sample"][:, 2:5]))


# ---------------------------------------------------------------------------------------- resampled GT
# (H, W, GH, GW, confidence at the GT's size, the kernel the dispatch takes)
GEOMS = [(384, 512, 512, 512, False, "loss_basic_kernel"),
         (40, 132, 64, 132, False, "loss_basic_kernel"),
         (97, 260, 128, 264, False, "loss_basic_kernel"),
         (224, 224, 512, 512, False, "loss_tile_kernel"),     # wide source segments: measured faster on the tile kernel
         (64, 96, 32, 48, False, "loss_tile_kernel"),         # upsampled
         (384, 512, 512, 512, True, "loss_tile_kernel")]      # pseudo-GT confidence at the GT's size


@pytest.mark.parametrize("bwd", [True, False], ids=["fwd_bwd", "fwd"])
@pytest.mark.parametrize("H,W,GH,GW,gt_conf,kernel", GEOMS)
def test_resampled_gt(dev, H, W, GH, GW, gt_conf, kernel, bwd):
    """A downsampled GT on loss_basic_kernel: bit for bit resample_bilinear + the same-size call.  Wide source segments
    (224x224 <- 512x512), an upsampled GT or a GT-sized confidence stay on the tile kernel's fused taps and agree to
    rounding."""
    from thermal3d_vision_b200.training import resample_bilinear
    B = 2
    P1, P2, G1, G2, C1, C2 = _case(B, H, W, seed=GH + W, dev=dev, GH=GH, GW=GW)
    rs = lambda t: resample_bilinear(t, (H, W))
    kw = dict(conf_min_only=True)
    if gt_conf:
        g = torch.Generator().manual_seed(9)
        C1, C2 = [(0.5 + 19.5 * torch.rand(B, GH, GW, generator=g)).to(dev) for _ in range(2)]
        kw["conf_grad"] = False
    call = (lambda *x: _fb(*x, **kw)) if bwd else (lambda *x: _fwd(*x, conf_min_only=True))
    fused, names = _launched(lambda: call(P1, P2, G1, G2, C1, C2))
    other = "loss_tile_kernel" if kernel == "loss_basic_kernel" else "loss_basic_kernel"
    assert kernel in names and other not in names, names
    two, names = _launched(lambda: call(P1, P2, rs(G1), rs(G2), rs(C1) if gt_conf else C1, rs(C2) if gt_conf else C2))
    _basic_ran(names)
    if kernel == "loss_basic_kernel":
        _assert_same(fused, two)
        return
    torch.testing.assert_close(fused["per_sample"][:, :5], two["per_sample"][:, :5], rtol=2e-6, atol=1e-7)
    for k in GRADS:
        if fused[k] is None or two[k] is None:
            assert fused[k] is None and two[k] is None, k
        else:
            torch.testing.assert_close(fused[k], two[k], rtol=1e-4, atol=1e-7)


def test_resampled_gt_persistent_grid_reuse(dev):
    """B = 16 at 384x512 <- 512x512: more work items than resident warps, so warps take several items each."""
    from thermal3d_vision_b200.training import resample_bilinear
    B, H, W = 16, 384, 512
    P1, P2, G1, G2, C1, C2 = _case(B, H, W, seed=16, dev=dev, GH=512, GW=512)
    fused, names = _launched(lambda: _fb(P1, P2, G1, G2, C1, C2, conf_min_only=True))
    _basic_ran(names)
    _assert_same(fused, _fb(P1, P2, resample_bilinear(G1, (H, W)), resample_bilinear(G2, (H, W)), C1, C2, conf_min_only=True))


def test_non_finite_gt_at_zero_weight_taps(dev):
    """gh = 3 H: f = 3 y + 1 exactly, so source rows 3 y + 2 are read only by zero-weight taps.  ATen (and the
    resample-first path) turn 0 * Inf into NaN; so does the fused call."""
    from thermal3d_vision_b200.training import resample_bilinear
    B, H, W, GH, GW = 2, 40, 128, 120, 128
    P1, P2, G1, G2, C1, C2 = _case(B, H, W, seed=3, dev=dev, GH=GH, GW=GW)
    G1 = G1.clone()
    G1[0, 3 * 5 + 2, 17, 2] = float("inf")
    G1[0, 3 * 11 + 2, 64, 0] = float("nan")
    G2 = G2.clone()
    G2[1, 3 * 20 + 2, 127, 1] = float("-inf")
    fused, names = _launched(lambda: _fb(P1, P2, G1, G2, C1, C2, rescale_invalid=False))
    _basic_ran(names)
    two = _fb(P1, P2, resample_bilinear(G1, (H, W)), resample_bilinear(G2, (H, W)), C1, C2, rescale_invalid=False)
    _assert_same(fused, two, nan=True)
    assert torch.isnan(fused["per_sample"][:, 0]).all()


# ---------------------------------------------------------------------------------------- forward only
def test_forward_only_rows_equal_fwd_bwd_rows(dev):
    B, H, W = 3, 97, 260
    args = _case(B, H, W, seed=21, dev=dev)
    for cmo in (True, False):
        fb = _fb(*args, conf_min_only=cmo)
        fo, names = _launched(lambda: _fwd(*args, conf_min_only=cmo))
        _basic_ran(names)
        assert torch.equal(fo["per_sample"], fb["per_sample"])
    # the validation loss (no confidence, alpha 0, forward only) runs on the new kernel too
    from thermal3d_vision_b200.training import validation_batch_loss
    r, names = _launched(lambda: validation_batch_loss(args[0], args[1], args[2], args[3]))
    _basic_ran(names)
    ref = torch.stack([((args[0][i] - args[2][i]).abs().mean() + (args[1][i] - args[3][i]).abs().mean()) / 2
                       for i in range(B)]).mean()
    assert r.loss.item() == pytest.approx(ref.item(), rel=1e-5)


# ---------------------------------------------------------------------------------------- edge values
def test_large_confidences_unclamped_with_conf_min_only(dev):
    B, H, W = 2, 40, 132
    P1, P2, G1, G2, C1, C2 = _case(B, H, W, seed=5, dev=dev)
    C1 = C1.clone()
    C1[:, ::3] = 37.5
    res, names = _launched(lambda: _fb(P1, P2, G1, G2, C1, C2, conf_min_only=True))
    _basic_ran(names)
    for i in range(B):
        want = ref_loss.plain_confidence_loss_torch(P1[i].cpu(), P2[i].cpu(), G1[i].cpu(), G2[i].cpu(), C1[i].cpu(), C2[i].cpu())
        assert res["per_sample"][i, 0].item() == pytest.approx(want.item(), rel=1e-5)
    assert (res["dconf1"][:, ::3] != 0).all()
    clamped = _fb(P1, P2, G1, G2, C1, C2, conf_min_only=False)
    assert (clamped["dconf1"][:, ::3] == 0).all()          # above 10: outside the clamp, no gradient


@pytest.mark.parametrize("conf_min_only", [True, False])
def test_values_at_the_clamp_bounds_keep_their_gradient(dev, conf_min_only):
    B, H, W = 2, 8, 128
    args = _case(B, H, W, seed=6, dev=dev)
    C1 = args[4].clone()
    C1[:, 0] = 1e-5
    C1[:, 1] = 10.0
    C1[:, 2] = 5e-6                                         # below the lower bound: clamped, no gradient
    args[4] = C1
    got = _fb(*args, conf_min_only=conf_min_only)
    ref = _fb(*[_misaligned(t) for t in args], conf_min_only=conf_min_only)
    for k in GRADS:
        assert torch.equal(got[k], ref[k]), k
    assert (got["dconf1"][:, :2] != 0).all()
    assert (got["dconf1"][:, 2] == 0).all()


def test_nan_invalidates_only_its_sample(dev):
    B, H, W = 3, 40, 132
    args = _case(B, H, W, seed=8, dev=dev)
    clean = _fb(*args, conf_min_only=True)
    P1 = args[0].clone()
    P1[1, 5, 7, 0] = float("nan")
    res = _fb(P1, *args[1:], conf_min_only=True)
    assert res["per_sample"][:, 5].tolist() == [1.0, 0.0, 1.0]
    assert res["batch"][5].item() == 2.0
    assert torch.equal(res["per_sample"][[0, 2]], clean["per_sample"][[0, 2]])
    for k in GRADS:
        assert (res[k][1] == 0).all(), k
        # the valid samples' gradients are those of the mean over 2 samples: x 3/2 of the mean over 3
        torch.testing.assert_close(res[k][[0, 2]], clean[k][[0, 2]] * 1.5, rtol=1e-6, atol=0)


# ---------------------------------------------------------------------------------------- determinism, batch independence
def test_deterministic_and_batch_independent(dev):
    B, H, W = 4, 97, 260
    args = _case(B, H, W, seed=10, dev=dev)
    a, b = _fb(*args, conf_min_only=True), _fb(*args, conf_min_only=True)
    _assert_same(a, b)
    perm = [2, 0, 3, 1]
    c = _fb(*[t[perm].contiguous() for t in args], conf_min_only=True)
    assert torch.equal(c["per_sample"], a["per_sample"][perm])
    for k in GRADS:
        assert torch.equal(c[k], a[k][perm]), k


def test_large_batch_equals_single_samples(dev):
    """B = 64 at 384x512: 9 216 work items (18 bands x 4 strips x 128 image-views), more than the resident warps -- each sample's row equals its B = 1 call."""
    B, H, W = 64, 384, 512
    args = _case(B, H, W, seed=11, dev=dev)
    big, names = _launched(lambda: _fb(*args, conf_min_only=True))
    _basic_ran(names)
    for i in range(B):
        one = _fb(*[t[i:i + 1] for t in args], conf_min_only=True)
        assert torch.equal(one["per_sample"][0], big["per_sample"][i]), i


# ---------------------------------------------------------------------------------------- HotPathStep
STEP_CASES = [(4, 384, 512, None), (4, 384, 512, (512, 512)), (8, 224, 224, None), (8, 224, 224, (512, 512))]
ARGS = ("raw1", "raw2", "pred1", "pred2", "gt1", "gt2", "conf1", "conf2", "gt_depth")
KW = dict(alpha=0.2, edge_weight=0.5, smoothness_weight=0.3, detail_weight=0.4)


def _step_inputs(B, H, W, seed, dev, gt_hw):
    import bench
    d = bench.make_inputs_torch(B, H, W, seed, dev, raw_hw=(512, 640))
    if gt_hw is not None:
        g = torch.Generator().manual_seed(seed + 100)
        d["gt1"], d["gt2"] = _gt(B, *gt_hw, g).to(dev), _gt(B, *gt_hw, g).to(dev)
    return d


def _snap(step, r):
    return r.clone(), {k: step.loss_out[k].clone() for k in GRADS}


def _same_step(a, b):
    assert torch.equal(a[0], b[0])
    for k in GRADS:
        assert torch.equal(a[1][k], b[1][k]), k


@pytest.mark.parametrize("B,H,W,gt_hw", STEP_CASES)
def test_step_plain_loss(dev, B, H, W, gt_hw):
    from thermal3d_vision_b200 import loss as t3d
    from thermal3d_vision_b200 import preprocessing as pp
    from thermal3d_vision_b200.pipeline import HotPathStep
    d = _step_inputs(B, H, W, 1, dev, gt_hw)
    step = HotPathStep(B, H, W, device=dev, gt_hw=gt_hw, use_thermal_aware_loss=False, **KW)
    r, names = _launched(lambda: step.run_device(*[d[k] for k in ARGS]))
    if gt_hw is not None and W == 224:          # 224x224 <- 512x512: the tile kernel's fused taps
        assert "loss_tile_kernel" in names and "loss_basic_kernel" not in names, names
    else:
        _basic_ran(names)
    got = _snap(step, r)
    rc = r.cpu()

    # the composition: preprocessing (the model's input, no statistics) + the plain loss + the validity fix-up
    raw_both = torch.cat([d["raw1"], d["raw2"]])
    tb = pp.preprocess_thermal_batch(raw_both, (W, H), path="train", histogram=False, grad_stats=False)
    assert tb.grad_stats is None
    assert torch.equal(tb.thermal, step.pre_both["thermal"])
    ref = t3d.fused_thermal_loss_fwd_bwd(d["pred1"], d["pred2"], d["gt1"], d["gt2"], d["conf1"], d["conf2"], None, None,
                                         conf_min_only=True, alpha=KW["alpha"], multi_scale=False)
    ps = ref["per_sample"].double().cpu()
    valid = ps[:, 5] != 0
    assert rc[5].item() == valid.sum().item() and rc[6].item() == B
    assert rc[0].item() == pytest.approx(ps[valid, 0].sum().item(), rel=1e-5)
    assert rc[1].item() == rc[0].item()
    assert rc[2:5].tolist() == [0.0, 0.0, 0.0]
    for k in GRADS:
        torch.testing.assert_close(got[1][k], ref[k], rtol=1e-4, atol=1e-6, msg=lambda m: f"{k}: {m}")
    # the metric slots and the thermal batches are those of the thermal-aware step
    ta = HotPathStep(B, H, W, device=dev, gt_hw=gt_hw, **KW)
    rt = ta.run_device(*[d[k] for k in ARGS]).cpu()
    assert torch.equal(rt[7:15], rc[7:15])
    assert torch.equal(ta.pre_both["thermal"], step.pre_both["thermal"])
    bytes_plain, bytes_ta = step.algorithmic_bytes()["loss"], ta.algorithmic_bytes()["loss"]
    assert bytes_ta - bytes_plain == B * 8 * H * W

    # pipelined, three steps on alternating inputs == the plain steps, bit for bit
    d2 = _step_inputs(B, H, W, 2, dev, gt_hw)
    plain = [got, _snap(step, step.run_device(*[d2[k] for k in ARGS])), got]
    pst = HotPathStep(B, H, W, device=dev, gt_hw=gt_hw, use_thermal_aware_loss=False, pipelined=True, **KW)
    for k, inp in enumerate((d, d2, d)):
        rr = pst.run_device(*[inp[a] for a in ARGS])
        pst.wait_result(rr)
        _same_step(_snap(pst, rr), plain[k])
    pst.finish()

    # graph replay == stream launches
    replay = step.capture_graph(*[d[k] for k in ARGS])
    rr = replay()
    torch.cuda.synchronize()
    _same_step(_snap(step, rr), got)

    # run_host == run_device
    host = {k: d[k].cpu().pin_memory() for k in ARGS}
    hs = HotPathStep(B, H, W, device=dev, gt_hw=gt_hw, use_thermal_aware_loss=False, **KW)
    rh = hs.run_host(host)
    torch.cuda.synchronize()
    assert torch.equal(rh, got[0].cpu())
    for k in GRADS:
        assert torch.equal(hs.loss_out[k], got[1][k]), k

    # an invalid sample: excluded from the sums, zero gradients
    bad = dict(d, pred1=d["pred1"].clone())
    bad["pred1"][1, 3, 5, 2] = float("nan")
    rb = step.run_device(*[bad[k] for k in ARGS]).cpu()
    assert rb[5].item() == rc[5].item() - 1
    assert (step.loss_out["dpred1"][1] == 0).all() and (step.loss_out["dconf2"][1] == 0).all()


def test_step_plain_loss_has_no_multi_scale(dev):
    from thermal3d_vision_b200.pipeline import HotPathStep
    with pytest.raises(ValueError):
        HotPathStep(2, 64, 96, device=dev, multi_scale=True, use_thermal_aware_loss=False)
