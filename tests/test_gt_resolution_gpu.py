"""Pseudo-GT at its stored resolution on the fast path: the marching loss kernel resamples the GT rows bilinearly as it
stages them (loss_march_rs_kernel), bit-identical to resampling first (t3d_interp_bilinear_f32) and then running the
loss on same-size GT; wider source segments (224x224 <- 512x512) keep the tile kernel, which measured faster there;
HotPathStep(gt_hw=...) on top of both."""
import pytest
import torch
import torch.nn.functional as F

from oracle import ref_loss

pytestmark = pytest.mark.gpu
KW = dict(alpha=0.2, edge_weight=0.5, smoothness_weight=0.3, detail_weight=0.4, multi_scale=False)
OUTS = ("per_sample", "batch", "dpred1", "dpred2", "dconf1", "dconf2")


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _gt(B, GH, GW, g):
    G = torch.randn(B, GH, GW, 3, generator=g)
    G[..., 2] = 1.5 + 3 * G[..., 2].abs()
    return G


def _case(B, H, W, GH, GW, thermal, seed, dev):
    """pred at (H, W), gt at (GH, GW); thermal 'one' [B,1,H,W], 'three' [B,3,H,W], 'rep' three identical planes."""
    g = torch.Generator().manual_seed(seed)
    G1, G2 = _gt(B, GH, GW, g), _gt(B, GH, GW, g)
    up = lambda G: F.interpolate(G.permute(0, 3, 1, 2), size=(H, W), mode="bilinear", align_corners=False).permute(0, 2, 3, 1)
    P1 = up(G1) + 0.1 * torch.randn(B, H, W, 3, generator=g)
    P2 = up(G2) + 0.1 * torch.randn(B, H, W, 3, generator=g)
    C1, C2 = 1 + 4 * torch.rand(B, H, W, generator=g), 1 + 4 * torch.rand(B, H, W, generator=g)
    planes = 1 if thermal == "one" else 3
    T1, T2 = torch.rand(B, planes, H, W, generator=g), torch.rand(B, planes, H, W, generator=g)
    if thermal == "rep":
        T1, T2 = T1[:, :1].expand(B, 3, H, W), T2[:, :1].expand(B, 3, H, W)
    d = lambda t: t.contiguous().to(dev)
    return [d(t) for t in (P1, P2, G1, G2, C1, C2, T1, T2)]


def _run(P1, P2, G1, G2, C1, C2, T1, T2, thermal_stats=None, **kw):
    from thermal3d_vision_b200 import loss as t3d
    rep = T1 is not None and T1.shape[1] == 3 and all(torch.equal(T[:, 0], T[:, c]) for T in (T1, T2) for c in (1, 2))
    return t3d.fused_thermal_loss_fwd_bwd(P1, P2, G1, G2, C1, C2, T1, T2, thermal_replicated=rep,
                                          thermal_stats=thermal_stats, **dict(KW, **kw))


def _launched(fn, substr="loss_"):
    """Names of the library's kernels whose name contains `substr` that `fn` launches."""
    from thermal3d_vision_b200 import _lib
    torch.cuda.synchronize()
    _lib.profile_begin(substr, 256)
    out = fn()
    torch.cuda.synchronize()
    names = {n for n, _, _ in _lib.profile_timeline(256)}
    _lib.profile_end()
    return out, names


def _assert_same(a, b, nan=False):
    for k in OUTS:
        if a[k] is None or b[k] is None:
            assert a[k] is None and b[k] is None, k
        elif nan:
            torch.testing.assert_close(a[k], b[k], rtol=0, atol=0, equal_nan=True, msg=k)
        else:
            assert torch.equal(a[k], b[k]), k


def _vs_resample_first(args, H, W, kernel="loss_march_rs_kernel", nan=False, **kw):
    from thermal3d_vision_b200.training import resample_bilinear
    P1, P2, G1, G2, C1, C2, T1, T2 = args
    fused, names = _launched(lambda: _run(P1, P2, G1, G2, C1, C2, T1, T2, **kw))
    assert kernel in names, names
    assert (kernel == "loss_tile_kernel") == ("loss_tile_kernel" in names), names
    two = _run(P1, P2, resample_bilinear(G1, (H, W)), resample_bilinear(G2, (H, W)), C1, C2, T1, T2, **kw)
    _assert_same(fused, two, nan=nan)
    return fused


@pytest.mark.parametrize("conf", ["pred", "none"])
@pytest.mark.parametrize("thermal", ["one", "three", "rep"])
@pytest.mark.parametrize("H,W,GH,GW", [(384, 512, 512, 512), (40, 132, 64, 132), (96, 256, 128, 260)])
def test_bit_identical_to_resample_then_loss(dev, H, W, GH, GW, thermal, conf):
    B = 2
    args = _case(B, H, W, GH, GW, thermal, seed=H + GW, dev=dev)
    if conf == "none":
        args[4] = args[5] = None
    _vs_resample_first(args, H, W)


def test_persistent_grid_reuse(dev):
    """B = 16 at 384x512 <- 512x512: ~2 300 work items, more than the resident warps -- every warp carries its ring
    position from item to item."""
    _vs_resample_first(_case(16, 384, 512, 512, 512, "rep", seed=16, dev=dev), 384, 512)


def test_non_finite_gt_at_zero_weight_taps(dev):
    """gh = 3 H: f = 3 y + 1 exactly, so source rows 3 y + 2 are read only by zero-weight taps.  ATen (and the
    resample-first path) turn 0 * Inf into NaN; so must the fused kernel."""
    B, H, W, GH, GW = 2, 40, 128, 120, 128
    args = _case(B, H, W, GH, GW, "rep", seed=3, dev=dev)
    G1 = args[2].clone()
    G1[0, 3 * 5 + 2, 17, 2] = float("inf")
    G1[0, 3 * 11 + 2, 64, 0] = float("nan")
    G1[1, 3 * 20 + 2, 127, 1] = float("-inf")
    args[2] = G1
    fused = _vs_resample_first(args, H, W, nan=True)
    assert torch.isnan(fused["per_sample"][:, 0]).all()


def test_thermal_statistics_of_the_preprocessing(dev):
    """With the preprocessing's grad_stats the resampled call skips its statistics pass and equals the same-size call
    given the same statistics."""
    from oracle import ref_preprocess
    from thermal3d_vision_b200 import preprocessing as pp
    from thermal3d_vision_b200.training import resample_bilinear
    B, H, W, GH, GW = 2, 384, 512, 512, 512
    raw = torch.from_numpy(ref_preprocess.make_raw_frames(2 * B, seed=4, hw=(256, 320)).astype("int32")).to(torch.uint16).to(dev)
    tb = pp.preprocess_thermal_batch(raw, (W, H), path="train")
    stats = (tb.grad_stats[:B].contiguous(), tb.grad_stats[B:].contiguous())
    P1, P2, G1, G2, C1, C2, _, _ = _case(B, H, W, GH, GW, "one", seed=5, dev=dev)
    T1, T2 = tb.thermal[:B].contiguous(), tb.thermal[B:].contiguous()
    from thermal3d_vision_b200 import loss as t3d
    call = lambda g1, g2: t3d.fused_thermal_loss_fwd_bwd(P1, P2, g1, g2, C1, C2, T1, T2, thermal_stats=stats,
                                                        thermal_replicated=True, **KW)
    fused, names = _launched(lambda: call(G1, G2), substr="")
    assert "loss_march_rs_kernel" in names and not any("thermal_stats" in n for n in names), names
    two = call(resample_bilinear(G1, (H, W)), resample_bilinear(G2, (H, W)))
    _assert_same(fused, two)


def test_reference_parity(dev):
    """Against the reference arithmetic on the CPU: F.interpolate, then the loss per sample (DESIGN §2 tolerances)."""
    B, H, W, GH, GW = 2, 40, 132, 64, 132
    args = _case(B, H, W, GH, GW, "three", seed=7, dev=dev)
    res, names = _launched(lambda: _run(*args, grad_scale=1.0 / B))
    assert "loss_march_rs_kernel" in names
    P1, P2, G1, G2, C1, C2, T1, T2 = [t.cpu() for t in args]
    p1, p2 = P1.clone().requires_grad_(), P2.clone().requires_grad_()
    c1, c2 = C1.clone().requires_grad_(), C2.clone().requires_grad_()
    down = lambda G: F.interpolate(G.permute(0, 3, 1, 2), size=(H, W), mode="bilinear", align_corners=False).permute(0, 2, 3, 1)
    g1, g2 = down(G1), down(G2)
    tot = 0.0
    for i in range(B):
        loss, _ = ref_loss.enhanced_thermal_aware_loss_torch(p1[i], p2[i], g1[i], g2[i], c1[i], c2[i], T1[i], T2[i], **KW)
        assert res["per_sample"][i, 0].item() == pytest.approx(loss.item(), rel=1e-5)
        tot = tot + loss
    (tot / B).backward()
    for got, ref in ((res["dpred1"], p1.grad), (res["dpred2"], p2.grad), (res["dconf1"], c1.grad), (res["dconf2"], c2.grad)):
        torch.testing.assert_close(got.cpu(), ref, rtol=1e-4, atol=1e-6)
    # forward only (no gradient buffers, detached inputs) on the same GT gives the same numbers
    from thermal3d_vision_b200 import loss as t3d
    f, names = _launched(lambda: t3d.fused_thermal_loss(*args, **KW))
    assert "loss_march_rs_kernel" in names
    assert torch.equal(f.per_sample, res["per_sample"])


@pytest.mark.parametrize("case", ["multi_scale", "upsampled", "gt_sized_conf", "wide_segment"])
def test_fallback_to_tile_kernel(dev, case):
    from thermal3d_vision_b200.training import resample_bilinear
    B, H, W = 2, 64, 96
    GH, GW = (32, 48) if case == "upsampled" else (128, 128)
    if case == "wide_segment":          # 224x224 <- 512x512 and alike: 2 x more source pixels per strip than output
        B, H, W, GH, GW = 2, 224, 224, 512, 512
    args = _case(B, H, W, GH, GW, "rep", seed=11, dev=dev)
    kw = {}
    if case == "multi_scale":
        kw["multi_scale"] = True
    if case == "gt_sized_conf":
        g = torch.Generator().manual_seed(12)
        args[4], args[5] = [(1 + 4 * torch.rand(B, GH, GW, generator=g)).to(dev) for _ in range(2)]
        P1, P2, G1, G2, C1, C2, T1, T2 = args
        fused, names = _launched(lambda: _run(P1, P2, G1, G2, C1, C2, T1, T2, conf_grad=False))
        assert "loss_tile_kernel" in names and "loss_march_rs_kernel" not in names, names
        rs = lambda t: resample_bilinear(t, (H, W))
        two = _run(P1, P2, rs(G1), rs(G2), rs(C1), rs(C2), T1, T2, conf_grad=False)
        torch.testing.assert_close(fused["per_sample"][:, :5], two["per_sample"][:, :5], rtol=2e-6, atol=1e-7)
        torch.testing.assert_close(fused["dpred1"], two["dpred1"], rtol=1e-4, atol=1e-7)
        return
    P1, P2, G1, G2, C1, C2, T1, T2 = args
    fused, names = _launched(lambda: _run(P1, P2, G1, G2, C1, C2, T1, T2, **kw))
    assert "loss_tile_kernel" in names and "loss_march_rs_kernel" not in names, names
    two = _run(P1, P2, resample_bilinear(G1, (H, W)), resample_bilinear(G2, (H, W)), C1, C2, T1, T2, **kw)
    torch.testing.assert_close(fused["per_sample"][:, :5], two["per_sample"][:, :5], rtol=2e-6, atol=1e-7)
    for k in ("dpred1", "dpred2", "dconf1", "dconf2"):
        torch.testing.assert_close(fused[k], two[k], rtol=1e-4, atol=1e-7)


# ---------------------------------------------------------------------------------------------------- HotPathStep
STEP_CASES = [(4, 384, 512, (512, 640)), (8, 224, 224, (512, 640))]


def _step_inputs(B, H, W, raw_hw, seed, dev, GH=512, GW=512):
    import bench
    d = bench.make_inputs_torch(B, H, W, seed, dev, raw_hw=raw_hw)
    g = torch.Generator().manual_seed(seed + 100)
    d["gt1"], d["gt2"] = _gt(B, GH, GW, g).to(dev), _gt(B, GH, GW, g).to(dev)
    return d


ARGS = ("raw1", "raw2", "pred1", "pred2", "gt1", "gt2", "conf1", "conf2", "gt_depth")
GRADS = ("dpred1", "dpred2", "dconf1", "dconf2")


def _snap(step, r):
    return r.clone(), {k: None if step.loss_out[k] is None else step.loss_out[k].clone() for k in GRADS}


def _same_step(a, b, exact=True):
    if exact:
        assert torch.equal(a[0], b[0])
    else:
        torch.testing.assert_close(a[0], b[0], rtol=1e-5, atol=1e-9)
    for k in GRADS:
        if a[1][k] is None or b[1][k] is None:
            assert a[1][k] is None and b[1][k] is None, k
        elif exact:
            assert torch.equal(a[1][k], b[1][k]), k
        else:
            torch.testing.assert_close(a[1][k], b[1][k], rtol=1e-4, atol=1e-9)


@pytest.mark.parametrize("B,H,W,raw_hw", STEP_CASES)
def test_step_gt_hw_equals_step_on_resampled_gt(dev, B, H, W, raw_hw):
    """384x512 <- 512x512 runs on loss_march_rs_kernel: bit for bit the step on resampled GT; 224x224 <- 512x512 on the
    tile kernel's fused taps: equal to rounding.  Pipelined steps, graph replay and run_host: bit for bit."""
    from thermal3d_vision_b200.pipeline import HotPathStep
    from thermal3d_vision_b200.training import resample_bilinear
    d = _step_inputs(B, H, W, raw_hw, 1, dev)
    step = HotPathStep(B, H, W, raw_hw=raw_hw, device=dev, gt_hw=(512, 512))
    (r, _), names = _launched(lambda: (step.run_device(*[d[k] for k in ARGS]), None))
    march = W == 512
    assert ("loss_march_rs_kernel" if march else "loss_tile_kernel") in names, names
    got = _snap(step, r)
    ref_step = HotPathStep(B, H, W, raw_hw=raw_hw, device=dev)
    e = dict(d, gt1=resample_bilinear(d["gt1"], (H, W)), gt2=resample_bilinear(d["gt2"], (H, W)))
    want = _snap(ref_step, ref_step.run_device(*[e[k] for k in ARGS]))
    _same_step(got, want, exact=march)
    assert got[1]["dconf1"] is not None

    # pipelined, three steps on alternating inputs == the plain steps
    d2 = _step_inputs(B, H, W, raw_hw, 2, dev)
    plain = [got, _snap(step, step.run_device(*[d2[k] for k in ARGS])), got]
    pst = HotPathStep(B, H, W, raw_hw=raw_hw, device=dev, gt_hw=(512, 512), pipelined=True)
    for k, inp in enumerate((d, d2, d)):
        r = pst.run_device(*[inp[a] for a in ARGS])
        pst.wait_result(r)
        _same_step(_snap(pst, r), plain[k])
    pst.finish()

    # graph replay == run_device
    replay = step.capture_graph(*[d[k] for k in ARGS])
    r = replay()
    torch.cuda.synchronize()
    _same_step(_snap(step, r), got)

    # run_host == run_device
    host = {k: d[k].cpu().pin_memory() for k in ARGS}
    hs = HotPathStep(B, H, W, raw_hw=raw_hw, device=dev, gt_hw=(512, 512))
    rh = hs.run_host(host)
    torch.cuda.synchronize()
    assert torch.equal(rh, got[0].cpu())
    for k in GRADS:
        assert torch.equal(hs.loss_out[k], got[1][k]), k


@pytest.mark.parametrize("B,H,W,raw_hw", STEP_CASES)
def test_step_gt_sized_confidence_takes_no_gradient(dev, B, H, W, raw_hw):
    from thermal3d_vision_b200.pipeline import HotPathStep
    d = _step_inputs(B, H, W, raw_hw, 3, dev)
    g = torch.Generator().manual_seed(31)
    gc1, gc2 = 1 + 4 * torch.rand(B, 512, 512, generator=g), 1 + 4 * torch.rand(B, 512, 512, generator=g)
    d["conf1"], d["conf2"] = gc1.to(dev), gc2.to(dev)
    step = HotPathStep(B, H, W, raw_hw=raw_hw, device=dev, gt_hw=(512, 512))
    r = step.run_device(*[d[k] for k in ARGS]).cpu()
    assert step.loss_out["dconf1"] is None and step.loss_out["dconf2"] is None
    assert step.loss_out["dpred1"] is not None
    # the reference loop on resampled GT and confidences, with the step's own preprocessed thermal
    down = lambda t: F.interpolate(t.permute(0, 3, 1, 2), size=(H, W), mode="bilinear", align_corners=False).permute(0, 2, 3, 1)
    th = step.pre_both["thermal"].cpu()
    g1, g2 = down(d["gt1"].cpu()), down(d["gt2"].cpu())
    c1, c2 = down(gc1.unsqueeze(-1))[..., 0], down(gc2.unsqueeze(-1))[..., 0]
    tot, nv = 0.0, 0
    for i in range(B):
        loss, _ = ref_loss.enhanced_thermal_aware_loss_torch(d["pred1"][i].cpu(), d["pred2"][i].cpu(), g1[i], g2[i], c1[i],
                                                             c2[i], th[i], th[B + i], **KW)
        if torch.isfinite(loss) and loss > 0:
            tot += loss.item(); nv += 1
    assert r[5].item() == nv
    assert r[0].item() / nv == pytest.approx(tot / nv, rel=1e-5)


def test_step_rejects_gt_of_the_wrong_shape(dev):
    from thermal3d_vision_b200.pipeline import HotPathStep
    B, H, W = 2, 64, 96
    d = _step_inputs(B, H, W, (128, 160), 4, dev, GH=128, GW=128)
    step = HotPathStep(B, H, W, raw_hw=(128, 160), device=dev, gt_hw=(128, 160))
    with pytest.raises(ValueError):
        step.run_device(*[d[k] for k in ARGS])
    with pytest.raises(ValueError):
        HotPathStep(B, H, W, raw_hw=(128, 160), device=dev, gt_hw=(128, 128)).run_device(
            *[dict(d, conf1=d["conf1"][:, :32])[k] for k in ARGS])
