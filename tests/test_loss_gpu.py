"""GPU parity: fused sm_100a loss (through the C ABI) vs the oracle.

Tolerances (BASELINE.json north_star): loss / components rtol 1e-5 (fp32),
input gradients rtol 1e-4 / atol 1e-6 against the fp32 reference graph.  We also
check the gradients against the float64 closed form with a tolerance scaled to
the gradient magnitude (atol 1e-6 alone is nearly vacuous at 512x384 where
|g| ~ 5e-6).
"""
import numpy as np
import pytest
import torch

from oracle import ref_loss

pytestmark = pytest.mark.gpu

KW = dict(alpha=0.2, edge_weight=0.5, smoothness_weight=0.3, detail_weight=0.4)


def _oracle_sample(p1, p2, g1, g2, c1, c2, t1, t2, multi, **kw):
    a = [None if x is None else x.detach().clone() for x in (p1, p2, g1, g2, c1, c2, t1, t2)]
    a[0].requires_grad_(); a[1].requires_grad_()
    if a[4] is not None:
        a[4].requires_grad_()
    if a[5] is not None:
        a[5].requires_grad_()
    loss, comp = ref_loss.enhanced_thermal_aware_loss_torch(*a, multi_scale=multi, **kw)
    loss.backward()
    return loss.item(), comp, a[0].grad, a[1].grad, None if a[4] is None else a[4].grad, None if a[5] is None else a[5].grad


def _launched(fn):
    """(fn(), names of the library's loss kernels it launched, the second stage left out)."""
    from thermal3d_vision_b200 import _lib
    torch.cuda.synchronize()
    _lib.profile_begin("loss_", 256)
    out = fn()
    torch.cuda.synchronize()
    names = {n for n, _, _ in _lib.profile_timeline(256)} - {"loss_finalize_kernel"}
    _lib.profile_end()
    return out, names


def _misaligned(t):
    """A contiguous copy at element offset 1 of its storage: not 16-byte aligned."""
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    return v


def _check_grad(name, got, ref32, ref64):
    got = got.detach().cpu()
    torch.testing.assert_close(got, ref32, rtol=1e-4, atol=1e-6, msg=lambda m: f"{name} vs fp32 oracle: {m}")
    # magnitude-aware check against exact arithmetic
    r64 = torch.from_numpy(np.asarray(ref64))
    scale = r64.abs().max().item()
    err = (got.double() - r64).abs()
    tol = 1e-4 * r64.abs() + 2e-6 * scale
    assert bool((err <= tol).all()), f"{name} vs f64 closed form: max err {err.max().item():.3e}, scale {scale:.3e}"


@pytest.mark.parametrize("H,W", [(224, 224), (38, 52), (37, 51), (16, 128), (17, 129), (5, 7), (64, 260)])
@pytest.mark.parametrize("multi", [False, True])
def test_per_sample_api_matches_oracle(cuda_device, H, W, multi):
    from thermal3d_vision_b200 import loss as t3d
    p1, p2, g1, g2, c1, c2, t1, t2 = ref_loss.make_kat_inputs(H, W, seed=H * 1000 + W)
    c1 = c1 * 3 - 1.0          # hit both clamps of the confidence
    ref = _oracle_sample(p1, p2, g1, g2, c1, c2, t1, t2, multi, **KW)
    f64 = ref_loss.loss_fwd_bwd_f64(p1, p2, g1, g2, c1, c2, t1, t2, multi_scale=multi, **KW)

    d = [x.to(cuda_device) for x in (p1, p2, g1, g2, c1, c2, t1, t2)]
    for k in (0, 1, 4, 5):
        d[k].requires_grad_()
    loss, comp = t3d.enhanced_thermal_aware_loss(*d, multi_scale=multi, **KW)
    assert loss.dim() == 0 and loss.is_cuda
    assert set(comp) == {"basic_loss", "edge_loss", "smoothness_loss", "detail_loss"}
    assert all(isinstance(v, float) for v in comp.values())
    loss.backward()

    assert loss.item() == pytest.approx(ref[0], rel=1e-5)
    assert loss.item() == pytest.approx(f64["total"], rel=1e-5)
    for k, k64 in (("basic_loss", "basic"), ("edge_loss", "edge"), ("smoothness_loss", "smooth"), ("detail_loss", "detail")):
        assert comp[k] == pytest.approx(ref[1][k], rel=1e-5), k
        assert comp[k] == pytest.approx(f64[k64], rel=1e-5), k
    _check_grad("dpred1", d[0].grad, ref[2], f64["dp1"])
    _check_grad("dpred2", d[1].grad, ref[3], f64["dp2"])
    _check_grad("dconf1", d[4].grad, ref[4], f64["dc1"])
    _check_grad("dconf2", d[5].grad, ref[5], f64["dc2"])


@pytest.mark.parametrize("multi", [True, False])      # True: tile kernel, False: TMA marching kernel
@pytest.mark.parametrize("variant", ["no_conf", "no_thermal", "one_channel", "conf_no_grad", "basic_only_fn"])
def test_optional_arguments(cuda_device, variant, multi):
    from thermal3d_vision_b200 import loss as t3d
    H, W = 40, 64
    p1, p2, g1, g2, c1, c2, t1, t2 = ref_loss.make_kat_inputs(H, W, seed=7)
    if variant == "no_conf":
        c1 = c2 = None
    if variant in ("no_thermal", "basic_only_fn"):
        t1 = t2 = None
    if variant == "one_channel":
        t1, t2 = t1[:1].contiguous(), t2[:1].contiguous()
    ref = _oracle_sample(p1, p2, g1, g2, c1, c2, t1, t2, multi, **KW)
    d = [None if x is None else x.to(cuda_device) for x in (p1, p2, g1, g2, c1, c2, t1, t2)]
    d[0].requires_grad_(); d[1].requires_grad_()
    if c1 is not None and variant != "conf_no_grad":
        d[4].requires_grad_(); d[5].requires_grad_()
    if variant == "basic_only_fn":
        loss = t3d.confidence_weighted_regression_loss(d[0], d[1], d[2], d[3], d[4], d[5], alpha=0.2)
    else:
        loss, comp = t3d.enhanced_thermal_aware_loss(*d, multi_scale=multi, **KW)
        if variant == "no_thermal":
            assert comp["edge_loss"] == 0 and comp["smoothness_loss"] == 0 and comp["detail_loss"] == 0
    loss.backward()
    assert loss.item() == pytest.approx(ref[0], rel=1e-5)
    torch.testing.assert_close(d[0].grad.cpu(), ref[2], rtol=1e-4, atol=1e-6)
    torch.testing.assert_close(d[1].grad.cpu(), ref[3], rtol=1e-4, atol=1e-6)
    if c1 is not None and variant != "conf_no_grad":
        torch.testing.assert_close(d[4].grad.cpu(), ref[4], rtol=1e-4, atol=1e-6)
    elif c1 is not None:
        assert d[4].grad is None


def test_training_loop_usage_views_and_grad_output(cuda_device):
    """train_thermal_dustr.py:182-360: per-sample calls on views of batched storage,
    losses summed, divided by the number of valid samples, one backward()."""
    from thermal3d_vision_b200 import loss as t3d
    B, H, W = 3, 48, 68
    P1, P2, G1, G2, C1, C2, T1, T2 = ref_loss.make_batch_inputs(B, H, W, seed=3)

    def loop(fn, dev):
        leaves = [x.detach().clone().to(dev).requires_grad_() for x in (P1, P2, C1, C2)]
        gs = [x.to(dev) for x in (G1, G2, T1, T2)]
        tot, nv = 0.0, 0
        for i in range(B):
            pm1, pm2 = leaves[0][i] * 1.0, leaves[1][i] * 1.0      # non-leaf views like a model output
            cf1 = torch.clamp(leaves[2][i], min=1e-5)              # train_thermal_dustr.py:278
            cf2 = torch.clamp(leaves[3][i], min=1e-5)
            loss, _ = fn(pm1, pm2, gs[0][i], gs[1][i], confidences1=cf1, confidences2=cf2,
                         thermal_img1=gs[2][i], thermal_img2=gs[3][i], multi_scale=False, **KW)
            if torch.isfinite(loss) and loss > 0:
                tot = tot + loss
                nv += 1
        tot = tot / nv
        tot.backward()
        return tot.item(), [x.grad.cpu() for x in leaves]

    ref_l, ref_g = loop(ref_loss.enhanced_thermal_aware_loss_torch, "cpu")
    got_l, got_g = loop(t3d.enhanced_thermal_aware_loss, cuda_device)
    assert got_l == pytest.approx(ref_l, rel=1e-5)
    for a, b in zip(got_g, ref_g):
        torch.testing.assert_close(a, b, rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize("multi", [False, True])
def test_batched_extension_with_invalid_sample(cuda_device, multi):
    from thermal3d_vision_b200 import loss as t3d
    B, H, W = 5, 32, 132
    P1, P2, G1, G2, C1, C2, T1, T2 = ref_loss.make_batch_inputs(B, H, W, seed=11, stress_conf=True)
    P1[2, 3, 4, 2] = float("nan")           # sample 2 becomes invalid (non-finite loss)
    Pa, Pb, Ca, Cb = (x.clone().requires_grad_() for x in (P1, P2, C1, C2))
    mean, rows, valid = ref_loss.batched_loss_torch(Pa, Pb, G1, G2, Ca, Cb, T1, T2, multi_scale=multi, **KW)
    mean.backward()
    assert valid.tolist() == [True, True, False, True, True]

    d = [x.to(cuda_device) for x in (P1, P2, G1, G2, C1, C2, T1, T2)]
    for k in (0, 1, 4, 5):
        d[k].requires_grad_()
    res = t3d.fused_thermal_loss(*d, multi_scale=multi, **KW)
    res.loss.backward()
    ps = res.per_sample.cpu().numpy()
    assert ps[:, 5].tolist() == [1, 1, 0, 1, 1]
    ok = valid
    np.testing.assert_allclose(ps[ok, :5], rows[ok], rtol=1e-5)
    assert res.batch[5].item() == 4 and res.batch[6].item() == B
    assert res.loss.item() == pytest.approx(mean.item(), rel=1e-5)
    for got, ref in ((d[0].grad, Pa.grad), (d[1].grad, Pb.grad), (d[4].grad, Ca.grad), (d[5].grad, Cb.grad)):
        got = got.cpu()
        assert torch.isfinite(got).all()
        assert got[2].abs().max().item() == 0.0          # invalid sample contributes nothing
        torch.testing.assert_close(got, ref, rtol=1e-4, atol=1e-6)


def test_full_size_properties_and_determinism(cuda_device):
    """BASELINE config 3 shape (batch 8 of it): oracle on one sample + size-independent properties."""
    from thermal3d_vision_b200 import loss as t3d
    B, H, W = 8, 384, 512
    P1, P2, G1, G2, C1, C2, T1, T2 = ref_loss.make_batch_inputs(B, H, W, seed=5)
    d = [x.to(cuda_device) for x in (P1, P2, G1, G2, C1, C2, T1, T2)]
    out1 = t3d.fused_thermal_loss_fwd_bwd(*d, multi_scale=False, **KW)
    out2 = t3d.fused_thermal_loss_fwd_bwd(*d, multi_scale=False, **KW)
    for k in ("per_sample", "batch", "dpred1", "dpred2", "dconf1", "dconf2"):
        assert torch.equal(out1[k], out2[k]), f"{k} not bit-identical across runs"
    # sample 3 against the oracle
    b = 3
    ref = _oracle_sample(P1[b], P2[b], G1[b], G2[b], C1[b], C2[b], T1[b], T2[b], False, **KW)
    ps = out1["per_sample"].cpu()
    assert ps[b, 0].item() == pytest.approx(ref[0], rel=1e-5)
    torch.testing.assert_close(out1["dpred1"][b].cpu() * B, ref[2], rtol=1e-4, atol=1e-7)
    torch.testing.assert_close(out1["dconf2"][b].cpu() * B, ref[5], rtol=1e-4, atol=1e-7)
    # batch mean == mean of per-sample totals; x,y gradients only carry the basic term:
    assert out1["batch"][0].item() == pytest.approx(ps[:, 0].double().mean().item(), rel=1e-6)
    gxy = out1["dpred1"][..., :2]
    cc = d[4].clamp(1e-5, 10.0)[..., None] / (3.0 * H * W * B)
    nz = (d[0][..., :2] != d[2][..., :2])            # sgn(0) = 0: an exact pred == gt coordinate has zero gradient
    torch.testing.assert_close(gxy.abs(), cc.expand_as(gxy) * nz, rtol=1e-5, atol=0)
    # permutation equivariance over the batch
    perm = torch.tensor([3, 0, 7, 1, 2, 6, 5, 4], device=cuda_device)
    out3 = t3d.fused_thermal_loss_fwd_bwd(*[x[perm].contiguous() for x in d], multi_scale=False, **KW)
    assert torch.equal(out3["per_sample"], out1["per_sample"][perm])
    assert torch.equal(out3["dpred2"], out1["dpred2"][perm])


def test_errors(cuda_device):
    from thermal3d_vision_b200 import loss as t3d
    p = torch.zeros(8, 8, 3, device=cuda_device)
    with pytest.raises(ValueError):
        t3d.enhanced_thermal_aware_loss(p, p, p, p, thermal_img1=torch.zeros(8, 8, device=cuda_device),
                                        thermal_img2=torch.zeros(8, 8, device=cuda_device))
    with pytest.raises(ValueError):
        t3d.fused_thermal_loss(p[None], p[None], p[None], torch.zeros(1, 8, 9, 3, device=cuda_device))


@pytest.mark.parametrize("H,W", [(40, 64), (37, 51)])
def test_v1_thermal_aware_loss(cuda_device, H, W):
    """utils/loss.py:4-72 (dead code in the reference's training loop; API completeness)."""
    from thermal3d_vision_b200 import loss as t3d
    ins = ref_loss.make_kat_inputs(H, W, seed=H)
    a = [x.clone() for x in ins]
    for k in (0, 1, 4, 5):
        a[k].requires_grad_()
    ref, rc = ref_loss.thermal_aware_loss_torch(*a, alpha=0.2, edge_weight=0.5, smoothness_weight=0.3)
    ref.backward()
    d = [x.to(cuda_device) for x in ins]
    for k in (0, 1, 4, 5):
        d[k].requires_grad_()
    got, gc = t3d.thermal_aware_loss(*d, alpha=0.2, edge_weight=0.5, smoothness_weight=0.3)
    got.backward()
    assert set(gc) == {"basic_loss", "edge_loss", "smoothness_loss"}
    assert got.item() == pytest.approx(ref.item(), rel=1e-5)
    for k in gc:
        assert gc[k] == pytest.approx(rc[k], rel=1e-5)
    for k in (0, 1, 4, 5):
        torch.testing.assert_close(d[k].grad.cpu(), a[k].grad, rtol=1e-4, atol=1e-6)


def test_v1_golden_value(cuda_device):
    import os
    from thermal3d_vision_b200 import loss as t3d
    kat = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "loss_kat.npz"))
    d = [x.to(cuda_device) for x in ref_loss.make_kat_inputs(224, 224, seed=0)]
    got, gc = t3d.thermal_aware_loss(*d, alpha=0.2, edge_weight=0.5, smoothness_weight=0.3)
    np.testing.assert_allclose([got.item(), gc["basic_loss"], gc["edge_loss"], gc["smoothness_loss"]], kat["v1"], rtol=1e-5)


def test_golden_table_full_size(cuda_device):
    """KAT-L rows of SURVEY.md Appendix C incl. 384x512 (values produced by the reference itself)."""
    import os
    from thermal3d_vision_b200 import loss as t3d
    kat = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "loss_kat.npz"))
    for row in kat["table"]:
        H, W, multi = int(row[0]), int(row[1]), bool(row[2])
        d = [x.to(cuda_device) for x in ref_loss.make_kat_inputs(H, W, seed=0)]
        for k in (0, 1, 4, 5):
            d[k].requires_grad_()
        loss, comp = t3d.enhanced_thermal_aware_loss(*d, multi_scale=multi, **KW)
        loss.backward()
        got = [loss.item(), comp["basic_loss"], comp["edge_loss"], comp["smoothness_loss"], comp["detail_loss"],
               d[0].grad.abs().double().sum().item(), d[1].grad.abs().double().sum().item(),
               d[4].grad.abs().double().sum().item(), d[5].grad.abs().double().sum().item()]
        np.testing.assert_allclose(got, row[3:], rtol=1e-5)


@pytest.mark.parametrize("H,W", [(33, 132), (1, 128), (2, 8), (130, 516)])
def test_marching_kernel_edge_shapes(cuda_device, H, W):
    """Shapes that stress the TMA marching path: odd heights, single row, partial strips, bands of 1 row."""
    from thermal3d_vision_b200 import loss as t3d
    B = 2
    P1, P2, G1, G2, C1, C2, T1, T2 = ref_loss.make_batch_inputs(B, H, W, seed=H + W, stress_conf=True, smooth=H >= 8 and W >= 8)
    Pa, Pb, Ca, Cb = (x.clone().requires_grad_() for x in (P1, P2, C1, C2))
    mean, rows, valid = ref_loss.batched_loss_torch(Pa, Pb, G1, G2, Ca, Cb, T1, T2, multi_scale=False, **KW)
    mean.backward()
    d = [x.to(cuda_device) for x in (P1, P2, G1, G2, C1, C2, T1, T2)]
    for k in (0, 1, 4, 5):
        d[k].requires_grad_()
    res, names = _launched(lambda: t3d.fused_thermal_loss(*d, multi_scale=False, **KW))
    assert names == {"loss_march_kernel"}, names
    res.loss.backward()
    np.testing.assert_allclose(res.per_sample[:, :5].cpu().numpy(), rows, rtol=1e-5)
    for got, ref in ((d[0].grad, Pa.grad), (d[1].grad, Pb.grad), (d[4].grad, Ca.grad), (d[5].grad, Cb.grad)):
        torch.testing.assert_close(got.cpu(), ref, rtol=1e-4, atol=1e-6)
    # a misaligned thermal image: the tile kernel, same loss
    args = [x.detach() for x in d[:7]] + [_misaligned(d[7])]
    out, names = _launched(lambda: t3d.fused_thermal_loss_fwd_bwd(*args, multi_scale=False, **KW))
    assert names == {"loss_tile_kernel"}, names
    np.testing.assert_allclose(out["per_sample"][:, :5].cpu().numpy(), rows, rtol=1e-5)
    for got, ref in ((out["dpred1"], Pa.grad), (out["dpred2"], Pb.grad), (out["dconf1"], Ca.grad), (out["dconf2"], Cb.grad)):
        torch.testing.assert_close(got.cpu(), ref, rtol=1e-4, atol=1e-6)


def test_nan_thermal_poisons_only_that_sample(cuda_device):
    """clamp(NaN) = NaN in the reference: a NaN thermal pixel makes the sample's loss NaN -> sample skipped."""
    from thermal3d_vision_b200 import loss as t3d
    B, H, W = 3, 32, 128
    P1, P2, G1, G2, C1, C2, T1, T2 = ref_loss.make_batch_inputs(B, H, W, seed=4)
    T2[1, :, 5, 7] = float("nan")
    for multi in (False, True):
        mean, rows, valid = ref_loss.batched_loss_torch(P1, P2, G1, G2, C1, C2, T1, T2, multi_scale=multi, **KW)
        assert valid.tolist() == [True, False, True]
        res = t3d.fused_thermal_loss(*(x.to(cuda_device) for x in (P1, P2, G1, G2, C1, C2, T1, T2)), multi_scale=multi, **KW)
        assert res.per_sample[:, 5].tolist() == [1.0, 0.0, 1.0]
        assert res.loss.item() == pytest.approx(mean.item(), rel=1e-5)


@pytest.mark.parametrize("multi", [False, True])
@pytest.mark.parametrize("H,W", [(48, 256), (33, 132)])
def test_replicated_thermal_planes_read_once(cuda_device, H, W, multi):
    """T3D_THERMAL_REPLICATED: reading plane 0 only and evaluating gray3(v, v, v) is bit-identical to reading the
    three replicated planes enhance_thermal_contrast returns (utils/preprocessing.py:22-28)."""
    from thermal3d_vision_b200 import loss as t3d
    B = 3
    P1, P2, G1, G2, C1, C2, T1, T2 = ref_loss.make_batch_inputs(B, H, W, seed=11)
    T1 = T1[:, :1].repeat(1, 3, 1, 1).contiguous()
    T2 = T2[:, :1].repeat(1, 3, 1, 1).contiguous()
    d = [x.to(cuda_device) for x in (P1, P2, G1, G2, C1, C2, T1, T2)]
    a = t3d.fused_thermal_loss_fwd_bwd(*d, multi_scale=multi, **KW)
    b = t3d.fused_thermal_loss_fwd_bwd(*d, multi_scale=multi, thermal_replicated=True, **KW)
    for k in ("per_sample", "batch", "dpred1", "dpred2", "dconf1", "dconf2"):
        if multi:   # three planes: split path (t3d_loss_scale2.cu + march); replicas: both scales in one pass -- other summation order
            torch.testing.assert_close(a[k], b[k], rtol=1e-4, atol=1e-6)
        else:
            assert torch.equal(a[k], b[k]), k
    mean, rows, _ = ref_loss.batched_loss_torch(P1, P2, G1, G2, C1, C2, T1, T2, multi_scale=multi, **KW)
    np.testing.assert_allclose(b["per_sample"][:, :5].cpu().numpy(), rows, rtol=1e-5)


def test_wrong_replicated_promise_is_caught_in_debug_mode(cuda_device):
    """thermal_replicated=True is a caller promise; in debug / test mode (T3D_DEBUG_CHECKS=1, tests/conftest.py) it is
    verified on the device, so a wrong flag raises instead of silently changing the result."""
    from thermal3d_vision_b200 import loss as t3d
    assert t3d.DEBUG_CHECKS
    d = [x.to(cuda_device) for x in ref_loss.make_batch_inputs(2, 32, 64, seed=1)]
    t3d.fused_thermal_loss_fwd_bwd(*d, multi_scale=False, thermal_replicated=True, **KW)     # replicas: fine
    d[6][1, 2, 5, 7] += 1e-3                                  # one pixel of one plane differs
    with pytest.raises(ValueError, match="not bit-identical"):
        t3d.fused_thermal_loss_fwd_bwd(*d, multi_scale=False, thermal_replicated=True, **KW)


def test_second_backward_raises(cuda_device):
    """The precomputed gradients are scaled in place and handed over once: a second backward through the same node
    raises instead of silently contributing zeros."""
    from thermal3d_vision_b200 import loss as t3d
    d = [x.to(cuda_device) for x in ref_loss.make_batch_inputs(1, 16, 32, seed=2)]
    d[0].requires_grad_()
    res = t3d.fused_thermal_loss(*d, multi_scale=False, **KW)
    res.loss.backward(retain_graph=True)
    with pytest.raises(RuntimeError, match="already consumed"):
        res.loss.backward()
    f = t3d.fused_thermal_loss(*(x.detach() for x in d), multi_scale=False, **KW)      # no grad: nothing to hand back
    assert not f.loss.requires_grad


@pytest.mark.parametrize("planes", ["three", "one", "replicated"])
@pytest.mark.parametrize("H,W", [(130, 516), (65, 132), (4, 8), (38, 52), (224, 224), (5, 4), (97, 260), (66, 128)])
def test_multi_scale_march_paths_edge_shapes(cuda_device, H, W, planes):
    """multi_scale=True on vector-aligned shapes.  Three distinct thermal planes: the half-resolution pass
    (t3d_loss_scale2.cu) + the marching kernel; one plane / replicated planes: both scales in one pass
    (loss_march_ms_kernel).  Odd heights (last row outside every pooled cell), ragged strips, bands with and without
    rows above / below, batch > 1, gradients included."""
    from thermal3d_vision_b200 import loss as t3d
    B = 2
    P1, P2, G1, G2, C1, C2, T1, T2 = ref_loss.make_batch_inputs(B, H, W, seed=3 * H + W, stress_conf=True)
    if planes == "one":
        T1, T2 = T1[:, :1].contiguous(), T2[:, :1].contiguous()
    elif planes == "replicated":
        T1, T2 = T1[:, :1].repeat(1, 3, 1, 1).contiguous(), T2[:, :1].repeat(1, 3, 1, 1).contiguous()
    Pa, Pb, Ca, Cb = (x.clone().requires_grad_() for x in (P1, P2, C1, C2))
    mean, rows, valid = ref_loss.batched_loss_torch(Pa, Pb, G1, G2, Ca, Cb, T1, T2, multi_scale=True, **KW)
    mean.backward()
    d = [x.to(cuda_device) for x in (P1, P2, G1, G2, C1, C2, T1, T2)]
    for k in (0, 1, 4, 5):
        d[k].requires_grad_()
    expect = {"loss_scale2_kernel", "loss_march_kernel"} if planes == "three" else {"loss_march_ms_kernel"}
    if planes == "replicated":          # the functional entry takes the caller's promise that the planes are replicas
        out, names = _launched(lambda: t3d.fused_thermal_loss_fwd_bwd(*(x.detach() for x in d), multi_scale=True,
                                                                      thermal_replicated=True, **KW))
        assert names == expect, names
        np.testing.assert_allclose(out["per_sample"][:, :5].cpu().numpy(), rows, rtol=1e-5)
        for got, ref in ((out["dpred1"], Pa.grad), (out["dpred2"], Pb.grad), (out["dconf1"], Ca.grad), (out["dconf2"], Cb.grad)):
            torch.testing.assert_close(got.cpu(), ref, rtol=1e-4, atol=1e-6)
        return
    res, names = _launched(lambda: t3d.fused_thermal_loss(*d, multi_scale=True, **KW))
    assert names == expect, names
    res.loss.backward()
    np.testing.assert_allclose(res.per_sample[:, :5].cpu().numpy(), rows, rtol=1e-5)
    for got, ref in ((d[0].grad, Pa.grad), (d[1].grad, Pb.grad), (d[4].grad, Ca.grad), (d[5].grad, Cb.grad)):
        torch.testing.assert_close(got.cpu(), ref, rtol=1e-4, atol=1e-6)
    # forward-only entry (no gradient buffers) gives the same numbers
    f = t3d.fused_thermal_loss(*(x.detach() for x in d), multi_scale=True, **KW)
    assert torch.equal(f.per_sample[:, :5], res.per_sample[:, :5])
