"""The persistent loss kernels past their first wave of work items, and HotPathStep at the benchmark's own workload,
sample by sample against the float64 closed form (oracle.ref_loss.loss_fwd_bwd_f64).

loss_march_kernel, loss_march_ms_kernel, loss_march_rs_kernel and loss_basic_kernel run one CTA per SM.  Each warp
pulls work items (one image-view, one 128-px strip, one band of rows) from an atomic queue and carries its ring
position -- hence the mbarrier parity -- from one item to the next.  A fault in that carried state corrupts only the
items a warp takes after its first, so every case here queues at least two items per launched warp, and proves it from
the run itself: word 1 of the loss workspace is the queue counter, zeroed when a call starts, and every warp draws
exactly one ticket past the last item, so after the call counter[1] = items + launched warps.  The check does not
depend on the SM count or on the warps per CTA: a launch change that leaves a case in one wave fails it.

Every sample is compared, each gradient with a bound scaled to that sample's own gradient magnitude (a batch-wide
scale would hide one sample's errors), and a failure names the work item that wrote the worst element.
"""
import os
from concurrent.futures import ThreadPoolExecutor
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import ref_loss, ref_metrics, ref_preprocess

KW = dict(alpha=0.2, edge_weight=0.5, smoothness_weight=0.3, detail_weight=0.4)     # bench.py's weights
GRADS = ("dpred1", "dpred2", "dconf1", "dconf2")
REF_GRAD = {"dpred1": "dp1", "dpred2": "dp2", "dconf1": "dc1", "dconf2": "dc2"}
ROWS = ("total", "basic", "edge", "smooth", "detail")

# plan_bands (t3d_loss.cu) with the launcher's constants: bands of kMarchRows = kBasicRows = 32 rows from the top, then
# the last ~1/kMarchTailDiv = 1/kBasicTailDiv = 1/8 of the image in tail bands of kMarchTailRows = kBasicTailRows = 8
# rows, or kMarchMsTailRows = 16 on loss_march_ms_kernel (its bands start on even rows); strips of 128 px
BAND_ROWS, TAIL_DIV, STRIP_PX = 32, 8, 128
TAIL_ROWS = {"march": 8, "ms": 16, "basic": 8}


def plan_bands(H, W, queue):
    """-> (large bands, rows of a small band, small bands, strips) of one image-view (plan_bands, restated)."""
    rows_s = TAIL_ROWS[queue]
    small_rows = -(-(H // TAIL_DIV) // rows_s) * rows_s
    if small_rows > 0:
        nl = max(0, H - small_rows) // BAND_ROWS
        ns = -(-(H - nl * BAND_ROWS) // rows_s)
    else:
        nl, ns = -(-H // BAND_ROWS), 0
        if nl * BAND_ROWS > H:
            nl, rows_s, ns = nl - 1, BAND_ROWS, 1
    return nl, rows_s, ns, -(-W // STRIP_PX)


def test_plan_bands_restatement():
    """The restatement gives the per-image-view item counts the launcher comments and DESIGN quote."""
    nl, rs, ns, st = plan_bands(384, 512, "march")
    assert (nl, rs, ns, st) == (10, 8, 8, 4) and (nl + ns) * st == 72
    nl, rs, ns, st = plan_bands(384, 512, "ms")
    assert (nl, rs, ns, st) == (10, 16, 4, 4) and (nl + ns) * st == 56
    assert plan_bands(67, 260, "march") == (1, 8, 5, 3)
    assert plan_bands(67, 260, "ms") == (1, 16, 3, 3)
    assert plan_bands(5, 7, "march") == (0, 32, 1, 1)          # too short for a tail: one ragged band


class Waves:
    """The work-item queue of one call, read back from its workspace."""

    def __init__(self, ws, B, H, W, queue):
        self.B, self.H, self.plan = B, H, plan_bands(H, W, queue)
        nl, _, ns, nstrips = self.plan
        self.items = B * 2 * (nl + ns) * nstrips
        counter = ws[:8].cpu().numpy().view(np.uint32)
        self.warps = int(counter[1]) - self.items

    def check(self, what):
        ratio = self.items / self.warps if self.warps > 0 else float("inf")
        assert self.warps > 0, f"{what}: queue counter below the item count ({self.items} items, {self.warps} warps)"
        assert self.items >= 2 * self.warps, (f"{what}: {self.items} work items for {self.warps} warps "
                                              f"({ratio:.2f} per warp): the case no longer reaches past the first wave")
        print(f"[waves] {what}: items {self.items}, warps {self.warps}, items per warp {ratio:.2f}")

    def item_of(self, b, view, row, col):
        """The work item that wrote pixel (row, col) of sample b, view `view`: its band, strip and queue ticket."""
        nl, rows_s, ns, nstrips = self.plan
        img, s = 2 * b + view, col // STRIP_PX
        if row < nl * BAND_ROWS:
            k = row // BAND_ROWS
            ticket, band = (img * nl + k) * nstrips + s, f"band {k} (rows {k * BAND_ROWS}..{(k + 1) * BAND_ROWS - 1})"
        else:
            k = (row - nl * BAND_ROWS) // rows_s
            r0 = nl * BAND_ROWS + k * rows_s
            ticket = self.B * 2 * nl * nstrips + (img * ns + k) * nstrips + s
            band = f"tail band {k} (rows {r0}..{min(r0 + rows_s, self.H) - 1})"
        wave = "first wave" if ticket < self.warps else f"wave {ticket // self.warps + 1}"
        return f"{band}, strip {s}, ticket {ticket} ({wave})"


def _pool():
    return ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1))


def f64_refs(P1, P2, G1, G2, C1, C2, T1, T2, multi_scale, **kw):
    """loss_fwd_bwd_f64 of every sample ([B, ...] CPU tensors; T None: no thermal images).  numpy releases the GIL in
    its array loops, so a thread pool overlaps the samples."""
    args = (P1, P2, G1, G2, C1, C2, T1, T2)
    kw = dict(KW, **kw)

    def one(b):
        return ref_loss.loss_fwd_bwd_f64(*(None if t is None else t[b].numpy() for t in args), multi_scale=multi_scale, **kw)
    with _pool() as ex:
        return list(ex.map(one, range(P1.shape[0])))


def _valid(ref):
    t = np.float32(ref["total"])
    return bool(np.isfinite(t) and t > 0)


def check_rows(what, per_sample, refs, samples):
    """Rows [total, basic, edge, smooth, detail] to rtol 1e-5 of float64; the valid flag exactly."""
    ps = per_sample.double().cpu().numpy()
    for b in samples:
        np.testing.assert_allclose(ps[b, :5], [refs[b][k] for k in ROWS], rtol=1e-5,
                                   err_msg=f"{what}: sample {b}, rows {ROWS}")
        assert ps[b, 5] == (1.0 if _valid(refs[b]) else 0.0), f"{what}: sample {b} valid flag {ps[b, 5]}"


def check_grads(what, out, refs, n_valid, waves, samples):
    """output x n_valid against each sample's float64 gradient: |err| <= 1e-4 |r| + 2e-6 max|r|, max per sample and per
    tensor.  A failure names the worst element and the work item that wrote it."""
    for k in GRADS:
        view = 0 if k.endswith("1") else 1
        got_all = out[k].cpu()
        for b in samples:
            r = refs[b][REF_GRAD[k]]
            got = got_all[b].double().numpy() * n_valid
            err = np.abs(got - r)
            tol = 1e-4 * np.abs(r) + 2e-6 * np.abs(r).max()
            ok = err <= tol                                    # NaN fails
            if ok.all():
                continue
            q = np.where(ok, 0.0, np.nan_to_num(err / np.maximum(tol, 1e-300), nan=np.inf))
            at = np.unravel_index(int(np.argmax(q)), q.shape)
            row, col = int(at[0]), int(at[1])
            comp = f" component {'xyz'[at[2]]}" if len(at) == 3 else ""
            pytest.fail(f"{what} {k}: {int((~ok).sum())} elements out of bound in sample {b}; worst at view {view + 1}, "
                        f"row {row}, col {col}{comp}: got {got[at]:.6e}, float64 {r[at]:.6e}, |err| {err[at]:.3e} > "
                        f"{tol[at]:.3e}; written by {waves.item_of(b, view, row, col)}")


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


# ============================================================================ the loss kernels on their own
# name: (B, H, W, thermal planes, multi_scale, kernels that run, work-item queue)
#   rep    three bit-identical planes, thermal_replicated=True: one staged plane, gray of (v, v, v)
#   one    a single plane
#   three  three distinct planes (loss_march_kernel<3>: 10 warps per CTA)
CASES = {
    "rep": (64, 384, 512, "rep", False, {"loss_march_kernel"}, "march"),
    "one": (64, 384, 512, "one", False, {"loss_march_kernel"}, "march"),
    "three": (64, 384, 512, "three", False, {"loss_march_kernel"}, "march"),
    "ms_one": (64, 384, 512, "one", True, {"loss_march_ms_kernel"}, "ms"),
    "ms_rep": (64, 384, 512, "rep", True, {"loss_march_ms_kernel"}, "ms"),
    # three distinct planes, multi-scale: loss_scale2_kernel, then loss_march_kernel<3> adding its pooled gradient
    "ms_three": (64, 384, 512, "three", True, {"loss_scale2_kernel", "loss_march_kernel"}, "march"),
    # many small images: an odd height, a 4-px last strip, W % 8 == 4 (the split path's pooled gradient is read by
    # each lane instead of staged), and short items that wrap the ring at many different positions
    "ragged_rep": (160, 67, 260, "rep", False, {"loss_march_kernel"}, "march"),
    "ragged_ms_one": (160, 67, 260, "one", True, {"loss_march_ms_kernel"}, "ms"),
    "ragged_ms_three": (160, 67, 260, "three", True, {"loss_scale2_kernel", "loss_march_kernel"}, "march"),
}


def _planes(T, planes):
    if planes == "one":
        return T[:, :1].contiguous()
    if planes == "three":                                   # distinct, still smooth: mirror images of the plane
        return torch.stack([T[:, 0], T[:, 0].flip(-1), T[:, 0].flip(-2)], 1).contiguous()
    return T                                                # make_batch_inputs replicates its plane


@pytest.fixture(scope="module", params=list(CASES))
def loss_case(request, cuda_device):
    """Inputs of one case (CPU and device) and their float64 reference, computed once for every test of the case."""
    name = request.param
    B, H, W, planes, multi, kernels, queue = CASES[name]
    P1, P2, G1, G2, C1, C2, T1, T2 = ref_loss.make_batch_inputs(B, H, W, seed=list(CASES).index(name) + 70,
                                                                stress_conf=True)
    cpu = [P1, P2, G1, G2, C1, C2, _planes(T1, planes), _planes(T2, planes)]
    refs = f64_refs(*cpu, multi_scale=multi)
    return SimpleNamespace(name=name, B=B, H=H, W=W, multi=multi, rep=planes == "rep", kernels=kernels, queue=queue,
                           cpu=cpu, dev=[t.to(cuda_device) for t in cpu], refs=refs)


def _workspace(c):
    from thermal3d_vision_b200 import _lib
    from thermal3d_vision_b200 import loss as t3d
    nbytes = _lib.lib().t3d_loss_workspace_bytes(c.B, c.H, c.W, t3d.LOSS_MULTI_SCALE if c.multi else 0)
    return torch.empty(nbytes, dtype=torch.uint8, device=c.dev[0].device)


def _fwd_bwd(c, args, ws=None, **kw):
    from thermal3d_vision_b200 import loss as t3d
    out = None if ws is None else {"workspace": ws}
    return t3d.fused_thermal_loss_fwd_bwd(*args, multi_scale=c.multi, thermal_replicated=c.rep, out=out, **KW, **kw)


def _fwd(c, args, ws):
    """The forward-only entry (no gradient buffers): what fused_thermal_loss runs without requires_grad."""
    from thermal3d_vision_b200 import loss as t3d
    P1, P2, G1, G2, C1, C2, T1, T2 = args
    ps, _, _, _, _, _ = t3d._launch(False, P1, P2, G1, G2, C1, C2, T1, T2, (False, False), KW["alpha"],
                                    KW["edge_weight"], KW["smoothness_weight"], KW["detail_weight"], c.multi,
                                    1.0 / P1.shape[0], False, out={"workspace": ws}, thermal_replicated=c.rep)
    return ps


@pytest.mark.gpu
def test_past_first_wave_matches_f64(loss_case):
    """Every sample's rows and gradients against float64, forward + backward and forward only, each call proven to
    run at least two work items per warp."""
    c = loss_case
    ws = _workspace(c)
    out, names = _launched(lambda: _fwd_bwd(c, c.dev, ws))
    assert names == c.kernels, names
    waves = Waves(ws, c.B, c.H, c.W, c.queue)
    waves.check(f"{c.name} fwd+bwd ({'+'.join(sorted(names))})")
    assert all(_valid(r) for r in c.refs)
    assert out["batch"][5].item() == c.B
    check_rows(c.name, out["per_sample"], c.refs, range(c.B))
    check_grads(c.name, out, c.refs, c.B, waves, range(c.B))

    ps, names = _launched(lambda: _fwd(c, c.dev, ws))
    assert names == c.kernels, names
    Waves(ws, c.B, c.H, c.W, c.queue).check(f"{c.name} fwd")
    assert torch.equal(ps, out["per_sample"]), "forward-only rows differ from the forward + backward rows"


@pytest.mark.gpu
@pytest.mark.parametrize("loss_case", ["rep", "ms_one", "ms_rep"], indirect=True)
def test_batch_independence(loss_case):
    """Samples at the head, middle and end of the batch -- sample B-1's tail bands are among the last tickets drawn --
    equal, bit for bit, the same sample called alone."""
    c = loss_case
    big = _fwd_bwd(c, c.dev, grad_scale=1.0, rescale_invalid=False)
    for b in (0, c.B // 2 - 1, c.B - 1):
        one = _fwd_bwd(c, [t[b:b + 1] for t in c.dev], grad_scale=1.0, rescale_invalid=False)
        assert torch.equal(one["per_sample"][0], big["per_sample"][b]), f"sample {b} rows"
        for k in GRADS:
            assert torch.equal(one[k][0], big[k][b]), f"sample {b} {k}"


@pytest.mark.gpu
@pytest.mark.parametrize("loss_case", ["rep", "ms_one", "ms_rep"], indirect=True)
def test_invalid_samples_late_in_the_queue(loss_case):
    """A NaN prediction inside sample B-1's last tail band and a NaN thermal pixel in sample B/2: both samples drop
    out (exact-zero gradients), the others carry 1 / n_valid."""
    c = loss_case
    B, H, W = c.B, c.H, c.W
    cpu = [t.clone() for t in c.cpu]
    cpu[0][B - 1, H - 3, W - 5, 2] = float("nan")
    cpu[7][B // 2, :, H // 3, 7] = float("nan")           # every plane: the replicated promise still holds
    bad = (B // 2, B - 1)
    for b in bad:
        ref = ref_loss.loss_fwd_bwd_f64(*(t[b].numpy() for t in cpu), multi_scale=c.multi, **KW)
        assert not _valid(ref), b
    refs = [None if b in bad else r for b, r in enumerate(c.refs)]
    ws = _workspace(c)
    out = _fwd_bwd(c, [t.to(c.dev[0].device) for t in cpu], ws)
    waves = Waves(ws, B, H, W, c.queue)
    waves.check(f"{c.name} invalid samples")
    ps = out["per_sample"].cpu()
    assert [b for b in range(B) if ps[b, 5] == 0] == list(bad)
    assert out["batch"][5].item() == B - 2 and out["batch"][6].item() == B
    for k in GRADS:
        for b in bad:
            assert torch.count_nonzero(out[k][b]).item() == 0, f"{k} of invalid sample {b}"
    valid = [b for b in range(B) if b not in bad]
    check_rows(f"{c.name} invalid samples", out["per_sample"], refs, valid)
    check_grads(f"{c.name} invalid samples", out, refs, B - 2, waves, valid)


# ============================================================================ the benchmark's step
# variant: (HotPathStep options, the loss kernel it runs, its work-item queue)
STEP_VARIANTS = {
    "default": (dict(), "loss_march_kernel", "march"),
    "multi_scale": (dict(multi_scale=True), "loss_march_ms_kernel", "ms"),       # the preprocessing's two-scale statistics
    "gt_hw": (dict(gt_hw=(512, 512)), "loss_march_rs_kernel", "march"),          # pseudo-GT at its stored resolution
    "plain": (dict(use_thermal_aware_loss=False), "loss_basic_kernel", "basic"),  # confidences in [1, 5]: no upper clamp
}


def _step_inputs(seed, dev, gt_hw):
    import bench
    d = bench.make_inputs_torch(64, 384, 512, seed, dev)
    if gt_hw is not None:
        g = torch.Generator().manual_seed(seed + 100)
        for k in ("gt1", "gt2"):
            G = torch.randn(64, *gt_hw, 3, generator=g)
            G[..., 2] = 1.5 + 3 * G[..., 2].abs()
            d[k] = G.to(dev)
    return d


def _check_step(what, step, i, d, opts, queue):
    B, H, W = step.B, step.H, step.W
    lo, pre, met, res = step.loss_sets[i], step.pre_sets[i], step.met_sets[i], step.results[i].cpu().numpy()
    c = {k: v.cpu() for k, v in d.items()}
    # the thermal batches: all 2B frames bit-exact (the resize's row ranges span many frames)
    raw = torch.cat([c["raw1"], c["raw2"]]).numpy()
    with _pool() as ex:
        frames = list(ex.map(lambda j: ref_preprocess.train_path(raw[j], (H, W))[0], range(2 * B)))
    th = pre["thermal"].cpu().numpy()
    for j in range(2 * B):
        assert np.array_equal(th[j], frames[j]), f"{what}: thermal frame {j} (view {j // B + 1}, sample {j % B})"
    T = torch.from_numpy(np.stack(frames))
    thermal = opts.get("use_thermal_aware_loss", True)
    G1, G2 = c["gt1"], c["gt2"]
    if "gt_hw" in opts:                  # train_thermal_dustr.py:234-271: the GT resampled to the prediction's size
        up = lambda G: F.interpolate(G.permute(0, 3, 1, 2), size=(H, W), mode="bilinear",
                                     align_corners=False).permute(0, 2, 3, 1).contiguous()
        G1, G2 = up(G1), up(G2)
    kw = {} if thermal else dict(edge_weight=0.0, smoothness_weight=0.0, detail_weight=0.0)
    refs = f64_refs(c["pred1"], c["pred2"], G1, G2, c["conf1"], c["conf2"], T[:B] if thermal else None,
                    T[B:] if thermal else None, multi_scale=opts.get("multi_scale", False), **kw)
    assert all(_valid(r) for r in refs)
    waves = Waves(lo["workspace"], B, H, W, queue)
    waves.check(what)
    # n_valid and the packed loss: sums over the valid samples
    assert lo["batch"][5].item() == B and res[5] == B and res[6] == B and res[14] == B
    np.testing.assert_allclose(res[0:5], [sum(r[k] for r in refs) for k in ROWS], rtol=1e-5, err_msg=f"{what}: packed loss")
    check_rows(what, lo["per_sample"], refs, range(B))
    check_grads(what, lo, refs, B, waves, range(B))
    # depth metrics of view 1: per image (the delta accuracies are exact counts), and the dataset means
    per = [ref_metrics.compute_depth_metrics(c["pred1"][b, ..., 2].numpy(), c["gt_depth"][b].numpy()) for b in range(B)]
    m = met["metrics_f64"].cpu().numpy()
    for b in range(B):
        np.testing.assert_allclose(m[b, :4], [per[b][k] for k in ref_metrics.KEYS7[:4]], rtol=1e-5,
                                   err_msg=f"{what}: metrics of image {b}")
        assert m[b, 4:7].tolist() == [per[b][k] for k in ref_metrics.KEYS7[4:]], f"{what}: delta accuracies of image {b}"
    acc = ref_metrics.accumulate_dataset(per)
    np.testing.assert_allclose(res[7:14] / res[14], [acc[k] for k in ref_metrics.KEYS7], rtol=1e-5,
                               err_msg=f"{what}: dataset metrics")


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(STEP_VARIANTS))
def test_bench_step_matches_f64(cuda_device, variant):
    """HotPathStep as bench.py runs it (batch 64, 384x512 from 512x640 raw frames, pipelined) for two consecutive steps
    on different inputs: the second writes the other output set and overlaps the first one's tail.  Both are checked."""
    import bench
    from thermal3d_vision_b200.pipeline import HotPathStep
    opts, kernel, queue = STEP_VARIANTS[variant]
    weights = dict(alpha=bench.ALPHA, edge_weight=bench.EDGE_W, smoothness_weight=bench.SMOOTH_W, detail_weight=bench.DETAIL_W)
    step = HotPathStep(64, 384, 512, device=cuda_device, pipelined=True, **weights, **opts)
    inputs = [_step_inputs(seed, cuda_device, opts.get("gt_hw")) for seed in (0, 1)]

    def run():
        for d in inputs:
            step.run_device(*[d[k] for k in bench.KEYS])
        step.finish()
    _, names = _launched(run)
    assert names == {kernel}, names
    for i, d in enumerate(inputs):                          # step i wrote output set i
        _check_step(f"{variant} step {i + 1}", step, i, d, opts, queue)


def test_f64_reference_keeps_fp32_pooled_signs():
    """Two 2x2 cells whose float64 means differ by 2^-25 pool to the same fp32 value in the reference, so the
    reference's scale-2 gradient of |dz| there is sign(0) = 0.  The float64 closed form follows it: otherwise it would
    be off by ~1e-6 exactly where the kernels agree with the reference (one such cell in ~10^6)."""
    p1, p2, g1, g2, c1, c2, t1, t2 = ref_loss.make_kat_inputs(8, 8, seed=3)
    p1[0:2, 0:4, 2] = 1.0
    p1[1, 3, 2] = 1.0 + 2.0 ** -23                          # cell (0, 1): fp32 ((1 + 1) + 1) + (1 + 2^-23) rounds to 4
    a = [x.clone() for x in (p1, p2, g1, g2, c1, c2, t1, t2)]
    a[0].requires_grad_()
    loss, _ = ref_loss.enhanced_thermal_aware_loss_torch(*a, multi_scale=True, **KW)
    loss.backward()
    f64 = ref_loss.loss_fwd_bwd_f64(*(x.numpy() for x in (p1, p2, g1, g2, c1, c2, t1, t2)), multi_scale=True, **KW)
    want = a[0].grad[..., 2].double().numpy()
    np.testing.assert_allclose(f64["dp1"][..., 2], want, rtol=1e-4, atol=1e-3 * np.abs(want).max())
