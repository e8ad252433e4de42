"""GPU parity of the benchmarked path itself: pipeline.HotPathStep (preprocessing of both views -> fused loss
forward + backward -> pointmap -> depth -> metrics -> packed result) against the oracle loop that mirrors
train_thermal_dustr.py:182-360 + utils/metrics.py:72-138 on the same inputs."""
import numpy as np
import pytest
import torch

from oracle import ref_loss, ref_metrics, ref_preprocess

pytestmark = pytest.mark.gpu
KW = dict(alpha=0.2, edge_weight=0.5, smoothness_weight=0.3, detail_weight=0.4)
NVEC = 24        # T3D_RESULT_SIZE


def _oracle_step(raw1, raw2, P1, P2, G1, G2, C1, C2, gt_depth, H, W, multi):
    B = P1.shape[0]
    T1 = torch.from_numpy(np.stack([ref_preprocess.train_path(raw1[i], (H, W))[0] for i in range(B)]))
    T2 = torch.from_numpy(np.stack([ref_preprocess.train_path(raw2[i], (H, W))[0] for i in range(B)]))
    lead = [x.clone().requires_grad_() for x in (P1, P2, C1, C2)]
    mean, rows, valid = ref_loss.batched_loss_torch(lead[0], lead[1], G1, G2, lead[2], lead[3], T1, T2,
                                                    multi_scale=multi, **KW)
    mean.backward()
    per = [ref_metrics.compute_depth_metrics(P1[i, ..., 2].numpy(), gt_depth[i].numpy()) for i in range(B)]
    return T1, T2, mean.item(), rows, valid, [x.grad for x in lead], ref_metrics.accumulate_dataset(per)


@pytest.mark.parametrize("B,H,W", [(3, 96, 160), (1, 224, 224), (2, 100, 260)])
@pytest.mark.parametrize("multi", [False, True])
def test_hot_path_step_matches_oracle_loop(cuda_device, multi, B, H, W):
    from thermal3d_vision_b200.pipeline import HotPathStep
    raw = ref_preprocess.make_raw_frames(2 * B, seed=13, hw=(128, 200))
    P1, P2, G1, G2, C1, C2, _, _ = ref_loss.make_batch_inputs(B, H, W, seed=17, stress_conf=True)
    gt_depth = G1[..., 2].clone()
    gt_depth[B - 1, :7] = 0.0                               # invalid GT region in one image
    T1, T2, mean, rows, valid, grads, metrics = _oracle_step(raw[:B], raw[B:], P1, P2, G1, G2, C1, C2, gt_depth, H, W, multi)

    step = HotPathStep(B, H, W, raw_hw=(128, 200), device=cuda_device, multi_scale=multi, **KW)
    both = torch.from_numpy(raw).to(cuda_device)
    d = [x.to(cuda_device) for x in (P1, P2, G1, G2, C1, C2, gt_depth)]
    r = step.run_device(both[:B], both[B:], *d).cpu()
    s = HotPathStep.summarize(r)
    # the thermal batches fed to the loss are bit-exact, hence everything downstream is comparable
    assert np.array_equal(step.pre_both["thermal"][:B].cpu().numpy(), T1.numpy())
    assert np.array_equal(step.pre_both["thermal"][B:].cpu().numpy(), T2.numpy())
    assert s["n_valid"] == float(valid.sum()) and s["n_pairs"] == B and s["n_images"] == B
    assert s["loss"] == pytest.approx(mean, rel=1e-5)
    np.testing.assert_allclose(step.loss_out["per_sample"][:, :5].cpu().numpy(), rows, rtol=1e-5)
    for name, got, ref in (("dpred1", step.loss_out["dpred1"], grads[0]), ("dpred2", step.loss_out["dpred2"], grads[1]),
                           ("dconf1", step.loss_out["dconf1"], grads[2]), ("dconf2", step.loss_out["dconf2"], grads[3])):
        torch.testing.assert_close(got.cpu(), ref, rtol=1e-4, atol=1e-6, msg=lambda m: f"{name}: {m}")
    for k in ref_metrics.KEYS7:
        assert s[k] == pytest.approx(metrics[k], rel=1e-5), k
    # the host-buffer entry point (pinned H2D inside) gives the same packed vector, bit for bit
    host = {"raw1": torch.from_numpy(raw[:B]).pin_memory(), "raw2": torch.from_numpy(raw[B:]).pin_memory(),
            "pred1": P1.pin_memory(), "pred2": P2.pin_memory(), "gt1": G1.pin_memory(), "gt2": G2.pin_memory(),
            "conf1": C1.pin_memory(), "conf2": C2.pin_memory(), "gt_depth": gt_depth.pin_memory()}
    rh = step.run_host(host)
    torch.cuda.synchronize()
    assert torch.equal(rh, r)


def test_hot_path_step_full_size_is_deterministic(cuda_device):
    """BASELINE configs[2] shape (512x384) at a small batch: two runs give bit-identical results and gradients;
    the histogram option does not change a bit."""
    from thermal3d_vision_b200.pipeline import HotPathStep
    import bench
    B, H, W = 4, 384, 512
    d = bench.make_inputs_torch(B, H, W, seed=5, device=cuda_device)
    args = (d["raw1"], d["raw2"], d["pred1"], d["pred2"], d["gt1"], d["gt2"], d["conf1"], d["conf2"], d["gt_depth"])
    step = HotPathStep(B, H, W, device=cuda_device)
    a = step.run_device(*args).clone()
    ga = [step.loss_out[k].clone() for k in ("dpred1", "dpred2", "dconf1", "dconf2")]
    b = step.run_device(*args).clone()
    assert torch.equal(a, b)
    for x, k in zip(ga, ("dpred1", "dpred2", "dconf1", "dconf2")):
        assert torch.equal(x, step.loss_out[k]), k
    step.histogram = True
    c = step.run_device(*args).clone()
    assert torch.equal(a, c)
    assert (step.pre_both["histogram"].sum(1) == H * W).all()
    s = HotPathStep.summarize(a.cpu())
    assert s["n_valid"] == B and 0 < s["loss"] < 100 and 0 <= s["abs_rel"] < 1


def test_graph_replay_equals_stream_launches(cuda_device):
    """HotPathStep.capture_graph: the whole step as one CUDA-graph launch gives the bits of the eager step."""
    from thermal3d_vision_b200.pipeline import HotPathStep
    import bench
    B, H, W = 8, 224, 224                               # BASELINE configs[1] shape: launch-bound
    d = bench.make_inputs_torch(B, H, W, seed=2, device=cuda_device)
    args = (d["raw1"], d["raw2"], d["pred1"], d["pred2"], d["gt1"], d["gt2"], d["conf1"], d["conf2"], d["gt_depth"])
    step = HotPathStep(B, H, W, device=cuda_device)
    eager = step.run_device(*args).clone()
    grads = [step.loss_out[k].clone() for k in ("dpred1", "dconf2")]
    replay = step.capture_graph(*args)
    for _ in range(3):
        for k in ("dpred1", "dconf2"):
            step.loss_out[k].zero_()
        r = replay()
        torch.cuda.synchronize()
        assert torch.equal(r, eager)
        assert torch.equal(step.loss_out["dpred1"], grads[0]) and torch.equal(step.loss_out["dconf2"], grads[1])


def test_hot_path_step_invalid_sample(cuda_device):
    """A sample whose loss is not finite is skipped as train_thermal_dustr.py:320 does: it drops out of the mean,
    its gradients are exact zeros and the other samples' gradients carry 1 / n_valid (loss_finalize_kernel +
    t3d_step_epilogue do this on the device, without a host round trip)."""
    from thermal3d_vision_b200.pipeline import HotPathStep
    B, H, W = 3, 64, 128
    raw = ref_preprocess.make_raw_frames(2 * B, seed=3, hw=(96, 160))
    P1, P2, G1, G2, C1, C2, _, _ = ref_loss.make_batch_inputs(B, H, W, seed=23)
    P1[1, 5, 7, 2] = float("nan")
    gt_depth = G1[..., 2].clone()
    T1, T2, mean, rows, valid, grads, metrics = _oracle_step(raw[:B], raw[B:], P1, P2, G1, G2, C1, C2, gt_depth, H, W, False)
    assert valid.tolist() == [True, False, True]
    step = HotPathStep(B, H, W, raw_hw=(96, 160), device=cuda_device, **KW)
    both = torch.from_numpy(raw).to(cuda_device)
    d = [x.to(cuda_device) for x in (P1, P2, G1, G2, C1, C2, gt_depth)]
    for _ in range(2):                                      # second call: the workspace counters were reset
        s = HotPathStep.summarize(step.run_device(both[:B], both[B:], *d).cpu())
        assert s["n_valid"] == 2.0 and s["n_pairs"] == B
        assert s["loss"] == pytest.approx(mean, rel=1e-5)
        for name, got, ref in (("dpred1", step.loss_out["dpred1"], grads[0]), ("dpred2", step.loss_out["dpred2"], grads[1]),
                               ("dconf1", step.loss_out["dconf1"], grads[2]), ("dconf2", step.loss_out["dconf2"], grads[3])):
            ref = torch.zeros_like(got.cpu()) if ref is None else ref
            assert torch.count_nonzero(got[1]) == 0, name
            torch.testing.assert_close(got.cpu(), ref, rtol=1e-4, atol=1e-6, msg=lambda m: f"{name}: {m}")


def test_peer_mailbox_exchange_world_of_one(cuda_device):
    """t3d_step_epilogue_peers + t3d_mailbox_reduce (the data-parallel exchange over peer memory) with this process as
    the only rank: the reduced vector is the packed vector of t3d_step_epilogue, step after step (both parities of
    the mailbox get reused); with two "ranks" pointing at the same mailbox the slots add up in rank order."""
    import ctypes as C
    from thermal3d_vision_b200 import _lib
    lib = _lib.lib()
    B, H, W = 3, 8, 16
    g = torch.Generator().manual_seed(5)
    per_sample = torch.rand(B, 8, generator=g).to(cuda_device)
    per_sample[:, 5] = torch.tensor([1.0, 0.0, 1.0])                         # sample 1 invalid
    batch = torch.tensor([0, 0, 0, 0, 0, 2.0, float(B), 0], dtype=torch.float32, device=cuda_device)
    m64 = torch.rand(B, 8, generator=g, dtype=torch.float64).to(cuda_device)
    mk = lambda: [torch.ones(B, H, W, 3, device=cuda_device), torch.ones(B, H, W, 3, device=cuda_device),
                  torch.ones(B, H, W, device=cuda_device), torch.ones(B, H, W, device=cuda_device)]
    grads = mk()
    ref = torch.zeros(NVEC, dtype=torch.float64, device=cuda_device)
    st = _lib.current_stream_ptr()
    _lib.check(lib.t3d_step_epilogue(*[_lib.ptr(x) for x in grads], _lib.ptr(per_sample), _lib.ptr(batch), _lib.ptr(m64),
                                     B, H, W, B, 0, None, 0, _lib.ptr(ref), st), "t3d_step_epilogue")
    assert torch.count_nonzero(grads[0][1]) == 0 and torch.all(grads[0][0] == 1.5)    # fix-up: B / n_valid = 3 / 2
    # deferred variant (data parallel): zeros only; t3d_rescale_global applies samples / valid of the all-reduced vector
    g2 = mk()
    out = torch.zeros(NVEC, dtype=torch.float64, device=cuda_device)
    _lib.check(lib.t3d_step_epilogue(*[_lib.ptr(x) for x in g2], _lib.ptr(per_sample), _lib.ptr(batch), _lib.ptr(m64),
                                     B, H, W, B, 1, None, 0, _lib.ptr(out), st), "t3d_step_epilogue")
    assert torch.equal(out, ref) and torch.count_nonzero(g2[0][1]) == 0 and torch.all(g2[0][0] == 1.0)
    glob = out.clone(); glob[5] += 3; glob[6] += 3                                  # a second rank with 3 valid samples
    _lib.check(lib.t3d_rescale_global(*[_lib.ptr(x) for x in g2], _lib.ptr(per_sample), _lib.ptr(glob), B, H, W, st),
               "t3d_rescale_global")
    assert torch.count_nonzero(g2[2][1]) == 0 and torch.all(g2[0][2] == 1.2) and torch.all(g2[3][0] == 1.2)   # 6 / 5
    mailbox = torch.zeros(int(lib.t3d_mailbox_bytes()) // 8, dtype=torch.float64, device=cuda_device)
    null = [None] * 5
    for world in (1, 2):
        mailbox.zero_()
        peers = (C.c_uint64 * world)(*([mailbox.data_ptr()] * world))
        for step in range(5):
            grads = mk()
            local = torch.zeros(NVEC, dtype=torch.float64, device=cuda_device)
            out = torch.full((NVEC,), -1.0, dtype=torch.float64, device=cuda_device)
            for rank in range(world):                                             # every "rank" posts into the one mailbox
                _lib.check(lib.t3d_step_epilogue_peers(*[_lib.ptr(x) for x in grads], _lib.ptr(per_sample), _lib.ptr(batch),
                                                       _lib.ptr(m64), B, H, W, B, None, 0, _lib.ptr(local), peers, world, rank, step, st),
                           "t3d_step_epilogue_peers")
            assert torch.count_nonzero(grads[0][1]) == 0 and torch.all(grads[0][0] == 1.0)     # zeros only
            if step % 2 == 0:       # vector only
                _lib.check(lib.t3d_mailbox_reduce(_lib.ptr(mailbox), world, step, _lib.ptr(out), *null, 0, 0, 0, st), "t3d_mailbox_reduce")
            else:                   # + the global validity factor: world * 3 samples, world * 2 valid
                _lib.check(lib.t3d_mailbox_reduce(_lib.ptr(mailbox), world, step, _lib.ptr(out), *[_lib.ptr(x) for x in grads],
                                                  _lib.ptr(per_sample), B, H, W, st), "t3d_mailbox_reduce")
                assert torch.count_nonzero(grads[1][1]) == 0 and torch.all(grads[0][0] == 1.5) and torch.all(grads[3][2] == 1.5)
            assert torch.equal(local, ref)
            assert torch.equal(out, ref * world), (world, step)


def test_two_rank_validity_matches_single_process(cuda_device):
    """Global validity semantics (train_thermal_dustr.py:320,357-360 over the data-parallel batch): two "ranks" of B
    samples each, one sample invalid on rank 1, exchanged through one shared mailbox, give every rank the gradients
    a single process computes on the 2B batch -- bit for bit (same kernels, same 1 / (2B) a-priori scale, same
    (2B) / n_valid factor) -- and the reduced vector equals the single process's packed vector."""
    import ctypes as C
    from thermal3d_vision_b200 import _lib
    from thermal3d_vision_b200 import loss as t3d
    lib = _lib.lib()
    B, H, W = 2, 40, 128
    P1, P2, G1, G2, C1, C2, T1, T2 = ref_loss.make_batch_inputs(2 * B, H, W, seed=31)
    P2[3, 4, 5, 0] = float("inf")                                    # global sample 3 = rank 1's sample 1
    d = [x.to(cuda_device) for x in (P1, P2, G1, G2, C1, C2, T1, T2)]
    st = _lib.current_stream_ptr()
    names = ("dpred1", "dpred2", "dconf1", "dconf2")

    # single process, batch 2B
    whole = t3d.fused_thermal_loss_fwd_bwd(*d, multi_scale=False, rescale_invalid=False, **KW)
    ref16 = torch.zeros(NVEC, dtype=torch.float64, device=cuda_device)
    _lib.check(lib.t3d_step_epilogue(*[_lib.ptr(whole[k]) for k in names], _lib.ptr(whole["per_sample"]), _lib.ptr(whole["batch"]),
                                     None, 2 * B, H, W, 0, 0, None, 0, _lib.ptr(ref16), st), "t3d_step_epilogue")
    assert whole["per_sample"][:, 5].tolist() == [1.0, 1.0, 1.0, 0.0]

    # two ranks of B samples: a-priori scale 1 / (B * world)
    mailbox = torch.zeros(int(lib.t3d_mailbox_bytes()) // 8, dtype=torch.float64, device=cuda_device)
    peers = (C.c_uint64 * 2)(mailbox.data_ptr(), mailbox.data_ptr())
    parts = []
    for rank in range(2):
        sl = slice(rank * B, (rank + 1) * B)
        r = t3d.fused_thermal_loss_fwd_bwd(*[x[sl].contiguous() for x in d], multi_scale=False, rescale_invalid=False,
                                           grad_scale=1.0 / (2 * B), **KW)
        local = torch.zeros(NVEC, dtype=torch.float64, device=cuda_device)
        _lib.check(lib.t3d_step_epilogue_peers(*[_lib.ptr(r[k]) for k in names], _lib.ptr(r["per_sample"]), _lib.ptr(r["batch"]),
                                               None, B, H, W, 0, None, 0, _lib.ptr(local), peers, 2, rank, 0, st), "t3d_step_epilogue_peers")
        parts.append(r)
    for rank in range(2):
        r = parts[rank]
        out = torch.zeros(NVEC, dtype=torch.float64, device=cuda_device)
        _lib.check(lib.t3d_mailbox_reduce(_lib.ptr(mailbox), 2, 0, _lib.ptr(out), *[_lib.ptr(r[k]) for k in names],
                                          _lib.ptr(r["per_sample"]), B, H, W, st), "t3d_mailbox_reduce")
        assert out[5].item() == 3.0 and out[6].item() == 4.0
        torch.testing.assert_close(out[:5], ref16[:5], rtol=1e-12, atol=0)      # sums of the same fp32 numbers, other order
        sl = slice(rank * B, (rank + 1) * B)
        for k in names:
            assert torch.equal(r[k], whole[k][sl]), (rank, k)
    assert torch.count_nonzero(parts[1]["dpred1"][1]) == 0 and torch.count_nonzero(parts[0]["dpred1"]) > 0


def test_pipelined_steps_equal_plain_steps(cuda_device):
    """pipelined=True (consecutive steps overlap on the internal streams, outputs alternate between two sets) gives
    the bits of the plain step, for every step of a sequence with changing inputs."""
    from thermal3d_vision_b200.pipeline import HotPathStep
    import bench
    B, H, W = 3, 96, 128
    seqs = [bench.make_inputs_torch(B, H, W, seed=40 + k, device=cuda_device, raw_hw=(128, 160)) for k in range(3)]
    order = [0, 1, 2, 1, 0]
    key = ("raw1", "raw2", "pred1", "pred2", "gt1", "gt2", "conf1", "conf2", "gt_depth")
    plain = HotPathStep(B, H, W, raw_hw=(128, 160), device=cuda_device, **KW)
    want = []
    for k in order:
        r = plain.run_device(*[seqs[k][n] for n in key]).clone()
        want.append((r, plain.loss_out["dpred1"].clone(), plain.loss_out["dconf2"].clone(), plain.pre_both["thermal"].clone()))
    piped = HotPathStep(B, H, W, raw_hw=(128, 160), device=cuda_device, pipelined=True, **KW)
    got = []
    for k in order:
        r = piped.run_device(*[seqs[k][n] for n in key])
        piped.wait_result(r)
        got.append((r.clone(), piped.loss_out["dpred1"].clone(), piped.loss_out["dconf2"].clone(), piped.pre_both["thermal"].clone()))
    # and without waiting in between: only the last two steps' sets are still around
    for k in order:
        r = piped.run_device(*[seqs[k][n] for n in key])
    piped.finish()
    torch.cuda.synchronize()
    for (a, b) in zip(want, got):
        for x, y in zip(a, b):
            assert torch.equal(x, y)
    assert torch.equal(r, want[-1][0]) and torch.equal(piped.loss_out["dpred1"], want[-1][1])


def test_bench_dump_outputs(cuda_device, tmp_path):
    """bench.py --dump-outputs: two runs with different step counts store the same outputs of their last timed step,
    and those are what one HotPathStep call on bench's inputs returns."""
    import json
    import os
    import subprocess
    import sys
    from thermal3d_vision_b200.pipeline import HotPathStep
    import bench
    B, H, W = 2, 64, 96
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dumps = []
    for steps in (2, 5):
        out = tmp_path / f"steps{steps}"
        res = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", str(steps), "--warmup", "0",
                              "--batch", str(B), "--height", str(H), "--width", str(W), "--no-extras", "--no-cpu-baseline",
                              "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-2000:]
        assert json.loads(res.stdout.strip().splitlines()[-1])["steps"] == steps
        dumps.append({f[:-4]: np.load(out / f) for f in sorted(os.listdir(out))})
    assert set(dumps[0]) == {"result", "per_sample", "batch", "metrics", "percentiles", "thermal",
                             "dpred1", "dpred2", "dconf1", "dconf2"}
    for name, a in dumps[0].items():
        assert a.dtype in (np.float32, np.float64), name
        np.testing.assert_array_equal(a, dumps[1][name], err_msg=name)
    d = bench.make_inputs_torch(B, H, W, seed=0, device=cuda_device)
    step = HotPathStep(B, H, W, device=cuda_device, pipelined=True, **KW)
    r = step.run_device(*[d[n] for n in bench.KEYS])
    step.finish()
    np.testing.assert_array_equal(dumps[0]["result"], r.cpu().numpy())
    for name in ("dpred1", "dpred2", "dconf1", "dconf2", "per_sample"):
        np.testing.assert_array_equal(dumps[0][name], step.loss_out[name].cpu().numpy(), err_msg=name)
    np.testing.assert_array_equal(dumps[0]["thermal"], step.pre_both["thermal"].cpu().numpy())
    np.testing.assert_array_equal(dumps[0]["metrics"], step.met_out["metrics_f64"].cpu().numpy())


def test_bench_configuration_matches_oracle(cuda_device):
    """The exact thing bench.py times -- HotPathStep at batch 64, 512x384 pointmaps, 640x512 raw frames from
    bench.make_inputs_torch, replicated-plane flag, statistics hand-off, internal streams, epilogue -- against the
    oracle loop (train_thermal_dustr.py:182-360 + utils/metrics.py:72-138 restated) on the same inputs."""
    from thermal3d_vision_b200.pipeline import HotPathStep
    import bench
    B, H, W = 64, 384, 512
    d = bench.make_inputs_torch(B, H, W, seed=0, device=cuda_device)
    key = ("raw1", "raw2", "pred1", "pred2", "gt1", "gt2", "conf1", "conf2", "gt_depth")
    step = HotPathStep(B, H, W, device=cuda_device, pipelined=True, **KW)
    for _ in range(3):                                   # as in the bench: steps in flight behind each other
        r = step.run_device(*[d[n] for n in key])
    step.finish()
    s = HotPathStep.summarize(r.cpu())
    c = {n: d[n].cpu() for n in key}
    T1, T2, mean, rows, valid, grads, metrics = _oracle_step(c["raw1"].numpy(), c["raw2"].numpy(), c["pred1"], c["pred2"],
                                                             c["gt1"], c["gt2"], c["conf1"], c["conf2"], c["gt_depth"], H, W, False)
    assert np.array_equal(step.pre_both["thermal"][:B].cpu().numpy(), T1.numpy())        # bit-exact preprocessing
    assert np.array_equal(step.pre_both["thermal"][B:].cpu().numpy(), T2.numpy())
    assert s["n_valid"] == B == float(valid.sum()) and s["n_images"] == B
    assert s["loss"] == pytest.approx(mean, rel=1e-5)
    np.testing.assert_allclose(step.loss_out["per_sample"][:, :5].cpu().numpy(), rows, rtol=1e-5)
    for name, ref in zip(("dpred1", "dpred2", "dconf1", "dconf2"), grads):
        got = step.loss_out[name].cpu()
        torch.testing.assert_close(got, ref, rtol=1e-4, atol=1e-6, msg=lambda m: f"{name}: {m}")
        # atol 1e-6 is loose at this size (|g| ~ 5e-6): also bound the error relative to the gradient's own scale
        scale = ref.abs().mean().item()
        assert (got - ref).abs().max().item() <= 2e-3 * scale, name
    for k in ref_metrics.KEYS7:
        assert s[k] == pytest.approx(metrics[k], rel=1e-5), k


def test_second_device(cuda_device):
    """Tensors on cuda:1 while cuda:0 is the current device: every entry point launches on the tensors' device
    (the library launches on the CURRENT device; the host side guards it).  Needs two GPUs."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from thermal3d_vision_b200.pipeline import HotPathStep
    import bench
    B, H, W = 2, 64, 128
    key = ("raw1", "raw2", "pred1", "pred2", "gt1", "gt2", "conf1", "conf2", "gt_depth")
    d0 = bench.make_inputs_torch(B, H, W, seed=3, device=torch.device("cuda:0"), raw_hw=(96, 160))
    a = HotPathStep(B, H, W, raw_hw=(96, 160), device="cuda:0", **KW).run_device(*[d0[n] for n in key]).cpu()
    assert torch.cuda.current_device() == 0
    d1 = {n: v.to("cuda:1") for n, v in d0.items()}
    both = torch.cat([d1["raw1"], d1["raw2"]])
    d1["raw1"], d1["raw2"] = both[:B], both[B:]
    step1 = HotPathStep(B, H, W, raw_hw=(96, 160), device="cuda:1", **KW)
    b = step1.run_device(*[d1[n] for n in key]).cpu()
    assert torch.cuda.current_device() == 0 and step1.loss_out["dpred1"].device.index == 1
    assert torch.equal(a, b)


def test_sobel_parameter_gradients_ride_the_exchange(cuda_device):
    """HotPathStep(sobel=True): ThermalDUSt3R's Sobel enhancer (thermal_dustr_model.py:110-142) in front of the model;
    the gradients of its two scalars -- the only parameters on this path -- travel in slots 16, 17 of the packed
    vector.  Single process: the enhanced batch and the gradients equal the reference arithmetic (oracle/ref_sobel +
    autograd) on the preprocessed thermal.  Two "ranks" of B pairs posting into one mailbox: the reduced slots are
    the sum over the ranks = the gradients of the 2B batch (the data-parallel gradient all-reduce of this path)."""
    import ctypes as C
    from oracle import ref_sobel
    from thermal3d_vision_b200 import _lib
    from thermal3d_vision_b200.pipeline import HotPathStep
    import bench
    lib = _lib.lib()
    B, H, W = 2, 64, 96
    key = ("raw1", "raw2", "pred1", "pred2", "gt1", "gt2", "conf1", "conf2", "gt_depth")
    g = torch.Generator(device=cuda_device).manual_seed(3)
    parts, want_e, want_t = [], 0.0, 0.0
    for rank in range(2):
        d = bench.make_inputs_torch(B, H, W, seed=70 + rank, device=cuda_device, raw_hw=(96, 160))
        dout = torch.randn(2 * B, 3, H, W, device=cuda_device, generator=g) / (2 * B * H * W)
        step = HotPathStep(B, H, W, raw_hw=(96, 160), device=cuda_device, sobel=True, **KW)
        r = step.run_device(*[d[n] for n in key], sobel_dout=dout).clone()
        # reference arithmetic on the same (bit-exact) preprocessed thermal
        th = step.pre_both["thermal"].cpu()
        ew, ts = torch.tensor(0.5, requires_grad=True), torch.tensor(1.0, requires_grad=True)
        ref = ref_sobel.preprocess_thermal_torch(th, ew, ts)
        (ref * dout.cpu()).sum().backward()
        torch.testing.assert_close(step.sobel_out["enhanced"].cpu(), ref.detach(), rtol=1e-6, atol=1e-6)
        assert r[16].item() == pytest.approx(ew.grad.item(), rel=1e-4, abs=1e-9)
        assert r[17].item() == pytest.approx(ts.grad.item(), rel=1e-4, abs=1e-9)
        assert r[18:].abs().sum().item() == 0.0 and r[15].item() == 0.0
        want_e += r[16].item(); want_t += r[17].item()
        parts.append((step, r))
    # the same two local vectors through the peer-memory exchange
    mailbox = torch.zeros(int(lib.t3d_mailbox_bytes()) // 8, dtype=torch.float64, device=cuda_device)
    peers = (C.c_uint64 * 2)(mailbox.data_ptr(), mailbox.data_ptr())
    st = _lib.current_stream_ptr()
    for rank, (step, r) in enumerate(parts):
        lo, me = step.loss_out, step.met_out
        local = torch.zeros(NVEC, dtype=torch.float64, device=cuda_device)
        _lib.check(lib.t3d_step_epilogue_peers(*[_lib.ptr(lo[k]) for k in ("dpred1", "dpred2", "dconf1", "dconf2")],
                                               _lib.ptr(lo["per_sample"]), _lib.ptr(lo["batch"]), _lib.ptr(me["metrics_f64"]),
                                               B, H, W, B, _lib.ptr(step.sobel_out["dparams"]), 2, _lib.ptr(local), peers, 2, rank, 0, st),
                   "t3d_step_epilogue_peers")
        assert torch.equal(local, r)
    out = torch.zeros(NVEC, dtype=torch.float64, device=cuda_device)
    _lib.check(lib.t3d_mailbox_reduce(_lib.ptr(mailbox), 2, 0, _lib.ptr(out), None, None, None, None, None, 0, 0, 0, st), "t3d_mailbox_reduce")
    assert torch.equal(out, parts[0][1] + parts[1][1])
    assert out[16].item() == want_e and out[17].item() == want_t and out[6].item() == 2 * B


def test_chain_phases_equal_the_whole_call(cuda_device):
    """T3D_PHASE_SAMPLE (thin sampling kernels, launched ahead of time by the pipelined step) followed by T3D_PHASE_REST
    gives the bits of the one-call form: same samples, same windows / brackets, same everything after."""
    from oracle import ref_preprocess
    from thermal3d_vision_b200 import _lib, metrics as tm, preprocessing as pp
    lib = _lib.lib()
    B, H, W = 6, 96, 160
    g = torch.Generator().manual_seed(5)
    pm = (torch.rand(B, H, W, 3, generator=g) * 5 + 0.3).to(cuda_device)
    gt = (torch.rand(B, H, W, generator=g) * 5).to(cuda_device)
    gt[1, :7] = 0.0
    pm[2, 3, 4, 2] = float("nan")
    a = tm.compute_depth_metrics_batch(pm, gt)
    out = {"state": torch.empty(lib.t3d_depth_metrics_state_bytes(B), dtype=torch.uint8, device=cuda_device),
           "workspace": torch.empty(lib.t3d_depth_metrics_workspace_bytes(B, H, W), dtype=torch.uint8, device=cuda_device)}
    assert tm.compute_depth_metrics_batch(pm, gt, out=out, phase=tm.PHASE_SAMPLE) is None
    b = tm.compute_depth_metrics_batch(pm, gt, out=out, phase=tm.PHASE_REST)
    assert torch.equal(a["metrics_f64"].view(torch.int64), b["metrics_f64"].view(torch.int64))
    assert torch.equal(a["medians"].view(torch.int32), b["medians"].view(torch.int32))
    # without a state block the sampling outputs live in the workspace
    out2 = {"workspace": out["workspace"]}
    tm.compute_depth_metrics_batch(pm, gt, out=out2, phase=tm.PHASE_SAMPLE)
    c = tm.compute_depth_metrics_batch(pm, gt, out=out2, phase=tm.PHASE_REST)
    assert torch.equal(a["metrics_f64"].view(torch.int64), c["metrics_f64"].view(torch.int64))

    raw = torch.from_numpy(ref_preprocess.make_raw_frames(4, seed=8)).to(cuda_device)
    for size in ((512, 384), (224, 224), (640, 512)):
        w, h = size
        ref = pp.preprocess_thermal_batch(raw, size, path="train", histogram=False)
        o = {"workspace": torch.empty(lib.t3d_preprocess_workspace_bytes(4, h, w), dtype=torch.uint8, device=cuda_device),
             "thermal": torch.empty(4, 3, h, w, device=cuda_device), "percentiles": torch.empty(4, 2, dtype=torch.float64, device=cuda_device),
             "grad_stats": torch.empty_like(ref.grad_stats) if ref.grad_stats is not None else None}
        pp.preprocess_thermal_batch(raw, size, path="train", histogram=False, out=o, phase=1)
        got = pp.preprocess_thermal_batch(raw, size, path="train", histogram=False, out=o, phase=2)
        assert torch.equal(ref.percentiles, got.percentiles), size
        assert torch.equal(ref.thermal, got.thermal), size
        if ref.grad_stats is not None:
            assert torch.equal(ref.grad_stats, got.grad_stats), size
    with pytest.raises(_lib.T3DError, match="phases"):
        pp.preprocess_thermal_batch(raw, (224, 224), path="train", histogram=True, phase=1)


def test_pipelined_soak_without_host_syncs(cuda_device):
    """60 pipelined steps enqueued back to back (no host synchronisation: the host runs ahead, the sampling kernels of
    step i+1 run during step i, output sets and metric streams alternate), two different input batches in an irregular
    order: every step's packed result and a stride of its thermal planes / gradients equal the plain step's bits."""
    import bench
    from thermal3d_vision_b200.pipeline import HotPathStep
    B, H, W = 4, 96, 256
    sets = [bench.make_inputs_torch(B, H, W, seed, cuda_device, raw_hw=(120, 320)) for seed in (0, 7)]
    args = [tuple(d[k] for k in bench.KEYS) for d in sets]
    plain = HotPathStep(B, H, W, raw_hw=(120, 320), device=cuda_device, pipelined=False)
    want = []
    for a in args:
        r = plain.run_device(*a).clone()
        torch.cuda.synchronize()
        want.append((r, plain.pre_both["thermal"].clone(), plain.loss_out["dpred2"].clone()))
    step = HotPathStep(B, H, W, raw_hw=(120, 320), device=cuda_device, pipelined=True)
    assert step.pipelined
    snaps, prev = [], None
    for k in range(60):
        j = (k * 5 // 2) & 1 if k % 3 else k & 1
        r = step.run_device(*args[j])
        if prev is not None:            # this call's lazy join ordered the stream after the previous step
            pj, pr, plo, ppre = prev
            snaps.append((pj, pr.clone(), ppre["thermal"].clone(), plo["dpred2"].clone()))
        prev = (j, r, step.loss_out, step.pre_both)
    step.finish()
    torch.cuda.synchronize()
    for n, (jj, rr, th, d2) in enumerate(snaps):
        assert torch.equal(rr.view(torch.int64), want[jj][0].view(torch.int64)), n
        assert torch.equal(th, want[jj][1]), n
        assert torch.equal(d2, want[jj][2]), n
