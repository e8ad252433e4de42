"""CPU, world_size 2 over gloo: the N>1 host logic (sharding by image, ONE packed all-reduce, summary)
reproduces the single-process result.  The per-rank numbers come from the oracle (no GPU here); the
packing layout is the one t3d_step_epilogue writes on the device (include/t3d.h)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import ref_loss, ref_metrics

KW = dict(alpha=0.2, edge_weight=0.5, smoothness_weight=0.3, detail_weight=0.4, multi_scale=False)


def _pack(rows, valid, metrics):
    """Host mirror of the device packing (test helper, same layout as t3d_step_epilogue)."""
    from thermal3d_vision_b200.distributed import RESULT_SIZE
    v = np.zeros(RESULT_SIZE)
    for r, ok in zip(rows, valid):
        if ok:
            v[0:5] += r[0:5]; v[5] += 1
    v[6] = len(rows)
    for m in metrics:
        for i, k in enumerate(ref_metrics.KEYS7):
            if np.isfinite(m[k]):
                v[7 + i] += m[k]
    v[14] = len(metrics)
    return v


def _rank_result(lo, hi, data):
    P1, P2, G1, G2, C1, C2, T1, T2 = (x[lo:hi] for x in data)
    _, rows, valid = ref_loss.batched_loss_torch(P1, P2, G1, G2, C1, C2, T1, T2, **KW)
    mets = [ref_metrics.compute_depth_metrics(P1[i, ..., 2].numpy(), G1[i, ..., 2].numpy()) for i in range(hi - lo)]
    return _pack(rows, valid, mets)


def _worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from thermal3d_vision_b200 import distributed as td
    data = ref_loss.make_batch_inputs(5, 24, 32, seed=1)
    data[0][3, 2, 2, 2] = float("nan")                     # one invalid sample, lands on rank 1
    lo, hi = td.shard_range(5, rank, world)
    vec = torch.from_numpy(_rank_result(lo, hi, data))
    td.all_reduce_result(vec)
    assert td.world() == (rank, world)
    assert td.global_grad_scale(3) == pytest.approx(1.0 / (3 * world))
    if rank == 0:
        q.put(vec.numpy())
    dist.destroy_process_group()


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def test_shard_range_is_a_partition():
    from thermal3d_vision_b200 import distributed as td
    for n in (0, 1, 5, 64, 20647):
        for w in (1, 2, 3, 8):
            rs = [td.shard_range(n, r, w) for r in range(w)]
            assert rs[0][0] == 0 and rs[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(rs, rs[1:]))
            sizes = [b - a for a, b in rs]
            assert max(sizes) - min(sizes) <= 1


def test_two_ranks_equal_one_process():
    from thermal3d_vision_b200 import distributed as td
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    data = ref_loss.make_batch_inputs(5, 24, 32, seed=1)
    data[0][3, 2, 2, 2] = float("nan")
    want = _rank_result(0, 5, data)
    np.testing.assert_allclose(got, want, rtol=1e-12)
    s = td.summarize(got)
    assert s["n_valid"] == 4 and s["n_pairs"] == 5 and s["n_images"] == 5
    # mean over VALID samples (train_thermal_dustr.py:359); metrics divided by ALL images (utils/metrics.py:134)
    mean, rows, valid = ref_loss.batched_loss_torch(*data, **KW)
    assert s["loss"] == pytest.approx(mean.item(), rel=1e-6)
