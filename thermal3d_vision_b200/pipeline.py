"""The hot path as one step: thermal preprocessing -> fused thermal-aware loss
(forward + backward) -> pointmap->depth + depth metrics, batched over B pairs.

This is the public API `bench.py` times.  One "pair" = one training sample =
two 16-bit thermal frames, two predicted and two pseudo-GT pointmaps with
confidences (train_thermal_dustr.py:136-360) + the depth metrics of view 1
(utils/metrics.py:72-138).  All arithmetic runs in libt3d_sm100.so; this class
only owns buffers, streams and the (optional) data-parallel all-reduce.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from . import _lib
from . import distributed as _dist
from . import loss as _loss
from . import metrics as _metrics
from . import preprocessing as _pre

RESULT_SIZE = 24   # packed result vector (float64): see HotPathStep.run_device


class HotPathStep:
    """One training-side step of the hot path on B pairs (see the module docstring).

    Streams.  The step runs on three internal streams -- preprocessing (the loss needs its thermal batches: the
    critical path), depth metrics (needed only by the step's epilogue) and loss + epilogue -- forked from the
    caller's stream at call time (the inputs are ready there).  Every per-step output exists twice and the two sets
    alternate, so consecutive steps may overlap: with ``pipelined=True`` the caller's stream is NOT ordered after the
    step by `run_device` itself but lazily (by the next call, after that call has forked its own work, or by
    `wait_result()` / `finish()`), which lets the preprocessing and metric kernels of step i + 1 fill the machine
    while the tail of step i (the loss kernel's last work items, its second-stage reduction, the epilogue) drains.
    Pipelined steps also SAMPLE AHEAD: the one-CTA-per-image sampling kernels at the head of both side chains (value
    windows for the percentiles, brackets for the medians) are launched for step i + 1 -- from its `run_device` call,
    on two more streams, in a thin 256-thread form -- while step i's streaming kernels run, so that step i + 1 starts
    with its heavy kernels when step i's loss kernel ends; the metric chains of consecutive steps alternate between
    two streams.  The first step after `finish()` has nothing in flight and samples inside its own chains.
    Every step still does all of its work on its own inputs; results are bit-identical to the plain step's.  With ``pipelined=False`` (default) the caller's stream
    waits for the step before `run_device` returns: plain stream semantics.  `loss_out`, `pre_both`, `met_out` and
    `result` always name the set of the latest call.

    Loss.  ``use_thermal_aware_loss=True`` (default) trains on the thermal-aware loss of utils/loss.py:100-305.
    ``False`` is train_thermal_dustr.py's other branch (:278-279,305-318, the run without --use_thermal_aware_loss):
    the plain confidence-weighted L1 with the confidence clamped from below only.  The thermal batches are still
    produced (they are the model's input) but the loss does not read them, and the preprocessing computes no
    thermal-gradient statistics; edge_weight / smoothness_weight / detail_weight do not apply and the packed vector's
    slots 2-4 are 0.  It has no multi-scale form.
    """

    def __init__(self, B: int, H: int, W: int, raw_hw=(512, 640), device=None, multi_scale: bool = False,
                 alpha=0.2, edge_weight=0.5, smoothness_weight=0.3, detail_weight=0.4, distributed: bool = False,
                 exchange: str = "peer", pipelined: bool = False, sobel: bool = False, gt_hw=None,
                 use_thermal_aware_loss: bool = True):
        if not use_thermal_aware_loss and multi_scale:
            raise ValueError("multi_scale is a form of the thermal-aware loss: use_thermal_aware_loss=False has none")
        self.use_thermal_aware_loss = bool(use_thermal_aware_loss)
        self.B, self.H, self.W, self.raw_hw = B, H, W, tuple(raw_hw)
        # pseudo-GT at its stored resolution (e.g. 512x512, scripts/pseudo_gt.py:620): the loss resamples it bilinearly
        # to (H, W) as train_thermal_dustr.py:234-271 does; None: the GT comes at (H, W)
        self.gt_hw = tuple(int(v) for v in gt_hw) if gt_hw is not None else None
        self.sobel = bool(sobel)
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.multi_scale = bool(multi_scale)
        self.kw = dict(alpha=alpha, edge_weight=edge_weight, smoothness_weight=smoothness_weight,
                       detail_weight=detail_weight, multi_scale=multi_scale)
        if not self.use_thermal_aware_loss:
            # train_thermal_dustr.py:305-318: no thermal terms, the confidence clamped from below only (:278-279)
            self.kw = dict(alpha=alpha, edge_weight=0.0, smoothness_weight=0.0, detail_weight=0.0, multi_scale=False,
                           conf_min_only=True)
        self.distributed = distributed
        self.pipelined = bool(pipelined)
        dev = self.device
        lib = _lib.lib()
        f32 = dict(dtype=torch.float32, device=dev)
        with _lib.device_guard(dev):
            self._alloc(lib, dev, f32, B, H, W, multi_scale)
            self._init_exchange(lib, dev, distributed, exchange)

    def _alloc(self, lib, dev, f32, B, H, W, multi_scale):
        # outputs / workspaces are allocated once (the library never allocates), twice each: steps alternate
        flags = _loss.LOSS_MULTI_SCALE if multi_scale else 0
        self.loss_sets = [{
            "workspace": torch.empty(lib.t3d_loss_workspace_bytes(B, H, W, flags), dtype=torch.uint8, device=dev),
            "per_sample": torch.empty(B, 8, **f32), "batch": torch.empty(8, **f32),
            "dpred1": torch.empty(B, H, W, 3, **f32), "dpred2": torch.empty(B, H, W, 3, **f32),
            "dconf1": torch.empty(B, H, W, **f32), "dconf2": torch.empty(B, H, W, **f32),
        } for _ in range(2)]
        # what the step exposes as its loss outputs, per set: the set itself, or -- a step whose confidences take no
        # gradient (pseudo-GT confidences at gt_hw, or none) -- the set without the dconf buffers the loss left unwritten
        self.loss_views = list(self.loss_sets)
        # both views are preprocessed by ONE call when the caller hands them over as the two halves of a single
        # [2B,...] tensor (what run_host's staging does): outputs are halves of one buffer as well
        self.pre_sets = [{
            "thermal": torch.empty(2 * B, 3, H, W, **f32),
            "percentiles": torch.empty(2 * B, 2, dtype=torch.float64, device=dev),
            "workspace": torch.empty(lib.t3d_preprocess_workspace_bytes(2 * B, H, W), dtype=torch.uint8, device=dev),
        } for _ in range(2)]
        if self.use_thermal_aware_loss:      # the thermal-gradient sums the loss reads (the plain loss reads none)
            for p in self.pre_sets:
                p["grad_stats"] = torch.empty(2 * B, max(lib.t3d_preprocess_stats_tiles(H, W), 1), 4, **f32)
        self._pre_halves = [None, None]      # separate-view fallback: allocated on first use
        self.met_sets = [{
            "workspace": torch.empty(lib.t3d_depth_metrics_workspace_bytes(B, H, W), dtype=torch.uint8, device=dev),
            "metrics": torch.empty(B, 8, **f32), "metrics_f64": torch.empty(B, 8, dtype=torch.float64, device=dev),
            "medians": torch.empty(B, 2, **f32),
        } for _ in range(2)]
        # scratch that lives inside one chain is shared by the two sets: the chains of consecutive steps run in order
        # on their own stream, only what the loss / the epilogue consume later exists twice.  (One metric workspace
        # also means ONE planar-Z scratch: the extraction pass parks it in the L2 for the sum pass, t3d_metrics.cu.)
        # Pipelined: the metric chains of consecutive steps alternate between two streams (and two workspaces), so that
        # step i+1's extraction pass does not queue behind the tail of step i's sum pass, which the loss kernel held
        # up (406.2 -> 403.4 us per step).
        if not self.pipelined:
            self.met_sets[1]["workspace"] = self.met_sets[0]["workspace"]
        # Sampling ahead (pipelined steps): the two chains' sampling kernels -- one CTA per image, latency-bound, 30 us
        # of nearly idle machine at the head of every step -- are launched for step i+1 as soon as its inputs are
        # known, in their thin form, on streams of their own: they run beside step i's streaming kernels, and at the
        # gate step i+1 starts with its heavy kernels.  What they write exists per set (the preprocessing workspace;
        # for the metric chain a small state block -- its big scratch stays shared).
        self._primed = False
        if self.pipelined:
            for m in self.met_sets:
                m["state"] = torch.empty(lib.t3d_depth_metrics_state_bytes(B), dtype=torch.uint8, device=dev)
        else:
            self.pre_sets[1]["workspace"] = self.pre_sets[0]["workspace"]
        self.loss_out, self.pre_both, self.met_out = self.loss_sets[0], self.pre_sets[0], self.met_sets[0]
        if self.sobel:
            # ThermalDUSt3R's Sobel enhancer in front of the model (thermal_dustr_model.py:110-142): its output is the
            # model's input, its two scalars (edge_weight 0.5, temp_scale 1.0, :104-107) are the only parameters on this
            # path -- their gradients ride along in the packed vector (slots 16, 17) and are summed over the ranks
            # with it: the data-parallel gradient all-reduce of this path.
            self.sobel_params = torch.tensor([0.5, 1.0], **f32)
            self.sobel_sets = [{"enhanced": torch.empty(2 * B, 3, H, W, **f32), "dparams": torch.zeros(2, **f32)} for _ in range(2)]
            self.sobel_ws = torch.empty(lib.t3d_sobel_workspace_bytes(2 * B, 3, H, W), dtype=torch.uint8, device=dev)
            self.sobel_out = self.sobel_sets[0]
        # preprocessing first in line for free SMs (the loss waits for it), the metric chain last (it has a whole
        # step of slack: only the epilogue needs it)
        try:
            lo_pri, hi_pri = torch.cuda.Stream.priority_range()      # (least, greatest), e.g. (0, -5)
        except Exception:
            lo_pri, hi_pri = 0, -1
        # the persistent loss kernel first (its CTAs must not queue behind the next step's preprocessing CTAs)
        self.s_loss = torch.cuda.Stream(device=dev, priority=hi_pri)
        self.s_pre = torch.cuda.Stream(device=dev, priority=min(hi_pri + 1, lo_pri))
        self.s_met = torch.cuda.Stream(device=dev, priority=lo_pri)
        self.s_met_alt = torch.cuda.Stream(device=dev, priority=lo_pri) if self.pipelined else self.s_met
        self.s_samp_p = torch.cuda.Stream(device=dev, priority=lo_pri)
        self.s_samp_m = torch.cuda.Stream(device=dev, priority=lo_pri)
        self.ev_sp = [torch.cuda.Event() for _ in range(2)]
        self.ev_sm = [torch.cuda.Event() for _ in range(2)]
        self.ev_ready = [torch.cuda.Event() for _ in range(2)]
        self.ev_pre = [torch.cuda.Event() for _ in range(2)]
        self.ev_met = [torch.cuda.Event() for _ in range(2)]
        self.ev_done = [torch.cuda.Event() for _ in range(2)]
        self.ev_main = [torch.cuda.Event() for _ in range(2)]     # the loss's main kernel of the step on set i has finished
        self._main_recorded = [False, False]
        self._joined = [True, True]          # the caller's stream has been ordered after the step that last used set i
        # percentiles from sampled value windows (bit-identical to the exact-histogram path, no per-pixel atomic);
        # set True to also get the 65 536-bin histograms of the resized frames in pre_both["histogram"]
        self.histogram = False
        self.results = [torch.zeros(RESULT_SIZE, dtype=torch.float64, device=dev) for _ in range(2)]
        self.pending = [None, None]
        self.calls = 0
        self.result = self.results[0]
        self.result_host = torch.zeros(RESULT_SIZE, dtype=torch.float64).pin_memory()
        self.staging = None        # two device staging sets of run_host (allocated on first use)

    def _init_exchange(self, lib, dev, distributed, exchange):
        # Data-parallel exchange of the packed result.  "peer" (NCCL process group on one NVLink node): every rank
        # owns a 4 KB mailbox in symmetric memory; the step's epilogue kernel stores the rank's 16 doubles straight
        # into every peer's mailbox and a small kernel adds them up one step later -- no collective call and no
        # host work per step beyond two launches (a per-step dist.all_reduce costs enough host time to make the
        # 0.43 ms step host-bound: 0.458 vs 0.435 ms).  "nccl": one asynchronous dist.all_reduce per step.
        # Either way the reduction also applies the GLOBAL validity factor to this rank's gradients
        # (train_thermal_dustr.py:320,357-360 over the whole data-parallel batch).
        self.exchange = None
        self.exchange_fallback = None
        self.reduced = [True, True]     # results[i] holds the global vector of the step that last used set i
        self.step_of = [-1, -1]
        if distributed and _dist.world()[1] > 1:
            if exchange not in ("peer", "nccl"):
                raise ValueError("exchange must be 'peer' or 'nccl'")
            self.exchange = exchange
        if self.exchange == "peer":
            import ctypes as C
            import warnings
            import torch.distributed as dist
            rank, world = _dist.world()
            if world > 16:
                raise ValueError("peer exchange: at most 16 ranks on one node (include/t3d.h T3D_MAX_PEERS)")
            nbytes = int(lib.t3d_mailbox_bytes())
            err = None
            try:
                import torch.distributed._symmetric_memory as symm_mem
                self.mailbox = symm_mem.empty(nbytes // 8, dtype=torch.float64, device=dev)
                self.mailbox.zero_()
                hdl = symm_mem.rendezvous(self.mailbox, dist.group.WORLD.group_name)
                self.peer_ptrs = (C.c_uint64 * world)(*[int(p) for p in hdl.buffer_ptrs])
                self._symm_handle = hdl
            except Exception as e:      # no peer-addressable memory on this system (e.g. GPUs without P2P access)
                err = e
            # the ranks must agree: one that cannot map its peers takes everybody to the NCCL exchange (still on the GPUs)
            ok = torch.tensor([0 if err is not None else 1], dtype=torch.int32, device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok.item()) == 0:
                warnings.warn(f"peer-memory exchange unavailable ({err!r}); using one NCCL all-reduce per step")
                self.exchange = "nccl"
                self.exchange_fallback = repr(err)
            else:
                self.local = [torch.zeros(RESULT_SIZE, dtype=torch.float64, device=dev) for _ in range(2)]
                torch.cuda.synchronize(dev)
                dist.barrier()                  # every mailbox is zeroed before anybody's first peer store
        if self.exchange == "nccl":
            self.local = [torch.zeros(RESULT_SIZE, dtype=torch.float64, device=dev) for _ in range(2)]

    # ------------------------------------------------------------------ bytes (SURVEY.md 8d)
    def algorithmic_bytes(self) -> Dict[str, int]:
        B, n = self.B, self.H * self.W
        raw = self.raw_hw[0] * self.raw_hw[1]
        # read 2x12 gt; with gt_hw: the source rows the bilinear y-taps touch, each read once
        gt = 24 * n if self.gt_hw is None else 24 * rows_touched(self.gt_hw[0], self.H) * self.gt_hw[1]
        # read 2x12 pred, the gt, 2x4 conf, 2x4 thermal (the 3 planes are replicas: one is read), write 32; the plain
        # loss reads no thermal
        per_px = 72 if self.use_thermal_aware_loss else 64
        return {
            "loss": B * (per_px * n + gt),
            "preprocess": 2 * B * (2 * raw + 12 * n),          # u16 frame in, 3 fp32 planes out
            "metrics": B * (12 * n + 4 * n + 64),              # pointmap (AoS sectors) + GT in, 64 B out
        }

    # ------------------------------------------------------------------ device-resident step
    def run_device(self, raw1, raw2, pred1, pred2, gt1, gt2, conf1, conf2, gt_depth, _ready=None, sobel_dout=None):
        """All inputs already in HBM (ready on the caller's current stream).  Returns the packed device result vector
        (float64): [0] sum of valid per-sample losses  [1..4] sums of components  [5] n_valid  [6] B
        [7..13] sums of finite per-image metrics (abs_rel..acc_3)  [14] n_images  [15] unused
        [16, 17] with sobel=True and `sobel_dout`: gradients of ThermalDUSt3R's edge_weight / temp_scale  [18..23] 0.
        With distributed=True the vector is summed over the ranks (peer-memory mailboxes, or one NCCL all-reduce with
        exchange="nccl") and the gradients carry the global validity factor once `wait_result()` / `finish()` / the
        next call has enqueued the reduction.  pipelined=True: see the class docstring -- call `wait_result()`
        before consuming this step's outputs on the caller's stream."""
        with _lib.device_guard(self.device):
            return self._run_device(raw1, raw2, pred1, pred2, gt1, gt2, conf1, conf2, gt_depth, _ready, sobel_dout)

    def _run_device(self, raw1, raw2, pred1, pred2, gt1, gt2, conf1, conf2, gt_depth, ready, sobel_dout=None):
        size = (self.W, self.H)
        B = self.B
        conf_grad = self._check_gt_hw(gt1, gt2, conf1, conf2) if self.gt_hw is not None else True
        lib = _lib.lib()
        main = torch.cuda.current_stream(self.device)
        i = self.calls & 1
        step_no = self.calls
        self.calls += 1
        lo, pre, met = self.loss_sets[i], self.pre_sets[i], self.met_sets[i]
        self.loss_views[i] = lo if conf_grad else dict(lo, dconf1=None, dconf2=None)
        self.loss_out, self.pre_both, self.met_out = self.loss_views[i], pre, met
        # fork: the inputs are ready on the caller's stream as of now (or, from run_host, when the H2D copies are done)
        if ready is None:
            ready = self.ev_ready[i]
            ready.record(main)
        # ... and only now order the caller's stream after the PREVIOUS step (lazy join): its tail overlaps this
        # step's preprocessing / metric kernels.  Set i was last used by step - 2, which the join of call - 1 covered.
        self._join(main)
        stacked = (raw1.is_contiguous() and raw2.is_contiguous() and raw1.shape == raw2.shape and
                   raw1.untyped_storage().data_ptr() == raw2.untyped_storage().data_ptr() and
                   raw2.storage_offset() == raw1.storage_offset() + raw1.numel())      # halves of one tensor
        if self.histogram and "histogram" not in pre:
            pre["histogram"] = torch.empty(2 * B, 65536, dtype=torch.int32, device=self.device)

        # pipelined: this step's side chains start when the PREVIOUS step's loss kernel has left the machine -- not
        # earlier (their CTAs would take SMs away from that persistent kernel), not later (its second-stage
        # reduction and epilogue, and this step's one-CTA-per-image sampling kernels, then run beside each other)
        gate = self.ev_main[i ^ 1] if (self.pipelined and self._main_recorded[i ^ 1]) else None
        raw_both = torch.as_strided(raw1, (2 * B,) + tuple(raw1.shape[1:]), raw1.stride(), raw1.storage_offset()) if stacked else None
        # (the first step after finish() has no step in flight to hide its sampling behind: it takes the one-call
        # form with the 1 024-thread sampling kernels, which are faster when they have the machine to themselves)
        ahead = self.pipelined and stacked and not self.histogram and self._primed
        self._primed = True
        if ahead:
            # ungated, on their own streams: ordered only after the inputs and after the last user of this set's
            # sampling state (step - 2: its preprocessing / metric chain)
            with torch.cuda.stream(self.s_samp_m):
                self.s_samp_m.wait_event(ready)
                self.s_samp_m.wait_event(self.ev_met[i])
                _metrics.compute_depth_metrics_batch(pred1, gt_depth, out=met, phase=_metrics.PHASE_SAMPLE)
                self.ev_sm[i].record(self.s_samp_m)
            with torch.cuda.stream(self.s_samp_p):
                self.s_samp_p.wait_event(ready)
                self.s_samp_p.wait_event(self.ev_pre[i])
                _pre.preprocess_thermal_batch(raw_both, size, path="train", out=pre, histogram=False,
                                              half_res_stats=self.multi_scale, phase=_metrics.PHASE_SAMPLE, shared=True,
                                              grad_stats=self.use_thermal_aware_loss)
                self.ev_sp[i].record(self.s_samp_p)
        phase = _metrics.PHASE_REST if ahead else _metrics.PHASE_ALL
        s_met = self.s_met_alt if (i & 1) else self.s_met
        with torch.cuda.stream(s_met):                      # depth metrics (Z of pred1 read in place)
            s_met.wait_event(ready)
            if gate is not None:
                s_met.wait_event(gate)
            if ahead:
                s_met.wait_event(self.ev_sm[i])
            me = _metrics.compute_depth_metrics_batch(pred1, gt_depth, out=met if ahead else {k: v for k, v in met.items() if k != "state"},
                                                      phase=phase)
            self.ev_met[i].record(s_met)
        with torch.cuda.stream(self.s_pre):                 # shared=True: the metric chain runs beside the preprocessing
            self.s_pre.wait_event(ready)
            if gate is not None:
                self.s_pre.wait_event(gate)
            if ahead:
                self.s_pre.wait_event(self.ev_sp[i])
            if stacked:
                tb = _pre.preprocess_thermal_batch(raw_both, size, path="train", out=pre, histogram=self.histogram,
                                                   half_res_stats=self.multi_scale, phase=phase, shared=True,
                                                   grad_stats=self.use_thermal_aware_loss)
                gs = tb.grad_stats
                stats_scales = tb.stats_scales
                (t1, t2), stats = (tb.thermal[:B], tb.thermal[B:]), ((None, None) if gs is None else (gs[:B], gs[B:]))
            else:
                if self._pre_halves[i] is None:
                    self._pre_halves[i] = [{k: (v[:B] if h == 0 else v[B:]) if k != "workspace" else
                                            torch.empty(lib.t3d_preprocess_workspace_bytes(B, self.H, self.W), dtype=torch.uint8,
                                                        device=self.device) for k, v in pre.items()} for h in range(2)]
                a = _pre.preprocess_thermal_batch(raw1, size, path="train", out=self._pre_halves[i][0], histogram=self.histogram,
                                                  half_res_stats=self.multi_scale, shared=True,
                                                  grad_stats=self.use_thermal_aware_loss)
                b = _pre.preprocess_thermal_batch(raw2, size, path="train", out=self._pre_halves[i][1], histogram=self.histogram,
                                                  half_res_stats=self.multi_scale, shared=True,
                                                  grad_stats=self.use_thermal_aware_loss)
                (t1, t2), stats = (a.thermal, b.thermal), (a.grad_stats, b.grad_stats)
                stats_scales = min(a.stats_scales, b.stats_scales)
            pgrads, n_pgrads = None, 0
            if self.sobel:
                # the model's input: Sobel-enhanced thermal of both views ([2B,3,H,W], view 1 first); given the
                # upstream gradient w.r.t. it (`sobel_dout`, what the model's backward hands back), the gradients
                # of the enhancer's two scalars
                so = self.sobel_sets[i]
                self.sobel_out = so
                th_both = pre["thermal"] if stacked else torch.cat([t1, t2])
                st = _lib.current_stream_ptr()
                rc = lib.t3d_sobel_enhance_fwd(_lib.ptr(th_both), _lib.ptr(self.sobel_params), 2 * B, 3, self.H, self.W, 1,
                                               _lib.ptr(so["enhanced"]), _lib.ptr(self.sobel_ws), self.sobel_ws.numel(), st)
                _lib.check(rc, "t3d_sobel_enhance_fwd")
                if sobel_dout is not None:
                    if tuple(sobel_dout.shape) != (2 * B, 3, self.H, self.W) or sobel_dout.dtype != torch.float32 \
                            or not sobel_dout.is_contiguous():
                        raise ValueError("sobel_dout must be a contiguous float32 [2B,3,H,W] tensor")
                    rc = lib.t3d_sobel_enhance_bwd_params(_lib.ptr(th_both), _lib.ptr(self.sobel_params), _lib.ptr(sobel_dout),
                                                          2 * B, 3, self.H, self.W, 1, _lib.ptr(so["dparams"]),
                                                          _lib.ptr(self.sobel_ws), self.sobel_ws.numel(), st)
                    _lib.check(rc, "t3d_sobel_enhance_bwd_params")
                    pgrads, n_pgrads = _lib.ptr(so["dparams"]), 2
            self.ev_pre[i].record(self.s_pre)
        with torch.cuda.stream(self.s_loss):
            self.s_loss.wait_event(ready)                   # pred / gt / conf
            self.s_loss.wait_event(self.ev_pre[i])
            # the normalisation kernel already summed the thermal gradients: the loss skips its statistics pass
            if self.pipelined and not self._main_recorded[i]:
                self.ev_main[i].record(self.s_loss)              # creates the CUDA event behind the torch object
                self._main_recorded[i] = True
            # (the plain loss: the thermal batches are the model's input only)
            lt1, lt2 = (t1, t2) if self.use_thermal_aware_loss else (None, None)
            _loss.fused_thermal_loss_fwd_bwd(pred1, pred2, gt1, gt2, conf1, conf2, lt1, lt2, conf_grad=conf_grad,
                                             out=lo, thermal_stats=stats, thermal_stats_scales=stats_scales,
                                             main_done_event=self.ev_main[i] if self.pipelined else None,
                                             thermal_replicated=True,   # preprocess_thermal_batch wrote 3 identical planes
                                             grad_scale=_dist.global_grad_scale(self.B) if self.distributed else None,
                                             rescale_invalid=False,     # done by the epilogue below
                                             **self.kw)
            self.s_loss.wait_event(self.ev_met[i])
            stream = _lib.current_stream_ptr()
            grads = [_lib.ptr(self.loss_views[i][k]) for k in ("dpred1", "dpred2", "dconf1", "dconf2")]
            if self.exchange == "peer":
                # reduce(step - 1) is enqueued before epilogue(step): the order that makes the two mailbox slots reusable
                self._reduce_pending()
                rank, world = _dist.world()
                rc = lib.t3d_step_epilogue_peers(*grads, _lib.ptr(lo["per_sample"]), _lib.ptr(lo["batch"]),
                                                 _lib.ptr(me["metrics_f64"]), B, self.H, self.W, B, pgrads, n_pgrads,
                                                 _lib.ptr(self.local[i]), self.peer_ptrs, world, rank, step_no, stream)
                _lib.check(rc, "t3d_step_epilogue_peers")
                self.reduced[i] = False
                self.step_of[i] = step_no
            elif self.exchange == "nccl":
                self._reduce_pending()
                # validity: zero the invalid samples now, the global factor follows the all-reduce (t3d_rescale_global)
                rc = lib.t3d_step_epilogue(*grads, _lib.ptr(lo["per_sample"]), _lib.ptr(lo["batch"]),
                                           _lib.ptr(me["metrics_f64"]), B, self.H, self.W, B, 1, pgrads, n_pgrads,
                                           _lib.ptr(self.results[i]), stream)
                _lib.check(rc, "t3d_step_epilogue")
                self.local[i].copy_(self.results[i])
                self.pending[i] = _dist.all_reduce_result(self.results[i], async_op=True)
                self.reduced[i] = False
                self.step_of[i] = step_no
            else:
                # validity fix-up of the gradients + packing of the step's scalars: one launch
                rc = lib.t3d_step_epilogue(*grads, _lib.ptr(lo["per_sample"]), _lib.ptr(lo["batch"]),
                                           _lib.ptr(me["metrics_f64"]), B, self.H, self.W, B, 0, pgrads, n_pgrads,
                                           _lib.ptr(self.results[i]), stream)
                _lib.check(rc, "t3d_step_epilogue")
            self.ev_done[i].record(self.s_loss)
        self._joined[i] = False
        self.result = self.results[i]
        if not self.pipelined:
            self._join(main)
        return self.result

    def _check_gt_hw(self, gt1, gt2, conf1, conf2) -> bool:
        """Shapes of a step with gt_hw; returns whether the confidences are predicted ones (at (H, W): they take a
        gradient) -- at gt_hw they are pseudo-GT confidences (train_thermal_dustr.py:274-275), None means ones."""
        B, H, W = self.B, self.H, self.W
        want = (B,) + self.gt_hw + (3,)
        for name, g in (("gt1", gt1), ("gt2", gt2)):
            if tuple(g.shape) != want:
                raise ValueError(f"{name} must be {want} (gt_hw={self.gt_hw}), got {tuple(g.shape)}")
        if conf1 is None and conf2 is None:
            return False
        shapes = {None if c is None else tuple(c.shape) for c in (conf1, conf2)}
        if len(shapes) != 1 or shapes.pop() not in ((B, H, W), (B,) + self.gt_hw):
            raise ValueError(f"conf1 / conf2 must both be [B,H,W]={B, H, W} or [B,*gt_hw]={(B,) + self.gt_hw}, got "
                             f"{None if conf1 is None else tuple(conf1.shape)} / {None if conf2 is None else tuple(conf2.shape)}")
        return tuple(conf1.shape[1:3]) == (H, W)

    def _join(self, main):
        """Order `main` after every step it has not been ordered after yet (not after their pending reductions)."""
        for k in range(2):
            if not self._joined[k]:
                main.wait_event(self.ev_done[k])
                self._joined[k] = True

    def capture_graph(self, raw1, raw2, pred1, pred2, gt1, gt2, conf1, conf2, gt_depth):
        """Capture one `run_device` on these (static) device tensors into a CUDA graph and return `replay()`, which
        re-runs the whole step (three streams, ~15 kernels) with one launch and returns the packed result vector.
        For launch-bound shapes (BASELINE configs[1]: batch 8 at 224x224 is ~45 MB of traffic, a few microseconds
        of HBM time) this is what removes the per-kernel launch latency.  Single-process only (the exchange of a
        distributed step is issued outside any graph).  The captured step always uses output set 0."""
        if self.distributed:
            raise ValueError("capture_graph is for single-process steps")
        args = (raw1, raw2, pred1, pred2, gt1, gt2, conf1, conf2, gt_depth)
        pipelined, self.pipelined = self.pipelined, False
        with _lib.device_guard(self.device):
            cur = torch.cuda.current_stream(self.device)
            warm = torch.cuda.Stream(device=self.device)
            warm.wait_stream(cur)
            with torch.cuda.stream(warm):
                for _ in range(2):                     # one-time attribute / occupancy queries happen outside the capture
                    self.run_device(*args)
            cur.wait_stream(warm)
            torch.cuda.synchronize(self.device)
            self.calls = 0                             # the captured step writes set 0
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                r = self.run_device(*args)
        self.pipelined = pipelined
        sets = (self.loss_views[0], self.pre_sets[0], self.met_sets[0])

        def replay():
            graph.replay()
            self.loss_out, self.pre_both, self.met_out = sets
            self.result = r
            return r
        replay.graph = graph
        return replay

    def _reduce_pending(self):
        """Data parallel: enqueue (on the loss stream) the reduction of every step whose global vector has not been
        formed yet, oldest first -- it also applies the global validity factor to that step's gradients."""
        if self.exchange is None:
            return
        lib, world = _lib.lib(), _dist.world()[1]
        with torch.cuda.stream(self.s_loss):
            stream = _lib.current_stream_ptr()
            for i in sorted(range(2), key=lambda k: self.step_of[k]):
                if self.reduced[i]:
                    continue
                lo = self.loss_views[i]
                grads = [_lib.ptr(lo[k]) for k in ("dpred1", "dpred2", "dconf1", "dconf2")]
                if self.exchange == "peer":
                    rc = lib.t3d_mailbox_reduce(_lib.ptr(self.mailbox), world, self.step_of[i], _lib.ptr(self.results[i]),
                                                *grads, _lib.ptr(lo["per_sample"]), self.B, self.H, self.W, stream)
                    _lib.check(rc, "t3d_mailbox_reduce")
                else:
                    self.pending[i].wait()             # orders the loss stream after the all-reduce
                    self.pending[i] = None
                    rc = lib.t3d_rescale_global(*grads, _lib.ptr(lo["per_sample"]), _lib.ptr(self.results[i]),
                                                self.B, self.H, self.W, stream)
                    _lib.check(rc, "t3d_rescale_global")
                self.reduced[i] = True
                self.ev_done[i].record(self.s_loss)    # "done" now includes the reduction
                self._joined[i] = False

    def wait_result(self, r: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Order the current stream after the step that produced `r` (default: the latest), including -- data
        parallel -- its reduction over the ranks and the global validity fix-up of its gradients."""
        r = self.result if r is None else r
        with _lib.device_guard(self.device):
            self._reduce_pending()
            self._join(torch.cuda.current_stream(self.device))
        return r

    def finish(self):
        """Order the current stream after every outstanding step / reduction (end of a run / of a timed region)."""
        self.wait_result()
        self._primed = False        # nothing in flight any more: the next step samples inside its own chains

    # ------------------------------------------------------------------ host-buffer step (e2e)
    def run_host(self, host: Dict[str, torch.Tensor]):
        """Inputs are PINNED HOST tensors (raw1, raw2 uint16; pred1, pred2, gt1, gt2, conf1, conf2, gt_depth float32).
        Copies them to the device, runs the step, copies the packed result back to pinned host memory.
        Asynchronous; `result_host` is valid after a synchronise of the current stream.

        The H2D copies go through a dedicated copy stream into one of two staging sets, so the copies of call
        i + 1 overlap the kernels of call i (the step is PCIe-bound: 839 MB of inputs per call at batch 64);
        every call still copies all of its own inputs and reads its own result back."""
        with _lib.device_guard(self.device):
            return self._run_host(host)

    def _run_host(self, host):
        dev = self.device
        main = torch.cuda.current_stream(dev)
        if self.staging is None:
            self.staging = []
            for _ in range(2):
                st = {k: torch.empty(v.shape, dtype=v.dtype, device=dev) for k, v in host.items() if k not in ("raw1", "raw2")}
                both = torch.empty((2 * self.B,) + tuple(host["raw1"].shape[1:]), dtype=host["raw1"].dtype, device=dev)
                st["raw1"], st["raw2"] = both[:self.B], both[self.B:]
                self.staging.append(st)
            self.copy_stream = torch.cuda.Stream(device=dev)
            self.copied = [torch.cuda.Event() for _ in range(2)]
            self.consumed = [torch.cuda.Event() for _ in range(2)]
            self.host_calls = 0
        i = self.host_calls & 1
        s = self.staging[i]
        with torch.cuda.stream(self.copy_stream):
            if self.host_calls >= 2:
                self.copy_stream.wait_event(self.consumed[i])      # the kernels of call - 2 are done with this set
            else:
                self.copy_stream.wait_stream(main)
            for k, v in host.items():
                s[k].copy_(v, non_blocking=True)
            self.copied[i].record(self.copy_stream)
        r = self._run_device(s["raw1"], s["raw2"], s["pred1"], s["pred2"], s["gt1"], s["gt2"], s["conf1"], s["conf2"],
                             s["gt_depth"], self.copied[i])
        self.wait_result(r)
        self.consumed[i].record(main)
        self.result_host.copy_(r, non_blocking=True)
        self.host_calls += 1
        return self.result_host

    @staticmethod
    def h2d_bytes(host: Dict[str, torch.Tensor]) -> int:
        return int(sum(v.numel() * v.element_size() for v in host.values()))

    @staticmethod
    def summarize(result_host: torch.Tensor) -> Dict[str, float]:
        return _dist.summarize(result_host.tolist())


def rows_touched(src: int, dst: int) -> int:
    """Source rows that the bilinear y-taps of `dst` output rows read (F.interpolate, align_corners=False; the fp32
    tap arithmetic of t3d_bilinear.cuh, one rounding for scale * (y + 0.5) - 0.5)."""
    import numpy as np
    scale = float(np.float32(src) / np.float32(dst))
    y = np.arange(dst, dtype=np.float64)
    f = np.maximum((scale * (y + 0.5) - 0.5).astype(np.float32), np.float32(0))   # exact in fp64, then one rounding
    i0 = f.astype(np.int64)
    i1 = i0 + (i0 < src - 1)
    return int(np.unique(np.concatenate([i0, i1])).size)


class EvalStep:
    """BASELINE.json configs[4]: full-resolution 16-bit frames -> preprocessing (the model's input) and, for the
    model's pointmaps (the caller's; synthetic in bench.py), pointmap -> depth -> depth metrics against the GT
    depth, accumulated over a dataset shard with the reference's semantics (utils/metrics.py:86-136: finite
    per-image metrics summed, divided by the count of ALL images).  One rank = one contiguous shard
    (distributed.shard_range); `finish()` does the single all-reduce of the 8-double accumulator.

    path='train': data/dataset_loader.py:237-249 + enhance_thermal_contrast (u16 resize, raw counts);
    path='inference': utils/evaluate_depth_metrics.py:162-197 (/65535, float resize, float percentiles).
    GT depth of another size is nearest-resampled inside the metric kernels (utils/evaluate_depth_metrics.py:320-323).
    """

    def __init__(self, B: int, H: int, W: int, raw_hw=(512, 640), gt_hw=None, device=None, path: str = "train"):
        self.B, self.H, self.W, self.raw_hw, self.path = B, H, W, tuple(raw_hw), path
        self.gt_hw = tuple(gt_hw) if gt_hw is not None else (H, W)
        self.device = torch.device(device if device is not None else "cuda")
        dev, lib = self.device, _lib.lib()
        f32 = dict(dtype=torch.float32, device=dev)
        # every buffer twice: batches alternate, so that `prefetch` can sample batch k+1 while batch k is in flight and
        # the thermal batch a call returns stays valid until the call after the next one
        self.pre_sets = [{"thermal": torch.empty(B, 3, H, W, **f32),
                          "percentiles": torch.empty(B, 2, dtype=torch.float64, device=dev),
                          "workspace": torch.empty(lib.t3d_preprocess_workspace_bytes(B, H, W), dtype=torch.uint8, device=dev)}
                         for _ in range(2)]
        self.met_sets = [{"workspace": torch.empty(lib.t3d_depth_metrics_workspace_bytes(B, H, W), dtype=torch.uint8, device=dev),
                          "state": torch.empty(lib.t3d_depth_metrics_state_bytes(B), dtype=torch.uint8, device=dev),
                          "metrics": torch.empty(B, 8, **f32), "metrics_f64": torch.empty(B, 8, dtype=torch.float64, device=dev),
                          "medians": torch.empty(B, 2, **f32)} for _ in range(2)]
        self.pre_out, self.met_out = self.pre_sets[0], self.met_sets[0]
        self.acc = _metrics.MetricAccumulator(dev)
        self.side = torch.cuda.Stream(device=dev, priority=-1)
        self.s_samp_p = torch.cuda.Stream(device=dev)
        self.s_samp_m = torch.cuda.Stream(device=dev)
        self.fork, self.join = torch.cuda.Event(), torch.cuda.Event()
        self.ev_ready = [torch.cuda.Event() for _ in range(2)]
        self.ev_sp = [torch.cuda.Event() for _ in range(2)]
        self.ev_sm = [torch.cuda.Event() for _ in range(2)]
        self.ev_pre_done = [torch.cuda.Event() for _ in range(2)]
        self.ev_met_done = [torch.cuda.Event() for _ in range(2)]
        self._next = 0
        self._prefetched = []          # [(raw ptr, pointmap ptr or None, set)], oldest first

    def algorithmic_bytes(self) -> int:
        """Per batch: u16 frame in + 3 fp32 planes out, AoS pointmap + GT depth in (SURVEY.md 8d)."""
        n, raw, gt = self.H * self.W, self.raw_hw[0] * self.raw_hw[1], self.gt_hw[0] * self.gt_hw[1]
        return self.B * ((2 * raw + 12 * n) + (12 * n + 4 * min(gt, n) + 64))

    def prefetch(self, raw, pointmap=None, gt_depth=None):
        """Sample a FUTURE batch ahead of time (train path): launches only the sampling kernels of the two chains for
        these tensors, in their thin form and on streams of their own, so that they run beside the streaming kernels
        of the batch in flight; the `run_batch` call for the same tensors then starts with its heavy kernels.  Call it
        BEFORE the `run_batch` of the batch in front (what is recorded now is that the inputs are ready now).  In a
        real evaluation loop the raw frames of batch k+1 are known while the model still works on batch k -- the
        pointmap is not: pass `pointmap=None` and only the preprocessing is sampled ahead."""
        if self.path != "train":
            return
        with _lib.device_guard(self.device):
            j = self._next
            self._next ^= 1
            main = torch.cuda.current_stream(self.device)
            self.ev_ready[j].record(main)
            with torch.cuda.stream(self.s_samp_p):
                self.s_samp_p.wait_event(self.ev_ready[j])
                self.s_samp_p.wait_event(self.ev_pre_done[j])          # the last batch on this set is done with it
                _pre.preprocess_thermal_batch(raw, (self.W, self.H), path="train", out=self.pre_sets[j], histogram=False,
                                              phase=_metrics.PHASE_SAMPLE, shared=True)
                self.ev_sp[j].record(self.s_samp_p)
            if pointmap is not None:
                with torch.cuda.stream(self.s_samp_m):
                    self.s_samp_m.wait_event(self.ev_ready[j])
                    self.s_samp_m.wait_event(self.ev_met_done[j])
                    _metrics.compute_depth_metrics_batch(pointmap, gt_depth, out=self.met_sets[j], phase=_metrics.PHASE_SAMPLE)
                    self.ev_sm[j].record(self.s_samp_m)
            self._prefetched.append((raw.data_ptr(), pointmap.data_ptr() if pointmap is not None else None, j))

    def run_batch(self, raw, pointmap, gt_depth):
        """raw [B,Hs,Ws] uint16, pointmap [B,H,W,3] float32, gt_depth [B,gh,gw] float32, all on the device.
        Returns the preprocessed thermal batch [B,3,H,W] (valid until the call after the next one); the metrics go
        into the accumulator.  No host sync."""
        with _lib.device_guard(self.device):
            main = torch.cuda.current_stream(self.device)
            pre_phase = met_phase = _metrics.PHASE_ALL
            if self._prefetched and self._prefetched[0][0] == raw.data_ptr():
                _, pm_ptr, j = self._prefetched.pop(0)
                pre_phase = _metrics.PHASE_REST
                if pm_ptr is not None and pm_ptr == pointmap.data_ptr():
                    met_phase = _metrics.PHASE_REST
            else:
                self._prefetched.clear()                # not what was sampled ahead: start over
                j = self._next
                self._next ^= 1
            pre, met = self.pre_sets[j], self.met_sets[j]
            self.pre_out, self.met_out = pre, met
            self.fork.record(main)
            with torch.cuda.stream(self.side):
                self.side.wait_event(self.fork)
                self.side.wait_event(self.ev_sm[j])          # this batch's sampling -- or a stale one on this set: let it finish
                self.side.wait_event(self.ev_met_done[j])
                me = _metrics.compute_depth_metrics_batch(pointmap, gt_depth, out=met, phase=met_phase)
                self.join.record(self.side)
                self.ev_met_done[j].record(self.side)
            main.wait_event(self.ev_sp[j])                   # likewise for the preprocessing's sampling state
            # shared=True: the metric pipeline runs beside the preprocessing (side stream)
            tb = _pre.preprocess_thermal_batch(raw, (self.W, self.H), path=self.path, out=pre, histogram=False, phase=pre_phase,
                                               shared=True)
            self.ev_pre_done[j].record(main)
            main.wait_event(self.join)
            self.acc.update(me["metrics_f64"])
            return tb.thermal

    def finish(self) -> Dict[str, float]:
        """All-reduce (SUM) the accumulator over the ranks and return the dataset-mean metrics (host sync)."""
        return self.acc.all_reduce().result()
