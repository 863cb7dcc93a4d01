"""One optimisation step of the ScorePerformer model as a reusable object: forward, backward, (all-reduce), clip, AdamW.

Mirrors what `Trainer.run_epoch` + `Optimizer.step` do per batch (experiments/trainer.py:449-452, optimizers.py:151-169:
backward, `clip_grad_norm_(2.0)`, AdamW(lr 2e-4, wd 1e-6), `zero_grad`) with two B200-first changes:

* parameters, gradients, both AdamW moments and a bf16 weight shadow live in flat buffers (every `p.data` / `p.grad` is a
  view), so data parallelism is a single NCCL all-reduce of 46 MB over NVLink per step and the optimiser is ONE kernel:
  clip-by-global-norm + AdamW in one pass over memory (csrc/optim.cu); weight-gradient kernels accumulate
  straight into the gradient buffer (fused.DIRECT_GRAD) and ONE cast kernel per step refreshes the bf16 shadow every
  forward GEMM reads its weight from (fused.SHADOW_ACTIVE);
* forward + backward (the whole kernel sequence, ~1 000 launches) is captured once in a CUDA graph and replayed, because
  at ~15 ms per step the Python dispatch of the eager path (~19 ms) would otherwise be the bottleneck.  Dropout stays
  random across replays through a device-side counter mixed into the kernels' seeds (kernels.RNG_OFFSET); the learning rate is a
  device scalar (`set_lr` never re-captures); one graph is kept per batch-shape signature, so a short last batch or another
  sequence length gets its own capture instead of a shape error.
* data parallelism (SURVEY section 8 row e): the gradient all-reduce is part of the step -- captured in the same graph -- and
  bucketed by transformer stack: the moment a stack's backward node has finished (its weight gradients are final), that
  stack's slice of the flat gradient buffer is handed to NCCL on the communication stream while the backward of the layers
  below it keeps running; the remaining slices (embeddings, heads, latent levels, classifiers) follow after backward, and the
  clip + AdamW kernel waits for all of them.  Buckets are issued in a fixed order on every rank.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch
import torch.distributed as dist
from torch import Tensor

import os

from . import fused, kernels as K
from .utils import join_side_streams


class TrainStep:
    def __init__(self, model: torch.nn.Module, lr: float = 2e-4, weight_decay: float = 1e-6, grad_clip: Optional[float] = 2.0,
                 use_graph: bool = True, process_group=None, betas=(0.9, 0.999), eps: float = 1e-8):
        self.model = model
        self.grad_clip = grad_clip
        self.lr, self.weight_decay, self.betas, self.eps = lr, weight_decay, tuple(betas), eps
        self.use_graph = use_graph
        self.group = process_group
        self.world = dist.get_world_size(process_group) if dist.is_initialized() else 1
        self.params = [p for p in model.parameters() if p.requires_grad]
        dev = self.params[0].device
        if not dev.type == "cuda":
            raise RuntimeError("TrainStep needs a CUDA model: scoreperformer_b200 has no CPU fallback")
        # parameters, gradients and the bf16 weight shadow are three flat buffers with identical layouts (offsets rounded to
        # 8 elements so every bf16 view is 16-byte aligned for TMA)
        offsets, n = [], 0
        for p in self.params:
            offsets.append(n)
            n += (p.numel() + 7) // 8 * 8
        self.flat_param = torch.zeros(n, dtype=torch.float32, device=dev)
        self.flat_grad = torch.zeros(n, dtype=torch.float32, device=dev)
        self.flat_shadow = torch.zeros(n, dtype=torch.bfloat16, device=dev)
        for p, off in zip(self.params, offsets):
            view = self.flat_param[off:off + p.numel()].view_as(p)
            view.copy_(p.data)
            p.data = view
            p.grad = self.flat_grad[off:off + p.numel()].view_as(p)
            p._spb_shadow = self.flat_shadow[off:off + p.numel()].view_as(p)
        self.offsets = offsets
        self.flat_m = torch.zeros(n, dtype=torch.float32, device=dev)        # AdamW exp_avg
        self.flat_v = torch.zeros(n, dtype=torch.float32, device=dev)        # AdamW exp_avg_sq
        self.opt_step = torch.zeros(1, dtype=torch.int64, device=dev)        # device-side step number (CUDA-graph safe)
        self.lr_dev = torch.full((1,), float(lr), dtype=torch.float32, device=dev)      # device-side learning rate
        if use_graph and getattr(model, "perf_encoder", None) is not None:
            model.perf_encoder.exact_latent_shapes = False      # static segment tables: the step must not sync with the host
        self.rng_offset = torch.zeros(1, dtype=torch.int64, device=dev)
        K.RNG_OFFSET = self.rng_offset
        self.graph: Optional[torch.cuda.CUDAGraph] = None                    # the graph of the current batch-shape signature
        self.static_batch: Optional[Dict[str, Tensor]] = None
        self.static_loss: Optional[Tensor] = None
        self.static_losses: Optional[Dict[str, Tensor]] = None
        self._graphs: Dict[tuple, tuple] = {}                                # signature -> (graph, batch, loss, losses, metrics)
        self._static_metrics = None
        self._update_in_graph = True
        self._sig: Optional[tuple] = None
        self.evaluator = None                                                # set_evaluator(): metrics computed inside the step
        self.metrics: Optional[Dict[str, Tensor]] = None
        self._shadow_stale = True                                            # bf16 weight shadow must be rebuilt from the fp32 weights
        # gradient buckets of the data-parallel all-reduce: [lo, hi) slices of the flat buffer, one per transformer stack
        self.overlap = self.world > 1 and os.environ.get("SPB_DDP_OVERLAP", "1") == "1"
        self.graph_update = os.environ.get("SPB_DDP_GRAPH", "1") == "1"      # world > 1: all-reduce + AdamW inside the graph
        self._buckets = self._stack_buckets() if self.overlap else []
        self._bucket_of = {id(prm): i for i, (_, _, prms) in enumerate(self._buckets) for prm in prms}
        self._ready = [False] * len(self._buckets)
        self._next_bucket = 0
        self._works = []
        self.launches_per_step = 0
        self._warm = 0
        self._copy_stream = None
        self._stage: Optional[Dict[str, Tensor]] = None
        self._pstage: Optional[Dict[str, Tensor]] = None
        self._pspec = None
        self._packed_pending = False

    # ------------------------------------------------------------------ pieces
    def _stack_buckets(self):
        """One bucket per transformer stack: the contiguous slice of the flat buffers that holds its parameters."""
        from .modules.transformer.transformer import Transformer
        index = {id(p): i for i, p in enumerate(self.params)}
        buckets = []
        for mod in self.model.modules():
            if not isinstance(mod, Transformer):
                continue
            ids = sorted(index[id(p)] for p in mod.parameters() if id(p) in index)
            if not ids or ids[-1] - ids[0] + 1 != len(ids):
                continue                                   # not contiguous (shared parameters): stays in the tail reduction
            lo = self.offsets[ids[0]]
            last = self.params[ids[-1]]
            hi = self.offsets[ids[-1]] + (last.numel() + 7) // 8 * 8
            buckets.append((lo, hi, [self.params[i] for i in ids]))
        # backward reaches the decoder first, the encoders after it: issue order = reverse registration order
        return buckets[::-1]

    def _on_stack_backward_done(self, params) -> None:
        """fused.TransformerStackFn.backward calls this when every weight gradient of its stack has been written."""
        i = next((self._bucket_of[id(p)] for p in params if id(p) in self._bucket_of), None)
        if i is None:
            return
        # the stack's gradients are complete on THIS stream (its backward node ran here); a bucket that has to wait for its turn is
        # launched later from another stack's stream, which must first wait for this point
        ev = torch.cuda.Event()
        ev.record()
        self._ready[i] = ev
        cur = torch.cuda.current_stream()
        while self._next_bucket < len(self._buckets) and self._ready[self._next_bucket] is not False:
            lo, hi, _ = self._buckets[self._next_bucket]
            cur.wait_event(self._ready[self._next_bucket])
            self._works.append(self._all_reduce(self.flat_grad[lo:hi]))
            self._next_bucket += 1

    def _all_reduce(self, t: Tensor):
        return dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group, async_op=True)

    def _forward_backward(self, batch: Dict[str, Tensor]):
        self.rng_offset.add_(1)
        self.flat_grad.zero_()
        if self._shadow_stale:                                   # otherwise the previous AdamW launch has already written it
            K.cast_bf16(self.flat_param, out=self.flat_shadow)
            self._shadow_stale = False
        fused.DIRECT_GRAD = fused.SHADOW_ACTIVE = True
        self._ready = [False] * len(self._buckets)
        self._next_bucket = 0
        self._works = []
        fused.STACK_BACKWARD_DONE = self._on_stack_backward_done if self.overlap else None
        try:
            out = self.model(**batch)
            out.loss.backward()
            join_side_streams()       # in-place gradient writes on branch streams: order them before whoever reads flat_grad
        finally:
            fused.DIRECT_GRAD = fused.SHADOW_ACTIVE = False
            fused.STACK_BACKWARD_DONE = None
        if self.evaluator is not None:                           # trainer.py:462-464: metrics of every step
            self.metrics = self.evaluator(batch, out)
        return out

    def _update(self):
        if self.world > 1:
            # what the stack buckets have not covered, in order, then wait for everything on the current stream
            pos = 0
            done = sorted((lo, hi) for (lo, hi, _), r in zip(self._buckets, range(len(self._buckets))) if r < self._next_bucket)
            for lo, hi in done + [(self.flat_grad.numel(), self.flat_grad.numel())]:
                if lo > pos:
                    self._works.append(self._all_reduce(self.flat_grad[pos:lo]))
                pos = max(pos, hi)
            for w in self._works:
                w.wait()
            self._works = []
        norm = torch.linalg.vector_norm(self.flat_grad) if self.grad_clip is not None else None
        self.opt_step.add_(1)
        # averaging over ranks, clipping, AdamW and the bf16 weight shadow of the next step: one pass over the flat buffers
        K.adamw_step(self.flat_param, self.flat_grad, self.flat_m, self.flat_v, self.flat_shadow, norm, self.opt_step, lr=self.lr,
                     betas=self.betas, eps=self.eps, weight_decay=self.weight_decay, max_norm=self.grad_clip or 0.0,
                     grad_scale=1.0 / self.world, lr_dev=self.lr_dev)

    def set_evaluator(self, evaluator) -> None:
        """Compute `evaluator(batch, outputs)` inside every step, as Trainer.run_epoch does (experiments/trainer.py:462-464); the
        metrics of the last step are in `self.metrics`.  With ScorePerformerEvaluator they are ratios of sums the head kernel
        accumulates, so this adds a few scalar kernels to the captured graph."""
        self.evaluator = evaluator
        self._graphs.clear()
        self.graph = None

    def close(self) -> None:
        """Drop the captured graphs (they hold NCCL kernels when world > 1: a process group must not be destroyed under them)."""
        torch.cuda.synchronize()
        self._graphs.clear()
        self.graph = None
        self._sig = None
        self.static_batch = self.static_loss = self.static_losses = self._static_metrics = None
        torch.cuda.synchronize()

    def segment_overflow_count(self) -> int:
        """Note-tuples (accumulated over all steps so far) whose bar / beat / onset id exceeded the static segment tables of the
        sync-free mode -- they were left out of their level's pooling.  Non-zero means: raise
        `model.perf_encoder.slot_capacity` (and re-capture) or train with use_graph=False.  Reading it synchronises."""
        enc = getattr(self.model, "perf_encoder", None)
        c = getattr(enc, "segment_overflow", None)
        return 0 if c is None else int(c)

    def unexpected_label_count(self) -> int:
        """Labels (accumulated over all steps so far) found in output fields outside the LM wrapper's frozen `label_fields`: they
        did not enter the loss (the reference re-checks the fields every batch, wrappers.py:49-59).  Reading it synchronises."""
        wrapper = getattr(self.model, "perf_decoder", None)
        fn = getattr(wrapper, "unexpected_label_count", None)
        return 0 if fn is None else fn()

    def mark_weights_changed(self) -> None:
        """Call after writing parameters from outside the step (load_state_dict, manual edits): rebuilds the bf16 shadow."""
        self._shadow_stale = True

    # ------------------------------------------------------------------ input pipeline (host batches)
    def prefetch(self, batch: Dict[str, Tensor]) -> None:
        """Start copying the NEXT step's (pinned) host batch to the device on a side stream, so the transfer overlaps the step
        that is currently running.  Consume it with `step_prefetched()`."""
        dev = self.flat_grad.device
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=dev)
            self._copied = torch.cuda.Event()
            self._stage_free = torch.cuda.Event()
            self._stage_free.record()
        if self._stage is None or any(self._stage[k].shape != v.shape for k, v in batch.items()):
            self._stage = {k: torch.empty(v.shape, dtype=v.dtype, device=dev) for k, v in batch.items()}
        self._copy_stream.wait_event(self._stage_free)           # the previous step has taken its copy out of the stage
        with torch.cuda.stream(self._copy_stream):
            for k, v in batch.items():
                self._stage[k].copy_(v, non_blocking=True)
            self._copied.record()

    def prefetch_packed(self, packed: Dict[str, Tensor], spec=None) -> None:
        """Like `prefetch`, for a batch packed by `data.pack_batch` (uint16 tokens, int32 segments, uint8 directions, lengths: 65
        bytes per note-tuple instead of 466): the compact tensors are copied on the side stream and `step_prefetched()` expands
        them -- MixedLM masking included -- with one kernel straight into the step's input tensors."""
        from .data.packed import PackedBatchSpec
        dev = self.flat_grad.device
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=dev)
            self._copied = torch.cuda.Event()
            self._stage_free = torch.cuda.Event()
            self._stage_free.record()
        if self._pstage is None or any(k not in self._pstage or self._pstage[k].shape != v.shape for k, v in packed.items()):
            self._pstage = {k: torch.empty(v.shape, dtype=v.dtype, device=dev) for k, v in packed.items()}
        self._pspec = spec or PackedBatchSpec()
        self._copy_stream.wait_event(self._stage_free)
        with torch.cuda.stream(self._copy_stream):
            for k, v in packed.items():
                self._pstage[k].copy_(v, non_blocking=True)
            self._copied.record()
        self._packed_pending = True

    def _step_prefetched_packed(self) -> Tensor:
        from .data.packed import unpack_batch
        cur = torch.cuda.current_stream()
        cur.wait_event(self._copied)
        self._packed_pending = False
        if self.use_graph and self._warm >= 3 and self.graph is not None:
            # expand straight into the captured step's input tensors (shape changes fall through to a fresh capture below)
            try:
                unpack_batch(self._pstage, self._pspec, out=self.static_batch)
                self._stage_free.record()
                return self._replay()
            except AssertionError:
                pass
        batch = unpack_batch(self._pstage, self._pspec)
        self._stage_free.record()
        return self.step(batch)

    def step_prefetched(self) -> Tensor:
        """One training step on the batch handed to the last `prefetch()` / `prefetch_packed()` call."""
        if self._packed_pending:
            return self._step_prefetched_packed()
        assert self._stage is not None, "call prefetch(batch) first"
        cur = torch.cuda.current_stream()
        cur.wait_event(self._copied)
        if not self.use_graph or self._warm < 3 or not self._select_graph(self._stage):
            batch = {k: v.clone() for k, v in self._stage.items()}
            self._stage_free.record()
            return self.step(batch)
        for k, v in self._stage.items():
            self.static_batch[k].copy_(v, non_blocking=True)      # device-to-device, ~10 us
        self._stage_free.record()
        return self._replay()

    def set_lr(self, lr: float):
        """ExponentialLR etc. (experiments/optimizers.py:121-149): the rate lives in a device scalar the AdamW kernel reads, so a
        captured graph keeps replaying."""
        if lr != self.lr:
            self.lr = lr
            self.lr_dev.fill_(float(lr))

    def optimizer_state_dict(self) -> dict:
        """`torch.optim.AdamW.state_dict()`-shaped view of the flat moments, so reference checkpoints interoperate."""
        state = {}
        for i, (p, off) in enumerate(zip(self.params, self.offsets)):
            state[i] = {"step": self.opt_step.clone().float().squeeze(0),
                        "exp_avg": self.flat_m[off:off + p.numel()].view_as(p).clone(),
                        "exp_avg_sq": self.flat_v[off:off + p.numel()].view_as(p).clone()}
        group = {"lr": self.lr, "betas": self.betas, "eps": self.eps, "weight_decay": self.weight_decay, "amsgrad": False,
                 "params": list(range(len(self.params)))}
        return {"state": state, "param_groups": [group]}

    def load_optimizer_state_dict(self, sd: dict):
        for i, (p, off) in enumerate(zip(self.params, self.offsets)):
            st = sd["state"].get(i)
            if st is None:
                continue
            self.flat_m[off:off + p.numel()].view_as(p).copy_(st["exp_avg"])
            self.flat_v[off:off + p.numel()].view_as(p).copy_(st["exp_avg_sq"])
            self.opt_step.fill_(int(st["step"]))
        g = sd["param_groups"][0]
        self.lr, self.betas, self.eps, self.weight_decay = g["lr"], tuple(g["betas"]), g["eps"], g["weight_decay"]
        self.lr_dev.fill_(float(self.lr))
        self._graphs.clear()                                      # betas / eps / weight decay are baked into the captures
        self.graph = None

    @staticmethod
    def _signature(batch: Dict[str, Tensor]) -> tuple:
        return tuple((k, tuple(v.shape), v.dtype) for k, v in sorted(batch.items()))

    def _select_graph(self, batch: Dict[str, Tensor]) -> bool:
        """Make the graph captured for this batch's shapes current; False if there is none yet."""
        sig = self._signature(batch)
        if sig != self._sig:
            entry = self._graphs.get(sig)
            if entry is None:
                return False
            self.graph, self.static_batch, self.static_loss, self.static_losses, self._static_metrics = entry
            self._sig = sig
        return self.graph is not None

    def _capture(self, batch: Dict[str, Tensor]):
        self.static_batch = {k: v.clone() for k, v in batch.items()}
        self.graph = torch.cuda.CUDAGraph()
        before = K.LAUNCHES
        in_graph = self.world == 1 or self.graph_update
        # thread-local capture mode: NCCL's watchdog thread polls CUDA events of earlier collectives while this thread captures
        with torch.cuda.graph(self.graph, capture_error_mode="thread_local" if self.world > 1 else "global"):
            out = self._forward_backward(self.static_batch)
            if in_graph:
                self._update()
        self._update_in_graph = in_graph
        self.launches_per_step = K.LAUNCHES - before
        self.static_loss = out.loss.detach()
        self.static_losses = {k: v.detach() for k, v in out.losses.items()}
        self._static_metrics = self.metrics
        self._sig = self._signature(batch)
        self._graphs[self._sig] = (self.graph, self.static_batch, self.static_loss, self.static_losses, self._static_metrics)

    def _replay(self) -> Tensor:
        self.graph.replay()
        if not self._update_in_graph:
            self._update()
        self.losses = self.static_losses
        self.metrics = self._static_metrics
        # the static tensors are overwritten by the next replay: hand out a copy a trainer may keep (trainer.py:457-466 accumulates
        # loss tensors and reads them later)
        return self.static_loss.clone()

    # ------------------------------------------------------------------ public
    def step(self, batch: Dict[str, Tensor]) -> Tensor:
        """Run one training step on `batch` (device tensors, or pinned host tensors: they are copied in asynchronously).
        Returns the loss tensor (device, detached; a fresh tensor every call).  Batches of a new shape signature (a short last
        batch, another sequence length) are captured on first sight."""
        dev = self.flat_grad.device
        if not self.use_graph or self._warm < 3:
            # eager (also used to warm up lazily-initialised state before capture)
            b = {k: v.to(dev, non_blocking=True) for k, v in batch.items()}
            before = K.LAUNCHES
            out = self._forward_backward(b)
            self._update()
            self.launches_per_step = K.LAUNCHES - before
            self._warm += 1
            self.losses = {k: v.detach() for k, v in out.losses.items()}
            return out.loss.detach()
        if not self._select_graph(batch):
            torch.cuda.synchronize()
            self._capture({k: v.to(dev) for k, v in batch.items()})
        # device-resident tensors of the right dtype go into the static inputs in one launch, anything else (pinned host memory,
        # another dtype or layout) through copy_
        fast = [(self.static_batch[k], v) for k, v in batch.items()
                if v.is_cuda and v.device == dev and v.dtype == self.static_batch[k].dtype and v.is_contiguous()
                and v.shape == self.static_batch[k].shape and self.static_batch[k].is_contiguous()]
        taken = {id(v) for _, v in fast}
        for k, v in batch.items():
            if id(v) not in taken:
                self.static_batch[k].copy_(v, non_blocking=True)
        K.multi_copy([d for d, _ in fast], [s for _, s in fast])
        return self._replay()
