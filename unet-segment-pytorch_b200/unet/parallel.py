"""Batch-sharded data-parallel training step — the B200 form of the reference's
gradient-accumulation loop (scripts/train.py:103-161).

The reference reaches its effective batch by running ``accumulation_steps`` micro-batches one
after another on one device: each micro-batch has its own BatchNorm batch statistics, its loss
is divided by ``accumulation_steps`` (train.py:133), gradients sum into ``.grad`` and one
clip + optimizer step follows (train.py:139-143).  Here the micro-batches run at the same time,
one per GPU (one process per GPU): rank r computes forward/backward on its shard with the loss
divided by ``world_size``, gradients are summed with NCCL all-reduce over NVLink, and every
rank then applies the identical clip + optimizer step.  Up to summation order this is the same
arithmetic (statistics stay per micro-batch, exactly as in the reference, unless the model's
BatchNorms were converted with ``nn.SyncBatchNorm.convert_sync_batchnorm``: see unet/syncbn.py).

Gradients live in a few flat fp32 buckets cut in backward order; a bucket's all-reduce is
launched from an autograd hook as soon as its last gradient has been accumulated, on NCCL's
own stream, so communication overlaps the rest of backward.  With ``world_size == 1`` the same
code runs without collectives.
"""
from __future__ import annotations

import os
from typing import List

import torch
import torch.distributed as dist

from . import ops
from .optim import FusedAdamW


class _Bucket:
    __slots__ = ("flat", "params", "pending", "work", "deferred", "seen")

    def __init__(self, flat, params):
        self.flat, self.params, self.pending, self.work = flat, params, 0, None
        self.deferred = []   # split-K folds of this bucket's conv weights, launched together
        self.seen = set()    # parameters already counted this step (a gradient is reported ONCE, see _bucket_ready)


class _GradSink:
    """What unet.ops talks to during the trainer's backward pass (see ops.GRAD_SINK)."""

    def __init__(self, trainer):
        self.trainer = trainer

    def __call__(self, param):
        self.trainer._grad_sink(param)

    def defer_reduce(self, param, item):
        self.trainer._defer_reduce(param, item)


class BatchShardedTrainer:
    """fwd + loss/world + bwd (+ overlapped gradient all-reduce) + clip + optimizer step.

    Parameters
    ----------
    model, criterion, optimizer : as built by the reference's train.py (:306-350)
    grad_clip : max gradient norm (train.py:141), 0 disables
    bucket_mb : flat gradient bucket size
    process_group : None -> default group if torch.distributed is initialised
    accumulation_steps : micro-batches each rank runs per optimizer step (train.py:127-147 on fewer
        GPUs than micro-batches): ``step`` is then called once per micro-batch, gradients of
        ``loss / (world * accumulation_steps)`` sum into the buckets, and the all-reduce, clip,
        optimizer step and EMA update happen on every ``accumulation_steps``-th call
    buffer_sync : what happens to the BatchNorm running buffers of the ranks (each rank only sees its own
        shard, so they drift apart exactly like the reference's buffers move from micro-batch to
        micro-batch): ``"rank0"`` — rank 0's buffers are THE buffers, broadcast to every rank before
        ``evaluate`` / by ``sync_buffers()`` (call it before writing a checkpoint on another rank);
        ``"average"`` — all-reduce mean of running_mean / running_var instead; ``"none"`` — leave them.
        Training arithmetic never reads the buffers, so the choice does not change any gradient.

    The loss ``step`` returns is a fresh 0-dim device tensor on every call (under graph replay a copy of
    the graph's static output), so a loop may keep the returned losses and read them later.
    """

    def __init__(self, model, criterion, optimizer, grad_clip: float = 0.0, bucket_mb: float = 24.0,
                 process_group=None, cuda_graph: bool = False, graph_warmup: int = 3, ema=None,
                 accumulation_steps: int = 1, buffer_sync: str = "rank0"):
        self.model, self.criterion, self.optimizer, self.grad_clip = model, criterion, optimizer, grad_clip
        if accumulation_steps < 1:
            raise ValueError("accumulation_steps must be >= 1")
        self.accumulation_steps = int(accumulation_steps)
        self._micro = 0          # micro-batches seen since the last optimizer step
        self._first = self._last = True   # phase of the micro-batch being run (set by step)
        self.group = process_group
        self.world = dist.get_world_size(process_group) if dist.is_available() and dist.is_initialized() else 1
        # measurement knobs (bench.py's collective-exposure figures; never set in production):
        #   UB2_SKIP_ALLREDUCE=1   run the multi-rank step WITHOUT its collectives (replicas then diverge)
        #   UB2_ALLREDUCE_AT_END=1 launch every bucket's all-reduce after backward instead of as it fills
        #   UB2_BUCKET_MB=<float>  bucket size override
        self._skip_collectives = os.environ.get("UB2_SKIP_ALLREDUCE", "0") == "1"
        self._collectives_at_end = os.environ.get("UB2_ALLREDUCE_AT_END", "0") == "1"
        bucket_mb = float(os.environ.get("UB2_BUCKET_MB", bucket_mb))
        self.buffer_sync = buffer_sync
        self._buffers_dirty = False
        if self.world > 1:
            # One model, replicated: every rank starts from rank 0's parameters and buffers (what DDP does at
            # construction) — ranks that seeded or loaded differently would otherwise average gradients of
            # different weights without any error.
            self._broadcast_state()
        self.buckets: List[_Bucket] = []
        self._bucket_of = {}
        self._build_buckets(bucket_mb)
        self._steps = 0
        # unet.utils.general.ModelEMA (or None): updated after every optimizer step like the
        # reference's loop does (scripts/train.py:146-147), as one launch inside the step graph
        self.ema = ema
        self._packer = None   # all bf16 weight packs of the model, rebuilt by one launch per step
        # CUDA-graph replay of the whole step: a 512^2 batch-4 step is ~800 kernel launches, more
        # host time than GPU time when issued one by one.  Every kernel of the path is
        # stream-ordered with no host synchronisation, so the step is captured once per input
        # shape (after `graph_warmup` eager steps) and replayed.
        self.cuda_graph = cuda_graph
        self.graph_warmup = graph_warmup
        self._graphs = {}
        self._eager_steps = {}
        self._copy_stream = None   # mask copies (see step)
        self._side = None          # weight gradients next to the BatchNorm passes (ops.SideStream)
        self._side_enabled = os.environ.get("UB2_WGRAD_SIDE", "1") != "0"
        dev0 = next(model.parameters()).device
        if self._side_enabled and dev0.type == "cuda":
            self._side = ops.SideStream(dev0)   # created here, never inside a graph capture
        self._masks_ready = self._step_done = None

    # ------------------------------------------------------------------ replicated state
    def _broadcast_state(self) -> None:
        with torch.no_grad():
            for t in list(self.model.parameters()) + list(self.model.buffers()):
                dist.broadcast(t, src=dist.get_global_rank(self.group, 0) if self.group is not None else 0,
                               group=self.group)

    @torch.no_grad()
    def sync_buffers(self, mode: str = None) -> None:
        """Make the BatchNorm buffers of all ranks equal (see ``buffer_sync``)."""
        mode = mode or self.buffer_sync
        self._buffers_dirty = False
        if self.world == 1 or mode == "none":
            return
        src = dist.get_global_rank(self.group, 0) if self.group is not None else 0
        for b in self.model.buffers():
            if mode == "average" and b.is_floating_point():
                dist.all_reduce(b, op=dist.ReduceOp.SUM, group=self.group)
                b.div_(self.world)
            else:   # rank0; integer counters (num_batches_tracked) are equal on all ranks anyway
                dist.broadcast(b, src=src, group=self.group)

    # ------------------------------------------------------------------ flat gradient buckets
    def _build_buckets(self, bucket_mb: float) -> None:
        params = [p for p in self.model.parameters() if p.requires_grad]
        limit = int(bucket_mb * (1 << 20) / 4)
        groups, cur, cur_n = [], [], 0
        for p in reversed(params):  # backward produces gradients roughly in reverse registration order
            cur.append(p)
            cur_n += p.numel()
            if cur_n >= limit:
                groups.append(cur)
                cur, cur_n = [], 0
        if cur:
            groups.append(cur)
        pad = lambda n: (n + 31) & ~31   # every view starts on a 128-byte boundary (vector access)
        for g in groups:
            flat = torch.zeros(sum(pad(p.numel()) for p in g), device=g[0].device, dtype=torch.float32)
            off = 0
            for p in g:
                p.grad = flat[off:off + p.numel()].view_as(p)  # autograd accumulates in place into the view
                off += pad(p.numel())
            b = _Bucket(flat, g)
            self.buckets.append(b)
            for p in g:
                self._bucket_of[id(p)] = b
                if self.world > 1:
                    p.register_post_accumulate_grad_hook(self._make_hook(b))

    def _bucket_ready(self, bucket: _Bucket, n: int = 1, param=None) -> None:
        """``param``'s gradient is complete in the bucket.  A parameter can be announced twice — by the kernel
        path's gradient sink AND by the post-accumulate hook autograd runs for the same leaf (the engine still
        visits the AccumulateGrad node of an input whose backward returned None) — and must count once: a
        bucket whose count reached zero early was all-reduced while half of its gradients were still being
        written, so every rank kept a different sum (found by bench.py's replica check, round 2)."""
        if param is not None:
            if id(param) in bucket.seen:
                return
            bucket.seen.add(id(param))
        bucket.pending -= n
        if bucket.deferred and bucket.pending == len(bucket.deferred):
            # every other gradient of the bucket is in: fold all its split-K partials in one go
            from .kernels import wgrad_reduce_multi
            items, bucket.deferred = bucket.deferred, []
            ops.wgrad_join()   # the last partial tiles may still be written on the side stream
            wgrad_reduce_multi(items, accumulate=True)
            bucket.pending -= len(items)
        if (bucket.pending == 0 and self.world > 1 and self._last and bucket.work is None
                and not self._skip_collectives and not self._collectives_at_end):
            bucket.work = dist.all_reduce(bucket.flat, op=dist.ReduceOp.SUM, group=self.group, async_op=True)

    def _defer_reduce(self, param, item) -> None:
        b = self._bucket_of.get(id(param))
        if b is None:   # not one of ours: fold it now
            from .kernels import wgrad_reduce
            wgrad_reduce(*item, accumulate=True)
            return
        b.seen.add(id(param))     # counted when its fold is launched
        b.deferred.append(item)
        self._bucket_ready(b, 0)

    def _flush_deferred(self) -> None:
        """End of backward: buckets in which some parameter received no gradient this step."""
        from .kernels import wgrad_reduce_multi
        ops.wgrad_join()
        for b in self.buckets:
            if b.deferred:
                items, b.deferred = b.deferred, []
                wgrad_reduce_multi(items, accumulate=True)
                b.pending -= len(items)

    def _make_hook(self, bucket: _Bucket):
        return lambda param: self._bucket_ready(bucket, 1, param)

    def _grad_sink(self, param) -> None:
        """Called by unet.ops when a kernel has accumulated ``param``'s gradient straight into its
        bucket view (no autograd AccumulateGrad node runs for it, hence no hook)."""
        b = self._bucket_of.get(id(param))
        if b is not None:
            self._bucket_ready(b, 1, param)

    # ------------------------------------------------------------------ one optimizer step
    def _forward(self, images: torch.Tensor):
        """First half of a micro-step: on the first micro-batch of an optimizer step zero the
        gradient buckets and rebuild the weight packs (one launch); run the model's forward pass.
        Does not touch the masks."""
        self.model.train()
        for b in self.buckets:
            if self._first:
                b.flat.zero_()
            b.pending = len(b.params)
            b.work = None
            b.deferred = []
            b.seen = set()
        dev = next(self.model.parameters()).device
        if dev.type == "cuda":
            if self._packer is None:
                from .kernels import WeightPacker
                self._packer = WeightPacker([m.weight for m in self.model.modules()
                                             if isinstance(m, torch.nn.Conv2d) and m.weight.is_cuda])
            if self._first:   # the weights only change at an optimizer step
                self._packer.run()
        prev_packs, ops.PACKS = ops.PACKS, self._packer
        try:
            return self.model(images)
        finally:
            ops.PACKS = prev_packs

    def _backward(self, outputs, masks: torch.Tensor) -> torch.Tensor:
        """Second half: loss, backward (gradient sink installed) and, on the last micro-batch of an
        optimizer step, all-reduce, clip + optimizer, EMA."""
        prev_sink, ops.GRAD_SINK = ops.GRAD_SINK, _GradSink(self)
        prev_side, ops.WGRAD_SIDE = ops.WGRAD_SIDE, self._wgrad_side(outputs)
        try:
            loss = self.criterion(outputs, masks)
            (loss / (self.world * self.accumulation_steps)).backward()
            self._flush_deferred()
        finally:
            ops.wgrad_join()
            ops.GRAD_SINK = prev_sink
            ops.WGRAD_SIDE = prev_side
        if not self._last:
            return loss.detach()
        self._optimizer_tail()
        return loss.detach()

    def _wgrad_side(self, outputs):
        """The side stream weight gradients run on (ops.SideStream), or None: UB2_WGRAD_SIDE=0, CPU."""
        if not self._side_enabled:
            return None
        t = outputs[0] if isinstance(outputs, (tuple, list)) else outputs
        if not (torch.is_tensor(t) and t.is_cuda):
            return None
        if self._side is None or self._side.stream.device != t.device:
            self._side = ops.SideStream(t.device)
        return self._side

    def _optimizer_tail(self) -> None:
        """All-reduce what is not in flight yet, wait, clip + optimizer step, EMA (train.py:139-147)."""
        self._buffers_dirty = True
        if self.world > 1 and not self._skip_collectives:
            for b in self.buckets:
                if b.work is None:  # a parameter without gradient this step (or UB2_ALLREDUCE_AT_END)
                    b.work = dist.all_reduce(b.flat, op=dist.ReduceOp.SUM, group=self.group, async_op=True)
            for b in self.buckets:
                b.work.wait()
        if isinstance(self.optimizer, FusedAdamW):
            # clip + AdamW in two multi-tensor launches (csrc/optim.cu)
            self.optimizer.max_grad_norm = float(self.grad_clip)
            self.optimizer.step()
        else:
            if self.grad_clip > 0:
                torch.nn.utils.clip_grad_norm_(self.model.parameters(), self.grad_clip, foreach=True)
            self.optimizer.step()
        if self.ema is not None:
            self.ema.update(self.model, _advance=False)

    def flush(self) -> bool:
        """End of an epoch whose number of micro-batches is not a multiple of ``accumulation_steps``
        (train.py:153-159): apply the optimizer step to the gradients accumulated so far.  Like the
        reference, the left-over gradients are NOT rescaled (each micro-batch already carried
        ``1 / accumulation_steps``).  Returns False if nothing was pending.  Runs eagerly (it happens
        once per epoch); the next ``step`` starts a fresh accumulation window."""
        if self._micro == 0:
            return False
        self._micro = 0
        self._steps += 1
        if self.ema is not None:
            self.ema.prepare(self.model)
        for b in self.buckets:
            b.work = None
        self._optimizer_tail()
        return True

    def _step_body(self, images: torch.Tensor, masks: torch.Tensor) -> torch.Tensor:
        return self._backward(self._forward(images), masks)

    def _optimizer_capturable(self) -> bool:
        if isinstance(self.optimizer, FusedAdamW):
            return True
        return all(g.get("capturable", False) for g in self.optimizer.param_groups)

    def step(self, images: torch.Tensor, masks: torch.Tensor) -> torch.Tensor:
        """One micro-batch per rank and one optimizer step.  ``images`` / ``masks`` may be host
        (pinned) tensors: they are copied to this rank's GPU asynchronously.  Returns the
        un-divided micro-batch loss as a 0-dim device tensor (no host sync)."""
        dev = next(self.model.parameters()).device
        self._first = self._micro == 0
        self._last = self._micro == self.accumulation_steps - 1
        self._micro = 0 if self._last else self._micro + 1
        if self._last:
            self._steps += 1
            if self.ema is not None:
                self.ema.prepare(self.model)   # host side: counter, warm-up decay -> device memory
        use_graph = self.cuda_graph and dev.type == "cuda" and self._optimizer_capturable()
        if dev.type != "cuda":
            return self._step_body(images.to(dev), masks.to(dev))
        # The masks are not needed before the loss: their host->device copy (8 of the 12.5 MB of a
        # batch-4 step) runs on a copy stream under the forward pass.
        main = torch.cuda.current_stream(dev)
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=dev)
            self._masks_ready = torch.cuda.Event()
            self._step_done = torch.cuda.Event()
        copy = self._copy_stream
        if masks.is_cuda:
            # device-resident masks (e.g. from unet.data.DeviceBatchPipeline) were produced by work the
            # caller's stream already waits for: order the copy stream behind it as well
            copy.wait_stream(main)
        if not use_graph:
            with torch.cuda.stream(copy):
                masks_dev = masks.to(dev, non_blocking=True)
                self._masks_ready.record(copy)
            outputs = self._forward(images.to(dev, non_blocking=True))
            main.wait_event(self._masks_ready)
            masks_dev.record_stream(main)
            return self._backward(outputs, masks_dev)
        # a micro-step's graph depends on its phase (zero + pack first, all-reduce + optimizer last)
        key = (tuple(images.shape), images.dtype, tuple(masks.shape), masks.dtype, self._first, self._last)
        entry = self._graphs.get(key)
        if entry is None:
            done = self._eager_steps.get(key, 0)
            if done < self.graph_warmup:
                # eager warm-up (lazy initialisation, allocator, NCCL) on a side stream, as
                # torch.cuda.graph requires
                self._eager_steps[key] = done + 1
                side = torch.cuda.Stream(device=dev)
                side.wait_stream(main)
                with torch.cuda.stream(side):
                    loss = self._step_body(images.to(dev, non_blocking=True), masks.to(dev, non_blocking=True))
                main.wait_stream(side)
                return loss
            gx = torch.empty(images.shape, dtype=images.dtype, device=dev)
            gt = torch.empty(masks.shape, dtype=masks.dtype, device=dev)
            gx.copy_(images, non_blocking=True)
            gt.copy_(masks, non_blocking=True)
            torch.cuda.synchronize(dev)
            # two graphs sharing one memory pool, always replayed in this order: forward | the rest.
            # Between them the main stream waits for the masks.
            g_fwd, g_bwd = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            cap = None
            if os.environ.get("UB2_CAPTURE_PRIORITY", "0") == "1":
                # the critical path (everything but the weight gradients) on a high-priority stream: its thread
                # blocks are dispatched ahead of the side stream's whenever both have work ready
                cap = torch.cuda.Stream(device=dev, priority=-1)
            with torch.cuda.graph(g_fwd, stream=cap):
                outputs = self._forward(gx)
            with torch.cuda.graph(g_bwd, pool=g_fwd.pool(), stream=cap):
                gloss = self._backward(outputs, gt)
            del outputs
            entry = self._graphs[key] = (g_fwd, g_bwd, gx, gt, gloss)
            self._step_done.record(main)
            # the capture itself does not execute: fall through and replay it for this step
        g_fwd, g_bwd, gx, gt, gloss = entry
        gx.copy_(images, non_blocking=True)
        copy.wait_event(self._step_done)          # the previous replay has finished reading `gt`
        with torch.cuda.stream(copy):
            gt.copy_(masks, non_blocking=True)
            self._masks_ready.record(copy)
        if self._last and isinstance(self.optimizer, FusedAdamW):
            self.optimizer.sync_hyperparams()   # a scheduler may have changed the learning rate
        g_fwd.replay()
        main.wait_event(self._masks_ready)
        g_bwd.replay()
        self._step_done.record(main)
        return gloss.clone()   # the graph's static output is overwritten by the next replay

    def release_graphs(self) -> None:
        """Drop the captured step graphs (they hold references to NCCL work and pool memory)."""
        self._graphs.clear()
        self._eager_steps.clear()

    @torch.no_grad()
    def evaluate(self, images: torch.Tensor, masks: torch.Tensor, metrics=None) -> torch.Tensor:
        """validate() of the reference (train.py:164-197) for one batch: eval-mode forward
        (BatchNorm folded, ReLU fused), loss, and device-side confusion-matrix update."""
        dev = next(self.model.parameters()).device
        if self._buffers_dirty:
            self.sync_buffers()   # every rank validates the same model (buffer_sync policy)
        images = images.to(dev, non_blocking=True)
        masks = masks.to(dev, non_blocking=True)
        self.model.eval()
        out = self.model(images)
        if metrics is not None:
            metrics.update(out, masks)
        return self.criterion(out, masks)

    def all_reduce_confusion(self, metrics) -> None:
        """Confusion matrices are additive over shards: sum them across ranks."""
        if self.world == 1:
            return
        cm = torch.from_numpy(metrics.confusion_matrix.copy()).to(next(self.model.parameters()).device)
        dist.all_reduce(cm, op=dist.ReduceOp.SUM, group=self.group)
        metrics.confusion_matrix = cm.cpu().numpy()
