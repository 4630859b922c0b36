"""The aligner training step, isolated: pack -> aligner forward -> masked loss -> backward (-> gradient all-reduce) -> AdamW.

This is the hot part of the reference's ``BaseTask._train_inner_loop`` (thinkdiff/tasks/base_task.py:169-272) with the
frozen T5 decoder excised (SURVEY.md section 3.1): ``samples -> .cuda() -> autocast(bf16) forward -> loss -> backward ->
optimizer.step -> zero_grad``. The optimizer is the reference's AdamW with its weight-decay split
(thinkdiff/runners/runner_base.py:98-127); it stays a PyTorch (fused) optimizer -- plumbing, not the product.
"""
from __future__ import annotations

import torch

from . import ops
from .aligner import ThinkDiffAligner
from .pack import FlatBatch, PackedBatch, pack_device


def reference_param_groups(module: torch.nn.Module, weight_decay: float = 0.05):
    """The reference's weight-decay split (runner_base.py:104-119): no decay for ndim < 2 or names with bias/ln/bn."""
    decay, no_decay = [], []
    for n, p in module.named_parameters():
        if not p.requires_grad:
            continue
        (no_decay if (p.ndim < 2 or "bias" in n or "ln" in n or "bn" in n) else decay).append(p)
    return [{"params": decay, "weight_decay": weight_decay}, {"params": no_decay, "weight_decay": 0.0}]


def make_reference_optimizer(module, lr: float = 1e-4, weight_decay: float = 0.05, beta2: float = 0.999):
    return torch.optim.AdamW(reference_param_groups(module, weight_decay), lr=lr, weight_decay=weight_decay,
                             betas=(0.9, beta2), fused=True)


def synthetic_lvlm_batch(num_seqs: int, max_len: int, din: int, d: int, seed: int, pin: bool = True,
                         with_target: bool = True, truncated: bool = False, world: int = 1, rank: int = 0,
                         balanced: bool = True) -> FlatBatch:
    """BASELINE config-2 style ragged batch (``synth.py``) as a ``FlatBatch`` of (pinned) host tensors: this rank's ``num_seqs``
    sequences of the global batch of ``world * num_seqs`` sequences with this seed. ``balanced``: length-balanced assignment of
    the global batch (``sharding.balanced_assignment``: equal sequence counts, even token counts) instead of a contiguous split.
    ``truncated``: only the kept rows are in the flat source (``FlatCollater(truncate_on_host=True)`` layout)."""
    from .sharding import balanced_assignment, contiguous_assignment
    from .synth import global_lengths, lvlm_sequences

    lens_all = global_lengths(num_seqs * world, max_len, seed)
    groups = balanced_assignment(lens_all.tolist(), world) if (balanced and world > 1) else contiguous_assignment(num_seqs * world, world)
    flat, start, lens, target = lvlm_sequences(groups[rank], lens_all, din, d, seed, with_target, truncated)
    extras = {}
    if with_target:
        extras["flat_target"] = target
    if pin and torch.cuda.is_available():
        flat, start, lens = flat.pin_memory(), start.pin_memory(), lens.pin_memory()
        if with_target:
            extras["flat_target"] = extras["flat_target"].pin_memory()
    return FlatBatch(flat, start, lens, int(lens.max()), extras)


def _optimizer_step(optimizer, loss_scale: float):
    """Unscale (``FusedAdamW`` folds 1 / loss_scale into its update; a torch optimizer gets the gradients divided first), step, and
    drop the gradients. No-op without an optimizer."""
    if optimizer is None:
        return
    from .optim import FusedAdamW

    if isinstance(optimizer, FusedAdamW):
        optimizer.grad_scale = 1.0 / loss_scale
    elif loss_scale != 1.0:
        for group in optimizer.param_groups:
            torch._foreach_mul_([p.grad for p in group["params"] if p.grad is not None], 1.0 / loss_scale)
    optimizer.step()
    optimizer.zero_grad(set_to_none=True)


class AlignerTrainStep:
    """One data-parallel training step of the aligner against T5-space targets (masked MSE).

    The fused-loss step runs WITHOUT autograd: ``aligner.mse_loss_backward_packed`` enqueues forward, loss, backward and the
    gradient exchange directly (same kernels as ``mse_loss_packed(...).backward()``), so the host cost of a step is a dozen
    C calls. ``grad_scaler`` (a ``DeviceGradScaler``), ``max_grad_norm`` and ``accum_grad_iters`` reproduce the reference loop's
    ``scaler.scale(loss).backward()`` / ``scaler.unscale_`` + ``clip_grad_norm_`` / ``scaler.step`` / ``scaler.update`` every
    ``accum_grad_iters`` iterations (thinkdiff/tasks/base_task.py:241-258) with every decision taken on the device."""

    def __init__(self, aligner: ThinkDiffAligner, optimizer=None, loss_scale: float = 1.0, fused_loss: bool = True,
                 pipelined: bool = False, grad_scaler=None, max_grad_norm: float = 0.0, accum_grad_iters: int = 1):
        self.aligner = aligner
        self.optimizer = optimizer
        self.loss_scale = float(loss_scale)  # GradScaler-style static scale (backward is linear in it)
        self.fused_loss = fused_loss         # True: fused norm + loss + norm-backward (y / dy stay on chip); False: module boundary path
        # pipelined (data parallel + FusedAdamW + fused loss): the parameter updates of step i are applied inside step
        # i+1, each just before its parameter is first read -- Linear1's after the next batch is packed, Linear2's
        # between the two forward GEMMs -- so both gradient all-reduces hide behind compute. Same arithmetic, same
        # order of updates as the sequential step; call flush() before reading parameters outside the loop.
        self.pipelined = pipelined
        self.grad_scaler = grad_scaler
        self.max_grad_norm = float(max_grad_norm)
        self.accum_grad_iters = int(accum_grad_iters)
        self._micro = 0          # micro-batches accumulated so far in the current optimizer step
        self._accum = None       # GradBuckets being accumulated into
        self._pending_t = None
        self._sharded = False
        self._peer = False
        self._upstream = None
        controlled = grad_scaler is not None or self.max_grad_norm > 0.0 or self.accum_grad_iters > 1
        if controlled:
            from .optim import FusedAdamW

            if not (isinstance(optimizer, FusedAdamW) and fused_loss):
                raise ValueError("grad_scaler / max_grad_norm / accum_grad_iters need FusedAdamW and fused_loss=True")
            if pipelined:
                raise ValueError("grad_scaler / max_grad_norm / accum_grad_iters: the update needs the whole step's gradient "
                                 "statistics first -- use pipelined=False")
            dp = aligner._dp
            if dp is not None and dp.world > 1 and (dp.sharded or dp.peer):
                raise NotImplementedError("grad_scaler / clipping / accumulation with sharded or peer data parallel")
            if grad_scaler is None:
                from .optim import DeviceGradScaler

                self.grad_scaler = DeviceGradScaler(next(aligner.parameters()).device, enabled=False)
        if aligner._dp is not None and aligner._dp.peer and not pipelined:
            raise ValueError("peer data parallel needs AlignerTrainStep(pipelined=True) with FusedAdamW (the owners' AdamW "
                             "kernels are what consume the gradient slots)")
        if pipelined:
            from .optim import FusedAdamW

            if not (isinstance(optimizer, FusedAdamW) and fused_loss):
                raise ValueError("pipelined=True needs FusedAdamW and fused_loss=True")
            aligner._bwd_order = "linear1_first"
            dp = aligner._dp
            # sharded data parallel (enable_data_parallel(sharded=True)): reduce-scatter -> AdamW on this rank's rows ->
            # all-gather of the bf16 rows, all on a side stream that runs beside the remaining GEMMs
            self._sharded = dp is not None and dp.sharded and dp.world > 1
            self._peer = dp is not None and dp.peer  # (also at world 1: the degenerate case exercises every kernel)
            self._ag, self._upd_done = {}, {}
            aligner._record_phase_events = not (self._sharded or self._peer)

    def _upstream_scalar(self, device):
        """Device scalar multiplied into every gradient (static loss scale), or None."""
        if self.loss_scale == 1.0:
            return None
        if self._upstream is None or self._upstream.device != device:
            self._upstream = torch.full((1,), self.loss_scale, dtype=torch.float32, device=device)
        return self._upstream

    def _fwd_bwd(self, packed, target) -> torch.Tensor:
        return self.aligner.mse_loss_backward_packed(packed.x, *target, upstream=self._upstream_scalar(packed.x.device),
                                                     set_grads=not self.pipelined)

    def step_device(self, flat, src_row_start, lens_dev, total_rows: int, l_max: int, flat_target) -> torch.Tensor:
        """Inputs already resident in HBM. Returns the (unscaled) loss as a device scalar; nothing syncs the host."""
        if self.fused_loss:
            # the fused loss reads each token's target row straight from the flat source (row index from the feature pack)
            cu = ops.cu_seqlens(lens_dev)
            x, index = ops.pack_varlen(flat, src_row_start, cu, total_rows, want_index=True)
            packed = PackedBatch(x, cu, None, l_max)
            target = (flat_target, index)
        else:
            packed = pack_device(flat, src_row_start, lens_dev, total_rows, l_max)
            target = ops.pack_varlen(flat_target, src_row_start, packed.cu_seqlens, total_rows)
        if self.pipelined:
            return self._step_pipelined(packed, target)
        if self.grad_scaler is not None:
            return self._step_controlled(packed, target)
        if self.fused_loss:
            loss = self._fwd_bwd(packed, target)
        else:
            with torch.autocast("cuda", dtype=torch.bfloat16):
                y = self.aligner.forward_packed(packed.x, packed.cu_seqlens)
            loss, dy = ops.masked_mse_fwd_bwd(y, target, None, self.loss_scale)
            y.backward(dy)
        _optimizer_step(self.optimizer, self.loss_scale)
        return loss

    def _step_controlled(self, packed, target) -> torch.Tensor:
        """The reference loop with a GradScaler / gradient clipping / accumulation (base_task.py:241-258), decisions on the
        device: backward with the scaler's current scale as upstream scalar; on the last micro-batch the gradient statistics
        (non-finite count, norm) are folded into the step's control block and the AdamW kernels read skip / unscale / clip /
        bias corrections from it."""
        a, opt, sc = self.aligner, self.optimizer, self.grad_scaler
        dp = a._dp
        first = self._micro == 0
        if first:
            sc.begin_step()
        last = self._micro + 1 == self.accum_grad_iters
        if self.accum_grad_iters > 1:
            # micro-batches accumulate locally (like DDP's no_sync); the all-reduce runs once, on the last one
            if first:
                from .aligner import GradBuckets

                self._accum = GradBuckets(a.mm_hidden_size, a.hidden_size, packed.x.device)
                for f in self._accum.flats().values():
                    f.zero_()
            loss = a.mse_loss_backward_packed(packed.x, *target, upstream=sc.scale_tensor, accumulate_into=self._accum)
            if last and dp is not None and dp.world > 1:
                a._pending = {"linear1": dp.all_reduce_async(self._accum.linear1), "linear2": dp.all_reduce_async(self._accum.linear2)}
        else:
            loss = a.mse_loss_backward_packed(packed.x, *target, upstream=sc.scale_tensor)
        self._micro += 1
        if not last:
            return loss
        self._micro = 0
        a.wait_grads()  # the statistics are taken from the REDUCED gradients, so every rank reaches the same decision
        flats = a._grad_flats
        sc.accumulate_stats(flats["linear1"], flats["linear2"])
        sc.update(opt, self.max_grad_norm)
        opt.step(ctl=sc.ctl)
        opt.zero_grad(set_to_none=True)
        self._accum = None
        return loss

    def _wait_update(self, name: str):
        """Order the compute stream after bucket ``name``'s sharded update (its bf16 all-gather + small-vector AdamW)."""
        ag = self._ag.pop(name, None)
        if ag is not None:
            ag.wait()
        ev = self._upd_done.pop(name, None)
        if ev is not None:
            torch.cuda.current_stream().wait_event(ev)

    def _step_pipelined_sharded(self, packed, target) -> torch.Tensor:
        a, opt = self.aligner, self.optimizer
        opt.grad_scale = 1.0 / self.loss_scale
        if self._pending_t is not None:
            self._wait_update("linear1")                                  # W1 / b1 copies are current before GEMM1
            a._between_fwd_stages = lambda: self._wait_update("linear2")  # W2 / b2 / g before GEMM2
            a._bf16_managed = True
        # (the previous step's gradient buckets stay alive in self._grads_hold until the end of this step: by then the compute
        #  stream is ordered after both of that step's updates, which read them on the update stream)
        try:
            loss = self._fwd_bwd(packed, target)
        finally:
            a._between_fwd_stages = None
        t = opt.next_step_number()
        self._pending_t = t
        # enqueue both buckets' updates now, on the update stream: each waits (on the device) for its reduce-scatter,
        # i.e. for its weight-gradient GEMM, and then runs beside whatever the compute stream does next
        if not hasattr(self, "_update_stream"):
            self._update_stream = torch.cuda.Stream()
        grads = list(a._grad_flats.values())
        if not hasattr(self, "_small_done"):
            self._small_done = torch.cuda.Event()
        with torch.cuda.stream(self._update_stream):
            # in the order the collectives were issued: reduce-scatter(dW1), all-reduce(small), reduce-scatter(dW2)
            self._ag["linear1"] = opt.launch_sharded_update("linear1", t)
            opt.launch_small_update(t)  # [b2 | g | b1]: 48 KB all-reduce, replicated AdamW
            self._small_done.record(self._update_stream)
            self._upd_done["linear1"] = self._small_done
            self._ag["linear2"] = opt.launch_sharded_update("linear2", t)
        # the gradient buckets were allocated on the compute stream and are last read on the update stream: keep them
        # alive until the compute stream has waited for the updates (next step), instead of record_stream(), which would
        # keep the caching allocator from recycling the 126 MB of buckets in time
        self._grads_hold = grads
        return loss

    def _step_pipelined_peer(self, packed, target) -> torch.Tensor:
        """The sharded pipeline with no collectives (peer.py): gradients reach their owner from the GEMM epilogues, updated bf16
        rows come back from the owners' AdamW kernels, and the compute stream only ever waits on two counters per step."""
        from .peer import ROW_W1, ROW_W2

        a, opt = self.aligner, self.optimizer
        px = a._ensure_peer()
        opt.grad_scale = 1.0 / self.loss_scale
        if self._pending_t is not None:
            prev = a._peer_epoch
            px.wait(ROW_W1, prev)             # every owner has stored its rows of W1 (and this rank its b1 / b2 / g) for the previous step

            def before_gemm2():
                px.wait(ROW_W2, prev)

            a._between_fwd_stages = before_gemm2
            a._bf16_managed = True
        # (the previous step's small-vector bucket stays alive in self._grads_hold until the end of this step: by then the compute
        #  stream is ordered after that step's updates, which read it on the update stream)
        try:
            loss = self._fwd_bwd(packed, target)
        finally:
            a._between_fwd_stages = None
        t = opt.next_step_number()
        self._pending_t = t
        e = a._peer_epoch
        if not hasattr(self, "_update_stream"):
            self._update_stream = torch.cuda.Stream()
        grads = list(a._grad_flats.values())
        with torch.cuda.stream(self._update_stream):
            # no event from the compute stream is needed: each update waits on a counter, and this rank's own +1 is issued by the
            # compute stream right after the GEMM that produced the data
            opt.launch_peer_update("linear1", t, e)   # (+ the three small vectors)
            opt.launch_peer_update("linear2", t, e)
        self._grads_hold = grads
        return loss

    def _step_pipelined(self, packed, target) -> torch.Tensor:
        if self._peer:
            return self._step_pipelined_peer(packed, target)
        if self._sharded:
            return self._step_pipelined_sharded(packed, target)
        a, opt = self.aligner, self.optimizer
        opt.grad_scale = 1.0 / self.loss_scale
        if self._pending_t is not None:
            self._wait_update("linear1")                                  # W1 / b1 (+ bf16 copies) before GEMM1 reads them
            a._between_fwd_stages = lambda: self._wait_update("linear2")  # W2 / b2 / g before GEMM2
            a._bf16_managed = True
        # (the previous step's gradient buckets stay alive in self._grads_hold until the end of this step: by then the compute
        #  stream is ordered after both of that step's updates, which read them on the update stream)
        try:
            loss = self._fwd_bwd(packed, target)
        finally:
            a._between_fwd_stages = None
        t = opt.next_step_number()
        self._pending_t = t
        # AdamW of each bucket on the update stream, as soon as that bucket's gradients exist (and, under data parallel,
        # are all-reduced): the HBM-bound updates run beside the tensor-bound GEMMs instead of after them
        if not hasattr(self, "_update_stream"):
            self._update_stream = torch.cuda.Stream()
        grads = list(a._grad_flats.values())
        with torch.cuda.stream(self._update_stream):
            for name in ("linear1", "linear2"):
                self._update_stream.wait_event(a._phase_done[name])
                opt.step_bucket(name, t=t, release_grads=True)
                ev = torch.cuda.Event()
                ev.record(self._update_stream)
                self._upd_done[name] = ev
        self._grads_hold = grads  # freed only after the compute stream has waited for the updates (next step / flush)
        return loss

    def flush(self, sync_masters: bool = True):
        """Apply the parameter updates still pending from the last pipelined step (no-op otherwise). In the sharded / peer modes
        every rank only holds current fp32 MASTER rows for its own shard (the bf16 compute copies are complete everywhere):
        ``sync_masters`` all-gathers the masters too (collective; needed before checkpointing or reading ``.weight``) --
        pass False inside a training loop that only needs the updates applied."""
        if self._pending_t is not None:
            if self._peer:
                from .peer import ROW_W1, ROW_W2

                px, e = self.aligner._ensure_peer(), self.aligner._peer_epoch
                px.wait(ROW_W1, e)
                px.wait(ROW_W2, e)
                self._grads_hold = None
                self._masters_stale = True
            elif self._sharded:
                self._wait_update("linear1")
                self._wait_update("linear2")
                self._grads_hold = None
                self._masters_stale = True
            else:
                self._wait_update("linear1")
                self._wait_update("linear2")
                self._grads_hold = None
            self.optimizer.mark_bf16_current()
            self._pending_t = None
            self.aligner._bf16_managed = False
        if sync_masters and getattr(self, "_masters_stale", False):
            self.aligner.sync_parameters()  # fp32 master rows of the other ranks (NCCL all-gather, off the hot path)
            self._masters_stale = False

    # -- host-fed path with the copy of batch i+1 overlapping the compute of batch i (what the reference's PrefetchLoader
    #    does on a side stream, thinkdiff/datasets/datasets/dataloader_utils.py:45-118)
    def prefetch(self, batch: FlatBatch, device="cuda"):
        """Start the H2D copies of ``batch`` (pinned host memory) on a dedicated copy stream; returns a handle for
        ``step_prefetched``. Nothing blocks the host."""
        k = max(1, int(getattr(self, "copy_streams", 2)))
        if not hasattr(self, "_copy_pool") or len(self._copy_pool) < k:
            self._copy_pool = [torch.cuda.Stream(device=device) for _ in range(k)]
        pool = self._copy_pool[:k]
        s0 = pool[0]
        with torch.cuda.stream(s0):
            # device buffers come from the caching allocator on the first copy stream; the others are ordered behind it
            flat = torch.empty(batch.flat.shape, dtype=batch.flat.dtype, device=device)
            tgt_h = batch.extras["flat_target"]
            tgt = torch.empty(tgt_h.shape, dtype=tgt_h.dtype, device=device)
            start = batch.src_row_start.to(device, non_blocking=True)
            lens = batch.lens.to(device, non_blocking=True)
        # the two big tensors are cut into row chunks spread over the copy streams: several DMA engines work in parallel,
        # which on these hosts is worth up to 2.6x over a single cudaMemcpyAsync stream
        jobs = []
        per = max(1, k // 2) if k > 1 else 1
        for dst, src, first in ((flat, batch.flat, 0), (tgt, tgt_h, per if k > 1 else 0)):
            rows = src.shape[0]
            step = (rows + per - 1) // per
            for c in range(per):
                lo, hi = c * step, min(rows, (c + 1) * step)
                if lo < hi:
                    jobs.append((pool[(first + c) % k], dst, src, lo, hi))
        events = []
        for st in pool[1:]:
            st.wait_stream(s0)
        for st, dst, src, lo, hi in jobs:
            with torch.cuda.stream(st):
                dst[lo:hi].copy_(src[lo:hi], non_blocking=True)
        for st in pool:
            ev = torch.cuda.Event()
            ev.record(st)
            events.append(ev)
        cb = batch.extras.get("_h2d_enqueued")
        if cb is not None:
            cb(events)  # the producer of the pinned buffers (EmbedShardReader) may recycle them once these have fired
        return (flat, start, lens, batch.total_rows, batch.l_max, tgt), events

    def tune_copy_streams(self, batch: FlatBatch, device="cuda", candidates=(1, 2, 4), reps: int = 2) -> int:
        """Pick how many copy streams ``prefetch`` spreads a batch over, by timing the H2D of ``batch`` alone for each candidate
        (hosts differ: on some a single cudaMemcpyAsync stream reaches PCIe line rate, on others several DMA engines are needed,
        on others more streams only add contention). Synchronises; call it once before the training loop."""
        import time

        best, best_t = int(getattr(self, "copy_streams", 2)), None
        for k in candidates:
            self.copy_streams = int(k)
            self.prefetch(batch, device)  # creates the streams / warms the allocator
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(reps):
                self.prefetch(batch, device)
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / reps
            if best_t is None or dt < best_t:
                best, best_t = int(k), dt
        self.copy_streams = best
        return best

    def step_prefetched(self, handle) -> torch.Tensor:
        tensors, events = handle
        cur = torch.cuda.current_stream()
        for ev in events:
            cur.wait_event(ev)
        for t in tensors:
            if isinstance(t, torch.Tensor):
                t.record_stream(cur)  # allocated on the copy stream, consumed here
        return self.step_device(*tensors)

    def step_host(self, batch: FlatBatch, device="cuda") -> torch.Tensor:
        """Inputs in (pinned) host memory: async H2D of the flat features/targets, then ``step_device``."""
        flat = batch.flat.to(device, non_blocking=True)
        tgt = batch.extras["flat_target"].to(device, non_blocking=True)
        start = batch.src_row_start.to(device, non_blocking=True)
        lens = batch.lens.to(device, non_blocking=True)
        cb = batch.extras.get("_h2d_enqueued")
        if cb is not None:
            ev = torch.cuda.Event()
            ev.record()
            cb([ev])
        return self.step_device(flat, start, lens, batch.total_rows, batch.l_max, tgt)


class AlignerT5TrainStep:
    """One training step of the aligner against the reference's objective (thinkdiff/models/mllama_vllm_t5_embed_decoder_2.py:585-598):
    the aligner output goes into the frozen T5 decoder as its encoder states and the loss is ``CrossEntropyLoss(ignore_index=-100)`` of
    the decoder's logits against the caption labels. Runs without autograd, as one direct call sequence: pack, aligner forward (fp32
    output with saved activations, the training regime), ``ops.t5_decoder_loss_fwd_bwd``, aligner backward from the fp32 encoder
    gradient into flat gradient buckets (the parameters' ``.grad`` are views of them), then the optimizer -- ``FusedAdamW`` with
    ``grad_scale = 1 / loss_scale``, or a torch optimizer with the gradients unscaled first. Without an optimizer the (scaled) gradients
    are left in ``.grad``. The static ``loss_scale`` is applied by the aligner backward, whose epilogues multiply in fp32, so a power of
    two scales every gradient exactly; the cross-entropy kernel folds its own ``grad_scale`` into the exponent of the softmax
    (``exp2(z log2 e - m + log2(scale / sum))``), where a scale moves the rounding of the logits' gradient.

    Same kernels and arithmetic as ``forward_packed`` under bf16 autocast + ``t5_decoder_loss(...).backward()``. One GPU: data
    parallel, a GradScaler, clipping and gradient accumulation are not built for this objective."""

    def __init__(self, aligner: ThinkDiffAligner, t5_weights, optimizer=None, loss_scale: float = 1.0, grad_scaler=None,
                 max_grad_norm: float = 0.0, accum_grad_iters: int = 1):
        if grad_scaler is not None or max_grad_norm > 0.0 or accum_grad_iters != 1:
            raise NotImplementedError("AlignerT5TrainStep: a GradScaler, gradient clipping and gradient accumulation are not built for "
                                      "the T5 objective (use a static loss_scale)")
        self._single_gpu(aligner)
        if aligner[0].weight.dtype != torch.float32:
            raise TypeError("AlignerT5TrainStep is a training step: the aligner's parameters must be float32 masters")
        self.aligner, self.t5, self.optimizer, self.loss_scale = aligner, t5_weights, optimizer, float(loss_scale)

    @staticmethod
    def _single_gpu(aligner):
        if aligner._dp is not None:
            raise NotImplementedError("AlignerT5TrainStep runs on one GPU: data parallel is not built for the T5 objective "
                                      "(call aligner.disable_data_parallel())")

    def step_device(self, flat, src_row_start, lens_dev, total_rows: int, l_max: int, labels, lens_q_dev, max_len_q: int) -> torch.Tensor:
        """Inputs already resident in HBM: the aligner's flat features with ``src_row_start`` / ``lens_dev`` (as ``AlignerTrainStep``),
        ``labels`` int64 [Mq] and ``lens_q_dev`` int32 [B] from ``t5.pack_labels``, ``max_len_q`` their longest sample. Returns the
        (unscaled) loss as a device scalar; nothing syncs the host."""
        from .aligner import GradBuckets

        a = self.aligner
        self._single_gpu(a)
        cu_k = ops.cu_seqlens(lens_dev)
        x = ops.pack_varlen(flat, src_row_start, cu_k, total_rows).to(torch.bfloat16)
        cu_q = ops.cu_seqlens(lens_q_dev)
        W1b, b1b, W2b, b2b = a._bf16_params()
        g = a[3].weight.detach()
        y, saved = ops.aligner_fwd(x, W1b, b1b, W2b, b2b, g, a.eps, False, True)
        loss, d_enc = ops.t5_decoder_loss_fwd_bwd(y, cu_k, l_max, labels, cu_q, max_len_q, self.t5)
        del y
        bwd = ops.AlignerBackward(x, saved, W2b, g, d_enc, grad_scale=self.loss_scale)
        gb = GradBuckets(a.mm_hidden_size, a.hidden_size, x.device)
        a._grad_flats = gb.flats()
        bwd.norm_and_linear2(gb.dW2, gb.db2, gb.dg)
        bwd.gelu_and_linear1(gb.dW1, gb.db1)
        for p, gr in zip((a[0].weight, a[0].bias, a[2].weight, a[2].bias, a[3].weight), gb.in_parameter_order()):
            p.grad = gr
        _optimizer_step(self.optimizer, self.loss_scale)
        return loss
