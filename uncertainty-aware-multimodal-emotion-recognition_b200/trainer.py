"""Data-parallel trainer step around the hot path (reference: src/training/training.py:121-150 AdamW parameter
groups, :176-245 train_epoch, :219 clip_grad_norm_, :224 optimizer.step).  The reference has no distributed code
(`setup_distributed_training` is `pass`, training.py:541-545); this is the north-star subsystem (4):

  * one process per GPU, batch sharded across ranks, weights and optimizer state replicated;
  * parameters and gradients live in ONE flat fp32 buffer each (encoder group first, then the rest), so the
    exchange step is a single NCCL all-reduce over the flat gradient buffer and the optimizer is two fused
    clip+AdamW launches (one per LR group) with the clip coefficient computed on the device - no host syncs;
  * the DEER loss is evaluated with exact GLOBAL-batch semantics: its 3x40 sufficient statistics (ECE bins, batch
    means) are all-reduced between the two loss phases, so N ranks x B/N samples give the same loss and gradients as
    one rank with B samples (BatchNorm statistics in the video encoder stay per-replica, as in stock DDP);
  * partially labelled batches: the optional batch key "target_mask" (targets' shape, bool / uint8, nonzero =
    labelled) reaches the fused loss; the per-dimension label counts are part of those statistics, so they are global
    too, and the mask is read on the device only (a captured step picks up a new mask content on every replay).
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import torch
import torch.distributed as dist
import torch.nn as nn

from . import ops
from ._lib import call, ptr
from .deer import EVIDENCE_KEY


class FlatBuffers:
    """Re-homes every parameter of `model` (and its .grad) into views of two flat fp32 buffers."""

    def __init__(self, model: nn.Module, group_fn):
        named = [(n, p) for n, p in model.named_parameters() if p.requires_grad]
        order = sorted(range(len(named)), key=lambda i: (group_fn(named[i][0]), i))
        self.names = [named[i][0] for i in order]
        params = [named[i][1] for i in order]
        dev = params[0].device
        # 16-byte aligned slots so float4 / TMA consumers can address any tensor
        offs, off = [], 0
        for p in params:
            offs.append(off)
            off += (p.numel() + 3) // 4 * 4
        self.numel = off
        self.params = torch.zeros(off, device=dev, dtype=torch.float32)
        self.grads = torch.zeros(off, device=dev, dtype=torch.float32)
        self.group_bounds: List[tuple] = []
        g_prev, start = None, 0
        for p, o, n in zip(params, offs, self.names):
            g = group_fn(n)
            if g != g_prev and g_prev is not None:
                self.group_bounds.append((g_prev, start, o))
                start = o
            g_prev = g
            self.params[o:o + p.numel()].copy_(p.data.reshape(-1))
            p.data = self.params[o:o + p.numel()].view_as(p)
            p.grad = self.grads[o:o + p.numel()].view_as(p)
        self.group_bounds.append((g_prev, start, off))
        self.payload = sum(p.numel() for p in params)
        self.offsets = offs

    def leading_prefix_end(self, prefix: str) -> int:
        """End offset of the run of parameters at the START of the buffer whose names begin with `prefix` (0 if none)."""
        end = 0
        for n, o in zip(self.names, self.offsets + [self.numel]):
            if not n.startswith(prefix):
                return o
            end = o
        return self.numel if self.names else end


def shard_batch(batch: Dict[str, torch.Tensor], rank: int, world: int) -> Dict[str, torch.Tensor]:
    """Contiguous equal shard of a global batch (SURVEY.md section 8e): rank r gets rows [r*B/world, (r+1)*B/world).
    Equal shard sizes keep mean-of-means == global mean for the batch-mean loss terms."""
    out = {}
    for k, v in batch.items():
        B = v.shape[0]
        if B % world != 0:
            raise ValueError(f"global batch {B} is not divisible by world size {world}")
        n = B // world
        out[k] = v[rank * n:(rank + 1) * n]
    return out


# Parameters that never receive a gradient in the REFERENCE (`p.grad is None`, so torch.optim.AdamW skips them
# entirely: no weight decay, no moment update): the never-executed uncertainty gate of HierarchicalMultimodalFusion
# (fusion.py:147-159, SURVEY app. B#4) and the pooled model's calibration layer, whose output does not feed the loss
# (complete_project.py:449).  Parameters with an exactly-zero gradient (Q/K rows of a single-key attention) DO take
# weight decay in the reference and stay in the optimised groups.
REFERENCE_NO_GRAD_PREFIXES = ("fusion.uncertainty_gate.", "calibration_layer.")
GROUP_ENCODER, GROUP_DEFAULT, GROUP_FROZEN = 0, 1, 2


def reference_lr_group(name: str) -> int:
    """training.py:128-142: names containing 'encoder' train at 0.5 x lr (group 0); everything else at lr (group 1);
    group 2 = parameters the reference optimizer never touches (grad is None), placed last and skipped."""
    if name.startswith(REFERENCE_NO_GRAD_PREFIXES):
        return GROUP_FROZEN
    return GROUP_ENCODER if "encoder" in name else GROUP_DEFAULT


def capture_forward(model: nn.Module, *inputs, warmup: int = 2, **kw_inputs):
    """CUDA-graph capture of an inference forward on static input tensors (refill them in place).  Returns
    (replay, outputs): `replay()` re-runs the captured launches and returns the static `outputs`."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.no_grad():
        with torch.cuda.stream(side):
            for _ in range(max(warmup, 1)):
                model(*inputs, **kw_inputs)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = model(*inputs, **kw_inputs)

    def replay():
        graph.replay()
        return out

    return replay, out


class DEERDataParallelTrainer:
    def __init__(self, model: nn.Module, learning_rate: float = 1e-4, weight_decay: float = 1e-5,
                 gradient_clip: float = 1.0, betas=(0.9, 0.999), eps: float = 1e-8,
                 process_group=None, exact_global_loss: bool = True, loss_weights=None, task_weights=None,
                 loss_eps: Optional[float] = None):
        self.model = model
        self._lr = float(learning_rate)
        self.wd, self.clip, self.betas, self.eps = weight_decay, gradient_clip, betas, eps
        self.pg = process_group
        self.world = dist.get_world_size(process_group) if (dist.is_available() and dist.is_initialized()) else 1
        self.exact_global_loss = exact_global_loss
        # the optimised objective is the model's own loss (what compute_loss reports): reg / kl / ece / cross-dimension
        # weights, task weights and epsilon are read from model.loss_fn (losses.MultiTaskDEERLoss) unless given
        lf = getattr(model, "loss_fn", None)
        if loss_weights is None:
            loss_weights = lf._weights()[0] if hasattr(lf, "_weights") else (0.1, 0.01, 0.05, 0.05)
        if task_weights is None and hasattr(lf, "_task_weight_list"):
            task_weights = lf._task_weight_list()
        if loss_eps is None:
            loss_eps = lf._weights()[1] if hasattr(lf, "_weights") else 1e-8
        self.loss_weights = tuple(float(w) for w in loss_weights)
        self.task_weights = task_weights
        self.loss_eps = float(loss_eps)
        self.flat = FlatBuffers(model, reference_lr_group)
        dev = self.flat.params.device
        self.m = torch.zeros_like(self.flat.params)
        self.v = torch.zeros_like(self.flat.params)
        self.sumsq = torch.zeros(1, device=dev, dtype=torch.float32)
        self.step_count = 0
        # device-side step counter and learning rate: a captured CUDA graph of the step replays unchanged while
        # both advance (dropout masks, AdamW bias corrections, LR schedule)
        self.step_tensor = torch.zeros(1, device=dev, dtype=torch.int64)
        # one learning rate PER GROUP on the device (training.py:138-142: encoder group at 0.5 x lr, and
        # CosineAnnealingLR anneals every group from ITS base value to the same eta_min, :155-159)
        self.group_scale = {GROUP_ENCODER: 0.5, GROUP_DEFAULT: 1.0}
        self.lr_tensor = torch.tensor([self.group_scale[GROUP_ENCODER] * float(learning_rate), float(learning_rate)],
                                      device=dev, dtype=torch.float32)
        self._graphs: Dict[int, tuple] = {}
        self._auto: Dict[tuple, dict] = {}
        self._graph_pool = None
        self.direct_grad = True   # backward kernels accumulate straight into the flat gradient buffer
        # Gradient exchange overlapped with BPTT: the audio encoder's parameters lead the flat buffer and its backward
        # (the LSTM recurrence, on its own stream) is the tail of the step, so everything behind them is all-reduced
        # as soon as the video / text / fusion / head backward has been issued, beside the audio backward.
        # Measured (round 2, B200 NVLink, graph replay): N = 2: 4.38 ms per step with one all-reduce at the end vs 4.39 ms
        # with the bucketed early exchange on a 32-CTA communicator, 4.53 ms on 8 CTAs, 5.12 ms on 2 CTAs (the collective
        # no longer fits the window); N = 8: 4.48 vs 4.53 ms.  The 2-rank timeline (profiles/r2_step_timeline_n2.txt)
        # shows what a step loses against one GPU: +43 us for the loss-statistics all-reduce between the two loss phases
        # and 109 us for the gradient all-reduce -- hiding the latter costs as much as it saves, because any CTA that is
        # resident beside the recurrence kernels pushes some of their 32 clusters into a second wave.  OFF by default.
        self.overlap_exchange = False
        self._audio_end = self.flat.leading_prefix_end("audio_encoder.")
        # Bucketed exchange (overlap_exchange): [0, _layer0_end) = the first LSTM layer (its gradients are the LAST to
        # complete), [_layer0_end, _audio_end) = rest of the audio encoder, [_audio_end, numel) = everything else.  The two
        # later buckets are all-reduced from a side stream on a separate NCCL communicator limited to `exchange_ctas`
        # CTAs, so that the collective fits beside the 128 CTAs of the recurrence kernels instead of pushing their
        # clusters into a second wave; only the first layer's 0.7 M gradients remain for the end of the step.
        self._layer0_end = self._leading_match_end(lambda n: n.startswith("audio_encoder.lstm.") and "_l0" in n)
        self.exchange_ctas = 8
        self._comm_group = None
        self._comm_stream = None
        self._grads_reduced = False
        self.last_losses: Optional[torch.Tensor] = None

    # ------------------------------------------------------------------ pieces
    def _leading_match_end(self, pred) -> int:
        """End offset of the run of parameters at the START of the flat buffer whose names satisfy `pred`."""
        f = self.flat
        for n, o in zip(f.names, f.offsets):
            if not pred(n):
                return o
        return f.numel

    def _comm(self):
        """(low-CTA NCCL communicator, launch stream) of the overlapped gradient buckets; created collectively on first use."""
        if self._comm_group is None:
            opts = dist.ProcessGroupNCCL.Options()
            opts.config.max_ctas = int(self.exchange_ctas)
            opts.config.min_ctas = 1
            ranks = dist.get_process_group_ranks(self.pg) if self.pg is not None else None
            self._comm_group = dist.new_group(ranks=ranks, backend="nccl", pg_options=opts)
            self._comm_stream = torch.cuda.Stream()
        return self._comm_group, self._comm_stream

    def _allreduce(self, t: torch.Tensor):
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.pg)

    def forward_backward(self, batch: Dict[str, torch.Tensor], loss_weight: float = 1.0) -> torch.Tensor:
        """fwd + fused head/loss + bwd; gradients are accumulated into the flat buffer.  Returns losses [5D+2].
        `loss_weight`: the per-batch dataset weight of training.py:211-212 (`weighted_loss = total_loss * w`): it scales
        the back-propagated gradient; the returned loss components stay unweighted (as the reference logs them)."""
        # one launch clears the flat gradient buffer and the gradient-norm accumulator -- on the weight-gradient stream,
        # beside the forward: nothing reads or accumulates into them before the backward starts (joined in front of it)
        cur = torch.cuda.current_stream()
        zs = ops._wgrad_stream() if self.flat.grads.is_cuda else None
        if zs is not None:
            zs.wait_stream(cur)
            with torch.cuda.stream(zs):
                call("deer_fill_zero", ptr(self.flat.grads), self.flat.numel, ptr(self.sumsq), 1)
            self._zero_stream = zs
        else:
            call("deer_fill_zero", ptr(self.flat.grads), self.flat.numel, ptr(self.sumsq), 1)
            self._zero_stream = None
        ops.set_direct_grad_accumulation(self.direct_grad)
        # this trainer's device step counter keys the dropout masks of ITS step only (restored afterwards)
        prev = ops.set_dropout_step_tensor(self.step_tensor)
        try:
            return self._forward_backward(batch, float(loss_weight))
        finally:
            ops.set_dropout_step_tensor(prev)
            ops.set_direct_grad_accumulation(False)

    def _forward_backward(self, batch: Dict[str, torch.Tensor], loss_weight: float = 1.0) -> torch.Tensor:
        model = self.model
        batch = {k: v for k, v in batch.items() if k != "dataset_id"}
        out = model(batch)   # both models accept the reference's batch dict (preprocessing.py:461-491)
        ev = out[EVIDENCE_KEY]
        targets = batch["targets"]
        target_mask = batch.get("target_mask")
        B = targets.shape[0]
        hook = self._allreduce if (self.exact_global_loss and self.world > 1) else None
        gb = B * self.world if self.exact_global_loss else B
        # with exact global semantics local gradients are SUMMED across ranks; otherwise they are averaged
        scale = (1.0 if self.exact_global_loss else 1.0 / self.world) * loss_weight
        ops.mark("head_out")
        losses, dE, _, _ = ops.nig_loss_raw(ev.detach(), None, targets, weights=self.loss_weights, eps=self.loss_eps,
                                            task_weights=self.task_weights, want_grad=True,
                                            grad_scale=scale, stats_hook=hook, global_batch=gb,
                                            target_mask=target_mask)
        ops.mark("loss_done")
        works = []
        handles = []
        fence = getattr(getattr(model, "video_encoder", None), "_first_bwd_node", None)
        lstm_nodes = getattr(getattr(model, "audio_encoder", None), "_lstm_bwd_nodes", None) or []
        if (self.world > 1 and self.overlap_exchange and fence is not None and ev.is_cuda and
                0 < self._audio_end < self.flat.numel and ops.branch_streams_enabled()):
            group, cs = self._comm()
            grads = self.flat.grads

            def _bucket(lo, hi, wait_sides=False):
                # issued from the autograd thread inside a node hook: the collective is launched on the communication
                # stream once the stream of that node AND the weight-gradient stream have drained up to here; neither
                # of them waits for it
                def hook(*_):
                    cs.wait_stream(torch.cuda.current_stream())
                    cs.wait_stream(ops._wgrad_stream())
                    if wait_sides:   # the text encoder's backward runs on its own stream (issued before this node)
                        for st_ in getattr(model, "branch_streams", lambda: [])():
                            cs.wait_stream(st_)
                    with torch.cuda.stream(cs):
                        works.append(dist.all_reduce(grads[lo:hi], op=dist.ReduceOp.SUM, group=group, async_op=True))
                return hook

            # (1) right after the LAST video/text/fusion/head backward node (the video encoder's first op has the lowest
            # sequence number on the main stream): every gradient behind the audio block is complete
            handles.append(fence.register_hook(_bucket(self._audio_end, self.flat.numel, wait_sides=True)))
            # (2) right after the BPTT + weight-gradient GEMMs of LSTM layer 1 (audio stream): the rest of the audio
            # encoder; it travels beside the BPTT of layer 0
            tail_lo = 0
            if len(lstm_nodes) >= 2 and lstm_nodes[1] is not None and 0 < self._layer0_end < self._audio_end:
                handles.append(lstm_nodes[1].register_hook(_bucket(self._layer0_end, self._audio_end)))
                tail_lo = self._layer0_end
            else:
                tail_lo = self._audio_end
        if getattr(self, "_zero_stream", None) is not None:
            torch.cuda.current_stream().wait_stream(self._zero_stream)   # the cleared gradient buffer
            self._zero_stream = None
        ev.backward(dE)
        for h_ in handles:
            h_.remove()
        ops.join_wgrad_stream()   # deferred weight-gradient GEMMs of the small layers (ops._Linear.backward)
        if works:
            # (3) what is left: the first LSTM layer (or the whole audio block), on the full-bandwidth communicator
            dist.all_reduce(self.flat.grads[:tail_lo], op=dist.ReduceOp.SUM, group=self.pg)
            for w in works:
                w.wait()
            self._grads_reduced = True
        self.last_losses = losses
        return losses

    @property
    def lr(self) -> float:
        return self._lr

    @lr.setter
    def lr(self, value: float):
        """Learning-rate schedule hook: updates the device scalars the (possibly graph-captured) AdamW launches read
        (every group at its multiple of `value`)."""
        self.set_group_lrs({g: sc * float(value) for g, sc in self.group_scale.items()})
        self._lr = float(value)

    def set_group_lrs(self, lrs: Dict[int, float]):
        """Per-group learning rates (group 0 = names containing 'encoder', group 1 = the rest), e.g. from a scheduler
        that anneals each group from its own base value (CosineAnnealingLR, training.py:155-159)."""
        vals = [float(lrs[GROUP_ENCODER]), float(lrs[GROUP_DEFAULT])]
        self.lr_tensor.copy_(torch.tensor(vals, dtype=torch.float32), non_blocking=False)
        self._lr = vals[1]

    def group_lrs(self) -> Dict[int, float]:
        v = self.lr_tensor.tolist()
        return {GROUP_ENCODER: v[0], GROUP_DEFAULT: v[1]}

    def optimizer_step(self):
        self.step_count += 1
        f = self.flat
        if not self._grads_reduced:
            self._allreduce(f.grads)
        self._grads_reduced = False
        ops.mark("grads_exchanged")
        call("deer_sumsq", ptr(f.grads), f.numel, ptr(self.sumsq))
        for g, lo, hi in f.group_bounds:
            n = hi - lo
            if n <= 0 or g == GROUP_FROZEN:   # the reference optimizer never sees these (grad is None): no decay either
                continue
            # lr = lr_tensor[group], step = *step_tensor + 1: both read on the device
            call("deer_adamw", f.params.data_ptr() + 4 * lo, f.grads.data_ptr() + 4 * lo, self.m.data_ptr() + 4 * lo,
                 self.v.data_ptr() + 4 * lo, n, 1.0, float(self.betas[0]),
                 float(self.betas[1]), float(self.eps), float(self.wd), 0, ptr(self.sumsq),
                 float(self.clip), 1.0, self.step_tensor.data_ptr(), self.lr_tensor.data_ptr() + 4 * g)
        call("deer_step_increment", self.step_tensor.data_ptr())

    def train_step(self, batch: Dict[str, torch.Tensor], loss_weight: float = 1.0) -> torch.Tensor:
        losses = self.forward_backward(batch, loss_weight)
        self.optimizer_step()
        return losses

    # ------------------------------------------------------------------ CUDA-graph replay of the whole step
    def capture(self, batch: Dict[str, torch.Tensor], warmup: int = 2, loss_weight: float = 1.0):
        """Capture fwd + loss + bwd + exchange + clip + AdamW on the tensors of `batch` (which become the static
        input buffers: refill them in place, e.g. with `copy_` from pinned host memory) into one CUDA graph.
        The ~300 kernel launches of a step then cost one `cudaGraphLaunch`; the step counter, dropout masks and the
        learning rate keep advancing because the kernels read them from device memory.  Returns a callable that
        replays the step and returns the (static) losses tensor."""
        key = tuple(sorted((k, v.data_ptr(), tuple(v.shape)) for k, v in batch.items() if torch.is_tensor(v)))
        key = key + (("loss_weight", float(loss_weight)),)   # a kernel argument of the captured launches
        hit = self._graphs.get(hash(key))
        if hit is not None:
            return hit[2]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):       # lazily created state (TMA descriptors, smem opt-ins, NCCL buffers)
                self.train_step(batch, loss_weight)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        if self._graph_pool is None:
            self._graph_pool = torch.cuda.graph_pool_handle()
        with torch.cuda.graph(graph, pool=self._graph_pool):
            losses = self.train_step(batch, loss_weight)
        self.step_count -= 1   # the capture pass itself launched nothing

        def replay() -> torch.Tensor:
            self.step_count += 1
            graph.replay()
            self.last_losses = losses
            return losses

        self._graphs[hash(key)] = (graph, losses, replay)
        return replay

    def train_step_auto(self, batch: Dict[str, torch.Tensor], eager_steps: int = 2,
                        loss_weight: float = 1.0, static_inputs: bool = False) -> torch.Tensor:
        """train_step for a stream of freshly allocated batches (a DataLoader): the first `eager_steps` batches of a
        given shape run eagerly (they double as the warm-up), then the step is captured once on static input buffers
        and every later batch of that shape is copied into them and replayed.  Batches of another shape (the last,
        short one of an epoch) get their own entry."""
        tens = {k: v for k, v in batch.items() if torch.is_tensor(v) and k != "dataset_id"}
        if static_inputs:
            # the batch already lives in static device buffers (data.DevicePrefetcher rotates a few sets): capture the
            # step on those addresses directly -- one graph per buffer set, no device-to-device copy per step
            sig = tuple(sorted((k, v.data_ptr(), tuple(v.shape)) for k, v in tens.items())) + (float(loss_weight),)
            ent = self._auto.setdefault(sig, {"seen": 0, "replay": None})
            if ent["replay"] is None:
                ent["seen"] += 1
                if ent["seen"] <= eager_steps or not all(v.is_cuda for v in tens.values()):
                    return self.train_step(tens, loss_weight)
                ent["replay"] = self.capture(tens, warmup=0, loss_weight=loss_weight)
            return ent["replay"]()
        sig = tuple(sorted((k, tuple(v.shape), v.dtype) for k, v in tens.items())) + (float(loss_weight),)
        ent = self._auto.setdefault(sig, {"seen": 0, "static": None, "replay": None})
        if ent["replay"] is None:
            ent["seen"] += 1
            if ent["seen"] <= eager_steps or not all(v.is_cuda for v in tens.values()):
                return self.train_step(batch, loss_weight)
            ent["static"] = {k: v.clone() for k, v in tens.items()}
            ent["replay"] = self.capture(ent["static"], warmup=0, loss_weight=loss_weight)
            # the capture pass launched nothing: fall through and replay this batch
        for k, v in tens.items():
            ent["static"][k].copy_(v, non_blocking=True)
        return ent["replay"]()

    def grad_norm(self) -> torch.Tensor:
        return self.sumsq.sqrt()
