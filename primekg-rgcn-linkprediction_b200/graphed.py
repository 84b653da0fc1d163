"""CUDA-graph replay of the hot step (forward + loss + backward) for launch-bound graph sizes.

At the reference's sizes one full-graph step is ~50 kernels of 3-80 us; issued eagerly from Python the host is the
limiter.  ``GraphedTrainStep`` captures one step — ``model(edge_index, edge_type, heads, tails, rels)`` ->
``BCEWithLogitsLoss`` -> ``backward()`` (reference src/train.py:291-306) — into a CUDA graph over static input buffers
and replays it; gradients land in the parameters' ``.grad`` as usual (each replay OVERWRITES them: the step owns the
buffers, so gradient accumulation over several batches needs ``flat_grads=True`` and a caller-side sum), so the
optimiser / clipping code of the caller (src/train.py:309-318) stays as it is — or, with ``optimizer=FusedAdam(...)``
(optim.py), the clipping and the Adam update become the last kernels of the captured step.  Dropout masks are re-drawn on every replay: the fused dropout is a counter-based hash of (seed, device-side
step counter, element index) and the counter is advanced by a kernel of the captured step itself (csrc/transform.cu,
csrc/decoder.cu; statistical quality: tests/test_gpu_parity.py::test_fused_dropout_hash_statistics).

Construct it before (or after dropping) any eager autograd graph of the same model: a live graph keeps the
parameters' AccumulateGrad nodes bound to the stream they were created on, which a capture cannot depend on.
"""
from __future__ import annotations

from typing import Callable, Optional

import torch

from .ops import bce_with_logits


class GraphedTrainStep:
    def __init__(self, model: torch.nn.Module, edge_index: torch.Tensor, edge_type: torch.Tensor, batch_size: int,
                 loss_fn: Optional[Callable] = None, warmup: int = 3, flat_grads: bool = False, sampler=None,
                 host_io: bool = False, allreduce: Optional[str] = None, optimizer=None):
        """``host_io``: the captured graph starts with the host-to-device copy of the batch from a pinned staging block
        (``self.host_batch``, int64 [4, B] in ``pack_batch`` layout) and ends with the device-to-host copy of the loss
        and the correct-count into pinned memory (``self.host_loss``, ``self.host_correct``): one graph launch per step
        is the whole host-side work.  Fill ``host_batch`` (``step.host_batch.copy_(packed)``), call ``replay_host()``,
        synchronise, read ``host_loss``; do not rewrite ``host_batch`` before the previous replay has consumed it
        (the reference's loop reads ``loss.item()`` every step, src/train.py:322, which is such a synchronisation).

        ``sampler`` (a ``NegativeSampler``): the captured step starts from ``batch_size / (1 + num_neg_samples)``
        POSITIVE edges and draws the negatives, the concatenation and the labels on the device inside the graph
        (reference src/train.py:276-288) — ``step.run_positives(pos_head, pos_tail, pos_rel)``; fresh negatives on every
        replay."""
        """``allreduce="peer"`` (needs ``flat_grads="arena"`` and an initialised process group of GPUs with peer access):
        data-parallel replicas — the backward kernels write the parameter gradients into a peer-visible flat buffer and the
        LAST kernels of the captured step average it over the ranks (``peer.PeerAllReduce``: our two-shot all-reduce over
        NVLink, no collective call); ``p.grad`` then are views of the averaged buffer.  Every rank must replay in step."""
        """``optimizer`` (an ``optim.FusedAdam`` / ``FusedAdamW`` over parameters of ``model``): its clipping and update
        kernels are captured as the last compute of the step (after the peer all-reduce, before the ``host_io`` copies),
        so one replay is the whole training iteration.  The warm-up steps run without it (construction moves neither
        the parameters nor the optimiser state).  Every replay first copies changed group hyperparameters (an LR
        scheduler's ``lr``) to the device and afterwards bumps the parameters' in-place versions; ``step.grad_norm`` is
        the optimiser's device-side total gradient norm.  The optimiser's state tensors must keep their addresses
        (``FusedAdam.load_state_dict`` loads into them)."""
        if not edge_index.is_cuda:
            raise RuntimeError("GraphedTrainStep needs CUDA tensors")
        dev = edge_index.device
        self.model, self.edge_index, self.edge_type = model, edge_index, edge_type
        self.loss_fn = loss_fn or bce_with_logits      # fused equivalent of nn.BCEWithLogitsLoss()
        # default loss + a model that offers it: decoder, loss and accuracy in one kernel pair (model.link_loss)
        self.fused_loss = loss_fn is None and hasattr(model, "link_loss")
        self.correct = None
        # the static input buffers are views of ONE int64 [4, B] block (heads, tails, rels; row 3 holds the float32
        # labels in its first 4 B bytes), so a caller that keeps its batch packed the same way in pinned host memory
        # (``pack_batch``) pays one host-to-device copy per step instead of four (``load_packed``)
        self.batch_size = batch_size
        self.batch_buf = torch.zeros(4, batch_size, dtype=torch.int64, device=dev)
        self.heads, self.tails, self.rels = self.batch_buf[0], self.batch_buf[1], self.batch_buf[2]
        self.labels = self.batch_buf[3].view(torch.float32)[:batch_size]
        self.host_io = bool(host_io)
        if self.host_io:
            self.host_batch = torch.zeros(4, batch_size, dtype=torch.int64).pin_memory()
            self.host_loss = torch.zeros(1, dtype=torch.float32).pin_memory()
            self.host_correct = torch.zeros(1, dtype=torch.int32).pin_memory()
        self.sampler = sampler
        if sampler is not None:
            if batch_size % (1 + sampler.num_neg_samples):
                raise ValueError("batch_size must be n_pos * (1 + num_neg_samples)")
            n_pos = batch_size // (1 + sampler.num_neg_samples)
            self.pos_heads = torch.zeros(n_pos, dtype=torch.int64, device=dev)
            self.pos_tails = torch.zeros(n_pos, dtype=torch.int64, device=dev)
            self.pos_rels = torch.zeros(n_pos, dtype=torch.int64, device=dev)
        self.params = [p for p in model.parameters() if p.requires_grad]
        self.optimizer = optimizer
        self._capturing = False
        if optimizer is not None:
            from .optim import FusedAdam
            if not isinstance(optimizer, FusedAdam):
                raise TypeError("optimizer must be a FusedAdam / FusedAdamW (its kernels are what the graph captures)")
            mine = {id(p) for p in self.params}
            if any(id(p) not in mine for g in optimizer.param_groups for p in g["params"]):
                raise ValueError("the optimizer holds a parameter that is not a trainable parameter of the model")
            optimizer.prepare_capture()        # state, workspace, hyperparameters: nothing is allocated under capture
            self._opt_params = [p for g in optimizer.param_groups for p in g["params"]]
        self.flat_grad = None
        self.arena = None
        self.peer_ar = None
        if allreduce not in (None, "peer"):
            raise ValueError("allreduce must be None or 'peer'")
        if allreduce == "peer" and flat_grads != "arena":
            raise ValueError("allreduce='peer' needs flat_grads='arena'")
        if flat_grads == "arena":
            # the backward kernels write the parameter gradients straight into one flat buffer (ops.GradArena): no zero
            # fill, no accumulate kernels, and ONE tensor to all-reduce
            from . import ops
            numel = sum((p.numel() + 63) // 64 * 64 for p in self.params)
            if allreduce == "peer":
                from .peer import PeerAllReduce
                self.peer_ar = PeerAllReduce(numel, dev)
                self.arena = ops.GradArena(numel, dev, buf=self.peer_ar.inp)
            else:
                self.arena = ops.GradArena(numel, dev)
            for p in self.params:
                p.grad = None
        elif flat_grads:
            # static gradient buffers: views into ONE flat tensor, so zeroing is a single fill and a data-parallel
            # caller all-reduces ``flat_grad`` in place (every p.grad sees the result); costs one accumulate per tensor
            self.flat_grad = torch.zeros(sum(p.numel() for p in self.params), dtype=torch.float32, device=dev)
            off = 0
            for p in self.params:
                p.grad = self.flat_grad[off:off + p.numel()].view_as(p)
                off += p.numel()
        else:
            # the kernels' own output buffers (static inside the captured graph) become p.grad: no zero fill and
            # no accumulate kernels
            for p in self.params:
                p.grad = None
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self._step()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        from . import ops as _ops
        _ops.raise_on_bad_pairs(dev)                     # an out-of-range index in the warm-up batch surfaces here
        # capture on the stream the warm-up ran on: the per-stream workspaces (ops._workspace, the fused loss's ticket
        # buffer) exist already, so no allocation — and no zero-fill node — ends up inside the graph
        self.graph = torch.cuda.CUDAGraph()
        self._capturing = True
        try:
            with torch.cuda.graph(self.graph, stream=side):
                self.loss, self.scores = self._step()
        finally:
            self._capturing = False
        if self.arena is not None:
            lo, hi = self.arena.buf.data_ptr(), self.arena.buf.data_ptr() + self.arena.buf.numel() * 4
            inside = all(g is not None and lo <= g.data_ptr() < hi for g in self._grads)
            if inside:
                self.flat_grad = self.arena.used        # every parameter gradient lives inside: all-reduce this one tensor
            # else (e.g. basis layers, whose gradients autograd assembles): p.grad are ordinary tensors, flat_grad stays None
            if self.peer_ar is not None:
                self._avg = self._step_grads()
                self.flat_grad = self.peer_ar.out[: self.arena.off]
        self._bind_grads()

    def _step(self):
        if self.arena is not None:
            from . import ops
            self.arena.reset()
            ops.set_grad_arena(self.arena)
            try:
                return self._step_body()
            finally:
                ops.set_grad_arena(None)
        return self._step_body()

    def _step_body(self):
        if self.host_io:
            self.batch_buf.copy_(self.host_batch, non_blocking=True)          # a memcpy node of the captured graph
        out = self._step_compute()
        if self.peer_ar is not None:
            self.peer_ar(self.arena.off)               # gradient exchange = the last kernels of the (captured) step
        if self.optimizer is not None and self._capturing:
            # every rank applies the same deterministic update to the same averaged gradients
            self.optimizer._launch(list(zip(self.params, self._step_grads())))
        if self.host_io:
            self.host_loss.copy_(out[0].reshape(1), non_blocking=True)
            if self.correct is not None:
                self.host_correct.copy_(self.correct.reshape(1), non_blocking=True)
        return out

    def _step_compute(self):
        if self.sampler is not None:
            self.sampler.batch(self.pos_heads, self.pos_tails, self.pos_rels,
                               out=(self.heads, self.tails, self.rels, self.labels))
        if self.fused_loss:
            loss, scores, self.correct = self.model.link_loss(self.edge_index, self.edge_type, self.heads, self.tails,
                                                              self.rels, self.labels)
        else:
            scores = self.model(self.edge_index, self.edge_type, self.heads, self.tails, self.rels)
            loss = self.loss_fn(scores, self.labels)
        if self.flat_grad is not None and self.arena is None:
            self.flat_grad.zero_()
            loss.backward()
        else:
            if getattr(self, "_one", None) is None or self._one.device != loss.device:
                self._one = torch.ones((), dtype=loss.dtype, device=loss.device)     # the seed gradient: no fill kernel per step
            self._grads = torch.autograd.grad(loss, self.params, grad_outputs=self._one, allow_unused=True)
        return loss.detach(), scores.detach()

    def _step_grads(self):
        """The gradients the step leaves, one per parameter (None: unused), before ``_bind_grads`` publishes them."""
        if self.peer_ar is not None:
            # the averaged gradients: same offsets as in the arena, in the exchange's output buffer
            lo = self.arena.buf.data_ptr()
            if any(g is None or not lo <= g.data_ptr() < lo + self.arena.buf.numel() * 4 for g in self._grads):
                raise RuntimeError("allreduce='peer': a parameter gradient was not written into the arena")
            return [self.peer_ar.out[(g.data_ptr() - lo) // 4: (g.data_ptr() - lo) // 4 + g.numel()].view_as(g)
                    for g in self._grads]
        if self.flat_grad is not None and self.arena is None:
            return [p.grad for p in self.params]
        return list(self._grads)

    @property
    def grad_norm(self) -> Optional[torch.Tensor]:
        """Total gradient norm of the last replay (device scalar; NaN when the optimizer does not clip)."""
        return None if self.optimizer is None else self.optimizer.grad_norm

    def _replay(self) -> None:
        if self.optimizer is not None:
            self.optimizer.sync_hparams()
        self.graph.replay()
        if self.optimizer is not None:
            torch.autograd.graph.increment_version(self._opt_params)

    def _bind_grads(self) -> None:
        if self.peer_ar is not None and getattr(self, "_avg", None) is not None:
            for p, g in zip(self.params, self._avg):
                p.grad = g
        elif self.flat_grad is None or self.arena is not None:
            for p, g in zip(self.params, self._grads):
                p.grad = g

    def load_batch(self, heads, tails, rels, labels, non_blocking: bool = True) -> None:
        """Copy one batch (host, pinned or device tensors) into the static input buffers."""
        self.heads.copy_(heads, non_blocking=non_blocking)
        self.tails.copy_(tails, non_blocking=non_blocking)
        self.rels.copy_(rels, non_blocking=non_blocking)
        self.labels.copy_(labels, non_blocking=non_blocking)

    @staticmethod
    def pack_batch(heads, tails, rels, labels, pin: bool = True) -> torch.Tensor:
        """One int64 [4, B] host tensor in the layout of the step's input block (pinned by default)."""
        b = heads.numel()
        out = torch.empty(4, b, dtype=torch.int64)
        if pin and torch.cuda.is_available():
            out = out.pin_memory()
        out[0].copy_(heads); out[1].copy_(tails); out[2].copy_(rels)
        out[3].zero_()
        out[3].view(torch.float32)[:b].copy_(labels)
        return out

    def load_packed(self, packed: torch.Tensor, non_blocking: bool = True) -> None:
        """Copy a ``pack_batch`` block (host or device) into the static input buffers: one copy."""
        if packed.shape != self.batch_buf.shape or packed.dtype != torch.int64:
            raise ValueError(f"packed batch must be int64 {tuple(self.batch_buf.shape)}")
        self.batch_buf.copy_(packed, non_blocking=non_blocking)

    def run_packed(self, packed: torch.Tensor) -> torch.Tensor:
        """One step from a ``pack_batch`` block."""
        if self.sampler is not None:
            raise RuntimeError("this step draws its own negatives: call run_positives(pos_heads, pos_tails, pos_rels)")
        self.load_packed(packed)
        self._replay()
        self._bind_grads()
        return self.loss

    def replay_host(self) -> torch.Tensor:
        """``host_io`` step: batch from ``host_batch``, results into ``host_loss`` / ``host_correct`` — one graph launch.
        Returns the pinned loss tensor (valid after a synchronisation)."""
        if not self.host_io:
            raise RuntimeError("replay_host needs a GraphedTrainStep built with host_io=True")
        self._replay()
        self._bind_grads()
        return self.host_loss

    def run_positives(self, pos_heads, pos_tails, pos_rels, non_blocking: bool = True) -> torch.Tensor:
        """One step from positive edges only (needs ``sampler``): negatives, labels, forward, loss, backward in the graph."""
        if self.sampler is None:
            raise RuntimeError("run_positives needs a GraphedTrainStep built with sampler=NegativeSampler(...)")
        self.pos_heads.copy_(pos_heads, non_blocking=non_blocking)
        self.pos_tails.copy_(pos_tails, non_blocking=non_blocking)
        self.pos_rels.copy_(pos_rels, non_blocking=non_blocking)
        self._replay()
        self._bind_grads()
        return self.loss

    def __call__(self, heads=None, tails=None, rels=None, labels=None) -> torch.Tensor:
        """Run one step; returns the (static) loss tensor.  With no arguments the buffers are used as they are."""
        if heads is not None:
            if self.sampler is not None:
                raise RuntimeError("this step draws its own negatives: call run_positives(pos_heads, pos_tails, pos_rels)")
            self.load_batch(heads, tails, rels, labels)
        self._replay()
        self._bind_grads()          # (a caller may have set .grad to None, e.g. optimizer.zero_grad())
        return self.loss
