"""Gradient clipping + Adam / AdamW as one device step (``rgcn_adam_step``, csrc/optim.cu).

``FusedAdam(params, lr, ..., max_grad_norm=1.0)`` does what the reference's ``clip_grad_norm_(params, 1.0)`` followed
by ``torch.optim.Adam.step()`` does (src/train.py:311-318), in two kernels (one without clipping): a deterministic
gradient-norm pass and one read-modify-write pass over parameters, gradients and both moments.  It subclasses
``torch.optim.Adam``, so ``param_groups``, ``state_dict`` / ``load_state_dict``, LR schedulers and hooks are torch's
own; the per-parameter state is torch's (``step`` a 0-dim fp32 tensor on the parameter's device, as with
``capturable=True``, ``exp_avg``, ``exp_avg_sq``) and a state dict moves both ways between it and ``torch.optim.Adam``.

The arithmetic is that of torch's single-tensor Adam, element by element in the same order.  One visible difference:
the clipped gradient is used on the fly and NOT written back to ``p.grad`` (torch's ``clip_grad_norm_`` scales
``p.grad`` in place).  ``grad_norm`` is the total norm before clipping (torch's return value) as a device scalar, NaN
when the optimiser does not clip.

``GraphedTrainStep(..., optimizer=FusedAdam(...))`` makes the two kernels the last of the captured training step.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from .graph import _ptr, _stream

_UNSUPPORTED = ("amsgrad", "maximize", "differentiable")


class FusedAdam(torch.optim.Adam):
    """``torch.optim.Adam`` (``decoupled_weight_decay=True``: AdamW) whose ``step()`` runs our sm_100a kernels, with
    ``clip_grad_norm_(params, max_grad_norm)`` folded in when ``max_grad_norm`` is given.  fp32 contiguous CUDA
    parameters on one device, at most 64 parameter tensors."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, amsgrad=False, *,
                 foreach=None, maximize=False, capturable=False, differentiable=False, fused=None,
                 decoupled_weight_decay=False, max_grad_norm: Optional[float] = None):
        for name, val in (("amsgrad", amsgrad), ("maximize", maximize), ("differentiable", differentiable)):
            if val:
                raise ValueError(f"FusedAdam does not implement {name}=True")
        if foreach:
            raise ValueError("FusedAdam runs its own kernels: foreach=True is not supported")
        if fused:
            raise ValueError("FusedAdam runs its own kernels: fused=True (torch's fused Adam) is not supported")
        if max_grad_norm is not None and not float(max_grad_norm) >= 0.0:
            raise ValueError(f"max_grad_norm must be None or >= 0, got {max_grad_norm}")
        # capturable=True: torch keeps 'step' on the parameter's device, which is where the kernels read it
        super().__init__(params, lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, amsgrad=False,
                         foreach=foreach, maximize=False, capturable=True, differentiable=False, fused=None,
                         decoupled_weight_decay=decoupled_weight_decay)
        self.max_grad_norm = None if max_grad_norm is None else float(max_grad_norm)
        dev = None
        n = 0
        for group in self.param_groups:
            for p in group["params"]:
                if not p.is_cuda:
                    raise RuntimeError("FusedAdam needs CUDA parameters: this package has no CPU implementation")
                if p.is_sparse or p.dtype != torch.float32 or not p.is_contiguous():
                    raise ValueError("FusedAdam needs dense, contiguous float32 parameters")
                if dev is not None and p.device != dev:
                    raise ValueError("FusedAdam needs every parameter on one device")
                dev = p.device
                n += 1
        if n > _lib.ADAM_MAX_SEGMENTS:
            raise ValueError(f"FusedAdam handles at most {_lib.ADAM_MAX_SEGMENTS} parameter tensors, got {n}")
        self._device = dev
        self._ws = None
        self._hp_dev = None
        self._hp_host = None
        self._table_key = None
        self._table = None
        self.grad_norm = None if dev is None else torch.full((), float("nan"), dtype=torch.float32, device=dev)

    # ---------------------------------------------------------------------------------------------------------------
    def load_state_dict(self, state_dict) -> None:
        for g in state_dict["param_groups"]:
            for name in _UNSUPPORTED:
                if g.get(name, False):
                    raise ValueError(f"FusedAdam does not implement {name}=True (found in the loaded state dict)")
        old = {p: dict(st) for p, st in self.state.items()}
        super().load_state_dict(state_dict)
        # a plain torch.optim.Adam's dict carries capturable=False and CPU steps: keep the steps on the device
        for group in self.param_groups:
            group["capturable"] = True
            group["foreach"] = group.get("foreach") or None
            group["fused"] = None
            for p in group["params"]:
                st = self.state.get(p)
                if not st:
                    continue
                st["step"] = torch.as_tensor(st["step"], dtype=torch.float32).to(p.device).reshape(())
                prev = old.get(p)
                if prev and all(k in prev for k in ("step", "exp_avg", "exp_avg_sq")):
                    # load INTO the existing state tensors: a captured training step keeps their addresses
                    for k in ("step", "exp_avg", "exp_avg_sq"):
                        prev[k].copy_(st[k])
                        st[k] = prev[k]
        self._table_key = None
        self._hp_host = None

    def _init_state(self, p: torch.Tensor) -> dict:
        st = self.state[p]
        if len(st) == 0:
            st["step"] = torch.zeros((), dtype=torch.float32, device=p.device)
            st["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
            st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
            self._table_key = None
        return st

    def prepare_capture(self) -> None:
        """Allocate everything a step touches (the state of every parameter, the workspace, the hyperparameter array)
        and load the kernels, so that a later step can be captured into a CUDA graph without allocating."""
        for group in self.param_groups:
            for p in group["params"]:
                self._init_state(p)
        self._device_buffers()

    def _device_buffers(self) -> None:
        if self._ws is None:
            total = sum(p.numel() for g in self.param_groups for p in g["params"])
            lib = _lib.load()
            nbytes = int(lib.rgcn_adam_workspace_bytes(total, _lib.ADAM_MAX_SEGMENTS))
            self._ws = torch.zeros(nbytes, dtype=torch.uint8, device=self._device)
            with torch.cuda.device(self._device):
                _lib.check(lib.rgcn_adam_step(None, 0, None, 0, -1.0, None, None, 0, _stream(self._device)),
                           "rgcn_adam_step")
        if not torch.cuda.is_current_stream_capturing():
            self.sync_hparams()

    def sync_hparams(self) -> None:
        """Copy the groups' lr / betas / eps / weight_decay to the device array the kernels read, when any changed
        since the last copy (an LR scheduler's change reaches the next step, captured or not)."""
        vals = tuple((float(g["lr"]), float(g["betas"][0]), float(g["betas"][1]), float(g["eps"]),
                      float(g["weight_decay"]), bool(g["decoupled_weight_decay"])) for g in self.param_groups)
        if vals == self._hp_host:
            return
        for g in self.param_groups:
            for name in _UNSUPPORTED:
                if g.get(name, False):
                    raise ValueError(f"FusedAdam does not implement {name}=True")
        host = (_lib.AdamHparams * len(vals))(*[_lib.AdamHparams(*v[:5], int(v[5])) for v in vals])
        src = torch.frombuffer(bytearray(bytes(host)), dtype=torch.uint8)
        if self._hp_dev is None or self._hp_dev.numel() != src.numel():
            self._hp_dev = torch.empty(src.numel(), dtype=torch.uint8, device=self._device)
            self._table_key = None
        self._hp_dev.copy_(src)
        self._hp_host = vals

    def _launch(self, pairs: Sequence[Tuple[torch.Tensor, Optional[torch.Tensor]]]) -> List[torch.Tensor]:
        """Enqueue the step for (param, grad) pairs on the current stream; pairs with grad None are skipped (their step
        does not advance, as in torch).  Returns the updated parameters."""
        if self._device is None:
            return []
        self._device_buffers()
        live = [(p, g) for p, g in pairs if g is not None]
        key = tuple((p.data_ptr(), g.data_ptr()) for p, g in live)
        if key != self._table_key:
            group_of = {p: gi for gi, group in enumerate(self.param_groups) for p in group["params"]}
            segs = []
            for p, g in live:
                if p not in group_of:
                    raise ValueError("FusedAdam: a gradient was given for a parameter this optimiser does not hold")
                if g.is_sparse or g.dtype != torch.float32 or not g.is_contiguous() or g.shape != p.shape \
                        or g.device != p.device:
                    raise ValueError("FusedAdam needs dense contiguous float32 gradients shaped like their parameters")
                st = self._init_state(p)
                segs.append(_lib.AdamSegment(p.data_ptr(), g.data_ptr(), st["exp_avg"].data_ptr(),
                                             st["exp_avg_sq"].data_ptr(), st["step"].data_ptr(), p.numel(),
                                             group_of[p]))
            self._table = ((_lib.AdamSegment * max(len(segs), 1))(*segs), len(segs))
            self._table_key = key
        table, n = self._table
        if n == 0:
            return []
        clip = -1.0 if self.max_grad_norm is None else self.max_grad_norm
        lib = _lib.load()
        _lib.check(lib.rgcn_adam_step(table, n, _ptr(self._hp_dev), len(self.param_groups), clip,
                                      _ptr(self.grad_norm), _ptr(self._ws), self._ws.numel(), _stream(self._device)),
                   "rgcn_adam_step")
        return [p for p, _ in live]

    @torch.no_grad()
    def step(self, closure=None):
        """One clip + Adam step over every parameter with a gradient; returns the closure's loss like torch."""
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        pairs = [(p, p.grad) for group in self.param_groups for p in group["params"]]
        updated = self._launch(pairs)
        if updated:
            # the kernels write through raw pointers: bump the in-place versions so that caches keyed on p._version
            # (DrugDiseaseRGCN's eval-mode encoding) see the change
            torch.autograd.graph.increment_version(updated)
        return loss


class FusedAdamW(FusedAdam):
    """``torch.optim.AdamW`` semantics (decoupled weight decay, default ``weight_decay=1e-2``) on ``FusedAdam``."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, amsgrad=False, *,
                 foreach=None, maximize=False, capturable=False, differentiable=False, fused=None,
                 max_grad_norm: Optional[float] = None):
        super().__init__(params, lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, amsgrad=amsgrad,
                         foreach=foreach, maximize=maximize, capturable=capturable, differentiable=differentiable,
                         fused=fused, decoupled_weight_decay=True, max_grad_norm=max_grad_norm)
