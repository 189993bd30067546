"""Single-box data parallelism: one process per GPU, NCCL over NVLink 5 / NVSwitch.

Replaces the reference's gradient sync — ``xm.optimizer_step(optimizer, barrier=True)`` (engine.py:185) on TPU and
``DistributedDataParallel`` (main.py:855-857) on GPU — with one all-reduce (SUM) of the whole flat gradient buffer after
backward.  The backward signals once, from its last stage; the all-reduce runs when the optimizer's pre-step hook (or
``engine.clip_grad_norm_``) calls ``finish_gradient_sync()``.  The 1/world_size of the mean is folded into the AdamW
kernel (``grad_scale``), so averaging costs no extra pass over the gradients.

Wire format: when the fused AdamW kernel consumes the result (an optimizer is attached and the gradient is on the GPU),
the flat fp32 gradient is cast into a persistent bf16 buffer (one vitk cast kernel, 0.09 ms for ViT-B) and THAT is
all-reduced (173 MB instead of 346 MB for ViT-B); AdamW reads the summed gradient from it.  Otherwise the fp32 buffer
is all-reduced in place.

Nothing overlaps backward (DESIGN.md section 6): on 8 B200 an all-reduce per block during backward measured 36.17 ms/step
against 34.98 ms for one after it, because NCCL's CTAs displace GEMM and attention kernels that are persistent with one
CTA per SM; reducing only the last blocks during backward landed inside the run-to-run spread.

With ``update_freq > 1`` the gradient is only reduced on the micro-batch that precedes ``optimizer.step()``
(``no_sync()`` context, like DDP).
"""
from __future__ import annotations

import contextlib

import torch
import torch.distributed as dist
import torch.nn as nn

from .store import get_store


class DataParallel(nn.Module):
    def __init__(self, module: nn.Module, optimizer=None, broadcast: bool = True):
        super().__init__()
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError("DataParallel needs an initialised torch.distributed process group")
        self.module = module
        self.world_size = dist.get_world_size()
        self.require_sync = True
        self._pending = False
        st = get_store(self._find_root(module))
        self.store = st
        if broadcast:
            dist.broadcast(st.flat, src=0)  # identical replicas (DDP does the same at construction)
            st._sig = None
        self._grad16 = None     # persistent bf16 wire buffer (allocated on first use)
        self._optimizer = None
        st.grad_ready_hooks.append(self._on_grad_ready)
        if optimizer is not None:
            self.attach_optimizer(optimizer)

    @staticmethod
    def _find_root(module: nn.Module) -> nn.Module:
        """The trainable vitk model inside ``module`` (e.g. the student of a StudentWithDistillation wrapper)."""
        from .models.vision_transformer import VisionTransformer

        roots = [m for m in module.modules()
                 if isinstance(m, VisionTransformer) and any(p.requires_grad for p in m.parameters())]
        if len(roots) > 1:
            raise NotImplementedError("DataParallel: more than one trainable vitk model inside the wrapped module")
        return roots[0] if roots else module

    def attach_optimizer(self, optimizer):
        optimizer.grad_scale = 1.0 / self.world_size
        optimizer.pre_step_hooks.append(lambda opt: self.finish_gradient_sync())
        self._optimizer = optimizer

    def _on_grad_ready(self):
        if self.require_sync and self.world_size > 1:
            self._pending = True

    def finish_gradient_sync(self):
        """Complete the gradient SUM over the replicas (idempotent: a second call before the next backward is a no-op)."""
        if self._pending:
            self._pending = False
            dist.all_reduce(self._wire(), op=dist.ReduceOp.SUM)
            if self._lowp():
                self._optimizer.grad_lowp = self._grad16   # AdamW reads the summed gradient from here (this step only)

    def _lowp(self) -> bool:
        """bf16 wire: the fused AdamW kernel reads the summed bf16 gradient, so it needs the optimizer and a CUDA store."""
        return self._optimizer is not None and self.store.grad.is_cuda

    def _wire(self) -> torch.Tensor:
        """The buffer that goes on the wire: the fp32 gradient itself, or its bf16 cast."""
        if not self._lowp():
            return self.store.grad
        from . import _lib as L

        if self._grad16 is None or self._grad16.numel() != self.store.grad.numel():
            self._grad16 = torch.empty_like(self.store.grad, dtype=torch.bfloat16)
        L.cast_bf16(self.store.grad, self._grad16)
        return self._grad16

    @contextlib.contextmanager
    def no_sync(self):
        old = self.require_sync
        self.require_sync = False
        try:
            yield
        finally:
            self.require_sync = old

    def forward(self, *args, **kwargs):
        return self.module(*args, **kwargs)

    def no_weight_decay(self):
        return self.module.no_weight_decay() if hasattr(self.module, "no_weight_decay") else set()
