"""Flat parameter / gradient / bf16-shadow storage for one model replica.

Data layout in HBM (DESIGN.md §3): every parameter of the root module lives in ONE fp32 buffer
(``flat``), padded to 64-element boundaries, in ``named_parameters()`` order — so the parameters of
``blocks.i`` are one contiguous range.  ``grad`` mirrors it (the
wgrad kernels ``red.add`` straight into it; ``p.grad`` are views), ``shadow`` is the bf16 copy the
tcgen05 GEMMs read as their B operand.  ``nn.Parameter`` objects keep their names and shapes (the
reference's state_dict contract, SURVEY Appendix B) but their ``.data`` is re-pointed into ``flat``.
"""
from __future__ import annotations

import threading
import weakref
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn

from . import _lib as L

ALIGN = 64  # elements; keeps every tensor 256-byte (fp32) / 128-byte (bf16) aligned


class ParamStore:
    def __init__(self, root: nn.Module, allow_cpu: bool = False):
        """``allow_cpu`` exists for the host-logic tests (gloo all-reduce plumbing); no kernel
        can run on such a store — every launch wrapper rejects CPU tensors."""
        named = list(root.named_parameters())
        if not named:
            raise L.VitkError("ParamStore: module has no parameters")
        dev = named[0][1].device
        if dev.type != "cuda" and not allow_cpu:
            raise L.VitkError("vitk kernels only run on CUDA (sm_100a); move the model with .cuda() first — "
                              "there is no CPU path")
        self.device = dev
        self.params: List[nn.Parameter] = []
        self.offsets: Dict[int, Tuple[int, int]] = {}
        off = 0
        for name, p in named:
            if p.dtype != torch.float32:
                raise L.VitkError(f"parameter {name} has dtype {p.dtype}; master weights must be fp32")
            if p.device != dev:
                raise L.VitkError(f"parameter {name} is on {p.device}, expected {dev}")
            n = p.numel()
            self.params.append(p)
            self.offsets[id(p)] = (off, n)
            off += (n + ALIGN - 1) // ALIGN * ALIGN
        self.total = off
        self.flat = torch.zeros(self.total, dtype=torch.float32, device=dev)
        self.grad = torch.zeros(self.total, dtype=torch.float32, device=dev)
        self.shadow = torch.empty(self.total, dtype=torch.bfloat16, device=dev)
        with torch.no_grad():
            for p in self.params:
                o, n = self.offsets[id(p)]
                view = self.flat[o:o + n].view(p.shape)
                view.copy_(p.data)
                p.data = view
        ref = weakref.ref(self)
        for p in self.params:
            p._vitk_store_ref = ref  # lets FusedAdamW find the store from a bare parameter
        self._ptrs = [p.data_ptr() for p in self.params]
        self._sig: Optional[int] = None
        self.grads_need_zero = False
        #: 1-element tensor that requires grad: makes autograd call the stage backward functions
        self.anchor = torch.zeros(1, device=dev, requires_grad=True)
        #: side channel between consecutive stage backwards: fp32 grad data_ptr -> bf16 copy (ops.py)
        self.chain: Dict[int, torch.Tensor] = {}
        #: callbacks() fired when a backward pass has enqueued its last gradient kernel (parallel.py)
        self.grad_ready_hooks: List = []
        self.attach_grads()

    # ------------------------------------------------------------------------------------
    def valid(self) -> bool:
        """False once any parameter's storage was replaced (e.g. by ``.to()`` / ``load(assign=True)``)."""
        for p, ptr in zip(self.params, self._ptrs):
            if p.data_ptr() != ptr:
                return False
        return True

    def view(self, p: nn.Parameter) -> torch.Tensor:
        return p.data

    def shadow_of(self, p: nn.Parameter) -> torch.Tensor:
        o, n = self.offsets[id(p)]
        return self.shadow[o:o + n].view(p.shape)

    def grad_of(self, p: nn.Parameter) -> torch.Tensor:
        o, n = self.offsets[id(p)]
        return self.grad[o:o + n].view(p.shape)

    # ------------------------------------------------------------------------------------
    def sync_shadow(self) -> None:
        """Re-cast the bf16 shadow if any parameter was modified through torch since the last cast.

        The fused AdamW kernel writes the shadow itself through raw pointers (no version bump), so in
        the steady state of training this is a cheap host-side check and launches nothing."""
        sig = 0
        for p in self.params:
            sig += p._version
        if sig != self._sig:
            L.cast_bf16(self.flat, self.shadow)
            self._sig = sig

    def mark_shadow_current(self) -> None:
        sig = 0
        for p in self.params:
            sig += p._version
        self._sig = sig

    def attach_grads(self) -> None:
        """Make ``p.grad`` a view of the flat gradient buffer for every trainable parameter.

        If an optimizer dropped the grads (``zero_grad(set_to_none=True)``) the flat buffer is zeroed
        so that accumulation starts from zero, exactly like autograd would."""
        missing = False
        for p in self.params:
            if not p.requires_grad:
                continue
            g = p.grad
            o, n = self.offsets[id(p)]
            if g is None or g.data_ptr() != self.grad.data_ptr() + 4 * o:
                missing = True
                p.grad = self.grad[o:o + n].view(p.shape)
        if missing:
            self.grad.zero_()

    def fire_grad_ready(self) -> None:
        for hook in self.grad_ready_hooks:
            hook()


_tls = threading.local()


def current() -> Optional[ParamStore]:
    return getattr(_tls, "store", None)


class use_store:
    """Context manager: the root module publishes its store to the sub-modules it calls."""

    def __init__(self, store: ParamStore):
        self.store = store

    def __enter__(self):
        self.prev = getattr(_tls, "store", None)
        _tls.store = self.store
        return self.store

    def __exit__(self, *exc):
        _tls.store = self.prev
        return False


def get_store(root: nn.Module) -> ParamStore:
    """Store owned by ``root`` (built lazily, rebuilt if the parameters moved)."""
    st = root.__dict__.get("_vitk_store")
    if st is None or not st.valid() or len(st.params) != sum(1 for _ in root.parameters()):
        st = ParamStore(root)
        root.__dict__["_vitk_store"] = st
    return st


def store_for(module: nn.Module) -> ParamStore:
    """The ambient store if a root module is executing, else ``module`` acts as its own root."""
    st = current()
    if st is not None:
        first = next(module.parameters(), None)
        if first is None or id(first) in st.offsets:
            return st
    return get_store(module)
