"""Fused Adam for the IntEL training loop.

Drop-in for ``torch.optim.Adam(model.customize_parameters(), lr=..., weight_decay=l2)`` as built by
``BaseRunner._build_optimizer`` (BaseRunner.py:182-188): same constructor arguments, same ``param_groups`` / ``state``
layout (``step``, ``exp_avg``, ``exp_avg_sq``), so ``state_dict()`` interchanges with torch's optimizer and
``torch.optim.lr_scheduler.StepLR`` works on it.  ``step()`` updates all parameters with one kernel launch per 48
tensors (``intel_adam_step``) instead of ~10 small kernels per tensor.

A group may mix dense and row-sparse (COO, one sparse dimension) gradients: ``IntEL(sparse_grad=1)`` gives its embedding
tables those.  A sparse gradient updates only the rows it lists (``intel_adam_rows_step``), each with the same per-element
arithmetic as the dense kernel, the group's L2 and its shared step count; the other rows keep parameter and moments bit
for bit.  That is not torch.optim.Adam on a dense gradient with zero rows (L2 and the moments' decay move every row there):
it is the lazy form of Adam, opted into with the model flag.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Hashable, Iterable

import torch

from . import _lib


# rows buffers of the COO gradients that IntEL's backward pass returns, by (model, table): their indices are ascending and
# unique, but autograd drops the coalesced flag on the way into .grad, so step() recognises them by this storage instead
_coalesced_rows: Dict[Hashable, torch.Tensor] = {}


def note_coalesced_rows(key: Hashable, rows: torch.Tensor) -> None:
    _coalesced_rows[key] = rows


def _rows_and_values(p: torch.Tensor, g: torch.Tensor):
    """(row ids int64 [U], gradient rows float32 [U, d]) of a row-sparse gradient, coalescing any other COO gradient
    (e.g. one accumulated over two backward passes, which has duplicate indices)"""
    if g.layout != torch.sparse_coo or g.sparse_dim() != 1 or g.shape != p.shape or p.dim() < 1:
        raise ValueError("optim.Adam: a sparse gradient must be a COO tensor of the parameter's shape with one sparse dimension")
    idx = g._indices()
    own = any(idx.data_ptr() == r.data_ptr() and idx.device == r.device and idx.numel() <= r.numel()
              for r in _coalesced_rows.values())
    if not own:
        g = g.coalesce()
        idx = g._indices()
    vals = g._values()
    d = p[0].numel()
    if vals.dtype != torch.float32 or vals.device != p.device:
        raise ValueError("intel_adam_rows_step needs float32 gradient rows on the parameter's device")
    return idx.reshape(-1).contiguous(), vals.reshape(-1, d).contiguous()


def customize_parameters(model: torch.nn.Module) -> list:
    """The reference's two parameter groups (BaseModel.customize_parameters, BaseModel.py:53-62)."""
    weight_p, bias_p = [], []
    for name, p in model.named_parameters():
        if p.requires_grad:
            (bias_p if "bias" in name else weight_p).append(p)
    return [{"params": weight_p}, {"params": bias_p, "weight_decay": 0}]


class Adam(torch.optim.Optimizer):
    def __init__(self, params: Iterable, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.0):
        if lr < 0 or eps < 0 or not 0 <= betas[0] < 1 or not 0 <= betas[1] < 1 or weight_decay < 0:
            raise ValueError("invalid Adam hyper-parameter")
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))
        self._cache = {}

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        lib = _lib.load()
        for gi, group in enumerate(self.param_groups):
            ps = [p for p in group["params"] if p.grad is not None]
            if not ps:
                continue
            key = [(id(p), p.grad.is_sparse) for p in ps]
            cache = self._cache.get(gi)
            if cache is None or cache["key"] != key or any(not self.state[p] for p in ps):
                cache = self._build_cache(ps, key)
                self._cache[gi] = cache
            step_t = cache["step"]
            step_t += 1                                   # one shared tensor: every parameter's state["step"] aliases it
            b1, b2 = group["betas"]
            wd = float(group["weight_decay"])
            sparse = [p for p in ps if p.grad.is_sparse]
            if sparse:
                self._rows_step(sparse, group, wd, int(step_t))
            ps = [p for p in ps if not p.grad.is_sparse]
            if not ps:
                continue
            n = len(ps)
            grads, params, ms, vs = cache["grads"], cache["params"], cache["m"], cache["v"]
            for i, p in enumerate(ps):
                g = p.grad
                if g.dtype != torch.float32 or not g.is_contiguous() or g.device != p.device:
                    raise ValueError("intel_adam_step needs contiguous float32 gradients on the parameter's device")
                grads[i] = g.data_ptr()
                # the Parameter object can outlive its storage (model.to(), p.data = ..., a replaced state tensor):
                # re-read the pointers every step like torch.optim.Adam re-reads the tensors
                st = self.state[p]
                params[i], ms[i], vs[i] = p.data_ptr(), st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr()
            if wd != cache["wd_value"]:
                cache["wd"] = (C.c_float * n)(*([wd] * n))
                cache["wd_value"] = wd
            _lib.check(lib.intel_adam_step(n, cache["params"], grads, cache["m"], cache["v"], cache["numel"], cache["wd"],
                                           float(group["lr"]), float(b1), float(b2), float(group["eps"]), int(step_t),
                                           _lib.stream_ptr(ps[0].device)))
        return loss

    def _rows_step(self, ps, group, wd: float, step: int) -> None:
        n = len(ps)
        arr = lambda vals, t=C.c_void_p: (t * n)(*vals)
        rows, vals = zip(*[_rows_and_values(p, p.grad) for p in ps])     # (kept alive until the launch is queued)
        st = [self.state[p] for p in ps]
        b1, b2 = group["betas"]
        _lib.check(_lib.load().intel_adam_rows_step(
            n, arr([_lib.ptr(p) for p in ps]), arr([_lib.ptr(s["exp_avg"]) for s in st]),
            arr([_lib.ptr(s["exp_avg_sq"]) for s in st]), arr([_lib.ptr(r) for r in rows]), arr([_lib.ptr(v) for v in vals]),
            arr([r.numel() for r in rows], C.c_int64), arr([p[0].numel() for p in ps], C.c_int32), arr([wd] * n, C.c_float),
            float(group["lr"]), float(b1), float(b2), float(group["eps"]), step, _lib.stream_ptr(ps[0].device)))

    def _build_cache(self, ps, key):
        """pointer tables of a group's dense-gradient tensors (parameters and moments keep their storage; gradients are
        refreshed every step); the state of every tensor of the group"""
        step_t = None
        for p in ps:
            if p.dtype != torch.float32 or not p.is_contiguous():
                raise ValueError("intel_adam_step needs contiguous float32 parameters")
            st = self.state[p]
            if not st:
                st["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                st["step"] = torch.tensor(0.0)
            if step_t is None:
                step_t = st["step"] if torch.is_tensor(st["step"]) else torch.tensor(float(st["step"]))
            elif float(st["step"]) != float(step_t):
                raise ValueError("parameters of one group must share their step count")
        for p in ps:
            self.state[p]["step"] = step_t
        ps = [p for p, (_, sparse) in zip(ps, key) if not sparse]
        n = len(ps)
        arr = lambda ts: (C.c_void_p * n)(*[_lib.ptr(t) for t in ts])
        return {"key": key, "step": step_t, "params": arr(ps),
                "m": arr([self.state[p]["exp_avg"] for p in ps]), "v": arr([self.state[p]["exp_avg_sq"] for p in ps]),
                "numel": (C.c_int64 * n)(*[p.numel() for p in ps]), "grads": (C.c_void_p * n)(), "wd": None, "wd_value": None}

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        self._cache = {}
