"""Fused Adam for the IntEL training loop.

Drop-in for ``torch.optim.Adam(model.customize_parameters(), lr=..., weight_decay=l2)`` as built by
``BaseRunner._build_optimizer`` (BaseRunner.py:182-188): same constructor arguments, same ``param_groups`` / ``state``
layout (``step``, ``exp_avg``, ``exp_avg_sq``), so ``state_dict()`` interchanges with torch's optimizer and
``torch.optim.lr_scheduler.StepLR`` works on it.  ``step()`` updates all parameters with one kernel launch per 48
tensors (``intel_adam_step``) instead of ~10 small kernels per tensor.

A group may mix dense and row-sparse (COO, one sparse dimension) gradients: ``IntEL(sparse_grad=1)`` and
``IntEL(sparse_grad=2)`` give their embedding tables those.  A sparse gradient updates only the rows it lists
(``intel_adam_rows_step``), each with the same per-element arithmetic as the dense kernel, the group's L2 and its shared
step count; the other rows keep parameter and moments bit for bit.  That is not torch.optim.Adam on a dense gradient with
zero rows (L2 and the moments' decay move every row there): it is the lazy form of Adam, opted into with
``sparse_grad=1``.

Parameters marked with ``defer_zero_updates`` (``IntEL(sparse_grad=2)`` marks its tables) stay on the dense trajectory
instead.  The update a dense step gives an unlisted row has a gradient of exactly +0.0, so it depends only on the row and
that step's scalars: the optimizer records each step's scalars per parameter and defers those updates, and
``intel_adam_deferred_rows_step`` replays a row's pending ones, in order and with the same arithmetic, before its next
update.  Rows are brought up to date without a new update by ``catch_up`` (the rows a forward pass is about to read) and
``flush`` (every row).  After ``flush()`` parameters and moments equal dense Adam's bit for bit; ``state_dict()`` and
``load_state_dict()`` flush first, so the saved state is torch's and interchanges with every mode.  A marked parameter that
receives a dense gradient is flushed and then takes the dense step.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Hashable, Iterable, Optional

import torch
from torch.utils.weak import WeakIdKeyDictionary

from . import _lib


# rows buffers of the COO gradients that IntEL's backward pass returns, by (model, table): their indices are ascending and
# unique, but autograd drops the coalesced flag on the way into .grad, so step() recognises them by this storage instead
_coalesced_rows: Dict[Hashable, torch.Tensor] = {}


def note_coalesced_rows(key: Hashable, rows: torch.Tensor) -> None:
    _coalesced_rows[key] = rows


class _Deferred:
    """Bookkeeping of a marked parameter (intel_adam_deferred_rows_step): ``n`` updates recorded since the last reset, their
    scalars in ``hist`` [cap, 8] (grown by doubling), ``done[r]`` = how many of them row r has received; ``state`` is the
    optimizer state (exp_avg, exp_avg_sq) the pending updates belong to."""

    def __init__(self, p: torch.Tensor, state: dict) -> None:
        self.state, self.n = state, 0
        self.hist = torch.zeros(16, 8, dtype=torch.float32, device=p.device)
        self.done = torch.zeros(p.shape[0], dtype=torch.int32, device=p.device)

    def record(self) -> None:
        """one more update; makes room for its entry in hist"""
        self.n += 1
        if self.n > self.hist.shape[0]:
            hist = torch.zeros(2 * self.hist.shape[0], 8, dtype=torch.float32, device=self.hist.device)
            hist[: self.n - 1] = self.hist[: self.n - 1]
            self.hist = hist


# parameters whose zero-gradient updates optim.Adam defers (IntEL(sparse_grad=2) marks its tables) -> their bookkeeping,
# None until the first deferred step
_deferred = WeakIdKeyDictionary()


def defer_zero_updates(params: Iterable[torch.Tensor]) -> None:
    """Mark parameters whose row-sparse gradients take the exact (deferred) row-wise step."""
    for p in params:
        _deferred.setdefault(p, None)


def _catch_up(ps, rows, counts) -> None:
    """intel_adam_deferred_catch_up over the pending parameters of ps (rows None: every row, then the count restarts)"""
    recs = [(p, _deferred.get(p), r, c) for p, r, c in zip(ps, rows, counts)]
    recs = [(p, d, r, c) for p, d, r, c in recs if d is not None and d.n > 0]
    if not recs:
        return
    n = len(recs)
    arr = lambda vals, t=C.c_void_p: (t * n)(*vals)
    _lib.check(_lib.load().intel_adam_deferred_catch_up(
        n, arr([_lib.ptr(p) for p, *_ in recs]), arr([_lib.ptr(d.state["exp_avg"]) for _, d, _, _ in recs]),
        arr([_lib.ptr(d.state["exp_avg_sq"]) for _, d, _, _ in recs]), arr([_lib.ptr(r) for _, _, r, _ in recs]),
        arr([_lib.ptr(c) for *_, c in recs]),
        arr([(r.numel() if r is not None else p.shape[0]) for p, _, r, _ in recs], C.c_int64),
        arr([p[0].numel() for p, *_ in recs], C.c_int32), arr([_lib.ptr(d.done) for _, d, _, _ in recs]),
        arr([_lib.ptr(d.hist) for _, d, _, _ in recs]), arr([d.n for _, d, _, _ in recs], C.c_int32),
        _lib.stream_ptr(recs[0][0].device)))
    for _, d, r, _ in recs:
        if r is None:
            d.n = 0


def catch_up(p: torch.Tensor, rows: torch.Tensor, count: torch.Tensor) -> None:
    """Bring the first ``count`` (a device int64 [1]) rows of ``rows`` of a marked parameter up to date, without a host
    synchronisation."""
    _catch_up([p], [rows], [count])


def flush(params: Iterable[torch.Tensor]) -> None:
    """Apply every pending update of the given (marked) parameters: they and their moments then equal dense Adam's."""
    ps = list(params)
    _catch_up(ps, [None] * len(ps), [None] * len(ps))


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
            deferred = [p for p in sparse if p in _deferred]
            if deferred:
                self._deferred_step(deferred, group, wd, int(step_t))
            lazy = [p for p in sparse if p not in _deferred]
            if lazy:
                self._rows_step(lazy, group, wd, int(step_t))
            ps = [p for p in ps if not p.grad.is_sparse]
            flush(p for p in ps if p in _deferred)         # a marked parameter with a dense gradient: current, then dense
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

    def _deferred_step(self, ps, group, wd: float, step: int) -> None:
        n = len(ps)
        arr = lambda vals, t=C.c_void_p: (t * n)(*vals)
        rows, vals = zip(*[_rows_and_values(p, p.grad) for p in ps])
        st = [self.state[p] for p in ps]
        recs = []
        for p, s in zip(ps, st):
            d = _deferred.get(p)
            if d is not None and d.state is not s:           # pending updates of another optimizer's state: apply them first
                flush([p])
                d = None
            if d is None:
                d = _deferred[p] = _Deferred(p, s)
            d.record()
            recs.append(d)
        b1, b2 = group["betas"]
        _lib.check(_lib.load().intel_adam_deferred_rows_step(
            n, arr([_lib.ptr(p) for p in ps]), arr([_lib.ptr(s["exp_avg"]) for s in st]),
            arr([_lib.ptr(s["exp_avg_sq"]) for s in st]), arr([_lib.ptr(r) for r in rows]), arr([_lib.ptr(v) for v in vals]),
            arr([r.numel() for r in rows], C.c_int64), arr([p[0].numel() for p in ps], C.c_int32), arr([wd] * n, C.c_float),
            arr([_lib.ptr(d.done) for d in recs]), arr([_lib.ptr(d.hist) for d in recs]), arr([d.n for d in recs], C.c_int32),
            float(group["lr"]), float(b1), float(b2), float(group["eps"]), step, _lib.stream_ptr(ps[0].device)))

    def flush(self, params: Optional[Iterable[torch.Tensor]] = None) -> None:
        """Apply the deferred updates of ``params`` (default: every parameter of this optimizer).  Afterwards parameters
        and moments equal what dense Adam would hold, bit for bit.  Call it before reading a marked table directly."""
        if params is None:
            params = [p for g in self.param_groups for p in g["params"]]
        flush(p for p in params if p in _deferred)

    def state_dict(self):
        self.flush()
        return super().state_dict()

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
        self.flush()                 # the pending updates belong to the weights as they are and to the state being replaced
        super().load_state_dict(state_dict)
        self._cache = {}
        for g in self.param_groups:
            for p in g["params"]:
                if _deferred.get(p) is not None:
                    _deferred[p] = None
