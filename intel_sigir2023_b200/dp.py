"""Session-sharded data parallelism (SURVEY.md 8e; absent in the reference, which is single process).

One process per GPU.  A global batch is cut into equal contiguous shards of sessions
(``synthetic.shard_batch`` keeps the global padded widths so pad keys take part in the unmasked
self-attention exactly as in a single-process run); tables and weights are replicated; the only
exchange step of the path is the gradient all-reduce (mean of the local batch-mean losses = global
batch mean), plus a sum of the additive evaluation terms.  NCCL over NVLink on the GPU box, gloo in
the CPU tests.
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch
import torch.distributed as dist


OVERLAP_SMS = 8     # measured on 2 x B200 (profiles/r02_summary.md): 8 hides the 79 MB exchange; 12 / 16 / 24 only slow the stack


def configure_nccl_for_overlap(sms: int = OVERLAP_SMS) -> None:
    """Call before ``init_process_group``: caps the CTAs of NCCL's kernels at the number of SMs the persistent backward
    kernel will leave free (``GradReducer(overlap_sms=...)``), so the collective that runs beside it never takes an SM
    away from one of its CTAs (a CTA that starts late would finish a whole wave late), and drops NCCL's thread-block
    clusters: a cluster of four needs four free SMs inside one GPC, which the scattered free SMs do not offer.
    Explicit settings in the environment win."""
    if os.environ.get("INTEL_DP_OVERLAP", "1") == "0":
        return
    os.environ.setdefault("NCCL_MAX_CTAS", str(int(os.environ.get("INTEL_DP_OVERLAP_SMS", sms))))
    os.environ.setdefault("NCCL_CGA_CLUSTER_SIZE", "0")


def _buffer_ptr(g: torch.Tensor) -> int:
    """storage of a gradient (the values of a sparse one)"""
    return (g._values() if g.is_sparse else g).untyped_storage().data_ptr()


class GradReducer:
    """Average the dense ``.grad`` buffers over the ranks after backward.

    The backward pass of ``IntEL`` writes every gradient into one flat buffer whose tail holds the parameters of the
    score stream, the last ones it completes.  With ``overlap`` the head of the buffer (everything else: ~all of the
    bytes, the embedding tables included) is all-reduced asynchronously as soon as it is final, beside the score stack's
    backward kernel, which leaves ``overlap_sms`` SMs free for it; ``allreduce()`` then exchanges the small tail and
    joins.  This needs ``p.grad is None`` before backward (``zero_grad(set_to_none=True)``, the torch default): gradient
    accumulation into existing ``.grad`` tensors is refused loudly.  Without the flat buffer (other models) the few
    large tensors are reduced in place, one collective each, and the small ones travel in one flat bucket.

    With ``IntEL(sparse_grad=1)`` the reducer also makes every rank build the same row sets: the model's forward pass
    all-gathers each table's ids (``_gather_ids``) and builds the union, so the compact table gradients in the flat
    buffer line up row for row across the ranks and the same all-reduce averages them."""

    def __init__(self, model: torch.nn.Module, world: int, small_numel: int = 1 << 16, overlap: bool = True,
                 overlap_sms: Optional[int] = None):
        self.model = model
        self.params: List[torch.nn.Parameter] = [p for p in model.parameters() if p.requires_grad]
        self.world = world
        self.small_numel = small_numel
        backend = dist.get_backend() if dist.is_initialized() else "none"
        self.avg_op = dist.ReduceOp.AVG if backend == "nccl" else dist.ReduceOp.SUM
        self.post_scale = 1.0 if backend == "nccl" else 1.0 / world
        self._pending = None
        self.overlap = (bool(overlap) and world > 1 and hasattr(model, "_early_reduce")
                        and os.environ.get("INTEL_DP_OVERLAP", "1") != "0")      # the environment switch is for A/B timing
        if world > 1 and hasattr(model, "_gather_ids"):
            model._gather_ids = self._gather_ids
        if self.overlap:
            model._early_reduce = self._early
            if backend == "nccl":
                from . import _lib
                n = int(os.environ.get("INTEL_DP_OVERLAP_SMS", OVERLAP_SMS)) if overlap_sms is None else int(overlap_sms)
                _lib.check(_lib.load().intel_reserve_sms(n))

    def _early(self, flat: torch.Tensor, late: int) -> None:
        """Called from inside the backward pass once flat[:late] is final (the score stack is still to come)."""
        if late > 0:
            self._pending = (dist.all_reduce(flat[:late], op=self.avg_op, async_op=True), flat, late)

    def _gather_ids(self, ids: torch.Tensor) -> torch.Tensor:
        """ids of every rank, concatenated (the shards have equal shapes: synthetic.shard_batch)"""
        parts = [torch.empty_like(ids) for _ in range(self.world)]
        dist.all_gather(parts, ids.contiguous())
        return torch.cat(parts)

    def allreduce(self) -> None:
        if self.world <= 1:
            return
        grads = [p.grad for p in self.params if p.grad is not None]
        pending, self._pending = self._pending, None
        if pending is not None:
            work, flat, late = pending
            base = flat.untyped_storage().data_ptr()
            if len(grads) != len(self.params) or any(_buffer_ptr(g) != base for g in grads):
                work.wait()
                raise RuntimeError("GradReducer(overlap=True): the .grad tensors do not alias the flat gradient buffer of this "
                                   "backward pass (gradient accumulation into existing .grad?); clear them with "
                                   "zero_grad(set_to_none=True) or build the reducer with overlap=False")
            if late < flat.numel():
                dist.all_reduce(flat[late:], op=self.avg_op)
            work.wait()
            if self.post_scale != 1.0:
                flat.mul_(self.post_scale)
            return
        # the backward pass writes all gradients into one zero-filled buffer (IntEL._IntelFn.backward): if every .grad
        # still aliases it (autograd adopted the views instead of copying them), one collective covers everything
        flat = getattr(self.model, "_flat_grad", None)
        if flat is not None and grads and len(grads) == len(self.params):
            base = flat.untyped_storage().data_ptr()
            if all(_buffer_ptr(g) == base for g in grads):
                dist.all_reduce(flat, op=self.avg_op)
                if self.post_scale != 1.0:
                    flat.mul_(self.post_scale)
                return
        if any(g.is_sparse for g in grads):
            raise RuntimeError("GradReducer: sparse table gradients are exchanged only inside the flat gradient buffer of the "
                               "backward pass that produced them")
        big = [g for g in grads if g.numel() > self.small_numel]
        small = [g for g in grads if g.numel() <= self.small_numel]
        works = [dist.all_reduce(g, op=self.avg_op, async_op=True) for g in big]
        if small:
            flat = torch.cat([g.reshape(-1) for g in small])
            dist.all_reduce(flat, op=self.avg_op)
            if self.post_scale != 1.0:
                flat.mul_(self.post_scale)
            off = 0
            for g in small:
                g.copy_(flat[off:off + g.numel()].view_as(g))
                off += g.numel()
        for w in works:
            w.wait()
        if self.post_scale != 1.0:
            for g in big:
                g.mul_(self.post_scale)


def global_max_len(session_len: torch.Tensor) -> int:
    """max(session_len) over every rank: evaluate_method's max_len is a global quantity (BaseRunner.py:66)."""
    m = session_len.max().reshape(1).clone()
    if dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(m, op=dist.ReduceOp.MAX)
    return int(m.item())


def evaluate_sharded(pred: torch.Tensor, ranking: torch.Tensor, pos_nums: Dict[str, torch.Tensor],
                     session_len: torch.Tensor, topk: Sequence[int], metrics: Sequence[str]) -> Dict[str, float]:
    """Every rank scores its shard of the eval sessions; the additive per-metric sums are all-reduced."""
    from . import evaluate
    max_len = max(global_max_len(session_len), max(topk))
    sums, counts = evaluate.ndcg_sums(pred, ranking, session_len, pos_nums['c_paynum_i'], pos_nums['c_favnum_i'],
                                      pos_nums['c_clicknum_i'], max_len, topk)
    if dist.is_initialized() and dist.get_world_size() > 1:
        both = torch.cat([sums, counts])
        dist.all_reduce(both, op=dist.ReduceOp.SUM)
        sums, counts = both[:sums.numel()], both[sums.numel():]
    return evaluate.metrics_from_sums(sums.cpu().numpy(), counts.cpu().numpy(), topk, metrics)
