"""Drop-in ``IntEL`` module: same constructor, ``state_dict`` and ``forward(batch) -> dict`` as the
reference (IntEL/src/models/IntEL/IntEL.py:13-124), with the forward/backward executed by the
hand-written sm_100a kernels of libintel_b200 through its C ABI.

The parameter containers below are the same torch modules the reference registers (so key names,
shapes and the PyTorch-default initialisation match, SURVEY.md 8b) but their ``forward`` is never
called: ``IntEL.forward`` hands raw device pointers to ``intel_intent_fwd`` / ``intel_ensemble_fwd``.
"""
from __future__ import annotations

import argparse
import logging
import os
from typing import Dict, Optional

import torch
import torch.nn as nn

from . import _lib, optim
from .config import IntelConfig

# embedding tables that --sparse_grad 1 and 2 cover: parameter, the batch fields whose ids index it (the backward scatters from
# exactly these), the row map's field in intel_row_maps_t
SPARSE_TABLES = (("iid_embeddings.weight", ("i_id_s", "his_item_id"), "iid"),
                 ("item_embeddings.weight", ("i_class_c",), "item"),
                 ("uid_embeddings.weight", ("u_id_c",), "uid"),
                 ("context_embeddings.weight", ("context_mh", "his_context_mh"), "ctx"))


def _encoder_container(cfg: IntelConfig, d: int) -> nn.Module:
    m = nn.Module()
    if cfg.encoder == "GRU4Rec":                                    # GeneralSeq.py:58-62
        m.rnn = nn.GRU(input_size=d, hidden_size=cfg.gru_hidden, batch_first=True)
        m.out = nn.Linear(cfg.gru_hidden, d, bias=False)
    elif cfg.encoder == "BERT4Rec":                                 # GeneralSeq.py:80-88, layers.py:62-80
        m.p_embeddings = nn.Embedding(cfg.history_max + 1, d)
        blocks = []
        for _ in range(cfg.bert_layers):
            b = nn.Module()
            b.masked_attn_head = nn.Module()
            b.masked_attn_head.q_linear = nn.Linear(d, d)
            b.masked_attn_head.k_linear = nn.Linear(d, d)
            b.masked_attn_head.v_linear = nn.Linear(d, d)
            b.layer_norm1 = nn.LayerNorm(d)
            b.linear1 = nn.Linear(d, d)
            b.linear2 = nn.Linear(d, d)
            b.layer_norm2 = nn.LayerNorm(d)
            blocks.append(b)
        m.transformer_block = nn.ModuleList(blocks)
    else:
        raise ValueError("Invalid sequence encoder.")
    return m


def _attn_container(d: int) -> nn.Module:
    m = nn.Module()
    m.q_linear = nn.Linear(d, d, bias=False)
    m.k_linear = nn.Linear(d, d, bias=False)
    m.v_linear = nn.Linear(d, d, bias=False)
    return m


def _cross_container(I: int, d: int) -> nn.Module:
    m = nn.Module()
    m.query_layer = nn.Linear(I, d, bias=False)
    m.key_layer = nn.Linear(d, d, bias=False)
    m.value_layer = nn.Linear(d, d, bias=False)
    return m


def _take_ws(model, nbytes: int, dev) -> torch.Tensor:
    """Workspaces are multi-GB at B=4096: keep them in a per-model pool instead of round-tripping the
    allocator every step.  Reuse is stream-ordered (same stream), so handing a buffer back right after the
    kernels that use it were queued is safe."""
    pool = model._ws_pool.setdefault((int(nbytes), str(dev)), [])
    return pool.pop() if pool else torch.empty(int(nbytes), dtype=torch.uint8, device=dev)


def _give_ws(model, t: torch.Tensor) -> None:
    pool = model._ws_pool.setdefault((t.numel(), str(t.device)), [])
    if len(pool) < 2:
        pool.append(t)


class _RowSets:
    """The row sets of one training step (IntEL with sparse_grad = 1 or 2): per covered table the ascending unique ids the
    batch feeds it, built on the device at the start of the forward pass.  The set sizes travel to pinned host memory behind
    an event that backward waits on (it has long completed by then), so the step gains no host synchronisation.  With
    sparse_grad = 2 the rows of each set are brought up to date (optim.catch_up) before any kernel reads the tables."""

    def __init__(self, model: "IntEL", batch: Dict[str, object], dev: torch.device, stream) -> None:
        self.model, self.dev, self.stream = model, dev, stream
        self.tables = []            # (parameter name, [id arrays], row count, rows buffer)
        for name, keys, _ in SPARSE_TABLES:
            if name not in model._param_names:
                continue
            ids = [batch[k].reshape(-1) for k in keys]
            if model._gather_ids is not None:       # data parallel: the union over the ranks (dp.GradReducer)
                ids = [model._gather_ids(torch.cat(ids))]
            n_rows = model.get_parameter(name).shape[0]
            rows = torch.empty(max(1, min(n_rows, sum(t.numel() for t in ids))), dtype=torch.int64, device=dev)
            self.tables.append((name, ids, n_rows, rows))
        self.count = torch.empty(len(self.tables), dtype=torch.int64, device=dev)
        self.build()
        if model.cfg.sparse_grad == 2:
            for j, (name, _, _, rows) in enumerate(self.tables):
                optim.catch_up(model.get_parameter(name), rows, self.count[j:j + 1])
        self.host = torch.empty(len(self.tables), dtype=torch.int64, pin_memory=dev.type == "cuda")
        self.host.copy_(self.count, non_blocking=True)
        self.event = torch.cuda.Event() if dev.type == "cuda" else None
        if self.event is not None:
            self.event.record(torch.cuda.current_stream(dev))

    def build(self) -> None:
        """(Re)writes the rows buffers and the model's row -> slot maps; the result depends on the ids alone."""
        lib, model = _lib.load(), self.model
        for j, (name, ids, n_rows, rows) in enumerate(self.tables):
            slot = model._row_slot.get(name)
            if slot is None or slot.device != self.dev or slot.numel() != n_rows:
                slot = model._row_slot[name] = torch.zeros(n_rows, dtype=torch.int32, device=self.dev)
            ws = torch.empty(lib.intel_rowset_workspace_bytes(n_rows), dtype=torch.uint8, device=self.dev)
            a, b = (ids + [None])[:2]
            _lib.check(lib.intel_rowset_build(n_rows, _lib.ptr(a, torch.int64), a.numel(), _lib.ptr(b, torch.int64),
                                              0 if b is None else b.numel(), _lib.ptr(slot), _lib.ptr(rows),
                                              _lib.ptr(self.count[j:j + 1]), _lib.ptr(ws), ws.numel(), self.stream))
        model._row_sets_current = self

    def sizes(self) -> Dict[str, int]:
        if self.event is not None:
            self.event.synchronize()
        if self.model._row_sets_current is not self:     # another training forward pass rewrote the shared maps since
            self.build()
        return {t[0]: int(u) for t, u in zip(self.tables, self.host.tolist())}

    def maps(self) -> "_lib.RowMaps":
        m = _lib.RowMaps()
        for name, _, field in SPARSE_TABLES:
            if any(t[0] == name for t in self.tables):
                setattr(m, field, _lib.ptr(self.model._row_slot[name]))
        return m


class _IntelFn(torch.autograd.Function):
    """(parameters...) -> (weights, ens_score, intents); backward = ensemble_bwd then intent_bwd."""

    @staticmethod
    def forward(ctx, model: "IntEL", batch: Dict[str, object], grad_mode: bool, *params: torch.Tensor):
        lib = _lib.load()
        cfg = model.cfg
        dev = params[0].device
        names = model._param_names
        tensors = dict(zip(names, params))
        B, L = batch["i_id_s"].shape
        H1, H2 = batch["his_context_mh"].shape[1], batch["his_item_id"].shape[1]
        p_drop = float(cfg.dropout) if model.training else 0.0
        if p_drop > 0.0:
            model._drop_step += 1
        keep = grad_mode and any(ctx.needs_input_grad)
        dims = _lib.make_dims(cfg, B, L, H1, H2, p_drop, model._drop_seed * 1000003 + model._drop_step, inference=not keep)
        P = _lib.make_tensors(cfg, tensors)
        bt = _lib.make_batch(batch, cfg)
        stream = _lib.stream_ptr(dev)
        ws_int = _take_ws(model, lib.intel_intent_workspace_bytes(dims), dev)
        ws_ens = _take_ws(model, lib.intel_ensemble_workspace_bytes(dims), dev)
        if model.validate_inputs:
            model._queue_input_check(lib, dims, bt, dev, stream)
        row_sets = _RowSets(model, batch, dev, stream) if keep and cfg.sparse_grad else None
        intents = torch.empty(B, cfg.intent_num, dtype=torch.float32, device=dev)
        weights = torch.empty(B, L, cfg.model_num, dtype=torch.float32, device=dev)
        ens = torch.empty(B, L, dtype=torch.float32, device=dev)
        _lib.check(lib.intel_intent_fwd(dims, P, bt, _lib.ptr(intents), _lib.ptr(ws_int), ws_int.numel(), stream))
        _lib.check(lib.intel_ensemble_fwd(dims, P, bt, _lib.ptr(intents), _lib.ptr(weights), _lib.ptr(ens),
                                          _lib.ptr(ws_ens), ws_ens.numel(), stream))
        # needs_input_grad stays True under torch.no_grad() (BaseRunner.predict) and the grad mode is always off inside
        # Function.forward: the caller's grad mode arrives as an argument
        if keep:
            ctx.model, ctx.batch, ctx.dims = model, batch, dims
            ctx.ws_int, ctx.ws_ens = ws_int, ws_ens
            ctx.params = params
            ctx.row_sets = row_sets
            # `intents` is an output: holding it as a plain attribute would close a ctx -> tensor -> grad_fn -> ctx
            # cycle that only the cyclic GC frees, and every leaked step costs the allocator a fresh cudaMalloc.
            ctx.save_for_backward(intents)
        else:                       # inference: nothing is kept for a backward pass
            _give_ws(model, ws_int)
            _give_ws(model, ws_ens)
        return weights, ens, intents

    @staticmethod
    def backward(ctx, d_weights, d_ens, d_intents):
        lib = _lib.load()
        if getattr(ctx, "ws_int", None) is None or ctx.ws_ens is None:
            raise RuntimeError("IntEL backward ran twice on one forward pass: the activations live in a pooled workspace "
                               "that the first backward handed back (retain_graph is not supported)")
        model, cfg, batch, dims = ctx.model, ctx.model.cfg, ctx.batch, ctx.dims
        params = ctx.params
        (intents,) = ctx.saved_tensors
        dev = params[0].device
        names = model._param_names
        P = _lib.make_tensors(cfg, dict(zip(names, params)))
        # one zero-filled buffer for all dense gradients (a single fill kernel instead of one per parameter); the
        # per-parameter gradients are 256-byte aligned views into it.  The score stream's parameters sit at the end: they
        # are the last gradients the pass below completes, so everything before `late` can be exchanged while they are
        # still being computed (dp.GradReducer installs model._early_reduce for that).
        # sparse_grad: a covered table's gradient is the compact [U, d] block of its row set (the table writes all happen
        # before the SCORE phase, so the blocks sit before `late` with the other early gradients)
        row_sets = ctx.row_sets
        U = row_sets.sizes() if row_sets is not None else {}
        numel = [U[n] * p[0].numel() if n in U else p.numel() for n, p in zip(names, params)]
        late_names = model._late_grad_names
        pack = [n for n in model._packed_grad_names if n in names]
        rest = [n for n in names if n not in late_names and n not in pack]
        order = [names.index(n) for n in rest + pack] + [i for i, n in enumerate(names) if n in late_names]
        offs, total, late = [0] * len(params), 0, None
        for i in order:
            if late is None and names[i] in late_names:
                late = total
            offs[i] = total
            # the three weights multiplied by the predicted intents sit back to back (no alignment gap): the library then
            # forms their gradients with one product (api_model.cu, intel_ensemble_bwd_phase)
            packed_next = names[i] in pack and names[i] != pack[-1]
            total += numel[i] if packed_next else (numel[i] + 63) // 64 * 64
        late = total if late is None else late
        flat = torch.zeros(total, dtype=torch.float32, device=dev)
        grads = [flat[o:o + n].view((U[k],) + p.shape[1:] if k in U else p.shape) for o, n, k, p in zip(offs, numel, names, params)]
        model._flat_grad = flat         # dp.GradReducer all-reduces this one buffer when the .grad tensors still alias it
        model._flat_late = late
        G = _lib.make_tensors(cfg, dict(zip(names, grads)))
        bt = _lib.make_batch(batch, cfg)
        stream = _lib.stream_ptr(dev)
        maps = row_sets.maps() if row_sets is not None else None
        have_ens = d_weights is not None or d_ens is not None
        d_int_ens: Optional[torch.Tensor] = None
        dw = de = None

        def ens_bwd(phases: int) -> None:
            _lib.check(lib.intel_ensemble_bwd_phase_rows(dims, P, bt, _lib.ptr(intents), _lib.ptr(dw), _lib.ptr(de), G,
                                                         _lib.ptr(d_int_ens), _lib.ptr(ctx.ws_ens), ctx.ws_ens.numel(), stream,
                                                         phases, maps))

        # order of the pass (SURVEY 8e): head + cross attentions (the gradient w.r.t. the predicted intents is final) ->
        # intent predictor -> item stack + embedding rows -> [every gradient but the score stream's is final] -> score stack
        single = getattr(model, "_single_call_backward", False)       # test hook: intel_ensemble_bwd in one call
        if have_ens:
            d_int_ens = torch.empty_like(intents)
            dw = d_weights.contiguous() if d_weights is not None else None
            de = d_ens.contiguous() if d_ens is not None else None
            ens_bwd(_lib.ENS_BWD_HEAD | _lib.ENS_BWD_ITEM | _lib.ENS_BWD_SCORE if single else _lib.ENS_BWD_HEAD)
        first = d_intents.contiguous() if d_intents is not None else d_int_ens
        extra = d_int_ens if d_intents is not None else None
        if first is not None:
            _lib.check(lib.intel_intent_bwd_rows(dims, P, bt, _lib.ptr(intents), _lib.ptr(first), _lib.ptr(extra), G,
                                                 _lib.ptr(ctx.ws_int), ctx.ws_int.numel(), stream, maps))
        if have_ens and not single:
            ens_bwd(_lib.ENS_BWD_ITEM)
        early = getattr(model, "_early_reduce", None)
        if early is not None and not single:
            early(flat, late)            # asynchronous: runs beside the score stack below
        if have_ens and not single:
            ens_bwd(_lib.ENS_BWD_SCORE)
        _give_ws(model, ctx.ws_int)
        _give_ws(model, ctx.ws_ens)
        ctx.ws_int = ctx.ws_ens = ctx.row_sets = None
        if row_sets is not None:
            # COO gradients whose values are the compact blocks; optim.Adam recognises these indices as coalesced (autograd
            # drops the flag on its way into .grad); the indices are valid by construction, so no invariant check
            with torch.sparse.check_sparse_tensor_invariants(enable=False):
                for name, _, _, rows in row_sets.tables:
                    i = names.index(name)
                    optim.note_coalesced_rows((id(model), name), rows)
                    grads[i] = torch.sparse_coo_tensor(rows[:U[name]].view(1, -1), grads[i], size=params[i].shape,
                                                       is_coalesced=True)
        return (None, None, None) + tuple(grads)


class IntEL(nn.Module):
    reader, runner = "SeqReader", "BaseRunner"
    extra_log_args = ['cross_attn_qsize', 'num_heads', 'num_layers', 'encoder', 'intent_emb_size']

    @staticmethod
    def parse_model_args(parser: argparse.ArgumentParser) -> argparse.ArgumentParser:
        """Same flags and defaults as IntEL.py:17-34 + GeneralSeq.py:15-17 + BaseModel.py:20-27."""
        parser.add_argument('--encoder', type=str, default='BERT4Rec', help='A sequence encoder for intent prediction.')
        parser.add_argument('--context_emb_size', type=int, default=16, help='Embedding size for context.')
        parser.add_argument('--i_emb_size', type=int, default=16, help='Embedding size for item id.')
        parser.add_argument('--u_emb_size', type=int, default=32, help='Embedding size for user.')
        parser.add_argument('--s_emb_size', type=int, default=32, help='Embedding size for score.')
        parser.add_argument('--im_emb_size', type=int, default=16, help='Embedding size for item metadata.')
        parser.add_argument('--intent_emb_size', type=int, default=16, help='Embedding size for intent.')
        parser.add_argument('--cross_attn_qsize', type=int, default=32, help='Embedding size for cross-attention query.')
        parser.add_argument('--num_heads', type=int, default=1, help='Number of attention heads.')
        parser.add_argument('--dropout', type=float, default=0, help='Dropout probability for each deep layer')
        parser.add_argument('--num_layers', type=int, default=1, help='Number of self-attention layers.')
        parser.add_argument('--cross_attention', type=int, default=1,
                            help='Using cross-attention structure or direct attention.')
        parser.add_argument('--history_max', type=int, default=20)
        parser.add_argument('--model_path', type=str, default='', help='Model save path.')
        parser.add_argument('--buffer', type=int, default=1, help='Whether to buffer feed dicts for dev/test')
        parser.add_argument('--model_num', type=int, default=2, help='Number of base models.')
        parser.add_argument('--sparse_grad', type=int, default=0,
                            help='Row-sparse (COO) gradients for the embedding tables; they need optim.Adam (BaseRunner_b200), '
                                 'since torch.optim.Adam rejects sparse gradients.  1: lazy Adam, the rows a step does not '
                                 'name keep their values (differs from dense Adam with L2).  2: exact, optim.Adam defers the '
                                 'updates of those rows and replays them when the rows are next read: bitwise dense Adam.')
        return parser

    def __init__(self, args, corpus=None, cfg: Optional[IntelConfig] = None):
        super().__init__()
        self.cfg = cfg if cfg is not None else IntelConfig.from_args(args, corpus)
        c = self.cfg
        self.device = getattr(args, "device", torch.device("cuda"))
        self.model_path = getattr(args, "model_path", "")
        self.buffer = getattr(args, "buffer", 1)
        self.optimizer, self.scheduler = None, None
        self.check_list = list()
        self._ws_pool = {}
        # index range check of every batch (nn.Embedding raises IndexError in the reference): the check kernel runs with
        # the forward pass, its verdict is read without a sync at the next forward / by check_inputs()
        self.validate_inputs = True
        self._check_flag = self._check_host = self._check_event = None
        self._drop_seed, self._drop_step = int(torch.initial_seed()) & 0x7FFFFFFF, 0
        self.intent_num, self.model_num = c.intent_num, c.model_num
        self.user_num, self.item_num = c.user_rows, c.item_rows
        self.max_his = c.history_max
        I, K, di, ds = c.intent_num, c.model_num, c.d_item, c.d_score
        # ---- parameter containers, registered in the reference's order (IntEL.py:43-115) ----
        self.iid_embeddings = nn.Embedding(c.item_rows, c.i_emb_size)
        if c.class_rows > 0:
            self.item_embeddings = nn.Embedding(c.class_rows, c.im_emb_size)
        self.uid_embeddings = nn.Embedding(c.user_rows, c.u_emb_size)
        self.intent_embeddings = nn.Linear(I, c.intent_emb_size)
        self.score_embeddings = nn.Linear(K, c.s_emb_size)
        self.i_attn_head = _attn_container(di)
        self.i_W1, self.i_W2 = nn.Linear(di, di), nn.Linear(di, di)
        self.i_layer_norm = nn.LayerNorm(di)
        self.s_attn_head = _attn_container(ds)
        self.s_W1, self.s_W2 = nn.Linear(ds, ds), nn.Linear(ds, ds)
        self.s_layer_norm = nn.LayerNorm(ds)
        if c.cross_attention:
            self.intent_score_attention = _cross_container(I, ds)
            self.intent_item_attention = _cross_container(I, di)
        else:
            self.intent_score_embeddings = nn.Sequential(nn.Linear(I, c.cross_attn_qsize), nn.ReLU(),
                                                         nn.Linear(c.cross_attn_qsize, ds, bias=False))
            self.intent_item_embeddings = nn.Sequential(nn.Linear(I, c.cross_attn_qsize), nn.ReLU(),
                                                        nn.Linear(c.cross_attn_qsize, di, bias=False))
        self.weight_embeddings = nn.Linear(c.d_head, K)
        self.context_embeddings = nn.Embedding(c.ctx_rows, c.context_emb_size)
        self.encoder = _encoder_container(c, c.d_his)
        self.item_encoder = _encoder_container(c, c.d_his_item)
        self.pred_layer = nn.Linear(c.d_pred, I)
        self._param_names = [n for n, _ in self.named_parameters()]
        # gradients that only the last phase of the backward pass (the score stream's stack) writes
        self._late_grad_names = {n for n in self._param_names
                                 if n.startswith(("s_attn_head.", "s_W1.", "s_W2.", "s_layer_norm.", "score_embeddings."))}
        self._early_reduce = None       # set by dp.GradReducer: callable(flat_grad, late_offset)
        # sparse_grad: persistent row -> slot map per table (intel_rowset_build), the row sets of the last training forward
        # pass, and dp.GradReducer's hook that gathers the ids of all ranks (every rank then builds the same row sets)
        self._row_slot: Dict[str, torch.Tensor] = {}
        self._row_sets_current = None
        self._gather_ids = None
        # gradients kept back to back in the flat buffer, in the row order of the library's stacked weight (Wcat)
        self._packed_grad_names = (["intent_item_attention.query_layer.weight", "intent_score_attention.query_layer.weight",
                                    "intent_embeddings.weight"] if c.cross_attention else [])
        shapes = c.param_shapes()
        for n, p in self.named_parameters():
            assert tuple(p.shape) == shapes[n], (n, tuple(p.shape), shapes[n])
        if c.sparse_grad not in (0, 1, 2):
            raise ValueError(f"sparse_grad must be 0, 1 or 2, not {c.sparse_grad}")
        if c.sparse_grad == 2:
            # optim.Adam defers the zero-gradient updates of these tables: whatever reads them whole sees them current
            optim.defer_zero_updates(self._deferred_tables())
            self.register_state_dict_pre_hook(lambda module, *_: module.flush_tables())
            self.register_load_state_dict_pre_hook(lambda module, *_: module.flush_tables())

    def _deferred_tables(self) -> list:
        return [self.get_parameter(n) for n, _, _ in SPARSE_TABLES if n in self._param_names] if self.cfg.sparse_grad == 2 else []

    def flush_tables(self) -> None:
        """sparse_grad = 2: apply the updates optim.Adam deferred on the embedding tables (a no-op when none are pending)."""
        optim.flush(self._deferred_tables())

    def _queue_input_check(self, lib, dims, bt, dev, stream) -> None:
        self.check_inputs(wait=False)
        if self._check_flag is None or self._check_flag.device != dev:
            self._check_flag = torch.zeros(1, dtype=torch.int32, device=dev)
            self._check_host = torch.zeros(1, dtype=torch.int32).pin_memory() if dev.type == "cuda" else torch.zeros(1, dtype=torch.int32)
            self._check_event = torch.cuda.Event() if dev.type == "cuda" else None
        _lib.check(lib.intel_batch_validate(dims, bt, _lib.ptr(self._check_flag), stream))
        self._check_host.copy_(self._check_flag, non_blocking=True)
        if self._check_event is not None:
            self._check_event.record(torch.cuda.current_stream(dev))

    def check_inputs(self, wait: bool = True) -> None:
        """Raise IndexError if a batch fed so far carried an id outside its embedding table (or a history length
        outside [1, H]).  wait=False only looks at verdicts that have already arrived (no device sync)."""
        if self._check_host is None:
            return
        if self._check_event is not None:
            if wait:
                self._check_event.synchronize()
            elif not self._check_event.query():
                return
        flags = int(self._check_host.item())
        if flags:
            self._check_flag.zero_()
            self._check_host.zero_()
            raise IndexError("IntEL batch out of range: " + _lib.describe_bad_input(flags))

    # ---- the hot path ----
    def forward(self, data: Dict[str, object]) -> Dict[str, torch.Tensor]:
        params = [p for _, p in self.named_parameters()]
        if self.cfg.sparse_grad == 2 and not (torch.is_grad_enabled() and any(p.requires_grad for p in params)):
            self.flush_tables()      # no row set is built (a training forward pass catches up its rows in _RowSets)
        weights, ens, intents = _IntelFn.apply(self, data, torch.is_grad_enabled(), *params)
        return {"weights": weights, "ens_score": ens, "intents": intents}

    # ---- auxiliary methods kept from BaseModel (BaseModel.py:53-78) ----
    def customize_parameters(self, define_dict={}) -> list:
        weight_p, bias_p = [], []
        for name, p in filter(lambda x: x[1].requires_grad, self.named_parameters()):
            (bias_p if 'bias' in name else weight_p).append(p)
        return [{'params': weight_p}, {'params': bias_p, 'weight_decay': 0}]

    def save_model(self, model_path=None):
        model_path = model_path or self.model_path
        os.makedirs(os.path.dirname(model_path) or ".", exist_ok=True)
        torch.save(self.state_dict(), model_path)

    def load_model(self, model_path=None):
        model_path = model_path or self.model_path
        self.load_state_dict(torch.load(model_path))
        logging.info('Load model from ' + model_path)

    def count_variables(self) -> int:
        return sum(p.numel() for p in self.parameters() if p.requires_grad)
