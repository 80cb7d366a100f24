"""ctypes binding of libintel_b200.so (the C ABI declared in include/intel_b200.h).

There is NO fallback: if the CUDA library is missing or a tensor is not on a CUDA device the
call raises.  PyTorch is only the owner of device memory and streams here.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Optional

import torch

from .config import IntelConfig

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libintel_b200.so")
MAX_BERT_LAYERS = 4
MAX_TOPK = 16

_p = C.c_void_p


class Dims(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("B", "L", "K", "I", "H1", "H2", "item_rows", "class_rows", "user_rows", "ctx_rows")] + \
               [(n, C.c_int32) for n in ("d_iid", "d_im", "d_u", "d_s", "d_int", "d_ctx", "qsize", "heads", "layers",
                                         "cross_attention", "encoder", "gru_hidden", "bert_layers", "bert_heads",
                                         "history_max")] + \
               [("dropout_p", C.c_float), ("dropout_seed", C.c_uint64), ("inference", C.c_int32)]


class BertLayer(C.Structure):
    _fields_ = [(n, _p) for n in ("qw", "qb", "kw", "kb", "vw", "vb", "ln1w", "ln1b", "l1w", "l1b", "l2w", "l2b",
                                  "ln2w", "ln2b")]


class Encoder(C.Structure):
    _fields_ = [("pos", _p), ("layer", BertLayer * MAX_BERT_LAYERS)] + \
               [(n, _p) for n in ("w_ih", "w_hh", "b_ih", "b_hh", "w_out")]


class SelfAtt(C.Structure):
    _fields_ = [(n, _p) for n in ("wq", "wk", "wv", "w1", "b1", "w2", "b2", "lnw", "lnb")]


class Tensors(C.Structure):
    _fields_ = [(n, _p) for n in ("iid_emb", "item_emb", "uid_emb", "ctx_emb", "intent_w", "intent_b", "score_w",
                                  "score_b")] + \
               [("item", SelfAtt), ("score", SelfAtt)] + \
               [(n, _p) for n in ("xq_item", "xk_item", "xv_item", "xq_score", "xk_score", "xv_score",
                                  "gate_item_w0", "gate_item_b0", "gate_item_w2",
                                  "gate_score_w0", "gate_score_b0", "gate_score_w2", "head_w", "head_b")] + \
               [("enc", Encoder), ("item_enc", Encoder), ("pred_w", _p), ("pred_b", _p)]


class RowMaps(C.Structure):
    _fields_ = [(n, _p) for n in ("iid", "item", "uid", "ctx")]


class Batch(C.Structure):
    _fields_ = [(n, _p) for n in ("u_id", "i_id", "i_class", "session_len", "scores", "context_mh", "his_context",
                                  "his_intents", "history_len", "his_item_id", "his_item_int", "history_item_len",
                                  "his_intents_idx", "his_intents_val", "his_item_int_idx", "his_item_int_val")] + \
               [("nz1", C.c_int32), ("nz2", C.c_int32)]


ENS_BWD_HEAD, ENS_BWD_ITEM, ENS_BWD_SCORE = 1, 2, 4     # INTEL_ENS_BWD_* of include/intel_b200.h

_lib: Optional[C.CDLL] = None
_allow_host_tensors = False     # flipped only by tests/emu (kernel-logic emulator), never by the package


def _declare(lib: C.CDLL) -> None:
    i64, i32, dbl, sz = C.c_int64, C.c_int, C.c_double, C.c_size_t
    PD, PT, PB, PM = C.POINTER(Dims), C.POINTER(Tensors), C.POINTER(Batch), C.POINTER(RowMaps)
    sig = {
        "intel_last_error": (C.c_char_p, []),
        "intel_abi_version": (i32, []),
        "intel_intent_workspace_bytes": (sz, [PD]),
        "intel_intent_fwd": (i32, [PD, PT, PB, _p, _p, sz, _p]),
        "intel_intent_bwd": (i32, [PD, PT, PB, _p, _p, _p, PT, _p, sz, _p]),
        "intel_ensemble_workspace_bytes": (sz, [PD]),
        "intel_ensemble_fwd": (i32, [PD, PT, PB, _p, _p, _p, _p, sz, _p]),
        "intel_ensemble_bwd": (i32, [PD, PT, PB, _p, _p, _p, PT, _p, _p, sz, _p]),
        "intel_ensemble_bwd_phase": (i32, [PD, PT, PB, _p, _p, _p, PT, _p, _p, sz, _p, i32]),
        "intel_ensemble_bwd_phase_rows": (i32, [PD, PT, PB, _p, _p, _p, PT, _p, _p, sz, _p, i32, PM]),
        "intel_intent_bwd_rows": (i32, [PD, PT, PB, _p, _p, _p, PT, _p, sz, _p, PM]),
        "intel_rowset_workspace_bytes": (sz, [i64]),
        "intel_rowset_build": (i32, [i64, _p, i64, _p, i64, _p, _p, _p, _p, sz, _p]),
        "intel_reserve_sms": (i32, [i32]),
        "intel_loss_pl_fwd_bwd": (i32, [i64, i64, i64, _p, _p, _p, _p, _p, i32, dbl, _p, _p, _p, _p]),
        "intel_loss_bpr_fwd_bwd": (i32, [i64, i64, i64, _p, _p, _p, _p, _p, _p, C.c_uint64, i32, dbl, _p, _p, _p, _p]),
        "intel_loss_mse_fwd_bwd": (i32, [i64, i64, i64, _p, _p, _p, _p, _p, i32, dbl, _p, _p, _p, _p]),
        "intel_intent_loss_fwd_bwd": (i32, [i64, i64, _p, _p, dbl, dbl, _p, _p, _p, _p]),
        "intel_scale_by_device_scalar": (i32, [i64, _p, _p, dbl, _p, dbl, _p, _p]),
        "intel_ndcg_workspace_bytes": (sz, [i64, i32]),
        "intel_ndcg_topk": (i32, [i64, i64, _p, _p, _p, _p, _p, _p, i64, C.POINTER(C.c_int32), i32, _p, _p, _p, sz, _p]),
        "intel_intent_topk_workspace_bytes": (sz, [i64, i32]),
        "intel_intent_topk": (i32, [i64, i64, _p, _p, C.POINTER(C.c_int32), i32, _p, _p, sz, _p]),
        "intel_fuse_fwd": (i32, [i64, i64, i64, _p, _p, _p, _p]),
        "intel_select_list": (i32, [i64, i64, i64, _p, i32, _p, _p]),
        "intel_rank_lists": (i32, [i64, i64, i64, _p, _p, _p]),
        "intel_batch_validate": (i32, [PD, PB, _p, _p]),
        "intel_batch_build": (i32, [_p, i64, _p, _p, i64, i64, i64, _p, _p]),
        "intel_gather_fwd": (i32, [i64, i32, _p, _p, _p, i32, i32, _p]),
        "intel_scatter_add_bwd": (i32, [i64, i32, _p, i32, _p, _p, _p]),
        "intel_linear_fwd": (i32, [i64, i64, i64, _p, _p, _p, _p, _p]),
        "intel_linear_dx": (i32, [i64, i64, i64, _p, _p, _p, _p, _p]),
        "intel_linear_dw": (i32, [i64, i64, i64, _p, _p, _p, _p, _p]),
        "intel_linear_fwd_ex": (i32, [i64, i64, i64, _p, i64, _p, _p, _p, i64, i32, _p]),
        "intel_linear_dx_ex": (i32, [i64, i64, i64, _p, _p, _p, i64, _p, i64, _p]),
        "intel_linear_dw_ex": (i32, [i64, i64, i64, _p, _p, i64, _p, _p, i32, _p]),
        "intel_softmax_rows_fwd": (i32, [i64, i64, _p, _p, _p]),
        "intel_softmax_rows_bwd": (i32, [i64, i64, _p, _p, _p, _p]),
        "intel_mha_fwd": (i32, [i64, i64, i32, i32, _p, _p, _p, _p]),
        "intel_mha_bwd": (i32, [i64, i64, i32, i32, _p, _p, _p, _p, _p]),
        "intel_debug_use_fused_stack": (i32, [i32]),
        "intel_debug_stack_sessions_per_cta": (i32, [i32]),
        "intel_debug_use_tcgen05_gemm": (i32, [i32]),
        "intel_debug_use_tcgen05_stack": (i32, [i32]),
        "intel_debug_use_tcgen05_gru": (i32, [i32]),
        "intel_debug_use_rows_gemm": (i32, [i32]),
        "intel_debug_gru_prep": (i32, [i64, i64, _p, _p, _p, _p, _p, _p]),
        "intel_debug_use_fused_bert": (i32, [i32]),
        "intel_host_pack_rows": (i64, [i64, i64, _p, i32, _p, _p, _p, i32, i64, _p]),
        "intel_awelv_fwd": (i32, [i64, i64, i32, i32, _p, _p, _p, _p, _p, _p, _p, _p]),
        "intel_awelv_bwd": (i32, [i64, i64, i32, i32, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
        "intel_pool_head_fwd": (i32, [i64, i64, i32, _p, _p, _p, _p, _p, _p, _p]),
        "intel_pool_head_bwd": (i32, [i64, i64, i32, _p, _p, _p, _p, _p, _p, _p]),
        "intel_lambdarank_lambdas": (i32, [i64, i64, _p, _p, _p, _p, _p]),
        "intel_adam_step": (i32, [i32, _p, _p, _p, _p, _p, _p, dbl, dbl, dbl, dbl, i64, _p]),
        "intel_adam_rows_step": (i32, [i32, _p, _p, _p, _p, _p, _p, _p, _p, dbl, dbl, dbl, dbl, i64, _p]),
        "intel_adam_deferred_rows_step": (i32, [i32, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, dbl, dbl, dbl, dbl, i64, _p]),
        "intel_adam_deferred_catch_up": (i32, [i32, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
        "intel_profile_enable": (i32, [i32]),
        "intel_profile_report": (i32, [C.c_char_p, sz]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)       # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args


EXPORTED = ["intel_ensemble_bwd_phase", "intel_reserve_sms", "intel_last_error", "intel_abi_version", "intel_intent_workspace_bytes", "intel_intent_fwd",
            "intel_intent_bwd", "intel_ensemble_workspace_bytes", "intel_ensemble_fwd", "intel_ensemble_bwd",
            "intel_loss_pl_fwd_bwd", "intel_loss_bpr_fwd_bwd", "intel_loss_mse_fwd_bwd", "intel_intent_loss_fwd_bwd",
            "intel_scale_by_device_scalar", "intel_ndcg_workspace_bytes", "intel_ndcg_topk",
            "intel_intent_topk_workspace_bytes", "intel_intent_topk", "intel_fuse_fwd", "intel_select_list",
            "intel_rank_lists", "intel_gather_fwd", "intel_scatter_add_bwd", "intel_linear_fwd",
            "intel_profile_enable", "intel_profile_report", "intel_linear_dx", "intel_linear_dw", "intel_mha_fwd",
            "intel_mha_bwd", "intel_debug_use_fused_stack", "intel_debug_stack_sessions_per_cta", "intel_debug_use_tcgen05_gemm", "intel_host_pack_rows", "intel_adam_step", "intel_awelv_fwd", "intel_awelv_bwd",
            "intel_lambdarank_lambdas", "intel_pool_head_fwd", "intel_pool_head_bwd",
            "intel_linear_fwd_ex", "intel_linear_dx_ex", "intel_linear_dw_ex", "intel_softmax_rows_fwd", "intel_softmax_rows_bwd",
            "intel_batch_validate", "intel_debug_use_tcgen05_stack", "intel_batch_build", "intel_debug_use_tcgen05_gru", "intel_debug_use_rows_gemm", "intel_debug_gru_prep", "intel_debug_use_fused_bert",
            "intel_rowset_workspace_bytes", "intel_rowset_build", "intel_ensemble_bwd_phase_rows", "intel_intent_bwd_rows",
            "intel_adam_rows_step", "intel_adam_deferred_rows_step", "intel_adam_deferred_catch_up"]


def load(path: Optional[str] = None) -> C.CDLL:
    """Load (once) and return the shared library; raises if it has not been built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise RuntimeError(f"{p} is missing: build it with `python -m intel_sigir2023_b200.build` "
                           "(there is no CPU fallback for the IntEL hot path)")
    lib = C.CDLL(p)
    _declare(lib)
    if lib.intel_abi_version() != 1:
        raise RuntimeError("libintel_b200 ABI version mismatch")
    if os.environ.get("INTEL_STACK_SESSIONS"):       # tuning knob for the fused stack kernels (1..4 sessions per CTA)
        lib.intel_debug_stack_sessions_per_cta(int(os.environ["INTEL_STACK_SESSIONS"]))
    if os.environ.get("INTEL_TCGEN05_GEMM"):
        lib.intel_debug_use_tcgen05_gemm(int(os.environ["INTEL_TCGEN05_GEMM"]))
    _lib = lib
    return lib


def check(status: int) -> None:
    if status != 0:
        msg = load().intel_last_error()
        raise RuntimeError(f"libintel_b200 error {status}: {msg.decode() if msg else ''}")


def ptr(t: Optional[torch.Tensor], dtype: Optional[torch.dtype] = None) -> Optional[int]:
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda and not _allow_host_tensors:
        raise RuntimeError("libintel_b200 needs CUDA tensors; there is no CPU path")
    if not t.is_contiguous():
        raise RuntimeError("libintel_b200 needs contiguous tensors")
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError(f"expected {dtype}, got {t.dtype}")
    return t.data_ptr()


def stream_ptr(device: torch.device) -> Optional[int]:
    if device.type != "cuda":
        return None
    return torch.cuda.current_stream(device).cuda_stream


def make_dims(cfg: IntelConfig, B: int, L: int, H1: int, H2: int, dropout_p: float = 0.0, seed: int = 0,
              inference: bool = False) -> Dims:
    d = Dims()
    d.inference = 1 if inference else 0
    d.dropout_p, d.dropout_seed = float(dropout_p), int(seed) & 0xFFFFFFFFFFFFFFFF
    d.B, d.L, d.K, d.I, d.H1, d.H2 = B, L, cfg.model_num, cfg.intent_num, H1, H2
    d.item_rows, d.class_rows, d.user_rows, d.ctx_rows = cfg.item_rows, cfg.class_rows, cfg.user_rows, cfg.ctx_rows
    d.d_iid, d.d_im = cfg.i_emb_size, (cfg.im_emb_size if cfg.class_rows > 0 else 0)
    d.d_u, d.d_s, d.d_int, d.d_ctx = cfg.u_emb_size, cfg.s_emb_size, cfg.intent_emb_size, cfg.context_emb_size
    d.qsize, d.heads, d.layers = cfg.cross_attn_qsize, cfg.num_heads, cfg.num_layers
    d.cross_attention = 1 if cfg.cross_attention else 0
    if cfg.encoder == "BERT4Rec":
        d.encoder = 0
    elif cfg.encoder == "GRU4Rec":
        d.encoder = 1
    else:
        raise ValueError("Invalid sequence encoder.")
    d.gru_hidden, d.bert_layers, d.bert_heads, d.history_max = cfg.gru_hidden, cfg.bert_layers, cfg.bert_heads, cfg.history_max
    return d


def make_tensors(cfg: IntelConfig, tensors: Dict[str, torch.Tensor]) -> Tensors:
    """Pointer struct from a {state_dict key: tensor} mapping (parameters or their gradient buffers)."""
    def g(key: str) -> Optional[int]:
        t = tensors.get(key)
        return ptr(t, torch.float32) if t is not None else None
    T = Tensors()
    T.iid_emb, T.item_emb = g("iid_embeddings.weight"), g("item_embeddings.weight")
    T.uid_emb, T.ctx_emb = g("uid_embeddings.weight"), g("context_embeddings.weight")
    T.intent_w, T.intent_b = g("intent_embeddings.weight"), g("intent_embeddings.bias")
    T.score_w, T.score_b = g("score_embeddings.weight"), g("score_embeddings.bias")
    for pre, st in (("i", T.item), ("s", T.score)):
        st.wq, st.wk, st.wv = (g(f"{pre}_attn_head.{n}_linear.weight") for n in "qkv")
        st.w1, st.b1, st.w2, st.b2 = g(f"{pre}_W1.weight"), g(f"{pre}_W1.bias"), g(f"{pre}_W2.weight"), g(f"{pre}_W2.bias")
        st.lnw, st.lnb = g(f"{pre}_layer_norm.weight"), g(f"{pre}_layer_norm.bias")
    T.xq_item, T.xk_item, T.xv_item = (g(f"intent_item_attention.{n}_layer.weight") for n in ("query", "key", "value"))
    T.xq_score, T.xk_score, T.xv_score = (g(f"intent_score_attention.{n}_layer.weight") for n in ("query", "key", "value"))
    T.gate_item_w0, T.gate_item_b0, T.gate_item_w2 = (g("intent_item_embeddings.0.weight"), g("intent_item_embeddings.0.bias"),
                                                      g("intent_item_embeddings.2.weight"))
    T.gate_score_w0, T.gate_score_b0, T.gate_score_w2 = (g("intent_score_embeddings.0.weight"), g("intent_score_embeddings.0.bias"),
                                                         g("intent_score_embeddings.2.weight"))
    T.head_w, T.head_b = g("weight_embeddings.weight"), g("weight_embeddings.bias")
    for name, e in (("encoder", T.enc), ("item_encoder", T.item_enc)):
        e.pos = g(f"{name}.p_embeddings.weight")
        for l in range(min(cfg.bert_layers, MAX_BERT_LAYERS)):
            b, bl = f"{name}.transformer_block.{l}", e.layer[l]
            bl.qw, bl.qb = g(f"{b}.masked_attn_head.q_linear.weight"), g(f"{b}.masked_attn_head.q_linear.bias")
            bl.kw, bl.kb = g(f"{b}.masked_attn_head.k_linear.weight"), g(f"{b}.masked_attn_head.k_linear.bias")
            bl.vw, bl.vb = g(f"{b}.masked_attn_head.v_linear.weight"), g(f"{b}.masked_attn_head.v_linear.bias")
            bl.ln1w, bl.ln1b = g(f"{b}.layer_norm1.weight"), g(f"{b}.layer_norm1.bias")
            bl.l1w, bl.l1b = g(f"{b}.linear1.weight"), g(f"{b}.linear1.bias")
            bl.l2w, bl.l2b = g(f"{b}.linear2.weight"), g(f"{b}.linear2.bias")
            bl.ln2w, bl.ln2b = g(f"{b}.layer_norm2.weight"), g(f"{b}.layer_norm2.bias")
        e.w_ih, e.w_hh = g(f"{name}.rnn.weight_ih_l0"), g(f"{name}.rnn.weight_hh_l0")
        e.b_ih, e.b_hh = g(f"{name}.rnn.bias_ih_l0"), g(f"{name}.rnn.bias_hh_l0")
        e.w_out = g(f"{name}.out.weight")
    T.pred_w, T.pred_b = g("pred_layer.weight"), g("pred_layer.bias")
    return T


def make_batch(batch: Dict[str, object], cfg: IntelConfig) -> Batch:
    """Pointer struct over the reference's batch dict (dtypes exactly as collate_batch delivers them)."""
    i64, f64 = torch.int64, torch.float64
    b = Batch()
    b.u_id = ptr(batch["u_id_c"], i64)
    b.i_id = ptr(batch["i_id_s"], i64)
    b.i_class = ptr(batch["i_class_c"], i64) if cfg.class_rows > 0 else None
    b.session_len = ptr(batch["session_len"], i64)
    b.scores = ptr(batch["scores"], f64)
    b.context_mh = ptr(batch["context_mh"], i64)
    b.his_context = ptr(batch["his_context_mh"], i64)
    b.history_len = ptr(batch["history_len"], i64)
    b.his_item_id = ptr(batch["his_item_id"], i64)
    if "his_intents_idx" in batch:       # opt-in compact layout (synthetic.make_batch(layout="compact"))
        b.his_intents_idx = ptr(batch["his_intents_idx"], torch.int32)
        b.his_intents_val = ptr(batch["his_intents_val"], torch.float32)
        b.nz1 = batch["his_intents_idx"].shape[2]
    else:
        b.his_intents = ptr(batch["his_intents"], f64)
    if "his_item_int_idx" in batch:
        b.his_item_int_idx = ptr(batch["his_item_int_idx"], torch.int32)
        b.his_item_int_val = ptr(batch["his_item_int_val"], torch.float32)
        b.nz2 = batch["his_item_int_idx"].shape[2]
    else:
        b.his_item_int = ptr(batch["his_item_int"], f64)
    b.history_item_len = ptr(batch["history_item_len"], i64)
    return b


BAD_INPUT_BITS = {1: "u_id_c outside uid_embeddings", 2: "i_id_s / his_item_id outside iid_embeddings",
                  4: "i_class_c outside item_embeddings", 8: "context_mh / his_context_mh outside context_embeddings",
                  16: "session_len outside [0, L]", 32: "history_len / history_item_len outside [1, H]",
                  64: "compact history intent index outside [0, intent_num)"}


def describe_bad_input(flags: int) -> str:
    return "; ".join(msg for bit, msg in BAD_INPUT_BITS.items() if flags & bit)


def profile(on) -> None:
    """True/1: per-kernel CUDA-event timing; 2: additionally one line per GEMM shape; False/0: off."""
    check(load().intel_profile_enable(int(on)))


def profile_report() -> Dict[str, Dict[str, float]]:
    """{kernel name: {launches, ms, bytes, flops}} of the launches recorded since profile(True)."""
    buf = C.create_string_buffer(1 << 16)
    check(load().intel_profile_report(buf, len(buf)))
    out: Dict[str, Dict[str, float]] = {}
    for line in buf.value.decode().splitlines():
        name, n, ms, by, fl = line.rsplit(None, 4)
        out[name] = {"launches": float(n), "ms": float(ms), "bytes": float(by), "flops": float(fl)}
    return out
