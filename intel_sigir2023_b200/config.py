"""Shape/config record of the IntEL hot path.

Field names follow the reference's command-line flags (IntEL/src/models/IntEL/IntEL.py:17-34,
GeneralSeq.py:15-17, BaseModel.py:25) so an ``argparse.Namespace`` produced by the
reference's ``main.py`` converts 1:1 with :func:`IntelConfig.from_args`.
"""
from __future__ import annotations

from dataclasses import dataclass, asdict
from typing import Dict, Tuple


@dataclass(frozen=True)
class IntelConfig:
    # corpus-derived sizes (what the reader reports)
    item_rows: int            # corpus.max_iid + 1            (BaseModel.py:155)
    class_rows: int           # prod(corpus.itemfnum)         (IntEL.py:38)
    user_rows: int            # corpus.max_uid + 1            (BaseModel.py:154)
    ctx_rows: int             # prod(corpus.contextfnum)      (IntEL.py:99)
    intent_num: int           # len(corpus.zero_int)          (IntEL.py:39)
    model_num: int = 3        # --model_num
    # model flags with the reference defaults (IntEL.py:18-33)
    encoder: str = "BERT4Rec"
    context_emb_size: int = 16
    i_emb_size: int = 16
    u_emb_size: int = 32
    s_emb_size: int = 32
    im_emb_size: int = 16
    intent_emb_size: int = 16
    cross_attn_qsize: int = 32
    num_heads: int = 1
    num_layers: int = 1
    cross_attention: int = 1
    dropout: float = 0.0
    history_max: int = 20
    gru_hidden: int = 128     # GRU4RecEncoder(hidden_size=128)  (IntEL.py:105-106)
    bert_layers: int = 2      # BERT4RecEncoder(num_layers=2, num_heads=2) (IntEL.py:108-109)
    bert_heads: int = 2
    # --sparse_grad: 0 dense table gradients; 1 and 2 give the four embedding tables row-sparse (COO) gradients over the
    # rows a step names, with lazy Adam (1: unnamed rows keep their values) or exact Adam (2: bitwise dense Adam)
    sparse_grad: int = 0

    # ---- derived widths ----
    @property
    def d_item(self) -> int:           # item stream width (IntEL.py:59)
        return self.i_emb_size + (self.im_emb_size if self.class_rows > 0 else 0)

    @property
    def d_score(self) -> int:          # score stream width (IntEL.py:67)
        return self.s_emb_size

    @property
    def d_his(self) -> int:            # session-history token width (IntEL.py:102)
        return self.intent_emb_size + self.context_emb_size

    @property
    def d_his_item(self) -> int:       # item-history token width (IntEL.py:103)
        return self.intent_emb_size + self.i_emb_size

    @property
    def d_head(self) -> int:           # weight_embeddings input width (IntEL.py:95-96)
        return self.d_item + self.s_emb_size + self.intent_emb_size + self.u_emb_size

    @property
    def d_pred(self) -> int:           # pred_layer input width (IntEL.py:112-115)
        return self.d_his + self.d_his_item + self.context_emb_size + self.u_emb_size

    @staticmethod
    def from_args(args, corpus) -> "IntelConfig":
        """Build from the reference's ``args`` namespace and reader ``corpus`` object."""
        def prod(xs):
            p = 1
            for x in xs:
                p *= int(x)
            return p
        g = lambda name, default: getattr(args, name, default)
        return IntelConfig(
            item_rows=int(corpus.max_iid + 1), class_rows=prod(corpus.itemfnum),
            user_rows=int(corpus.max_uid + 1), ctx_rows=prod(corpus.contextfnum),
            intent_num=len(corpus.zero_int), model_num=int(g("model_num", 2)),
            encoder=g("encoder", "BERT4Rec"), context_emb_size=g("context_emb_size", 16),
            i_emb_size=g("i_emb_size", 16), u_emb_size=g("u_emb_size", 32),
            s_emb_size=g("s_emb_size", 32), im_emb_size=g("im_emb_size", 16),
            intent_emb_size=g("intent_emb_size", 16), cross_attn_qsize=g("cross_attn_qsize", 32),
            num_heads=g("num_heads", 1), num_layers=g("num_layers", 1),
            cross_attention=int(g("cross_attention", 1)), dropout=float(g("dropout", 0.0)),
            history_max=int(g("history_max", 20)), sparse_grad=int(g("sparse_grad", 0)))

    def to_dict(self) -> Dict[str, object]:
        return asdict(self)

    def param_shapes(self) -> Dict[str, Tuple[int, ...]]:
        """``state_dict`` contract of the reference module (SURVEY.md 8b), key -> shape."""
        c = self
        di, ds, dint, I, K = c.d_item, c.d_score, c.intent_emb_size, c.intent_num, c.model_num
        s: Dict[str, Tuple[int, ...]] = {}
        s["iid_embeddings.weight"] = (c.item_rows, c.i_emb_size)
        if c.class_rows > 0:
            s["item_embeddings.weight"] = (c.class_rows, c.im_emb_size)
        s["uid_embeddings.weight"] = (c.user_rows, c.u_emb_size)
        s["intent_embeddings.weight"] = (dint, I)
        s["intent_embeddings.bias"] = (dint,)
        s["score_embeddings.weight"] = (ds, K)
        s["score_embeddings.bias"] = (ds,)
        for p, d in (("i", di), ("s", ds)):
            for n in "qkv":
                s[f"{p}_attn_head.{n}_linear.weight"] = (d, d)
            for n in ("W1", "W2"):
                s[f"{p}_{n}.weight"] = (d, d)
                s[f"{p}_{n}.bias"] = (d,)
            s[f"{p}_layer_norm.weight"] = (d,)
            s[f"{p}_layer_norm.bias"] = (d,)
        if c.cross_attention:
            for name, d in (("intent_score_attention", ds), ("intent_item_attention", di)):
                s[f"{name}.query_layer.weight"] = (d, I)
                s[f"{name}.key_layer.weight"] = (d, d)
                s[f"{name}.value_layer.weight"] = (d, d)
        else:
            for name, d in (("intent_score_embeddings", ds), ("intent_item_embeddings", di)):
                s[f"{name}.0.weight"] = (c.cross_attn_qsize, I)
                s[f"{name}.0.bias"] = (c.cross_attn_qsize,)
                s[f"{name}.2.weight"] = (d, c.cross_attn_qsize)
        s["weight_embeddings.weight"] = (K, c.d_head)
        s["weight_embeddings.bias"] = (K,)
        s["context_embeddings.weight"] = (c.ctx_rows, c.context_emb_size)
        for name, d in (("encoder", c.d_his), ("item_encoder", c.d_his_item)):
            if c.encoder == "GRU4Rec":
                h = c.gru_hidden
                s[f"{name}.rnn.weight_ih_l0"] = (3 * h, d)
                s[f"{name}.rnn.weight_hh_l0"] = (3 * h, h)
                s[f"{name}.rnn.bias_ih_l0"] = (3 * h,)
                s[f"{name}.rnn.bias_hh_l0"] = (3 * h,)
                s[f"{name}.out.weight"] = (d, h)
            elif c.encoder == "BERT4Rec":
                s[f"{name}.p_embeddings.weight"] = (c.history_max + 1, d)
                for l in range(c.bert_layers):
                    b = f"{name}.transformer_block.{l}"
                    for n in "qkv":
                        s[f"{b}.masked_attn_head.{n}_linear.weight"] = (d, d)
                        s[f"{b}.masked_attn_head.{n}_linear.bias"] = (d,)
                    for n in ("layer_norm1", "layer_norm2"):
                        s[f"{b}.{n}.weight"] = (d,)
                        s[f"{b}.{n}.bias"] = (d,)
                    for n in ("linear1", "linear2"):
                        s[f"{b}.{n}.weight"] = (d, d)
                        s[f"{b}.{n}.bias"] = (d,)
            else:
                raise ValueError("Invalid sequence encoder.")
        s["pred_layer.weight"] = (I, c.d_pred)
        s["pred_layer.bias"] = (I,)
        return s
