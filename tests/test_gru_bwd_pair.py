"""Backward recurrence of the two GRU encoders: one launch for both when both histories are length-sorted (T <= 63), one
launch each otherwise.  The gradients of every parameter (both encoders' w_ih, w_hh, b_ih, b_hh, w_out and the embedding
rows of the history tokens) are checked against the float64 oracle for length profiles the synthetic batches do not
reach: one encoder all at its longest and the other all at length 1, batches that are not a multiple of the 16-session
tile or smaller than one, and a history longer than 63 slots next to a sorted one.  Runs on the emulator and on the GPU;
the large GPU case is big enough for the products to walk the live-row lists, where the recurrence leaves the gradient
rows of padding slots unwritten."""
import os
import sys

import numpy as np
import pytest
import torch

import parity_checks as P
from conftest import LOSS_KW, assert_grad_close, rel_err
from oracle import intel_oracle as O

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "emu"))


def _lengths(profile, B, H, gen):
    if profile == "max":
        return torch.full((B,), H, dtype=torch.long)
    if profile == "one":
        return torch.ones(B, dtype=torch.long)
    lens = torch.randint(1, H + 1, (B,), generator=gen)
    lens[0] = H
    return lens


def _resize(x, T, mask):
    """x [B, H, ...] -> [B, T, ...]: slots tiled from the original ones, padding slots zeroed"""
    idx = torch.arange(T) % x.shape[1]
    y = x[:, idx]
    m = mask.reshape(mask.shape + (1,) * (y.dim() - 2)).to(y.dtype)
    return y * m


def _with_lengths(batch, his_len, item_len):
    """the batch with new history lengths: the history tensors take the width of the longest history"""
    b = dict(batch)
    for key_len, new, keys in (("history_len", his_len, ("his_context_mh", "his_intents", "his_intents_idx", "his_intents_val")),
                               ("history_item_len", item_len, ("his_item_id", "his_item_int", "his_item_int_idx", "his_item_int_val"))):
        T = int(new.max())
        mask = torch.arange(T)[None, :] < new[:, None]
        b[key_len] = new.clone()
        for k in keys:
            if k in b:
                b[k] = _resize(b[k], T, mask)
    b["position"] = his_len.clone()
    return b


def run_case(device, B, history_max, his_profile, item_profile, seed=0, L=7):
    from intel_sigir2023_b200 import losses, synthetic
    from intel_sigir2023_b200.config import IntelConfig
    corpus = synthetic.CorpusSpec(n_item=300, n_class=11, n_user=40, n_ctx=23, model_num=3, intent_num=48, history_max=history_max)
    cfg = IntelConfig(item_rows=corpus.item_rows, class_rows=corpus.n_class, user_rows=corpus.user_rows, ctx_rows=corpus.n_ctx,
                      intent_num=corpus.intent_num, model_num=corpus.model_num, history_max=history_max, encoder="GRU4Rec",
                      num_heads=2, num_layers=1)
    base = synthetic.make_batch(corpus, synthetic.BatchSpec(batch_size=B, max_len=L, min_len=3), seed=seed)
    gen = torch.Generator().manual_seed(seed + 7)
    batch_cpu = _with_lengths(base, _lengths(his_profile, B, history_max, gen), _lengths(item_profile, B, history_max, gen))
    state = O.init_state(cfg, seed=seed + 1)
    model = P.make_model(cfg, {k: v.to(device) for k, v in state.items()}, device).train()
    batch = {k: (v.to(device) if torch.is_tensor(v) else v) for k, v in batch_cpu.items()}
    crit = losses.IntListloss(P.loss_args())
    out = model(batch)
    loss, _, _ = crit(out, batch)
    loss.backward()
    sd = {k: v.clone().requires_grad_(True) for k, v in state.items()}
    ref = O.forward(sd, cfg, batch_cpu)
    rl, _, _ = O.total_loss("list", ref, batch_cpu, **LOSS_KW)
    rl.backward()
    assert rel_err(out["intents"].detach().cpu().numpy(), ref["intents"].detach().numpy()) < P.TOL
    gmax = max(float(p.grad.abs().max()) for p in sd.values() if p.grad is not None)
    for k, p in model.named_parameters():
        ref_g = sd[k].grad.numpy() if sd[k].grad is not None else np.zeros(tuple(p.shape), np.float32)
        assert_grad_close(p.grad.cpu().numpy(), ref_g, gmax, k)


# (B, history_max, session-history lengths, item-history lengths)
CASES = {
    "max_vs_one": (37, 20, "max", "one"),          # pair launch; the item history has no row longer than 1
    "one_vs_max": (9, 20, "one", "max"),           # fewer sessions than one tile
    "random_pair": (40, 20, "random", "random"),
    "unsorted_70": (21, 70, "random", "random"),   # T > 63: no length order, one launch per encoder
    "unsorted_vs_one": (18, 70, "max", "one"),     # one encoder sorted, the other not
}


@pytest.fixture(scope="module")
def emu_lib():
    from build_emu import build_emu
    from intel_sigir2023_b200 import _lib
    path = build_emu()
    old = (_lib._lib, _lib._allow_host_tensors)
    _lib._lib = None
    _lib.load(path)
    _lib._allow_host_tensors = True
    yield
    _lib._lib, _lib._allow_host_tensors = old


@pytest.mark.parametrize("name", sorted(CASES))
def test_gru_bwd_pair_emu(name, emu_lib):
    run_case("cpu", *CASES[name])


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_gru_bwd_pair_gpu(name):
    run_case("cuda", *CASES[name])


@pytest.mark.gpu
def test_gru_bwd_pair_gpu_live_rows():
    """B T >= 16 384 history rows: the products take the live-row lists and padding rows are not written"""
    run_case("cuda", 1100, 20, "random", "random", seed=3)
