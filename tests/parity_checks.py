"""Parity checks shared by the emulator tests (CPU, kernel logic) and the GPU tests (the real thing).
Every check drives the product's Python host layer -> C ABI -> kernels and compares with the golden
vectors of the unmodified reference and with the CPU oracle."""
import argparse
import os

import numpy as np
import torch

from conftest import GOLDEN, LOSS_KW, assert_grad_close, load_model_case, rel_err
from oracle import intel_oracle as O

TOL = 1e-5   # north_star: scores / losses within 1e-5 relative (to the tensor's inf-norm), fp32


def loss_args(**kw):
    a = argparse.Namespace(**LOSS_KW)
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def make_model(cfg, state, device):
    from intel_sigir2023_b200.IntEL import IntEL
    args = argparse.Namespace(device=torch.device(device), model_path="", buffer=1)
    m = IntEL(args, cfg=cfg).to(device)
    missing = m.load_state_dict(state, strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    return m


def check_linear(device):
    from intel_sigir2023_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(0)
    for (M, N, K) in [(7, 5, 3), (130, 33, 17), (64, 64, 64), (300, 8, 40), (20, 100, 70), (3001, 32, 32), (2500, 24, 32), (200, 32, 1071), (130, 48, 300), (77, 9, 515), (300, 176, 600)]:
        A = torch.randn(M, K, generator=g).to(device)
        W = torch.randn(N, K, generator=g).to(device)
        b = torch.randn(N, generator=g).to(device)
        Cout = torch.empty(M, N, device=device)
        _lib.check(lib.intel_linear_fwd(M, N, K, _lib.ptr(A), _lib.ptr(W), _lib.ptr(b), _lib.ptr(Cout), _lib.stream_ptr(A.device)))
        ref = A.cpu() @ W.cpu().t() + b.cpu()
        assert rel_err(Cout.cpu().numpy(), ref.numpy()) < 2e-6, (M, N, K)


def check_linear_grads(device):
    """input / weight gradient GEMM variants on awkward shapes (tails in every dimension, split-K)."""
    from intel_sigir2023_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(2)
    for (M, N, K) in [(9, 5, 3), (1000, 33, 17), (4100, 32, 32), (257, 96, 40), (70, 130, 50), (150, 1071, 32), (90, 300, 24), (300, 600, 176)]:
        dY = torch.randn(M, N, generator=g).to(device)
        X = torch.randn(M, K, generator=g).to(device)
        W = torch.randn(N, K, generator=g).to(device)
        U = torch.randn(M, K, generator=g).to(device)
        st = _lib.stream_ptr(dY.device)
        dX = torch.empty(M, K, device=device)
        _lib.check(lib.intel_linear_dx(M, N, K, _lib.ptr(dY), _lib.ptr(W), _lib.ptr(dX), _lib.ptr(U), st))
        ref = (dY.cpu() @ W.cpu()) * (U.cpu() > 0)
        assert rel_err(dX.cpu().numpy(), ref.numpy()) < 2e-6, ("dx", M, N, K)
        dW = torch.zeros(N, K, device=device)
        db = torch.zeros(N, device=device)
        _lib.check(lib.intel_linear_dw(M, N, K, _lib.ptr(dY), _lib.ptr(X), _lib.ptr(dW), _lib.ptr(db), st))
        assert rel_err(dW.cpu().numpy(), (dY.cpu().t() @ X.cpu()).numpy()) < 3e-6, ("dw", M, N, K)
        assert rel_err(db.cpu().numpy(), dY.cpu().sum(0).numpy()) < 3e-6, ("db", M, N, K)


def check_linear_large(device):
    """shapes large enough for the tcgen05 / TMEM kernel (all three passes, tails in every dimension, split-K with
    atomics, relu / mask / bias epilogues), against float64 and against the mma.sync kernels"""
    from intel_sigir2023_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(7)
    st = _lib.stream_ptr(torch.device(device))
    for (M, N, K) in [(4096, 128, 256), (8192, 100, 176), (20000, 384, 48), (4099, 72, 1000), (4096, 1068, 176)]:
        X = torch.randn(M, K, generator=g).to(device)
        W = torch.randn(N, K, generator=g).to(device)
        b = torch.randn(N, generator=g).to(device)
        dY = torch.randn(M, N, generator=g).to(device)
        U = torch.randn(M, K, generator=g).to(device)
        ref_y = (X.double() @ W.double().t() + b.double()).cpu().numpy()
        ref_dx = ((dY.double() @ W.double()) * (U > 0)).cpu().numpy()
        ref_dw = (dY.double().t() @ X.double()).cpu().numpy()
        outs = []
        for on in (1, 0):
            _lib.check(lib.intel_debug_use_tcgen05_gemm(on))
            try:
                Y = torch.empty(M, N, device=device)
                _lib.check(lib.intel_linear_fwd(M, N, K, _lib.ptr(X), _lib.ptr(W), _lib.ptr(b), _lib.ptr(Y), st))
                dX = torch.empty(M, K, device=device)
                _lib.check(lib.intel_linear_dx(M, N, K, _lib.ptr(dY), _lib.ptr(W), _lib.ptr(dX), _lib.ptr(U), st))
                dW = torch.zeros(N, K, device=device)
                db = torch.zeros(N, device=device)
                _lib.check(lib.intel_linear_dw(M, N, K, _lib.ptr(dY), _lib.ptr(X), _lib.ptr(dW), _lib.ptr(db), st))
            finally:
                _lib.check(lib.intel_debug_use_tcgen05_gemm(1))
            assert rel_err(Y.cpu().numpy(), ref_y) < 3e-6, ("fwd", M, N, K, on)
            assert rel_err(dX.cpu().numpy(), ref_dx) < 3e-6, ("dx", M, N, K, on)
            assert rel_err(dW.cpu().numpy(), ref_dw) < 3e-6, ("dw", M, N, K, on)
            outs.append((Y, dX, dW))
        for a, c in zip(*outs):
            assert rel_err(a.cpu().numpy(), c.cpu().numpy()) < 4e-6


def check_rows_gemm(device):
    """the persistent warp-specialised tcgen05 kernel for tall products with a resident weight (gemm_rows_tc.cu): forward
    (several N blocks per row tile) and input gradient (several K chunks per block), ragged row / column tails, against
    float64 and against the generic kernel"""
    from intel_sigir2023_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(11)
    st = _lib.stream_ptr(torch.device(device))
    for (M, N, K) in [(20000, 384, 64), (16500, 384, 48), (33001, 96, 40), (81920, 384, 64), (86016, 384, 128), (17000, 128, 32)]:
        X = torch.randn(M, K, generator=g).to(device)
        W = torch.randn(N, K, generator=g).to(device)
        b = torch.randn(N, generator=g).to(device)
        dY = torch.randn(M, N, generator=g).to(device)
        ref_y = (X.double() @ W.double().t() + b.double()).cpu().numpy()
        ref_dx = (dY.double() @ W.double()).cpu().numpy()
        ref_dw = (dY.double().t() @ X.double()).cpu().numpy()
        outs = []
        for on in (1, 0):
            _lib.check(lib.intel_debug_use_rows_gemm(on))
            try:
                Y = torch.full((M, N), float("nan"), device=device)
                _lib.check(lib.intel_linear_fwd(M, N, K, _lib.ptr(X), _lib.ptr(W), _lib.ptr(b), _lib.ptr(Y), st))
                dX = torch.full((M, K), float("nan"), device=device)
                _lib.check(lib.intel_linear_dx(M, N, K, _lib.ptr(dY), _lib.ptr(W), _lib.ptr(dX), None, st))
                dW = torch.zeros(N, K, device=device)         # weight gradient: both operands contracted over the rows
                _lib.check(lib.intel_linear_dw(M, N, K, _lib.ptr(dY), _lib.ptr(X), _lib.ptr(dW), None, st))
            finally:
                _lib.check(lib.intel_debug_use_rows_gemm(1))
            assert rel_err(Y.cpu().numpy(), ref_y) < 3e-6, ("fwd", M, N, K, on, rel_err(Y.cpu().numpy(), ref_y))
            assert rel_err(dX.cpu().numpy(), ref_dx) < 3e-6, ("dx", M, N, K, on, rel_err(dX.cpu().numpy(), ref_dx))
            assert rel_err(dW.cpu().numpy(), ref_dw) < 3e-6, ("dw", M, N, K, on, rel_err(dW.cpu().numpy(), ref_dw))
            outs.append((Y, dX, dW))
        for a, c in zip(*outs):
            assert rel_err(a.cpu().numpy(), c.cpu().numpy()) < 4e-6


def check_mha(device, shapes=((3, 12, 32, 2), (2, 50, 32, 2), (2, 100, 32, 1), (1, 130, 48, 2))):
    """attention core vs torch on list lengths that span several 64-row query blocks, with and without key masks."""
    from intel_sigir2023_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(4)
    for (B, T, d, h) in shapes:
        for masked in (False, True):
            qkv = torch.randn(B, T, 3 * d, generator=g)
            lens = torch.randint(1, T + 1, (B,), generator=g) if masked else None
            dO = torch.randn(B, T, d, generator=g)
            q = qkv.clone().requires_grad_(True)
            dk = d // h
            Q, K, V = (q[:, :, i * d:(i + 1) * d].view(B, T, h, dk).transpose(1, 2) for i in range(3))
            s = Q @ K.transpose(-1, -2) / dk ** 0.5
            if masked:
                keym = torch.arange(T)[None, :] < lens[:, None]
                s = s.masked_fill(~keym[:, None, None, :], float("-inf"))
            ref = (s.softmax(-1) @ V).transpose(1, 2).reshape(B, T, d)
            ref.backward(dO)
            qd, dOd = qkv.to(device), dO.to(device)
            ld = lens.to(device) if masked else None
            out = torch.empty(B, T, d, device=device)
            dq = torch.empty(B, T, 3 * d, device=device)
            st = _lib.stream_ptr(qd.device)
            _lib.check(lib.intel_mha_fwd(B, T, d, h, _lib.ptr(qd), _lib.ptr(ld), _lib.ptr(out), st))
            _lib.check(lib.intel_mha_bwd(B, T, d, h, _lib.ptr(qd), _lib.ptr(ld), _lib.ptr(dOd), _lib.ptr(dq), st))
            assert rel_err(out.cpu().numpy(), ref.detach().numpy()) < 3e-6, ("fwd", B, T, d, h, masked)
            assert rel_err(dq.cpu().numpy(), q.grad.numpy()) < 1e-5, ("bwd", B, T, d, h, masked)


def check_gather_scatter(device):
    from intel_sigir2023_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(1)
    for d in (16, 32, 6):
        table = torch.randn(11, d, generator=g).to(device)
        idx = torch.randint(0, 11, (37,), generator=g).to(device)
        out = torch.empty(37, d, device=device)
        _lib.check(lib.intel_gather_fwd(37, d, _lib.ptr(table), _lib.ptr(idx), _lib.ptr(out), d, 0, _lib.stream_ptr(out.device)))
        assert torch.equal(out.cpu(), table.cpu()[idx.cpu()])          # index work: bit exact
        gout = torch.randn(37, d, generator=g).to(device)
        gt = torch.zeros(11, d, device=device)
        _lib.check(lib.intel_scatter_add_bwd(37, d, _lib.ptr(gout), d, _lib.ptr(idx), _lib.ptr(gt), _lib.stream_ptr(out.device)))
        ref = torch.zeros(11, d).index_add_(0, idx.cpu(), gout.cpu())
        assert rel_err(gt.cpu().numpy(), ref.numpy()) < 1e-6


def check_forward(name, device):
    cfg, batch, state, gold = load_model_case(name, device)
    model = make_model(cfg, state, device).eval()
    with torch.no_grad():
        out = model(batch)
    cpu_batch = {k: (v.cpu() if torch.is_tensor(v) else v) for k, v in batch.items()}
    ora = O.forward({k: v.cpu() for k, v in state.items()}, cfg, cpu_batch)
    for k in ("intents", "weights", "ens_score"):
        got = out[k].cpu().numpy()
        assert got.shape == gold["out." + k].shape, k
        assert rel_err(got, gold["out." + k]) < TOL, (name, k, "vs reference golden", rel_err(got, gold["out." + k]))
        assert rel_err(got, ora[k].numpy()) < TOL, (name, k, "vs oracle")
    # per-session rankings identical to the reference's (no exact ties in these fixtures)
    n = cpu_batch["session_len"].numpy()
    for b in range(len(n)):
        a = np.argsort(-out["ens_score"][b, :n[b]].cpu().numpy(), kind="stable")
        r = np.argsort(-gold["out.ens_score"][b, :n[b]], kind="stable")
        gaps = np.abs(np.diff(np.sort(gold["out.ens_score"][b, :n[b]])))
        if gaps.size == 0 or gaps.min() > 1e-4:
            assert np.array_equal(a, r), (name, b)


def check_backward(name, kind, device):
    from intel_sigir2023_b200 import losses
    cfg, batch, state, gold = load_model_case(name, device)
    model = make_model(cfg, state, device).train()
    crit = {"list": losses.IntListloss, "bpr": losses.IntBPRloss, "mse": losses.IntMSEloss}[kind](loss_args())
    if kind == "bpr":
        crit.bpr_noise = torch.from_numpy(gold["bpr_noise"]).to(device)
    out = model(batch)
    loss, ens_l, int_l = crit(out, batch)
    got = np.array([loss.item(), ens_l.item(), int_l.item()])
    ref = gold[f"loss.{kind}"]
    assert np.allclose(got, ref, rtol=TOL, atol=1e-7), (name, kind, got, ref)
    loss.backward()
    names = [n for n, _ in model.named_parameters()]
    gmax = max(np.abs(gold[f"grad.{kind}.{k}"]).max() for k in names)
    for k, p in model.named_parameters():
        assert p.grad is not None, k
        assert_grad_close(p.grad.cpu().numpy(), gold[f"grad.{kind}.{k}"], gmax, f"{name}/{kind}/{k}")


def check_loss_edge_cases(device):
    """no-diversity variants, a session without positives (NaN like the reference), in-kernel BPR RNG."""
    from intel_sigir2023_b200 import losses
    cfg, batch, state, gold = load_model_case("default_bert", device)
    cpu_batch = {k: (v.cpu() if torch.is_tensor(v) else v) for k, v in batch.items()}
    out = {"ens_score": torch.from_numpy(gold["out.ens_score"]).to(device).requires_grad_(True),
           "weights": torch.from_numpy(gold["out.weights"]).to(device).requires_grad_(True),
           "intents": torch.from_numpy(gold["out.intents"]).to(device).requires_grad_(True)}
    for kind, cls in (("list", losses.Listloss), ("mse", losses.MSEloss), ("bpr", losses.BPRloss)):
        crit = cls(loss_args(cal_diversity=0))
        noise = torch.from_numpy(gold["bpr_noise"])
        crit.bpr_noise = noise.to(device)
        l, _, _ = crit(out, batch)
        o = {k: v.detach().cpu().requires_grad_(True) for k, v in out.items()}
        if kind == "list":
            ref = O.list_loss(o, cpu_batch, 0, 0.0)
        elif kind == "mse":
            ref = O.mse_loss(o, cpu_batch, 0, 0.0)
        else:
            ref = O.bpr_loss(o, cpu_batch, 0, 0.0, noise)
        assert abs(l.item() - ref.item()) <= TOL * abs(ref.item()) + 1e-7, (kind, l.item(), ref.item())
        out["ens_score"].grad = None
        l.backward()
        ref.backward()
        assert rel_err(out["ens_score"].grad.cpu().numpy(), o["ens_score"].grad.numpy()) < 1e-4, kind
    # in-kernel RNG: finite, and differs from seed to seed only through the negative choice
    crit = losses.BPRloss(loss_args(cal_diversity=1))
    l1, _, _ = crit(out, batch)
    assert np.isfinite(l1.item())
    # a session with no positive item: 0/0 -> NaN, as in the reference (Listloss.py:14)
    nb = dict(batch)
    nb["ranking"] = batch["ranking"].clone()
    nb["ranking"][1] = 0
    l, _, _ = losses.Listloss(loss_args(cal_diversity=0))(out, nb)
    assert np.isnan(l.item())
    # intent loss soft branch (prediction with an exact zero, BaseIntloss.py:32-35)
    p = out["intents"].detach().clone()
    p[0, 0] = 0.0
    il = losses._IntentLossFn.apply(p.requires_grad_(True), batch["intents"], 0.5, 2.0)
    ref, ce, kl = O.intent_loss(p.detach().cpu().requires_grad_(True), cpu_batch["intents"], 0.5, 2.0)
    assert np.allclose(il.detach().cpu().numpy(), [ref.item(), ce.item(), kl.item()], rtol=TOL), (il, ref, ce, kl)


def check_list_loss_forms(device, B=37, L=41, K=4, seed=5):
    """the rank-bucket (O(L K)) Plackett-Luce kernel on ragged sessions with ties, empty levels, unlabeled (-1) slots and pad
    positives, and the pair form it falls back to when a session has more than three rank levels: both against the oracle's
    literal [B,L,L,K] restatement of Listloss.py:12-43 (loss, d ens_score, d weights)"""
    from intel_sigir2023_b200 import losses
    g = torch.Generator().manual_seed(seed)
    for levels in (3, 5):
        n = torch.randint(1, L + 1, (B,), generator=g)
        n[0], n[1] = L, 1
        ranking = torch.randint(-1, levels + 1, (B, L), generator=g)
        ranking[2] = torch.where(ranking[2] > 0, 2, 0)                    # a single positive level
        ranking[3, : int(n[3])] = 1                                       # only positives: nothing ranked below them
        ranking[:, 0] = torch.maximum(ranking[:, 0], torch.ones(B, dtype=torch.long))      # every session has a positive
        valid = torch.arange(L)[None, :] < n[:, None]
        batch = {"ranking": ranking, "session_len": n, "scores": torch.rand(B, L, K, generator=g, dtype=torch.float64) * valid[:, :, None],
                 "batch_size": B}
        out = {"ens_score": (torch.randn(B, L, generator=g) * 1.5 * valid).requires_grad_(True),
               "weights": torch.randn(B, L, K, generator=g).requires_grad_(True)}
        ref = O.list_loss(out, batch, 1, 0.07)
        ref.backward()
        dev_out = {k: v.detach().to(device).requires_grad_(True) for k, v in out.items()}
        dev_batch = {k: (v.to(device) if torch.is_tensor(v) else v) for k, v in batch.items()}
        l, _, _ = losses.Listloss(loss_args(cal_diversity=1, diversity_alpha=0.07))(dev_out, dev_batch)
        l.backward()
        assert abs(l.item() - ref.item()) <= TOL * abs(ref.item()) + 1e-7, (levels, l.item(), ref.item())
        for k in ("ens_score", "weights"):
            assert rel_err(dev_out[k].grad.cpu().numpy(), out[k].grad.numpy()) < 2e-5, (levels, k)


def check_evaluate(tag, device):
    from intel_sigir2023_b200 import evaluate
    z = np.load(f"{GOLDEN}/eval.npz")
    pos = {k: z[f"{tag}.pos.{k}"] for k in ("c_paynum_i", "c_favnum_i", "c_clicknum_i")}
    topk, metrics = [3, 1, 5, 10], ["NDCG", "HR"]
    res = evaluate.evaluate_method(list(z[f"{tag}.pred"]), list(z[f"{tag}.ranking"]), pos, topk, metrics,
                                   z[f"{tag}.session_len"], device=device)
    ora = O.evaluate_method(list(z[f"{tag}.pred"]), list(z[f"{tag}.ranking"]), pos, topk, metrics, z[f"{tag}.session_len"])
    assert set(res.keys()) == set(ora.keys())
    for k, v in ora.items():       # same tie rule as the oracle: every key, including fav_*
        assert (np.isnan(v) and np.isnan(res[k])) or abs(res[k] - v) < 1e-9, (tag, k, res[k], v)
    for k in res:                  # and the reference itself wherever it is well defined
        if k.startswith("fav_") and tag != "B":
            continue
        ref = float(z[f"{tag}.metric.{k}"])
        assert (np.isnan(ref) and np.isnan(res[k])) or abs(res[k] - ref) < 1e-6, (tag, k, res[k], ref)


def check_evaluate_ties(device):
    """exact ties (zero scores vs pad slots, duplicated scores): the documented stable tie rule == oracle."""
    from intel_sigir2023_b200 import evaluate
    z = np.load(f"{GOLDEN}/eval.npz")
    pred = z["A.pred"].copy()
    pred = np.round(pred * 4) / 4          # many duplicates, including exact zeros
    pos = {k: z[f"A.pos.{k}"] for k in ("c_paynum_i", "c_favnum_i", "c_clicknum_i")}
    topk, metrics = [3, 1, 5, 10], ["NDCG", "HR"]
    res = evaluate.evaluate_method(list(pred), list(z["A.ranking"]), pos, topk, metrics, z["A.session_len"], device=device)
    ora = O.evaluate_method(list(pred), list(z["A.ranking"]), pos, topk, metrics, z["A.session_len"])
    for k, v in ora.items():
        assert (np.isnan(v) and np.isnan(res[k])) or abs(res[k] - v) < 1e-9, (k, res[k], v)


def check_evaluate_intents(device):
    from intel_sigir2023_b200 import evaluate
    z = np.load(f"{GOLDEN}/eval.npz")
    res = evaluate.evaluate_intents(z["I.true"], z["I.pred"], topk=[1, 3, 5, 10, 30], device=device)
    for k, v in res.items():
        assert abs(v - float(z[f"I.metric.{k}"])) < 1e-6, (k, v)
    # config-3 shape (12 intent classes): the reference's default cut-offs [1,5,10,30] fail on a numpy broadcast
    # (BaseRunner.py:142-144, verified against the unmodified method); cut-offs <= I work and match the oracle
    import pytest
    t12 = z["I.true"][:, :12] + 1e-3
    t12 = t12 / t12.sum(axis=1, keepdims=True)
    p12 = z["I.pred"][:, :12] / z["I.pred"][:, :12].sum(axis=1, keepdims=True)
    with pytest.raises(ValueError):
        evaluate.evaluate_intents(t12, p12, topk=[1, 5, 10, 30], device=device)
    with pytest.raises(ValueError):
        O.evaluate_intents(t12, p12, [1, 5, 10, 30])
    got, ref = evaluate.evaluate_intents(t12, p12, topk=[1, 3, 5, 10], device=device), O.evaluate_intents(t12, p12, [1, 3, 5, 10])
    for k, v in ref.items():
        assert abs(got[k] - v) < 1e-6, (k, got[k], v)


def check_baselines(device):
    from intel_sigir2023_b200 import baselines
    z = np.load(f"{GOLDEN}/eval.npz")
    batch = {"scores": torch.from_numpy(z["F.scores"]).to(device)}
    s = baselines.SingleSort(choose_list="pCVR")(batch)["ens_score"].cpu().numpy()
    assert np.array_equal(s, z["F.single_pCVR"])
    b = baselines.Borda()(batch)["ens_score"].cpu().numpy()
    assert np.allclose(b, O.borda({"scores": torch.from_numpy(z["F.scores"])})["ens_score"].numpy(), rtol=1e-6, atol=0)
    untied = (z["F.scores"] > 0).all(axis=2)
    assert np.allclose(b[untied], z["F.borda"][untied])
    raw = torch.rand(z["F.scores"].shape, generator=torch.Generator().manual_seed(3))
    r = baselines.RandomFusion()(batch, raw.to(device))["ens_score"].cpu().numpy()
    ref = O.random_fusion({"scores": torch.from_numpy(z["F.scores"])}, raw)["ens_score"].numpy()
    assert rel_err(r, ref) < 1e-6


def check_against_oracle(device, seed=0, B=70, L=21, min_len=3, kind="list", corpus_kw=None, **cfg_kw):
    """Seeded synthetic batch + random weights: product (forward, loss, parameter gradients) vs the CPU oracle.
    Used for shapes the golden fixtures do not cover (B beyond one CTA tile, long lists, other widths)."""
    from intel_sigir2023_b200 import losses, synthetic
    from intel_sigir2023_b200.config import IntelConfig
    ck = dict(n_item=300, n_class=11, n_user=40, n_ctx=23, model_num=3, intent_num=48, history_max=9)
    ck.update(corpus_kw or {})
    corpus = synthetic.CorpusSpec(**ck)
    cfg = IntelConfig(item_rows=corpus.item_rows, class_rows=corpus.n_class, user_rows=corpus.user_rows,
                      ctx_rows=corpus.n_ctx, intent_num=corpus.intent_num, model_num=corpus.model_num,
                      history_max=corpus.history_max, **cfg_kw)
    batch_cpu = synthetic.make_batch(corpus, synthetic.BatchSpec(batch_size=B, max_len=L, min_len=min_len), seed=seed)
    state = O.init_state(cfg, seed=seed + 1)
    model = make_model(cfg, {k: v.to(device) for k, v in state.items()}, device).train()
    batch = {k: (v.to(device) if torch.is_tensor(v) else v) for k, v in batch_cpu.items()}
    crit = {"list": losses.IntListloss, "bpr": losses.IntBPRloss, "mse": losses.IntMSEloss}[kind](loss_args())
    noise = torch.rand(B, L, L, generator=torch.Generator().manual_seed(seed))
    crit.bpr_noise = noise.to(device)
    out = model(batch)
    loss, _, _ = crit(out, batch)
    loss.backward()
    sd = {k: v.clone().requires_grad_(True) for k, v in state.items()}
    ref = O.forward(sd, cfg, batch_cpu)
    rl, _, _ = O.total_loss(kind, ref, batch_cpu, noise=noise, **LOSS_KW)
    rl.backward()
    for k in ("intents", "weights", "ens_score"):
        assert rel_err(out[k].detach().cpu().numpy(), ref[k].detach().numpy()) < TOL, (k, cfg_kw)
    assert abs(loss.item() - rl.item()) <= TOL * abs(rl.item()) + 1e-7, (loss.item(), rl.item())
    gmax = max(float(p.grad.abs().max()) for p in sd.values() if p.grad is not None)
    for k, p in model.named_parameters():
        ref_g = sd[k].grad.numpy() if sd[k].grad is not None else np.zeros(tuple(p.shape), np.float32)
        assert_grad_close(p.grad.cpu().numpy(), ref_g, gmax, f"{k} {cfg_kw}")


C3_MODEL = dict(encoder="GRU4Rec", num_heads=2, num_layers=2, context_emb_size=32, intent_emb_size=32, cross_attn_qsize=64)


def check_config3_shapes(device, intent_num, B=6, kind="list"):
    """BASELINE.json configs[2] (LifeData-shaped, SURVEY.md 8d): K = 2 basic lists, four context features with
    cardinalities (24,7,16,8) -> 21 504 context rows, I = 12 (the code hint) or 2048 (the stress size), L = 50, the
    script's GRU4Rec sizes: forward, loss and every parameter gradient against the oracle"""
    check_against_oracle(device, seed=3, B=B, L=50, min_len=20, kind=kind,
                         corpus_kw=dict(model_num=2, intent_num=intent_num, n_ctx=24 * 7 * 16 * 8, history_max=20, n_item=500,
                                        n_user=60), **C3_MODEL)


def check_compact_layout(device):
    """the opt-in index form of his_intents / his_item_int gives the same forward and gradients as the dense API"""
    from intel_sigir2023_b200 import losses, synthetic
    from intel_sigir2023_b200.config import IntelConfig
    corpus = synthetic.CorpusSpec(n_item=200, n_class=9, n_user=30, n_ctx=19, model_num=3, intent_num=40, history_max=6)
    for enc in ("GRU4Rec", "BERT4Rec"):
        cfg = IntelConfig(item_rows=corpus.item_rows, class_rows=corpus.n_class, user_rows=corpus.user_rows,
                          ctx_rows=corpus.n_ctx, intent_num=corpus.intent_num, model_num=3, history_max=6, encoder=enc,
                          num_heads=2)
        both = synthetic.make_batch(corpus, synthetic.BatchSpec(batch_size=11, max_len=13, min_len=2), seed=5, layout="both")
        both = {k: (v.to(device) if torch.is_tensor(v) else v) for k, v in both.items()}
        dense = {k: v for k, v in both.items() if not k.endswith(("_idx", "_val"))}
        compact = {k: v for k, v in both.items() if k not in ("his_intents", "his_item_int")}
        state = O.init_state(cfg, seed=3)
        res = []
        for b in (dense, compact):
            model = make_model(cfg, {k: v.to(device) for k, v in state.items()}, device).train()
            out = model(b)
            loss, _, _ = losses.IntListloss(loss_args())(out, b)
            loss.backward()
            res.append((out, loss, {k: p.grad.clone() for k, p in model.named_parameters()}))
        for k in ("intents", "weights", "ens_score"):
            assert rel_err(res[1][0][k].detach().cpu().numpy(), res[0][0][k].detach().cpu().numpy()) < 2e-6, (enc, k)
        gmax = max(float(g.abs().max()) for g in res[0][2].values())
        for k, g in res[0][2].items():
            assert_grad_close(res[1][2][k].cpu().numpy(), g.cpu().numpy(), gmax, f"{enc}/{k}")


def _fresh(cfg, state, device, batch, train=True, fused=True, drop_step=0):
    from intel_sigir2023_b200 import _lib, losses
    _lib.check(_lib.load().intel_debug_use_fused_stack(1 if fused else 0))
    try:
        model = make_model(cfg, {k: v.to(device) for k, v in state.items()}, device)
        model.train(train)
        model._drop_seed, model._drop_step = 1234, drop_step
        out = model(batch)
        loss, _, _ = losses.IntListloss(loss_args())(out, batch)
        loss.backward()
        return out, loss, {k: p.grad.clone() for k, p in model.named_parameters()}
    finally:
        _lib.check(_lib.load().intel_debug_use_fused_stack(1))


def check_fused_vs_staged(device, dropout=0.0, B=19, L=23, heads=2, layers=2, sessions_per_cta=4):
    """the fused per-session stack kernel and the staged kernels implement the same math (also under dropout:
    both draw the mask from the same counter-based hash)"""
    from intel_sigir2023_b200 import synthetic
    from intel_sigir2023_b200.config import IntelConfig
    corpus = synthetic.CorpusSpec(n_item=200, n_class=9, n_user=30, n_ctx=19, model_num=3, intent_num=40, history_max=6)
    cfg = IntelConfig(item_rows=corpus.item_rows, class_rows=corpus.n_class, user_rows=corpus.user_rows, ctx_rows=corpus.n_ctx,
                      intent_num=corpus.intent_num, model_num=3, history_max=6, encoder="GRU4Rec", num_heads=heads,
                      num_layers=layers, dropout=dropout)
    batch = synthetic.make_batch(corpus, synthetic.BatchSpec(batch_size=B, max_len=L, min_len=min(2, L)), seed=8)
    batch = {k: (v.to(device) if torch.is_tensor(v) else v) for k, v in batch.items()}
    state = O.init_state(cfg, seed=4)
    from intel_sigir2023_b200 import _lib
    _lib.check(_lib.load().intel_debug_stack_sessions_per_cta(sessions_per_cta))
    try:
        a = _fresh(cfg, state, device, batch, fused=True)
    finally:
        _lib.check(_lib.load().intel_debug_stack_sessions_per_cta(4))
    b = _fresh(cfg, state, device, batch, fused=False)
    for k in ("intents", "weights", "ens_score"):
        assert rel_err(a[0][k].detach().cpu().numpy(), b[0][k].detach().cpu().numpy()) < 5e-6, (k, dropout)
    gmax = max(float(g.abs().max()) for g in b[2].values())
    for k, g in b[2].items():
        assert_grad_close(a[2][k].cpu().numpy(), g.cpu().numpy(), gmax, f"{k} p={dropout}", rtol=2e-4, afrac=3e-6)
    return cfg, state, batch, a


def check_tc_stack(device, cases=((10, 30, 2, 2), (7, 50, 2, 2), (5, 64, 1, 1), (9, 17, 1, 2))):
    """the tcgen05 / tensor-memory forward kernel of the fused stack (trunk_tc.cu) against the mma.sync kernel (trunk.cu):
    outputs, and the gradients the (shared) backward kernel computes from the activations each of them saved"""
    from intel_sigir2023_b200 import _lib
    for (B, L, heads, layers) in cases:
        cfg, state, batch, a = check_fused_vs_staged(device, B=B, L=L, heads=heads, layers=layers)
        _lib.check(_lib.load().intel_debug_use_tcgen05_stack(0))
        try:
            b = _fresh(cfg, state, device, batch, fused=True)
        finally:
            _lib.check(_lib.load().intel_debug_use_tcgen05_stack(1))
        for k in ("intents", "weights", "ens_score"):
            assert rel_err(a[0][k].detach().cpu().numpy(), b[0][k].detach().cpu().numpy()) < 5e-6, (k, B, L, heads, layers)
        gmax = max(float(g.abs().max()) for g in b[2].values())
        for k, g in b[2].items():
            assert_grad_close(a[2][k].cpu().numpy(), g.cpu().numpy(), gmax, f"{k} {(B, L, heads, layers)}", rtol=2e-4, afrac=3e-6)


def check_gru_tc(device, B=300, L=9, history_max=11):
    """the tcgen05 cluster kernel of the GRU recurrence (gru_tc.cu) against the mma.sync kernel (gru.cu): several session
    tiles with a ragged tail, history lengths 1..H, outputs and every parameter gradient.  Histories longer than 63 slots
    run without the length-sorted order, forward and backward."""
    from intel_sigir2023_b200 import _lib, synthetic
    from intel_sigir2023_b200.config import IntelConfig
    corpus = synthetic.CorpusSpec(n_item=200, n_class=9, n_user=30, n_ctx=19, model_num=3, intent_num=40, history_max=history_max)
    cfg = IntelConfig(item_rows=corpus.item_rows, class_rows=corpus.n_class, user_rows=corpus.user_rows, ctx_rows=corpus.n_ctx,
                      intent_num=corpus.intent_num, model_num=3, history_max=history_max, encoder="GRU4Rec", num_heads=2, num_layers=1,
                      context_emb_size=32, intent_emb_size=32)
    batch = synthetic.make_batch(corpus, synthetic.BatchSpec(batch_size=B, max_len=L, min_len=2), seed=21)
    batch = {k: (v.to(device) if torch.is_tensor(v) else v) for k, v in batch.items()}
    state = O.init_state(cfg, seed=9)
    a = _fresh(cfg, state, device, batch)
    _lib.check(_lib.load().intel_debug_use_tcgen05_gru(0))
    try:
        b = _fresh(cfg, state, device, batch)
    finally:
        _lib.check(_lib.load().intel_debug_use_tcgen05_gru(1))
    for k in ("intents", "weights", "ens_score"):
        assert rel_err(a[0][k].detach().cpu().numpy(), b[0][k].detach().cpu().numpy()) < 5e-6, k
    gmax = max(float(g.abs().max()) for g in b[2].values())
    for k, g in b[2].items():
        assert_grad_close(a[2][k].cpu().numpy(), g.cpu().numpy(), gmax, k, rtol=2e-5, afrac=3e-6)


def check_fused_shapes(device, cases=((5, 7, 2, 1, 1), (9, 16, 1, 2, 2), (7, 40, 2, 1, 4), (6, 50, 2, 2, 3), (5, 64, 1, 1, 2),
                                      (4, 70, 2, 2, 4), (3, 100, 1, 1, 4), (3, 128, 2, 1, 4), (10, 30, 2, 2, 4),
                                      (3, 200, 1, 1, 4), (2, 150, 2, 2, 4), (3, 208, 2, 1, 4), (2, 129, 1, 2, 4))):
    """every padded-length / head-count instantiation of the fused stack kernels, and every sessions-per-CTA
    setting, against the staged kernels: cases are (B, L, heads, layers, sessions per CTA)"""
    for (B, L, heads, layers, ns) in cases:
        check_fused_vs_staged(device, B=B, L=L, heads=heads, layers=layers, sessions_per_cta=ns)


def check_dropout(device):
    """training-mode dropout: deterministic per (seed, step), off in eval mode, changes the output, unbiased scale,
    and the backward pass uses the same mask (directional finite difference with the mask held fixed)."""
    from intel_sigir2023_b200 import losses
    cfg, state, batch, a = check_fused_vs_staged(device, dropout=0.3)
    again = _fresh(cfg, state, device, batch)
    assert torch.equal(a[0]["ens_score"], again[0]["ens_score"])                      # same seed and step -> same mask
    other = _fresh(cfg, state, device, batch, drop_step=7)
    assert not torch.equal(a[0]["ens_score"], other[0]["ens_score"])                  # new step -> new mask
    ev = _fresh(cfg, state, device, batch, train=False)
    import dataclasses
    cfg0 = dataclasses.replace(cfg, dropout=0.0)
    ref = _fresh(cfg0, state, device, batch)
    assert torch.equal(ev[0]["ens_score"], ref[0]["ens_score"])                       # eval mode: no dropout
    assert not torch.equal(a[0]["ens_score"], ref[0]["ens_score"])
    # finite differences along a random direction of the stack weights, mask fixed by (seed, step)
    g = torch.Generator().manual_seed(0)
    keys = [k for k in state if k.startswith(("i_", "s_"))]
    direction = {k: torch.randn(state[k].shape, generator=g) for k in keys}
    analytic = sum(float((a[2][k].cpu().double() * direction[k].double()).sum()) for k in keys)
    eps = 2e-3
    lp = _fresh(cfg, {k: (v + eps * direction[k] if k in direction else v) for k, v in state.items()}, device, batch)[1]
    lm = _fresh(cfg, {k: (v - eps * direction[k] if k in direction else v) for k, v in state.items()}, device, batch)[1]
    num = (lp.item() - lm.item()) / (2 * eps)
    assert abs(analytic - num) <= 3e-2 * abs(num) + 1e-4, (analytic, num)


def check_adam(device, steps=4):
    """optim.Adam (one fused launch) against torch.optim.Adam with the reference's two parameter groups (L2 on the
    weights, none on the biases), several steps, including a StepLR decay and a state_dict round trip"""
    from intel_sigir2023_b200 import optim
    g = torch.Generator().manual_seed(3)

    def make():
        torch.manual_seed(0)
        m = torch.nn.Module()
        m.emb = torch.nn.Embedding(257, 16)
        m.table = torch.nn.Embedding(9001, 32)          # > 2^18 elements: the one-launch-per-table path
        m.lin = torch.nn.Linear(33, 7)
        m.odd = torch.nn.Parameter(torch.randn(5, 3, 2))
        return m.to(device)
    ma, mb = make(), make()
    oa = optim.Adam(optim.customize_parameters(ma), lr=3e-3, weight_decay=1e-4)
    ob = torch.optim.Adam(optim.customize_parameters(mb), lr=3e-3, weight_decay=1e-4)
    sa = torch.optim.lr_scheduler.StepLR(oa, step_size=2, gamma=0.5)
    sb = torch.optim.lr_scheduler.StepLR(ob, step_size=2, gamma=0.5)
    for it in range(steps):
        for (na, pa), (nb, pb) in zip(ma.named_parameters(), mb.named_parameters()):
            gr = torch.randn(pa.shape, generator=g).to(device)
            pa.grad, pb.grad = gr.clone(), gr.clone()
        oa.step(); ob.step(); sa.step(); sb.step()
        if it == 1:                         # interchangeable state
            import copy
            oa.load_state_dict(copy.deepcopy(ob.state_dict()))     # (load_state_dict keeps references to the step tensors)
    for (na, pa), (nb, pb) in zip(ma.named_parameters(), mb.named_parameters()):
        assert rel_err(pa.detach().cpu().numpy(), pb.detach().cpu().numpy()) < 2e-6, na
        ea, eb = oa.state[pa]["exp_avg_sq"], ob.state[pb]["exp_avg_sq"]
        assert rel_err(ea.cpu().numpy(), eb.cpu().numpy()) < 2e-6, na


def load_awelv_case(device="cpu"):
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "awelv.npz"))
    batch = {k[6:]: torch.from_numpy(z[k]).to(device) for k in z.files if k.startswith("batch.")}
    batch["batch_size"] = int(batch["i_id_s"].shape[0])
    state = {k[6:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("state.")}
    return z, batch, state


def check_awelv(device):
    """baselines.aWELv (one fused kernel per direction) + Listloss with the diversity term against arrays produced by the
    unmodified reference model (oracle/make_golden.py:make_awelv)"""
    import argparse
    from intel_sigir2023_b200 import baselines, losses
    z, batch, state = load_awelv_case(device)
    args = argparse.Namespace(hidden_size=int(z["hidden_size"][0]), model_num=int(z["model_num"][0]), device=device)
    model = baselines.aWELv(args, user_num=int(z["user_rows"][0]))
    model.load_state_dict(state)
    model = model.to(device)
    out = model(batch)
    assert rel_err(out["weights"].detach().cpu().numpy(), z["out.weights"]) < TOL
    assert rel_err(out["ens_score"].detach().cpu().numpy(), z["out.ens_score"]) < TOL
    crit = losses.Listloss(argparse.Namespace(cal_diversity=1, diversity_alpha=0.05, intent_weight=0.1, ensemble_weight=1.0,
                                              kl_weight=0.5, kl_temp=2.0))
    loss = crit(out, batch)
    loss = loss[0] if isinstance(loss, (tuple, list)) else loss
    assert abs(float(loss.detach()) - float(z["loss.list"][0])) <= TOL * abs(float(z["loss.list"][0]))
    loss.backward()
    gmax = max(float(np.abs(z["grad.list." + n]).max()) for n, _ in model.named_parameters())
    for n, p in model.named_parameters():
        assert_grad_close(p.grad.cpu().numpy(), z["grad.list." + n], gmax, n)


def load_awelv_int_case(name, device="cpu", prefix="awelv_int"):
    """-> (cfg, batch, state, npz) from tests/golden/awelv_int_<name>.npz (oracle/make_golden.py:make_awelv_int)"""
    import json
    from intel_sigir2023_b200.config import IntelConfig
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", f"{prefix}_{name}.npz"))
    cfg = IntelConfig(**json.loads(bytes(z["cfg"]).decode()))
    batch = {k[6:]: torch.from_numpy(z[k]).to(device) for k in z.files if k.startswith("batch.")}
    batch["batch_size"] = int(batch["i_id_s"].shape[0])
    batch["phase"] = "train"
    state = {k[6:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("state.")}
    return cfg, batch, state, z


def check_awelv_int(device, name):
    """baselines.aWELv_Int (intent predictor + per-session softmax fusion) + IntListloss against arrays produced by the
    unmodified reference model (models/supervise/aWELv_Int.py, script/baselines.sh:40)"""
    import argparse
    from intel_sigir2023_b200 import baselines, losses
    cfg, batch, state, z = load_awelv_int_case(name, device)
    model = baselines.aWELv_Int(argparse.Namespace(device=device, model_path="", buffer=1), cfg=cfg)
    assert [n for n, _ in model.named_parameters()] == list(state.keys())       # the reference's registration order
    model.load_state_dict(state)
    model = model.to(device)
    out = model(batch)
    for k in ("intents", "weights", "ens_score"):
        assert rel_err(out[k].detach().cpu().numpy(), z["out." + k]) < TOL, k
    crit = losses.IntListloss(argparse.Namespace(**LOSS_KW))
    loss, ens_l, int_l = crit(out, batch)
    for got, ref in zip((loss, ens_l, int_l), z["loss.list"]):
        assert abs(float(got.detach()) - float(ref)) <= TOL * abs(float(ref)), (float(got.detach()), float(ref))
    loss.backward()
    gmax = max(float(np.abs(z["grad.list." + n]).max()) for n, _ in model.named_parameters())
    for n, p in model.named_parameters():
        if n == "item_embeddings.weight":           # declared, never read: no gradient on either side
            assert p.grad is None and not np.any(z["grad.list." + n])
            continue
        assert_grad_close(p.grad.cpu().numpy(), z["grad.list." + n], gmax, n)


def load_lambdarank_case(tag, device="cpu"):
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "lambdarank.npz"))
    return tuple(torch.from_numpy(z[f"{tag}.{k}"]).to(device) for k in ("ranking", "scores", "session_len")) + (z[f"{tag}.lambdas"],)


def assert_lambdas_close(got, ref):
    """NaN rows (sessions without a positive item: 0/0 in the reference) must coincide; the rest within TOL of the inf-norm"""
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    ok = ~np.isnan(ref)
    assert rel_err(got[ok], ref[ok]) < TOL, rel_err(got[ok], ref[ok])


def check_lambdarank(device):
    """lambdarank.compute_lambda_new (one kernel) against arrays produced by the unmodified reference method
    (helpers/LambdaRankRunner.py:315-344; oracle/make_golden.py:make_lambdarank), then against the oracle on a larger set"""
    from intel_sigir2023_b200 import lambdarank, synthetic
    for tag in ("S", "W", "Z", "L"):
        ranking, scores, slen, ref = load_lambdarank_case(tag, device)
        got = lambdarank.compute_lambda_new(ranking, scores, slen)                         # raw ranking: clamped by the kernel
        assert_lambdas_close(got.cpu().numpy(), ref)
        got2 = lambdarank.compute_lambda_new(torch.clamp(ranking, min=0), scores, slen)    # the reference's own call (:241-246)
        assert np.array_equal(got.cpu().numpy(), got2.cpu().numpy(), equal_nan=True)
        pad = torch.arange(ranking.shape[1], device=device)[None, :] >= slen[:, None]
        assert not np.any(got.cpu().numpy()[(pad & ~torch.isnan(got)).cpu().numpy()])      # pad slots of live sessions: 0
    pred, ranking, _, slen = synthetic.eval_set(37, 70, 5, seed=11)
    scores = pred.float().softmax(dim=-1)
    got = lambdarank.compute_lambda_new(ranking.to(device), scores.to(device), slen.to(device))
    assert_lambdas_close(got.cpu().numpy(), O.compute_lambda(ranking, scores, slen).numpy())
    empty = lambdarank.compute_lambda_new(ranking[:0].to(device), scores[:0].to(device), slen[:0].to(device))
    assert tuple(empty.shape) == (0, 70)


def check_awelv_intel(device, name):
    """baselines.aWELv_IntEL (IntEL's gate path + the pooled, twice-softmaxed head) + IntListloss against arrays produced by
    the unmodified reference model (models/supervise/aWELv_IntEL.py, script/baselines.sh:47)"""
    import argparse
    from intel_sigir2023_b200 import baselines, losses
    cfg, batch, state, z = load_awelv_int_case(name, device, prefix="awelv_intel")
    model = baselines.aWELv_IntEL(argparse.Namespace(device=device, model_path="", buffer=1), cfg=cfg)
    assert [n for n, _ in model.named_parameters()] == list(state.keys())       # the reference's registration order
    model.load_state_dict(state)
    model = model.to(device)
    out = model(batch)
    for k in ("intents", "weights", "ens_score"):
        assert rel_err(out[k].detach().cpu().numpy(), z["out." + k]) < TOL, k
    crit = losses.IntListloss(argparse.Namespace(**LOSS_KW))
    loss, ens_l, int_l = crit(out, batch)
    for got, ref in zip((loss, ens_l, int_l), z["loss.list"]):
        assert abs(float(got.detach()) - float(ref)) <= TOL * abs(float(ref)), (float(got.detach()), float(ref))
    loss.backward()
    gmax = max(float(np.abs(z["grad.list." + n]).max()) for n, _ in model.named_parameters())
    for n, p in model.named_parameters():
        assert_grad_close(p.grad.cpu().numpy(), z["grad.list." + n], gmax, n)


def load_lambdarank_model_case(name, device="cpu"):
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", f"lambdarank_model_{name}.npz"))
    batch = {k[6:]: torch.from_numpy(z[k]).to(device) for k in z.files if k.startswith("batch.")}
    state = {k[6:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("state.")}
    return z, batch, state


def check_lambdarank_model(device, name):
    """lambdarank.LambdaRank (gather + MLP + list softmax) and one training signal of LambdaRankRunner.fit (lambdas, then
    ens_score.backward(lambdas)) against arrays produced by the unmodified reference model and runner method"""
    import argparse
    from intel_sigir2023_b200 import lambdarank
    z, batch, state = load_lambdarank_model_case(name, device)
    args = argparse.Namespace(hidden_size=bytes(z["hidden_size"]).decode(), i_emb_size=32, model_num=int(z["model_num"][0]),
                              device=device)
    model = lambdarank.LambdaRank(args, item_num=int(z["item_rows"][0]))
    assert [n for n, _ in model.named_parameters()] == list(state.keys())
    model.load_state_dict(state)
    model = model.to(device)
    out = model(batch)
    assert rel_err(out["ens_score"].detach().cpu().numpy(), z["out.ens_score"]) < TOL
    assert out["weights"].shape == z["out.weights"].shape and not out["weights"].any()
    lam = lambdarank.compute_lambda_new(torch.clamp(batch["ranking"], min=0), out["ens_score"].detach(), batch["session_len"])
    lam = torch.nan_to_num(lam, nan=0.0)
    assert rel_err(lam.cpu().numpy(), z["lambdas"]) < 5 * TOL
    out["ens_score"].backward(torch.from_numpy(z["lambdas"]).to(device))
    gmax = max(float(np.abs(z["grad." + n]).max()) for n, _ in model.named_parameters())
    for n, p in model.named_parameters():
        assert_grad_close(p.grad.cpu().numpy(), z["grad." + n], gmax, n)


def check_phased_backward(device, name="script_pl_gru"):
    """IntEL's backward pass runs intel_ensemble_bwd_phase (HEAD -> intent predictor -> ITEM -> SCORE, the order a data-parallel
    caller overlaps its gradient exchange with); the one-call intel_ensemble_bwd must give the same gradients, and the flat
    gradient buffer must end with the score stream's parameters."""
    from intel_sigir2023_b200 import losses
    cfg, batch, state, _ = load_model_case(name, device)
    grads = []
    for single in (False, True):
        model = make_model(cfg, state, device).train()
        model._single_call_backward = single
        crit = losses.IntListloss(loss_args())
        out = model(batch)
        crit(out, batch)[0].backward()
        grads.append({n: p.grad.detach().cpu().numpy().copy() for n, p in model.named_parameters()})
        if not single:
            late, flat = model._flat_late, model._flat_grad
            assert 0 < late < flat.numel()
            base = flat.data_ptr()
            for n, p in model.named_parameters():
                off = (p.grad.data_ptr() - base) // 4
                assert (off >= late) == (n in model._late_grad_names), n
            pk = [dict(model.named_parameters())[n].grad for n in model._packed_grad_names]
            for a, b in zip(pk, pk[1:]):        # the three intent-projection gradients sit back to back
                assert b.data_ptr() == a.data_ptr() + 4 * a.numel()
    gmax = max(float(np.abs(g).max()) for g in grads[1].values())
    for n, g in grads[1].items():
        err = float(np.abs(grads[0][n] - g).max())
        # same kernels, same inputs: the only difference is the order of the fp32 atomic adds into the shared tables
        assert err <= 3e-6 * float(np.abs(g).max()) + 3e-7 * gmax, (n, err)


def check_gru_prep(device):
    """The index kernels of the packed GRU path against numpy: stable order by decreasing (clamped) length, the list of live
    (session, step) rows in (b, t) order, their count.  Index work: bit exact.  Sizes cross the 1024-session chunk of the kernels."""
    from intel_sigir2023_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(3)
    for B, T in ((1, 1), (37, 5), (1024, 20), (1025, 20), (4096, 20), (3000, 63)):
        lens_np = rng.integers(0, T + 3, size=B).astype(np.int64)          # 0 and > T occur: both are clamped
        lens_np[rng.integers(0, B)] = T
        lens = torch.from_numpy(lens_np).to(device)
        order = torch.full((B + 1,), -7, dtype=torch.int32, device=device)
        rows_t = torch.full((B * T,), -1, dtype=torch.int32, device=device)
        rows_t1 = torch.full((B * T,), -1, dtype=torch.int32, device=device)
        count = torch.zeros(1, dtype=torch.int32, device=device)
        _lib.check(lib.intel_debug_gru_prep(B, T, _lib.ptr(lens), _lib.ptr(order), _lib.ptr(rows_t), _lib.ptr(rows_t1), _lib.ptr(count),
                                            _lib.stream_ptr(torch.device(device))))
        cl = np.clip(lens_np, 0, T)
        ref_order = np.argsort(-cl, kind="stable").astype(np.int32)
        got = order.cpu().numpy()
        assert np.array_equal(got[:B], ref_order), (B, T)
        assert got[B] == 0
        n = int(cl.sum())
        assert int(count.cpu()[0]) == n
        b = np.repeat(np.arange(B), cl)
        t = np.concatenate([np.arange(k) for k in cl]) if n else np.zeros(0, dtype=np.int64)
        assert np.array_equal(rows_t.cpu().numpy()[:n], (b * T + t).astype(np.int32))
        assert np.array_equal(rows_t1.cpu().numpy()[:n], (b * (T + 1) + t).astype(np.int32))
        assert (rows_t.cpu().numpy()[n:] == -1).all()


def check_bert_fused_vs_staged(device, names=("default_bert", "wide_intent_bert_full")):
    """The one-kernel BERT4Rec encoder forward (bert_fused.cu) against the staged path (~25 launches per encoder): same
    outputs, and - through the activations it leaves for the staged backward pass - the same gradients."""
    from intel_sigir2023_b200 import _lib, losses
    lib = _lib.load()
    for name in names:
        cfg, batch, state, _ = load_model_case(name, device)
        res = []
        for on in (1, 0):
            _lib.check(lib.intel_debug_use_fused_bert(on))
            try:
                model = make_model(cfg, state, device).train()
                out = model(batch)
                losses.IntListloss(loss_args())(out, batch)[0].backward()
                res.append(({k: v.detach().cpu().numpy() for k, v in out.items()},
                            {n: p.grad.detach().cpu().numpy().copy() for n, p in model.named_parameters()}))
                model.eval()
                with torch.no_grad():
                    res[-1][0]["intents_eval"] = model(batch)["intents"].cpu().numpy()
            finally:
                _lib.check(lib.intel_debug_use_fused_bert(1))
        (oa, ga), (ob, gb) = res
        for k in ob:
            assert rel_err(oa[k], ob[k]) < 3e-6, (name, k, rel_err(oa[k], ob[k]))
        gmax = max(float(np.abs(g).max()) for g in gb.values())
        for n, g in gb.items():
            assert_grad_close(ga[n], g, gmax, f"{name}:{n}")


def check_bert_fused_token_tiles(device, B=10):
    """The fused BERT4Rec encoder is instantiated per token tile (history slots rounded up to 12 / 16 / 20 / 24): each one
    against the CPU oracle (forward, loss and - through the activations it leaves for the staged backward - gradients);
    one and two encoder heads."""
    for hm, heads, bh in ((7, 1, 2), (13, 2, 1), (19, 2, 2), (23, 1, 2)):
        check_against_oracle(device, seed=hm, B=B, L=9, min_len=2, encoder="BERT4Rec", num_heads=heads, bert_heads=bh,
                             corpus_kw=dict(history_max=hm))
