"""Exact row-sparse Adam (IntEL sparse_grad = 2) against dense (0) and lazy (1) table gradients, C2 shape, over an epoch of
distinct batches.

    python profiles/tools/sparse_exact.py [--n_items 1000000 10000000 50000000] [--steps 50] [--reps 5]

A row that no batch of an epoch names collects one pending update per step in exact mode, and the flush at the end of the
epoch replays them all.  So the batches must be distinct: they are built on the device from a synthetic columnar corpus
(corpus.synthetic_columns + DeviceCorpus.batch), `steps` batches of `batch` sessions, built before the timing.  One step =
zero_grad, forward, loss, backward, optim.Adam.step.  The three arms start from the same weights and run the same epochs
alternately in one process (after a warm-up epoch, `reps` rounds, CUDA events around each epoch); the exact arm's epoch
ends with optimizer.flush(), timed separately and included in its per-epoch total.  Then fresh models run one epoch each
(exact + flush, dense, and a second dense run): the rows no batch named are compared between exact and dense (bitwise), and
the largest difference elsewhere is reported beside that between the two dense runs.

A last line times the flush of a 50 M x 16 table with k pending updates on every row (replay rate), and one dense Adam
step over the same table for comparison.  The GPU's name and power limit are read by nvidia-smi in the same process.
"""
from __future__ import annotations

import argparse
import dataclasses
import gc
import json
import os
import statistics
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

from intel_sigir2023_b200 import _lib, corpus as corpus_mod, losses, optim, synthetic  # noqa: E402
from intel_sigir2023_b200.config import IntelConfig  # noqa: E402
from intel_sigir2023_b200.IntEL import IntEL, SPARSE_TABLES  # noqa: E402
from sparse_tables import gpu_info  # noqa: E402

ARMS = {"dense": 0, "lazy": 1, "exact": 2}


def events():
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def epoch_c2(n_item: int, a, dev, crit) -> dict:
    corpus = synthetic.CorpusSpec(n_item=n_item, n_class=357, n_user=a.n_user, n_ctx=931, model_num=4, intent_num=1071,
                                  history_max=20)
    cfg = IntelConfig(item_rows=corpus.item_rows, class_rows=corpus.n_class, user_rows=corpus.user_rows, ctx_rows=corpus.n_ctx,
                      intent_num=corpus.intent_num, model_num=corpus.model_num, history_max=20, encoder="GRU4Rec",
                      context_emb_size=32, intent_emb_size=32, cross_attn_qsize=64, num_heads=2, num_layers=2)
    n_sess = a.steps * a.batch
    cols, shared, nz = corpus_mod.synthetic_columns(n_sess, 50, n_item, corpus.n_class, a.n_user, corpus.n_ctx, corpus.model_num,
                                                    corpus.intent_num, max_his=20, seed=17)
    dc = corpus_mod.DeviceCorpus(cols, shared, corpus.model_num, corpus.intent_num, 20, nz, dev)
    del cols, shared
    order = np.random.default_rng(5).permutation(n_sess)
    batches = [dc.batch(order[i * a.batch:(i + 1) * a.batch], shuffle=False) for i in range(a.steps)]
    del dc
    arms = {}
    for arm, sp in ARMS.items():
        torch.manual_seed(0)
        with torch.device(dev):
            model = IntEL(argparse.Namespace(device=dev, model_path="", buffer=1), cfg=dataclasses.replace(cfg, sparse_grad=sp))
        arms[arm] = (model, optim.Adam(optim.customize_parameters(model), lr=1e-3, weight_decay=1e-6))

    def epoch(arm):
        model, opt = arms[arm]
        e0, e1, e2 = events()
        e0.record()
        for b in batches:
            opt.zero_grad(set_to_none=True)
            crit(model(b), b)[0].backward()
            opt.step()
        e1.record()
        if arm == "exact":
            opt.flush()
        e2.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), e1.elapsed_time(e2)

    gc.collect()
    for arm in arms:
        epoch(arm)
    ms = {arm: [] for arm in arms}
    for _ in range(a.reps):
        for arm in arms:
            ms[arm].append(epoch(arm))
    out = {"n_item": n_item, "config": "c2/pl", "batch": a.batch, "list_len": 50, "steps_per_epoch": a.steps, "rounds": a.reps,
           "weight_decay": 1e-6}
    for arm in arms:
        steps_ms = [s for s, _ in ms[arm]]
        tot = [s + f for s, f in ms[arm]]
        out[arm] = {"ms_per_step": round(statistics.median(steps_ms) / a.steps, 4),
                    "ms_per_step_incl_flush": round(statistics.median(tot) / a.steps, 4),
                    "epoch_ms_rounds": [round(x, 3) for x in tot]}
        if arm == "exact":
            out[arm]["flush_ms"] = round(statistics.median(f for _, f in ms[arm]), 4)
    out["dense_over_exact"] = round(out["dense"]["ms_per_step_incl_flush"] / out["exact"]["ms_per_step_incl_flush"], 4)
    out["dense_over_lazy"] = round(out["dense"]["ms_per_step_incl_flush"] / out["lazy"]["ms_per_step_incl_flush"], 4)
    del arms
    gc.collect()
    out["exact_vs_dense"] = check_epoch(cfg, batches, dev, crit)
    del batches
    gc.collect()
    torch.cuda.empty_cache()
    return out


def check_epoch(cfg, batches, dev, crit) -> dict:
    """fresh models, one epoch (+ flush for exact): the rows no batch named, exact against dense (bitwise); elsewhere the
    largest difference relative to the tensor's largest entry, exact against dense and, for scale, a second dense run
    (gradient atomics order the sums differently from run to run)"""
    runs = {}
    for arm, sp in (("dense", 0), ("dense2", 0), ("exact", 2)):
        torch.manual_seed(0)
        with torch.device(dev):
            model = IntEL(argparse.Namespace(device=dev, model_path="", buffer=1), cfg=dataclasses.replace(cfg, sparse_grad=sp))
        opt = optim.Adam(optim.customize_parameters(model), lr=1e-3, weight_decay=1e-6)
        for b in batches:
            opt.zero_grad(set_to_none=True)
            crit(model(b), b)[0].backward()
            opt.step()
        opt.flush()
        runs[arm] = {n: (p.detach(), opt.state[p]["exp_avg"], opt.state[p]["exp_avg_sq"]) for n, p in model.named_parameters()}
        del model, opt
    tables = {n: keys for n, keys, _ in SPARSE_TABLES}
    rel = lambda x, y: float((x - y).abs().max()) / max(float(x.abs().max()), 1e-30) if x.numel() else 0.0
    out = {"untouched_rows_bitwise": True, "max_rel_diff": {"exact_vs_dense": {}, "dense_vs_dense": {}}, "rows_named": {}}
    for n, dense in runs["dense"].items():
        mask = None
        if n in tables:
            mask = torch.zeros(dense[0].shape[0], dtype=torch.bool, device=dev)
            for b in batches:
                for k in tables[n]:
                    ids = b[k].reshape(-1)
                    mask[ids[(ids >= 0) & (ids < mask.numel())]] = True
            out["rows_named"][n] = int(mask.sum())
            out["untouched_rows_bitwise"] &= all(bool(torch.equal(x[~mask], y[~mask])) for x, y in zip(dense, runs["exact"][n]))
        for other, key in (("exact", "exact_vs_dense"), ("dense2", "dense_vs_dense")):
            for kind, x, y in zip(("param", "exp_avg", "exp_avg_sq"), dense, runs[other][n]):
                if mask is not None:
                    x, y = x[mask], y[mask]
                d = out["max_rel_diff"][key]
                d[kind] = max(d.get(kind, 0.0), rel(x, y))
    return out


def replay_rate(rows: int, d: int, ks, reps: int, dev) -> dict:
    p = torch.nn.Parameter(torch.randn(rows, d, device=dev))
    optim.defer_zero_updates([p])
    opt = optim.Adam([p], lr=1e-3, weight_decay=1e-6)
    empty = torch.sparse_coo_tensor(torch.zeros(1, 0, dtype=torch.int64, device=dev), torch.zeros(0, d, device=dev), size=(rows, d))
    out = {"table": [rows, d], "flush": {}}
    for k in ks:
        t = []
        for _ in range(reps + 1):
            for _ in range(k):               # a step that names no row: one more pending update on every row
                p.grad = empty
                opt.step()
            e0, e1, _ = events()
            e0.record()
            opt.flush()
            e1.record()
            torch.cuda.synchronize()
            t.append(e0.elapsed_time(e1))
        ms = statistics.median(t[1:])
        out["flush"][str(k)] = {"ms": round(ms, 4), "ns_per_element_update": round(ms * 1e6 / (rows * d * k), 5),
                                "ms_rounds": [round(x, 4) for x in t[1:]]}
    q = torch.nn.Parameter(torch.randn(rows, d, device=dev))
    dense = optim.Adam([q], lr=1e-3, weight_decay=1e-6)
    q.grad = torch.zeros_like(q)
    t = []
    for _ in range(reps + 1):
        e0, e1, _ = events()
        e0.record()
        dense.step()
        e1.record()
        torch.cuda.synchronize()
        t.append(e0.elapsed_time(e1))
    out["dense_adam_step_ms"] = round(statistics.median(t[1:]), 4)
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--n_items", type=int, nargs="+", default=[1_000_000, 10_000_000, 50_000_000])
    ap.add_argument("--n_user", type=int, default=100_000)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=50, help="distinct batches (steps) per epoch")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--replay_rows", type=int, default=50_000_000)
    ap.add_argument("--replay_k", type=int, nargs="+", default=[1, 8, 64])
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sparse_exact.py times the B200 kernels: it needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    _lib.load()
    info = gpu_info(0)
    crit = losses.IntListloss(argparse.Namespace(cal_diversity=1, diversity_alpha=1e-4, intent_weight=0.1, ensemble_weight=1.0,
                                                 kl_temp=2.0, kl_weight=0.5))
    for n_item in a.n_items:
        print(json.dumps({**info, **epoch_c2(n_item, a, dev, crit)}), flush=True)
    print(json.dumps({**info, "replay": replay_rate(a.replay_rows, 16, a.replay_k, a.reps, dev)}), flush=True)


if __name__ == "__main__":
    main()
