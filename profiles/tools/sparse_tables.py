"""Full training step with dense against row-sparse embedding-table gradients (IntEL sparse_grad = 0 / 1), C2 shape.

    python profiles/tools/sparse_tables.py [--n_items 1000000 10000000 50000000] [--steps 10] [--reps 5]
    torchrun --nproc_per_node 2 profiles/tools/sparse_tables.py ...      # the data-parallel leg

One step = zero_grad, forward, loss, backward, GradReducer.allreduce (world > 1), optim.Adam.step.  Both models start from
the same weights and see the same resident batches; after a warm-up the two are timed alternately in one process (reps
rounds of `steps` steps each, CUDA events around each round), so drift of the shared machine hits both alike.  The row-set
build (all four tables, started at the top of the sparse forward pass) is timed on its own the same way.  One JSON line
per catalogue size goes to stdout (rank 0), with the GPU's name and power limit read by nvidia-smi in the same process.
"""
from __future__ import annotations

import argparse
import dataclasses
import gc
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from intel_sigir2023_b200 import _lib, dp, losses, optim, synthetic  # noqa: E402
from intel_sigir2023_b200.config import IntelConfig  # noqa: E402
from intel_sigir2023_b200.IntEL import IntEL, _RowSets  # noqa: E402


def gpu_info(index: int) -> dict:
    q = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = ([s.strip() for s in q.stdout.strip().split(",")] + ["?", "?", "?"])[:3]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--n_items", type=int, nargs="+", default=[1_000_000, 10_000_000, 50_000_000])
    ap.add_argument("--n_user", type=int, default=100_000)
    ap.add_argument("--batch", type=int, default=4096, help="sessions per step per GPU")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()

    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dp.configure_nccl_for_overlap()
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()
    info = gpu_info(local)
    # C2: the 'pl' run of script/IntEL.sh (GRU4Rec, list loss), 50 candidates, 4 lists, 1071 intents, 931 contexts
    crit = losses.IntListloss(argparse.Namespace(cal_diversity=1, diversity_alpha=1e-4, intent_weight=0.1, ensemble_weight=1.0,
                                                 kl_temp=2.0, kl_weight=0.5))
    for n_item in a.n_items:
        corpus = synthetic.CorpusSpec(n_item=n_item, n_class=357, n_user=a.n_user, n_ctx=931, model_num=4, intent_num=1071,
                                      history_max=20)
        cfg = IntelConfig(item_rows=corpus.item_rows, class_rows=corpus.n_class, user_rows=corpus.user_rows, ctx_rows=corpus.n_ctx,
                          intent_num=corpus.intent_num, model_num=corpus.model_num, history_max=20, encoder="GRU4Rec",
                          context_emb_size=32, intent_emb_size=32, cross_attn_qsize=64, num_heads=2, num_layers=2)
        spec = synthetic.BatchSpec(batch_size=a.batch, max_len=50, min_len=50)
        batches = [synthetic.make_batch(corpus, spec, seed=1000 * rank + i, device=dev) for i in range(3)]
        arms = {}
        for sp in (0, 1):
            torch.manual_seed(0)
            with torch.device(dev):
                model = IntEL(argparse.Namespace(device=dev, model_path="", buffer=1), cfg=dataclasses.replace(cfg, sparse_grad=sp))
            opt = optim.Adam(optim.customize_parameters(model), lr=1e-3, weight_decay=1e-6)
            red = dp.GradReducer(model, world) if world > 1 else None
            arms["sparse" if sp else "dense"] = (model, opt, red)

        def step(arm, i):
            model, opt, red = arms[arm]
            opt.zero_grad(set_to_none=True)
            b = batches[i % len(batches)]
            loss = crit(model(b), b)[0]
            loss.backward()
            if red is not None:
                red.allreduce()
            opt.step()

        def timed(fn, n):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(n):
                fn(i)
            e1.record()
            torch.cuda.synchronize()
            ms = torch.tensor([e0.elapsed_time(e1) / n], device=dev)
            if world > 1:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            return float(ms.item())

        gc.collect()
        for arm in arms:
            for i in range(a.warmup):
                step(arm, i)
        ms = {arm: [] for arm in arms}
        for _ in range(a.reps):
            for arm in arms:
                ms[arm].append(timed(lambda i, arm=arm: step(arm, i), a.steps))
        sparse_model = arms["sparse"][0]
        stream = _lib.stream_ptr(dev)
        build_ms = [timed(lambda i: _RowSets(sparse_model, batches[i % len(batches)], dev, stream), a.steps) for _ in range(a.reps)]
        rows = {n: int(p.grad._values().shape[0]) for n, p in sparse_model.named_parameters() if p.grad is not None and p.grad.is_sparse}
        if rank == 0:
            med = {k: statistics.median(v) for k, v in ms.items()}
            print(json.dumps({"n_item": n_item, "world": world, "batch_per_gpu": a.batch, "list_len": 50, "config": "c2/pl",
                              **info, "dense_ms_per_step": round(med["dense"], 4), "sparse_ms_per_step": round(med["sparse"], 4),
                              "speedup": round(med["dense"] / med["sparse"], 4),
                              "dense_ms_rounds": [round(x, 4) for x in ms["dense"]],
                              "sparse_ms_rounds": [round(x, 4) for x in ms["sparse"]],
                              "rowset_build_ms": round(statistics.median(build_ms), 4),
                              "rows_touched_last_step": rows,
                              "table_rows": {"iid_embeddings.weight": corpus.item_rows, "item_embeddings.weight": corpus.n_class,
                                             "uid_embeddings.weight": corpus.user_rows, "context_embeddings.weight": corpus.n_ctx},
                              "steps_per_round": a.steps, "rounds": a.reps}), flush=True)
        del arms, batches
        gc.collect()
        torch.cuda.empty_cache()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
