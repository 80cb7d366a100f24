"""Exact row-sparse Adam for the embedding tables (IntEL sparse_grad = 2): optim.Adam defers the zero-gradient updates of
the rows a step does not name and replays them when the rows are next read, so parameters and moments follow dense Adam bit
for bit.  The CPU tests run the kernels on the emulator build (tests/emu); the gpu-marked tests run them on the device."""
import argparse
import copy
import dataclasses
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "emu"))

import parity_checks as P  # noqa: E402
from conftest import load_model_case  # noqa: E402
from test_sparse_tables import _setup_emu, emu, expected_rows  # noqa: E402,F401


def _slice(batch, lo, hi, flip=False):
    out = {k: (v[lo:hi] if torch.is_tensor(v) and v.dim() > 0 else v) for k, v in batch.items()}
    if flip:
        out = {k: (v.flip(0) if torch.is_tensor(v) and v.dim() > 0 else v) for k, v in out.items()}
    out["batch_size"] = hi - lo
    return out


def _opt_state(opt, p):
    st = opt.state[p]
    return p.detach(), st["exp_avg"], st["exp_avg_sq"], float(st["step"])


def assert_same_state(ma, oa, mb, ob, what):
    for (n, pa), pb in zip(ma.named_parameters(), mb.parameters()):
        a, b = _opt_state(oa, pa), _opt_state(ob, pb)
        for k, x, y in zip(("param", "exp_avg", "exp_avg_sq"), a[:3], b[:3]):
            assert torch.equal(x, y), (what, n, k, float((x - y).abs().max()))
        assert a[3] == b[3], (what, n, a[3], b[3])


# ---- optimizer only --------------------------------------------------------------------------------------------------

def _tables(device, rows):
    torch.manual_seed(0)
    m = torch.nn.Module()
    m.table = torch.nn.Embedding(rows, 16)       # float4 rows
    m.odd = torch.nn.Embedding(50, 3)            # d % 4 != 0
    m.lin = torch.nn.Linear(7, 5)
    return m.to(device)


def check_deferred_adam(device, rows=300, steps=12, wd=1e-3, lr=3e-3):
    """dense optim.Adam fed dense gradients against the deferred optimizer fed COO gradients of the same rows"""
    from intel_sigir2023_b200 import optim
    g = torch.Generator().manual_seed(5)
    ma, mb = _tables(device, rows), _tables(device, rows)
    optim.defer_zero_updates([mb.table.weight, mb.odd.weight])
    oa = optim.Adam(optim.customize_parameters(ma), lr=lr, weight_decay=wd)
    ob = optim.Adam(optim.customize_parameters(mb), lr=lr, weight_decay=wd)
    sa = torch.optim.lr_scheduler.StepLR(oa, step_size=3, gamma=0.5)
    sb = torch.optim.lr_scheduler.StepLR(ob, step_size=3, gamma=0.5)
    for it in range(steps):
        for (n, pa), pb in zip(ma.named_parameters(), mb.parameters()):
            if n.startswith("lin"):
                gr = torch.randn(pa.shape, generator=g).to(device)
                pa.grad, pb.grad = gr.clone(), gr.clone()
                continue
            if n == "odd.weight" and it == 4:           # no gradient: dense Adam skips the parameter, so does the history
                pa.grad = pb.grad = None
                continue
            n_rows, d = pa.shape
            # the last rows are never named; the band below them only in the first and the last step (idle for long)
            live = n_rows - n_rows // 10
            band = live - n_rows // 5
            pool = torch.arange(live if it in (0, steps - 1) else band)
            pick = pool[torch.randperm(pool.numel(), generator=g)[: max(1, pool.numel() // 4)]].sort().values
            vals = torch.randn(pick.numel(), d, generator=g)
            if it == 2 and n == "table.weight":        # accumulated over two passes: duplicate, unsorted indices (pairs)
                half = pick.numel() // 2
                idx = torch.cat([pick.flip(0), pick[:half]])
                v = torch.cat([vals.flip(0), torch.randn(half, d, generator=g)])
            else:
                idx, v = pick, vals
            coo = torch.sparse_coo_tensor(idx.view(1, -1), v, size=pa.shape, check_invariants=True).to(device)
            pb.grad = coo
            pa.grad = coo.to_dense()
        oa.step()
        ob.step()
        sa.step()
        sb.step()
        if it == steps // 2:
            # state_dict() flushes: it equals the dense optimizer's; the round trip through torch.optim.Adam and back
            sd = ob.state_dict()
            da = oa.state_dict()
            for k in da["state"]:
                for f in ("exp_avg", "exp_avg_sq"):
                    assert torch.equal(sd["state"][k][f], da["state"][k][f]), (it, k, f)
            assert_same_state(ma, oa, mb, ob, "mid-run flush")
            tor = torch.optim.Adam(optim.customize_parameters(mb), lr=lr, weight_decay=wd)
            tor.load_state_dict(copy.deepcopy(sd))
            ob.load_state_dict(copy.deepcopy(tor.state_dict()))
    ob.flush()
    assert_same_state(ma, oa, mb, ob, "final flush")


def test_deferred_adam_equals_dense(emu):
    check_deferred_adam("cpu")


def test_untouched_rows_pending_until_flush(emu):
    """before the flush an untouched row still holds its old value; the flush alone brings it to the dense one"""
    from intel_sigir2023_b200 import optim
    ma, mb = _tables("cpu", 64), _tables("cpu", 64)
    optim.defer_zero_updates([mb.table.weight])
    oa = optim.Adam([ma.table.weight], lr=1e-2, weight_decay=1e-2)
    ob = optim.Adam([mb.table.weight], lr=1e-2, weight_decay=1e-2)
    before = mb.table.weight.detach().clone()
    for _ in range(3):
        coo = torch.sparse_coo_tensor(torch.tensor([[1, 5]]), torch.ones(2, 16), size=(64, 16))
        ma.table.weight.grad, mb.table.weight.grad = coo.to_dense(), coo
        oa.step()
        ob.step()
    w = mb.table.weight.detach()
    assert torch.equal(w[[1, 5]], ma.table.weight.detach()[[1, 5]])
    assert torch.equal(w[0], before[0]) and not torch.equal(w[0], ma.table.weight.detach()[0])
    ob.flush()
    assert torch.equal(mb.table.weight, ma.table.weight)


# ---- model ----------------------------------------------------------------------------------------------------------

def _batches(device):
    out = []
    for name in ("script_pl_gru", "default_bert"):
        cfg, batch, state, _ = load_model_case(name, device)
        B = batch["batch_size"]
        out.append((name, cfg, state, [_slice(batch, 0, B), _slice(batch, 0, B // 2, flip=True), _slice(batch, B // 3, B),
                                       _slice(batch, 1, B - 1, flip=True), _slice(batch, 0, max(2, B // 4))]))
    return out


def _train(cfg, state, batches, sparse, device, probe=None, reads=True):
    """optim.Adam(weight_decay=1e-4) + StepLR over the batches, with (reads) a no_grad eval forward after step 2 and a
    model.state_dict() read after step 4, both of which flush; returns (model, optimizer) after a final flush"""
    from intel_sigir2023_b200 import losses, optim
    model = P.make_model(dataclasses.replace(cfg, sparse_grad=sparse), state, device).train()
    crit = losses.IntListloss(P.loss_args())
    opt = optim.Adam(optim.customize_parameters(model), lr=1e-2, weight_decay=1e-4)
    sched = torch.optim.lr_scheduler.StepLR(opt, step_size=2, gamma=0.5)
    for it, b in enumerate(batches):
        opt.zero_grad(set_to_none=True)
        out = model(b)
        if probe is not None:
            probe(it, model, opt, b)
        crit(out, b)[0].backward()
        opt.step()
        sched.step()
        if reads and it == 1:
            model.eval()
            with torch.no_grad():
                model(batches[0])
            model.train()
        elif reads and it == 3:
            model.state_dict()
    opt.flush()
    return model, opt


@pytest.mark.parametrize("idx", [0, 1])
def test_model_mode2_equals_dense(emu, idx):
    from intel_sigir2023_b200.IntEL import SPARSE_TABLES
    name, cfg, state, batches = _batches("cpu")[idx]
    dense = _train(cfg, state, batches, 0, "cpu")
    exact = _train(cfg, state, batches, 2, "cpu")
    assert_same_state(*dense, *exact, name)
    # the lazy mode leaves the rows no batch named where they were: the comparison above can fail
    lazy, _ = _train(cfg, state, batches, 1, "cpu")
    tables = {n: keys for n, keys, _ in SPARSE_TABLES}
    pd = dict(dense[0].named_parameters())
    differ = 0
    for n, p in lazy.named_parameters():
        if n in tables:
            named = np.unique(np.concatenate([expected_rows(b, tables[n], p.shape[0]) for b in batches]))
            untouched = np.setdiff1d(np.arange(p.shape[0]), named)
            if untouched.size:
                differ += int(not torch.equal(p.detach()[untouched], pd[n].detach()[untouched]))
    assert differ > 0


def test_catch_up_brings_row_set_current(emu):
    """after a training forward pass in mode 2 the rows of its row set equal the dense run's at that step; the other rows
    are still pending"""
    from intel_sigir2023_b200.IntEL import SPARSE_TABLES
    name, cfg, state, batches = _batches("cpu")[0]
    tables = {n: keys for n, keys, _ in SPARSE_TABLES}
    seen = {}

    def record(tag):
        def probe(it, model, opt, b):
            if it < 2:
                return
            for n in tables:
                p = model.get_parameter(n)
                st = opt.state[p]
                seen[(tag, it, n)] = (p.detach().clone(), st["exp_avg"].clone(), st["exp_avg_sq"].clone(),
                                      expected_rows(b, tables[n], p.shape[0]))
        return probe

    _train(cfg, state, batches, 0, "cpu", record("dense"), reads=False)
    _train(cfg, state, batches, 2, "cpu", record("exact"), reads=False)
    pending = 0
    for (tag, it, n), (p, m, v, rows) in seen.items():
        if tag != "exact":
            continue
        dp_, dm, dv, _ = seen[("dense", it, n)]
        for x, y in ((p, dp_), (m, dm), (v, dv)):
            assert torch.equal(x[rows], y[rows]), (it, n)
        other = np.setdiff1d(np.arange(p.shape[0]), rows)
        pending += int(not torch.equal(p[other], dp_[other]))
    assert pending > 0


# ---- two ranks (gloo) ------------------------------------------------------------------------------------------------

def _dp_run(rank, world, sparse):
    from intel_sigir2023_b200 import dp, losses, optim, synthetic
    cfg, batch, state, _ = load_model_case("script_pl_gru")
    B = batch["batch_size"] - batch["batch_size"] % 2
    batches = [_slice(batch, 0, B), _slice(batch, 0, B, flip=True)]
    model = P.make_model(dataclasses.replace(cfg, sparse_grad=sparse), state, "cpu").train()
    crit = losses.IntListloss(P.loss_args())
    opt = optim.Adam(optim.customize_parameters(model), lr=1e-2, weight_decay=1e-4)
    reducer = dp.GradReducer(model, world, overlap=True)
    for b in batches:
        shard = synthetic.shard_batch(b, rank, world)
        opt.zero_grad(set_to_none=True)
        crit(model(shard), shard)[0].backward()
        reducer.allreduce()
        opt.step()
    opt.flush()
    return {n: [t.numpy().copy() for t in _opt_state(opt, p)[:3]] for n, p in model.named_parameters()}


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.set_num_threads(1)
    _setup_emu()
    dist.init_process_group("gloo", rank=rank, world_size=world)
    res = [_dp_run(rank, world, sp) for sp in (0, 2)]
    if rank == 0:
        q.put(res)
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_mode2_equals_dense():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 33500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    dense, exact = q.get(timeout=300)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for n in dense:
        for k, a, b in zip(("param", "exp_avg", "exp_avg_sq"), dense[n], exact[n]):
            assert np.array_equal(a, b), (n, k)


# ---- on the B200 ----------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_gpu_deferred_adam_equals_dense():
    check_deferred_adam("cuda", rows=2_000_000, steps=40)


@pytest.mark.gpu
def test_gpu_c2_mode2_matches_dense():
    """C2 shape (4096 sessions x 50 items, 1M items, GRU4Rec + the IntEL.sh 'pl' widths), 5 distinct batches and a flush:
    the rows no batch named are bitwise the dense run's; everything else is within the weight gate of config 1 (gradient
    atomics order the sums differently from run to run on the device, as between two dense runs)"""
    from intel_sigir2023_b200 import losses, optim, synthetic
    from intel_sigir2023_b200.config import IntelConfig
    from intel_sigir2023_b200.IntEL import IntEL, SPARSE_TABLES
    dev = torch.device("cuda")
    corpus = synthetic.CorpusSpec(n_item=1_000_000, n_class=357, n_user=100_000, n_ctx=931, model_num=4, intent_num=1071,
                                  history_max=20)
    cfg = IntelConfig(item_rows=corpus.item_rows, class_rows=corpus.n_class, user_rows=corpus.user_rows, ctx_rows=corpus.n_ctx,
                      intent_num=corpus.intent_num, model_num=corpus.model_num, history_max=20, encoder="GRU4Rec",
                      context_emb_size=32, intent_emb_size=32, cross_attn_qsize=64, num_heads=2, num_layers=2)
    batches = [synthetic.make_batch(corpus, synthetic.BatchSpec(batch_size=4096, max_len=50, min_len=50), seed=100 + s, device=dev)
               for s in range(5)]
    crit = losses.IntListloss(argparse.Namespace(cal_diversity=1, diversity_alpha=1e-4, intent_weight=0.1, ensemble_weight=1.0,
                                                 kl_temp=2.0, kl_weight=0.5))
    runs = []
    for sp in (0, 2):
        torch.manual_seed(0)
        model = IntEL(argparse.Namespace(device=dev, model_path="", buffer=1), cfg=dataclasses.replace(cfg, sparse_grad=sp)).to(dev)
        opt = optim.Adam(optim.customize_parameters(model), lr=1e-3, weight_decay=1e-6)
        sched = torch.optim.lr_scheduler.StepLR(opt, step_size=2, gamma=0.5)
        for b in batches:
            opt.zero_grad(set_to_none=True)
            crit(model(b), b)[0].backward()
            opt.step()
            sched.step()
        opt.flush()
        runs.append((model, opt))
    (dense, od), (exact, oe) = runs
    tables = {n: keys for n, keys, _ in SPARSE_TABLES}
    pe = dict(exact.named_parameters())
    for n, p in dense.named_parameters():
        for k, a, b in zip(("param", "exp_avg", "exp_avg_sq"), _opt_state(od, p)[:3], _opt_state(oe, pe[n])[:3]):
            if n in tables:
                named = torch.from_numpy(np.unique(np.concatenate([expected_rows(bt, tables[n], p.shape[0]) for bt in batches])))
                untouched = torch.ones(p.shape[0], dtype=torch.bool)
                untouched[named] = False
                untouched = untouched.to(dev)
                assert torch.equal(a[untouched], b[untouched]), (n, k)
            scale = float(a.abs().max())
            assert float((a - b).abs().max()) <= 5e-4 * scale, (n, k)
