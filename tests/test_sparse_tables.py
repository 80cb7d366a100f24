"""Row-sparse embedding-table gradients (IntEL sparse_grad = 1): the row-set kernel, the sparse-mode backward pass against
the dense one and the reference goldens, the row-wise Adam step, and the two-rank exchange.  The CPU tests run the kernels
on the emulator build (tests/emu); the gpu-marked tests run them on the device at the C2 shape."""
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
from conftest import assert_grad_close, load_model_case, rel_err  # noqa: E402

CASES = ["script_pl_gru", "default_bert", "direct_att_bert", "script_bpr_gru_k4"]


def _setup_emu():
    from build_emu import build_emu
    from intel_sigir2023_b200 import _lib
    _lib._lib = None
    _lib.load(build_emu())
    _lib._allow_host_tensors = True


@pytest.fixture
def emu():
    from intel_sigir2023_b200 import _lib
    old = (_lib._lib, _lib._allow_host_tensors)
    _setup_emu()
    yield
    _lib._lib, _lib._allow_host_tensors = old


def expected_rows(batch, keys, n_rows):
    ids = np.concatenate([batch[k].cpu().numpy().reshape(-1) for k in keys])
    return np.unique(ids[(ids >= 0) & (ids < n_rows)])


def rowset(n_rows, a, b=None, slot=None, device="cpu"):
    from intel_sigir2023_b200 import _lib
    lib = _lib.load()
    slot = torch.zeros(n_rows, dtype=torch.int32, device=device) if slot is None else slot
    rows = torch.full((max(1, min(n_rows, a.numel() + (0 if b is None else b.numel()))),), -7, dtype=torch.int64, device=device)
    count = torch.zeros(1, dtype=torch.int64, device=device)
    ws = torch.empty(lib.intel_rowset_workspace_bytes(n_rows), dtype=torch.uint8, device=device)
    _lib.check(lib.intel_rowset_build(n_rows, _lib.ptr(a), a.numel(), _lib.ptr(b), 0 if b is None else b.numel(), _lib.ptr(slot),
                                      _lib.ptr(rows), _lib.ptr(count), _lib.ptr(ws), ws.numel(), _lib.stream_ptr(torch.device(device))))
    U = int(count.item())
    return rows[:U].cpu().numpy(), slot


def check_rowset_cases(device):
    g = torch.Generator().manual_seed(11)
    cases = [(5000, torch.randint(0, 5000, (4096,), generator=g), torch.randint(0, 5000, (700,), generator=g)),
             (10000, torch.randint(0, 10000, (1,), generator=g), None),                           # one id (B = 1, no history)
             (9000, torch.full((300,), 4321, dtype=torch.int64), torch.full((20,), 4321, dtype=torch.int64)),   # all ids equal
             (1, torch.zeros(64, dtype=torch.int64), None),                                        # a one-row table
             (700, torch.randint(-50, 800, (2000,), generator=g), torch.tensor([-1, 700, 10 ** 12, 3]))]     # out of range
    slot = None
    for n_rows, a, b in cases:
        ids = a.numpy() if b is None else np.concatenate([a.numpy(), b.numpy()])
        want = np.unique(ids[(ids >= 0) & (ids < n_rows)])
        a_d, b_d = a.to(device), (None if b is None else b.to(device))
        got, slot_t = rowset(n_rows, a_d, b_d, device=device)
        assert np.array_equal(got, want), (n_rows, got[:10], want[:10])
        s = slot_t.cpu().numpy()
        assert (s >= 0).all() and np.array_equal(s[want], np.arange(want.size))
        # the map is reused without a reset: a second set built over the first one's state
        again, _ = rowset(n_rows, torch.flip(a_d, [0]), None, slot=slot_t, device=device)
        ids2 = a.numpy()
        assert np.array_equal(again, np.unique(ids2[(ids2 >= 0) & (ids2 < n_rows)]))
        slot = slot_t
    # a table bigger than one chunk of the compaction, ids on both ends
    a = torch.tensor([0, 123456, 4095, 4096, 123455, 8191, 8192, 0], dtype=torch.int64).to(device)
    got, _ = rowset(123457, a, device=device)
    assert np.array_equal(got, [0, 4095, 4096, 8191, 8192, 123455, 123456])


def test_rowset_matches_unique(emu):
    check_rowset_cases("cpu")


def run_step(cfg, state, batch, device, sparse, kind="list", noise=None):
    from intel_sigir2023_b200 import losses
    model = P.make_model(dataclasses.replace(cfg, sparse_grad=sparse), state, device).train()
    crit = {"list": losses.IntListloss, "bpr": losses.IntBPRloss}[kind](P.loss_args())
    if noise is not None:
        crit.bpr_noise = noise
    out = model(batch)
    loss, ens_l, int_l = crit(out, batch)
    loss.backward()
    return model, out, torch.stack([loss.detach(), ens_l.detach(), int_l.detach()])


def check_sparse_backward(name, device, kind="list"):
    from intel_sigir2023_b200.IntEL import SPARSE_TABLES
    cfg, batch, state, gold = load_model_case(name, device)
    noise = torch.from_numpy(gold["bpr_noise"]).to(device) if kind == "bpr" else None
    dense, out_d, loss_d = run_step(cfg, state, batch, device, 0, kind, noise)
    sparse, out_s, loss_s = run_step(cfg, state, batch, device, 1, kind, noise)
    for k in out_d:
        assert torch.equal(out_d[k], out_s[k]), (name, k)
    if device == "cpu":
        assert torch.equal(loss_d, loss_s), (name, loss_d, loss_s)
    else:
        # the loss kernels sum the per-session terms with float64 atomics, whose order varies from run to run on the
        # device: two dense runs of the same batch differ in the last bits as well
        assert torch.allclose(loss_d, loss_s, rtol=1e-12, atol=0.0), (name, loss_d, loss_s)
    tables = {n: keys for n, keys, _ in SPARSE_TABLES}
    names = [n for n, _ in sparse.named_parameters()]
    gmax = max(np.abs(gold[f"grad.{kind}.{k}"]).max() for k in names)
    for (n, p), pd in zip(sparse.named_parameters(), dense.parameters()):
        g = p.grad
        if n in tables:
            assert g.is_sparse and g.shape == p.shape, n
            want = expected_rows(batch, tables[n], p.shape[0])
            assert np.array_equal(g._indices().cpu().numpy(), want[None]), n
            assert g._values().shape == (want.size, p.shape[1]), n
            g = g.to_dense()
        else:
            assert not g.is_sparse, n
        assert_grad_close(g.cpu().numpy(), gold[f"grad.{kind}.{n}"], gmax, f"{name}/{n} sparse vs reference")
        assert_grad_close(g.cpu().numpy(), pd.grad.cpu().numpy(), gmax, f"{name}/{n} sparse vs dense")


@pytest.mark.parametrize("name", CASES)
def test_sparse_backward_matches_dense_and_reference(emu, name):
    check_sparse_backward(name, "cpu", "bpr" if "bpr" in name else "list")


def test_inference_builds_no_row_set(emu):
    cfg, batch, state, _ = load_model_case("script_pl_gru")
    model = P.make_model(dataclasses.replace(cfg, sparse_grad=1), state, "cpu").train()
    with torch.no_grad():
        model(batch)
    assert model._row_sets_current is None and not model._row_slot


def test_interleaved_forward_passes(emu):
    """Two training forward passes before their backward passes: each backward still writes through its own row set."""
    cfg, batch, state, _ = load_model_case("script_pl_gru")
    from intel_sigir2023_b200 import losses
    b2 = {k: (v.flip(0) if torch.is_tensor(v) and v.dim() > 0 else v) for k, v in batch.items()}
    b2 = {k: (v[:3] if torch.is_tensor(v) and v.dim() > 0 else v) for k, v in b2.items()}
    b2["batch_size"] = 3
    crit = losses.IntListloss(P.loss_args())
    ref = []
    for b in (batch, b2):
        m, _, _ = run_step(cfg, state, b, "cpu", 1)
        ref.append(m.iid_embeddings.weight.grad.to_dense())
    model = P.make_model(dataclasses.replace(cfg, sparse_grad=1), state, "cpu").train()
    l1 = crit(model(batch), batch)[0]
    l2 = crit(model(b2), b2)[0]
    l1.backward()
    g1 = model.iid_embeddings.weight.grad.to_dense()
    model.zero_grad(set_to_none=True)
    l2.backward()
    assert torch.equal(g1, ref[0]) and torch.equal(model.iid_embeddings.weight.grad.to_dense(), ref[1])


# ---- optimizer ------------------------------------------------------------------------------------------------------

def _opt_model(device):
    torch.manual_seed(0)
    m = torch.nn.Module()
    m.table = torch.nn.Embedding(300, 16)        # float4 rows
    m.odd = torch.nn.Embedding(50, 3)            # d % 4 != 0
    m.lin = torch.nn.Linear(7, 5)
    return m.to(device)


def _sparse_grad(n_rows, rows, vals, device, own_key=None):
    from intel_sigir2023_b200 import optim
    idx = torch.as_tensor(rows, dtype=torch.int64).to(device)
    if own_key is not None:                      # as IntEL's backward registers its own (coalesced) row buffers
        optim.note_coalesced_rows(own_key, idx)
    return torch.sparse_coo_tensor(idx.view(1, -1), vals.to(device), size=(n_rows, vals.shape[1]), is_coalesced=True,
                                   check_invariants=False)


def _restated_rows_step(p, m, v, rows, g, step, lr, wd):
    """torch.optim.Adam on the gathered rows and their moments"""
    q = torch.nn.Parameter(p[rows].clone())
    opt = torch.optim.Adam([q], lr=lr, weight_decay=wd)
    opt.state[q] = {"step": torch.tensor(float(step - 1)), "exp_avg": m[rows].clone(), "exp_avg_sq": v[rows].clone()}
    q.grad = g.clone()
    opt.step()
    st = opt.state[q]
    return q.detach(), st["exp_avg"], st["exp_avg_sq"]


def check_rows_adam(device, steps=5, wd=1e-4, lr=3e-3):
    from intel_sigir2023_b200 import optim
    g = torch.Generator().manual_seed(7)
    model = _opt_model(device)
    opt = optim.Adam(optim.customize_parameters(model), lr=lr, weight_decay=wd)
    sched = torch.optim.lr_scheduler.StepLR(opt, step_size=2, gamma=0.5)
    ref = {n: [p.detach().cpu().clone(), torch.zeros(p.shape), torch.zeros(p.shape)] for n, p in model.named_parameters()}
    for it in range(steps):
        lr_now = opt.param_groups[0]["lr"]
        for n, p in model.named_parameters():
            if n.startswith("lin"):
                p.grad = torch.randn(p.shape, generator=g).to(device)
                continue
            n_rows, d = p.shape
            rows = torch.randperm(n_rows, generator=g)[: max(1, n_rows // 3)].sort().values
            vals = torch.randn(rows.numel(), d, generator=g)
            if it == 2 and n == "table.weight":             # an accumulated gradient: duplicate and unsorted indices
                half = rows.numel() // 2
                idx = torch.cat([rows.flip(0), rows[:half]])
                extra = torch.randn(half, d, generator=g)
                p.grad = torch.sparse_coo_tensor(idx.view(1, -1).to(device), torch.cat([vals.flip(0), extra]).to(device),
                                                 size=p.shape, check_invariants=False)
                vals = vals.clone()
                vals[:half] += extra
            else:
                p.grad = _sparse_grad(n_rows, rows, vals, device, own_key=("test", n) if it % 2 == 0 else None)
            rp, rm, rv = ref[n]
            before = [t.clone() for t in (rp, rm, rv)]
            nq, nm, nv = _restated_rows_step(rp, rm, rv, rows, vals, it + 1, lr_now, wd)
            rp[rows], rm[rows], rv[rows] = nq, nm, nv
            ref[n].append((rows, before))
        opt.step()
        sched.step()
        for n, p in model.named_parameters():
            if n.startswith("lin"):
                continue
            rp, rm, rv, (rows, before) = ref[n][0], ref[n][1], ref[n][2], ref[n].pop()
            st = opt.state[p]
            got = [t.detach().cpu() for t in (p, st["exp_avg"], st["exp_avg_sq"])]
            untouched = torch.ones(p.shape[0], dtype=torch.bool)
            untouched[rows] = False
            for x, want_all, was in zip(got, (rp, rm, rv), before):
                assert torch.equal(x[untouched], was[untouched]), (n, it, "untouched rows moved")
                assert rel_err(x[rows].numpy(), want_all[rows].numpy()) < 2e-6, (n, it)
            # keep the restatement on the optimizer's values (torch's kernels may differ in the last ulp)
            rp.copy_(got[0]); rm.copy_(got[1]); rv.copy_(got[2])
    assert opt.state[model.table.weight]["step"] == steps


def test_rows_adam_matches_restatement(emu):
    check_rows_adam("cpu")


def test_rows_adam_all_rows_equals_dense(emu):
    """every row touched: the sparse step is bitwise the dense optim.Adam step, also across a state_dict round trip"""
    from intel_sigir2023_b200 import optim
    g = torch.Generator().manual_seed(9)
    ma, mb = _opt_model("cpu"), _opt_model("cpu")
    oa = optim.Adam(optim.customize_parameters(ma), lr=2e-3, weight_decay=1e-3)
    ob = optim.Adam(optim.customize_parameters(mb), lr=2e-3, weight_decay=1e-3)
    for it in range(4):
        for (n, pa), pb in zip(ma.named_parameters(), mb.parameters()):
            gr = torch.randn(pa.shape, generator=g)
            pb.grad = gr.clone()
            if n.startswith("lin"):
                pa.grad = gr.clone()
            else:
                pa.grad = _sparse_grad(pa.shape[0], torch.arange(pa.shape[0]), gr, "cpu", own_key=("all", n))
        oa.step()
        ob.step()
        if it == 1:                      # dense state into the sparse optimizer and back
            oa.load_state_dict(copy.deepcopy(ob.state_dict()))
            ob.load_state_dict(copy.deepcopy(oa.state_dict()))
    for (n, pa), pb in zip(ma.named_parameters(), mb.parameters()):
        assert torch.equal(pa, pb), n
        for k in ("exp_avg", "exp_avg_sq"):
            assert torch.equal(oa.state[pa][k], ob.state[pb][k]), (n, k)


def test_model_step_with_sparse_tables(emu):
    """one training step of IntEL(sparse_grad=1) + optim.Adam: the listed rows move like the dense step's rows, the others
    keep their values (the L2 of the weight group moves every row in the dense step)"""
    from intel_sigir2023_b200 import optim
    cfg, batch, state, _ = load_model_case("script_pl_gru")
    res = []
    for sp in (0, 1):
        model, _, _ = run_step(cfg, state, batch, "cpu", sp)
        opt = optim.Adam(optim.customize_parameters(model), lr=1e-2, weight_decay=0.0)
        opt.step()
        res.append(model)
    for (n, pd), ps in zip(res[0].named_parameters(), res[1].parameters()):
        assert torch.equal(pd, ps), n


# ---- two ranks (gloo) ------------------------------------------------------------------------------------------------

def _sparse_grads_dp(rank, world, case, overlap):
    from intel_sigir2023_b200 import dp, losses, synthetic
    cfg, batch, state, _ = load_model_case(case)
    B = batch["batch_size"]
    keep = B - (B % 2)
    batch = {k: (v[:keep] if torch.is_tensor(v) else v) for k, v in batch.items()}
    batch["batch_size"] = keep
    shard = synthetic.shard_batch(batch, rank, world)
    model = P.make_model(dataclasses.replace(cfg, sparse_grad=1), state, "cpu").train()
    crit = losses.IntListloss(P.loss_args())
    reducer = dp.GradReducer(model, world, overlap=overlap)
    loss, _, _ = crit(model(shard), shard)
    loss.backward()
    reducer.allreduce()
    out = {}
    for n, p in model.named_parameters():
        g = p.grad
        out[n] = (g._indices().numpy().copy(), g._values().numpy().copy()) if g.is_sparse else (None, g.numpy().copy())
    return out


def _worker(rank, world, port, case, overlap, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.set_num_threads(1)
    _setup_emu()
    dist.init_process_group("gloo", rank=rank, world_size=world)
    grads = _sparse_grads_dp(rank, world, case, overlap)
    if rank == 0:
        q.put(grads)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("case,overlap", [("script_bpr_gru_k4", True), ("default_bert", False)])
def test_two_rank_sparse_grads_match_single_process(case, overlap):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + (os.getpid() % 2000) + (7 if overlap else 0)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, case, overlap, q)) for r in range(2)]
    for p in procs:
        p.start()
    two = q.get(timeout=300)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    from intel_sigir2023_b200 import _lib
    old = (_lib._lib, _lib._allow_host_tensors)
    _setup_emu()
    try:
        one = _sparse_grads_dp(0, 1, case, overlap)
    finally:
        _lib._lib, _lib._allow_host_tensors = old
    gmax = max(float(np.abs(v).max()) for _, v in one.values())
    for k, (idx, v) in one.items():
        idx2, v2 = two[k]
        if idx is not None:
            assert np.array_equal(idx, idx2), k
        err = np.abs(v - v2).max()
        assert err <= 1e-4 * float(np.abs(v).max()) + 2e-6 * gmax, (k, err)


# ---- on the B200 ----------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_gpu_rowset_matches_unique():
    check_rowset_cases("cuda")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["script_pl_gru", "default_bert"])
def test_gpu_sparse_backward_golden(name):
    check_sparse_backward(name, "cuda")


@pytest.mark.gpu
def test_gpu_rows_adam_matches_restatement():
    check_rows_adam("cuda")


@pytest.mark.gpu
def test_gpu_c2_sparse_matches_dense():
    """C2 shape (4096 sessions x 50 items, 1M items, GRU4Rec + the IntEL.sh 'pl' widths) on the tcgen05 paths: sparse
    gradients agree with the dense ones, and three optimizer steps match the row-gathered torch.optim.Adam restatement."""
    import argparse
    from intel_sigir2023_b200 import losses, optim, synthetic
    from intel_sigir2023_b200.config import IntelConfig
    from intel_sigir2023_b200.IntEL import IntEL, SPARSE_TABLES
    dev = torch.device("cuda")
    corpus = synthetic.CorpusSpec(n_item=1_000_000, n_class=357, n_user=100_000, n_ctx=931, model_num=4, intent_num=1071,
                                  history_max=20)
    cfg = IntelConfig(item_rows=corpus.item_rows, class_rows=corpus.n_class, user_rows=corpus.user_rows, ctx_rows=corpus.n_ctx,
                      intent_num=corpus.intent_num, model_num=corpus.model_num, history_max=20, encoder="GRU4Rec",
                      context_emb_size=32, intent_emb_size=32, cross_attn_qsize=64, num_heads=2, num_layers=2)
    batches = [synthetic.make_batch(corpus, synthetic.BatchSpec(batch_size=4096, max_len=50, min_len=50), seed=s, device=dev)
               for s in range(3)]
    crit = losses.IntListloss(argparse.Namespace(cal_diversity=1, diversity_alpha=1e-4, intent_weight=0.1, ensemble_weight=1.0,
                                                 kl_temp=2.0, kl_weight=0.5))
    models = []
    for sp in (0, 1):
        torch.manual_seed(0)
        models.append(IntEL(argparse.Namespace(device=dev, model_path="", buffer=1), cfg=dataclasses.replace(cfg, sparse_grad=sp)).to(dev))
    dense, sparse = models
    tables = {n: keys for n, keys, _ in SPARSE_TABLES}
    opt = optim.Adam(optim.customize_parameters(sparse), lr=1e-3, weight_decay=1e-6)
    for it, b in enumerate(batches):
        grads = []
        for m in models:
            m.zero_grad(set_to_none=True)
            out = m(b)
            loss = crit(out, b)[0]
            loss.backward()
            grads.append({n: p.grad for n, p in m.named_parameters()})
        if it == 0:
            gmax = max(float(g.abs().max()) for g in grads[0].values())
            for n, g in grads[1].items():
                if n in tables:
                    assert g.is_sparse
                    want = expected_rows(b, tables[n], g.shape[0])
                    assert np.array_equal(g._indices()[0].cpu().numpy(), want), n
                    g = g.to_dense()
                assert_grad_close(g.cpu().numpy(), grads[0][n].cpu().numpy(), gmax, f"c2/{n}")
        # restatement of the step for the item table: torch.optim.Adam on the gathered rows and their moments
        p = sparse.iid_embeddings.weight
        g = p.grad
        rows, vals = g._indices()[0], g._values()
        st = opt.state.get(p)
        m0 = st["exp_avg"][rows] if st else torch.zeros_like(vals)
        v0 = st["exp_avg_sq"][rows] if st else torch.zeros_like(vals)
        want = _restated_rows_step(p.detach(), torch.zeros_like(p).index_copy_(0, rows, m0),
                                   torch.zeros_like(p).index_copy_(0, rows, v0), rows, vals, it + 1, 1e-3, 1e-6)
        before = p.detach().clone()
        opt.step()
        assert rel_err(p.detach()[rows].cpu().numpy(), want[0].cpu().numpy()) < 2e-6
        assert rel_err(opt.state[p]["exp_avg_sq"][rows].cpu().numpy(), want[2].cpu().numpy()) < 2e-6
        untouched = torch.ones(p.shape[0], dtype=torch.bool, device=dev)
        untouched[rows] = False
        assert torch.equal(p.detach()[untouched], before[untouched])
        dense.load_state_dict(sparse.state_dict())
