#!/usr/bin/env python
"""IntEL hot-path benchmark (BASELINE.json metric: sessions/sec, train fwd+bwd and eval; one JSON line on stdout, rank 0).

    python bench.py --gpus N --steps K --warmup W [--config c2|c3|c4|c5]     # B200 path (one rank per GPU under torchrun)
    python bench.py --impl reference --steps K --warmup W [--config ...]      # the reference's own CPU PyTorch path

Workloads (BASELINE.json `configs`; SURVEY.md 8d; synthetic Tmall-schema data, random-init weights):
  c2 (default, the configuration the metric is quoted on): configs[1], 50 candidates x K = 4 lists, I = 1071, IntEL-PL flags
      of IntEL/script/IntEL.sh:21, batches of 4096 sessions per GPU; step = model forward + criterion + backward (optimizer
      excluded, SURVEY 8d).  The eval rate (forward under no_grad + evaluate_method) rides along with its own roofline.
  c3: configs[2], LifeData-shaped: K = 2 lists, 21 504 context rows, I = 2048, same step.
  c4: configs[3], eval only: 200 candidates, default BERT4Rec sizes, step = forward + NDCG/HR@{3,1,5,10}.
  c5: configs[4], the fixed-weight ensembles of script/baselines.sh (SingleSort x K, Borda, random-softmax fusion) + NDCG.
`value`: inputs resident in HBM (three batches larger than L2, cycled).  `e2e`: the same step fed from the HOST through the
public API: the step's session indices (pinned host memory, what a sampler yields) are copied to the device, the batch is
built there from the device-resident columnar corpus (corpus.DeviceCorpus), the result is read back; every step.
`--impl reference`: the UNMODIFIED reference modules from oracle/_ref (oracle/make_ref.py) on the host cores, on a bounded
sample of the same workload; the oracle port only if that copy is absent.
`--dump-outputs DIR`: after the timed steps, what the last of them returned (model outputs, losses and parameter gradients
of a train step; outputs and NDCG sums of an eval or baselines step) as DIR/<name>.npy.  The inputs and initial weights
are drawn from fixed seeds, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from intel_sigir2023_b200 import synthetic                     # noqa: E402
from intel_sigir2023_b200.config import IntelConfig             # noqa: E402

VARIANTS = {
    # the three runs of IntEL/script/IntEL.sh (lines 9, 15, 21) + the bare flag defaults
    "pl": dict(loss="list", encoder="GRU4Rec", context_emb_size=32, intent_emb_size=32, cross_attn_qsize=64,
               num_heads=2, num_layers=2, intent_weight=0.1, diversity_alpha=1e-4),
    "bpr": dict(loss="bpr", encoder="GRU4Rec", context_emb_size=64, intent_emb_size=32, cross_attn_qsize=32,
                num_heads=2, num_layers=2, intent_weight=0.01, diversity_alpha=1e-5),
    "mse": dict(loss="mse", encoder="BERT4Rec", intent_weight=0.003, diversity_alpha=1e-5),
    "default": dict(loss="list", encoder="BERT4Rec", intent_weight=0.1, diversity_alpha=1e-4),
}
MODEL_KEYS = ("encoder", "context_emb_size", "intent_emb_size", "cross_attn_qsize", "num_heads", "num_layers")
CONFIGS = {
    "c2": dict(mode="train", list_len=50, model_num=4, intent_num=1071, n_ctx=931, variant="pl", batch=4096,
               name="BASELINE.json configs[1]: IntEL synthetic Tmall-schema, 1M sessions x 50 candidates x K=4 basic lists"),
    "c3": dict(mode="train", list_len=50, model_num=2, intent_num=2048, n_ctx=21504, variant="pl", batch=4096,
               name="BASELINE.json configs[2]: IntEL synthetic LifeData-shaped (K=2 lists, 21 504 context rows, I=2048)"),
    "c4": dict(mode="eval", list_len=200, model_num=4, intent_num=1071, n_ctx=931, variant="default", batch=2048,
               name="BASELINE.json configs[3]: eval-only scoring + NDCG@3 sweep, 10M sessions x 200 candidates"),
    "c5": dict(mode="baselines", list_len=50, model_num=4, intent_num=1071, n_ctx=931, variant="default", batch=4096,
               name="BASELINE.json configs[4]: fixed-weight ensembles of script/baselines.sh (SingleSort x K, Borda, random fusion) + NDCG"),
}
TOPK, METRICS = [3, 1, 5, 10], ["NDCG", "HR"]
TENSOR_KERNELS = {"trunk_fwd", "trunk_bwd", "gru_seq_fwd", "gru_seq_bwd", "gemm_fwd", "gemm_dgrad", "gemm_wgrad", "mha_fwd", "mha_bwd"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--variant", default=None, choices=sorted(VARIANTS))
    ap.add_argument("--batch", type=int, default=None, help="sessions per step per GPU")
    ap.add_argument("--list_len", type=int, default=None)
    ap.add_argument("--model_num", type=int, default=None)
    ap.add_argument("--intent_num", type=int, default=None)
    ap.add_argument("--n_item", type=int, default=1_000_000)
    ap.add_argument("--n_user", type=int, default=100_000)
    ap.add_argument("--resident_batches", type=int, default=3, help="distinct batches kept in HBM and cycled")
    ap.add_argument("--cpu_batch", type=int, default=512, help="sessions per step of the CPU reference sample")
    ap.add_argument("--corpus_batches", type=int, default=16, help="device-resident corpus of the e2e leg, in batches")
    ap.add_argument("--no_cpu_baseline", action="store_true")
    ap.add_argument("--no_e2e", action="store_true")
    ap.add_argument("--e2e_dense_api", action="store_true", help="also time the host-packed dense-API input path of round 1")
    ap.add_argument("--eval_steps", type=int, default=10)
    ap.add_argument("--profile_mode", action="store_true", help="under ncu: only warm-up + timed steps, nothing else")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (see dump_outputs), to compare builds")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 path (--impl b200)")
    c = CONFIGS[a.config]
    for k in ("variant", "batch", "list_len", "model_num", "intent_num"):
        if getattr(a, k) is None:
            setattr(a, k, c[k])
    a.mode, a.n_ctx = c["mode"], c["n_ctx"]
    return a


def make_cfg(a) -> tuple:
    v = VARIANTS[a.variant]
    n_ctx = getattr(a, "n_ctx", 931)
    corpus = synthetic.CorpusSpec(n_item=a.n_item, n_class=357, n_user=a.n_user, n_ctx=n_ctx, model_num=a.model_num,
                                  intent_num=a.intent_num, history_max=20)
    cfg = IntelConfig(item_rows=corpus.item_rows, class_rows=corpus.n_class, user_rows=corpus.user_rows,
                      ctx_rows=corpus.n_ctx, intent_num=corpus.intent_num, model_num=corpus.model_num,
                      history_max=20, **{k: v[k] for k in MODEL_KEYS if k in v})
    loss_args = argparse.Namespace(cal_diversity=1, diversity_alpha=v["diversity_alpha"], intent_weight=v["intent_weight"],
                                   ensemble_weight=1.0, kl_temp=2.0, kl_weight=0.5)
    return corpus, cfg, v["loss"], loss_args


def batch_bytes(batch) -> int:
    return sum(t.numel() * t.element_size() for t in batch.values() if torch.is_tensor(t))


DUMP_BYTES = 60 << 20        # array data; with the .npy headers the files stay under 64 MB


def dump_outputs(arrays, out_dir: str) -> None:
    """Writes every tensor of `arrays` as <out_dir>/<name>.npy: float64 stays float64, other floating types become
    float32, integers float64.  Their data totals DUMP_BYTES at most: the smaller arrays are written whole, and an array
    beyond its share of what is left keeps a seeded sample of its rows along the first axis (of its elements if one row
    is already too large), drawn first among the rows that are not all zero, so that a sparse gradient such as that of
    an embedding table keeps the rows the step touched.  The indices of the kept rows go to <name>.rows.npy (float64,
    ascending); they are part of what two builds compare."""
    os.makedirs(out_dir, exist_ok=True)

    def dtype_of(t):
        return torch.float32 if t.is_floating_point() and t.dtype != torch.float64 else torch.float64

    items = sorted(arrays.items(), key=lambda kv: kv[1].numel() * dtype_of(kv[1]).itemsize)
    left = DUMP_BYTES
    for j, (name, t) in enumerate(items):
        t = t.detach().to(dtype_of(t))
        share = left // (len(items) - j)
        if t.dim() > 0 and t.numel() * t.element_size() > share:
            if t[0].numel() * t.element_size() + 8 > share:
                t = t.reshape(-1)
            n, row_bytes = t.shape[0], t[0].numel() * t.element_size()
            k = min(n, share // (row_bytes + 8))                  # + 8: the row's entry in <name>.rows.npy
            live = (t.reshape(n, -1) != 0).any(1).nonzero().flatten().cpu().numpy()
            rng = np.random.default_rng(0)
            if len(live) >= k:
                rows = rng.choice(live, k, replace=False)
            else:
                rows = np.concatenate([live, rng.choice(np.setdiff1d(np.arange(n), live), k - len(live), replace=False)])
            rows = np.sort(rows)
            t = t.index_select(0, torch.from_numpy(rows).to(t.device))
            np.save(os.path.join(out_dir, name + ".rows.npy"), rows.astype(np.float64))
            left -= rows.size * 8
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())
        left -= t.numel() * t.element_size()


def metric_name(mode: str) -> str:
    return {"train": "sessions/sec (train fwd+bwd)", "eval": "sessions/sec (eval: forward + NDCG/HR@k)",
            "baselines": "sessions/sec (fixed-weight ensembles + NDCG/HR@k)"}[mode]


def workload_config(a, cfg, loss_kind, batch):
    return {"workload": f"{CONFIGS[a.config]['name']}; streamed in batches of {batch} sessions"
                        + (f" (1M sessions = {1_000_000 // max(batch, 1)} such steps)" if a.config == "c2" else ""),
            "config_id": a.config, "step": a.mode, "list_len": a.list_len, "model_num": a.model_num, "intent_num": a.intent_num,
            "context_rows": cfg.ctx_rows, "variant": f"IntEL-{a.variant} (IntEL/script/IntEL.sh flags)", "loss": loss_kind,
            "cal_diversity": 1, "encoder": cfg.encoder, "num_heads": cfg.num_heads, "num_layers": cfg.num_layers,
            "batch_per_gpu": batch, "history_max": 20, "n_item": cfg.item_rows - 1,
            "input_layout": "dense reference API (float64 [B,H,I] history intents) for `value`; device-built compact batches for `e2e`",
            "l2_policy": "inputs larger than L2 (resident batches of 0.1-1.5 GB, cycled)"}


# ------------------------------------------------------------------------------------------------
def cpu_reference_rate(a, corpus, cfg, loss_kind, loss_args, steps: int, warmup: int):
    """The reference's CPU PyTorch path on this host's cores on a bounded sample (B = --cpu_batch sessions per step):
    the UNMODIFIED reference modules when oracle/_ref is present (kind "reference"), else the oracle port (kind "port")."""
    from oracle import intel_oracle as O
    from oracle import ref_run
    ncores = os.cpu_count() or 1
    torch.set_num_threads(ncores)
    B, L = a.cpu_batch, a.list_len
    batch = synthetic.make_batch(corpus, synthetic.BatchSpec(batch_size=B, max_len=L, min_len=L), seed=11)
    kind = "reference" if ref_run.available() else "port"
    kw = dict(cal_diversity=1, diversity_alpha=loss_args.diversity_alpha, intent_weight=loss_args.intent_weight,
              ensemble_weight=1.0, kl_weight=0.5, kl_temp=2.0)
    pos = {k: batch[k].numpy() for k in ("c_paynum_i", "c_favnum_i", "c_clicknum_i")}
    if a.mode == "baselines":
        kind = "port"

        def step():
            for fn in [lambda b, k=k: O.single_sort(b, k) for k in range(3)] + [O.borda, lambda b: O.random_fusion(b, torch.rand(b["scores"].shape))]:
                ens = fn(batch)["ens_score"].numpy()
                O.evaluate_method(list(ens), list(batch["ranking"].numpy()), pos, TOPK, METRICS, batch["session_len"].numpy())
    elif kind == "reference":
        model, crit = ref_run.reference_on_synthetic(cfg, loss_kind, dict(diversity_alpha=loss_args.diversity_alpha,
                                                                          intent_weight=loss_args.intent_weight))
        runner_cls = ref_run._cls("helpers", "BaseRunner")
        if a.mode == "train":
            def step():
                model.zero_grad()
                loss, _, _ = crit(model(batch), batch)
                loss.backward()
        else:
            model.eval()

            def step():
                with torch.no_grad():
                    ens = model(batch)["ens_score"].numpy()
                runner_cls.evaluate_method(list(ens), list(batch["ranking"].numpy()), pos, TOPK, METRICS, batch["session_len"].numpy())
    else:
        sd = {k: v.requires_grad_(a.mode == "train") for k, v in O.init_state(cfg, seed=0).items()}
        noise = torch.rand(B, L, L) if loss_kind == "bpr" else None

        def step():
            if a.mode == "train":
                for p in sd.values():
                    p.grad = None
                loss, _, _ = O.total_loss(loss_kind, O.forward(sd, cfg, batch), batch, noise=noise, **kw)
                loss.backward()
            else:
                with torch.no_grad():
                    ens = O.forward(sd, cfg, batch)["ens_score"].numpy()
                O.evaluate_method(list(ens), list(batch["ranking"].numpy()), pos, TOPK, METRICS, batch["session_len"].numpy())
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    what = {"train": "fwd+loss+bwd", "eval": "forward + evaluate_method", "baselines": "3 SingleSort + Borda + random fusion, each + evaluate_method"}[a.mode]
    return (B * steps / dt, dt / steps * 1e3, ncores, kind,
            f"{steps} steps x {B} sessions (L={L}, K={a.model_num}, I={a.intent_num}), {what}, torch {torch.__version__} on {ncores} threads")


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    corpus, cfg, loss_kind, loss_args = make_cfg(a)
    # a step of this arm is a --cpu_batch sample of the same workload (~0.1-0.3 s on 16 cores): K <= 100 keeps the run short
    steps, warmup = max(1, min(a.steps, 100)), max(1, min(a.warmup, 5))
    rate, ms, ncores, kind, sample = cpu_reference_rate(a, corpus, cfg, loss_kind, loss_args, steps, warmup)
    conf = workload_config(a, cfg, loss_kind, a.cpu_batch)
    conf["batch_note"] = f"this arm runs {a.cpu_batch}-session steps of the workload (the B200 arm: {a.batch}); rates are per session"
    line = {
        "impl": "reference", "metric": metric_name(a.mode), "value": rate, "unit": "sessions/s",
        "n_gpus": a.gpus, "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": conf,
        "cpu_baseline": {"value": rate, "unit": "sessions/s", "cores": ncores, "kind": kind, "sample": sample},
        "e2e": {"value": rate, "unit": "sessions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm = sorted(float(r[1]) for r in rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            if len(r) >= 9:
                for n, v in zip(names, r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(n)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(rows)}


def load_peaks():
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    hbm_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    tc = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0)))
    tc_src = ("measured (MEASURED_PEAKS.json bf16_tflops_sustained; the TF32 rate is half of it)" if peaks
              else "fallback 1590 TFLOP/s dense bf16 (B200_PROFILING.md)")
    return hbm, hbm_src, tc, tc_src


def roofline_of(prof, prof_steps, traffic, pick=None):
    """roofline object of the kernel with the largest share (or of `pick`) from a live per-kernel profile"""
    hbm_peak, hbm_src, tc_peak, tc_src = load_peaks()
    total_ms = sum(v["ms"] for v in prof.values())
    name, rec = max(prof.items(), key=lambda kv: kv[1]["ms"]) if pick is None else (pick, prof[pick])
    sec = rec["ms"] * 1e-3
    gbs = rec["bytes"] / sec / 1e9 if sec > 0 else 0.0
    if name in TENSOR_KERNELS:
        achieved = 3.0 * rec["flops"] / sec / 1e12 if sec > 0 else 0.0
        roof = {"kernel": name, "bound": "tensor", "achieved": achieved, "peak": tc_peak, "unit": "TFLOP/s", "frac": achieved / tc_peak,
                "peak_source": tc_src, "flops_counted": "TF32 MMA flops issued = 3 x the fp32 product's flops (3xTF32 split for 1e-5 parity)",
                "hbm_gbs_algorithmic": gbs}
    else:
        roof = {"kernel": name, "bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak, "peak_source": hbm_src}
    tr = traffic.get(name)
    roof.update({
        "traffic": tr.get("dram_bytes_per_launch") if isinstance(tr, dict) else None,
        "algorithmic_bytes_per_launch": rec["bytes"] / rec["launches"],
        "share_of_step": rec["ms"] / total_ms if total_ms else None,
        "avg_launch_us": rec["ms"] * 1e3 / rec["launches"],
        "per_kernel": {k: {"share": v["ms"] / total_ms, "ms_per_step": v["ms"] / prof_steps,
                           "gbs": (v["bytes"] / (v["ms"] * 1e-3) / 1e9) if v["ms"] > 0 else 0.0,
                           "tflops_3xtf32": (3.0 * v["flops"] / (v["ms"] * 1e-3) / 1e12) if (v["ms"] > 0 and k in TENSOR_KERNELS) else None,
                           "launches_per_step": v["launches"] / prof_steps}
                       for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])}})
    return roof


def run_b200(a):
    import torch.distributed as dist
    from intel_sigir2023_b200 import _lib, baselines, corpus as corpus_mod, dp, evaluate, loader, losses
    from intel_sigir2023_b200.IntEL import IntEL

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dp.configure_nccl_for_overlap()      # the gradient exchange runs beside the tail of the backward pass (dp.GradReducer)
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()
    spec_corpus, cfg, loss_kind, loss_args = make_cfg(a)
    torch.manual_seed(0)
    model = IntEL(argparse.Namespace(device=dev, model_path="", buffer=1), cfg=cfg).to(dev)
    crit = {"list": losses.IntListloss, "bpr": losses.IntBPRloss, "mse": losses.IntMSEloss}[loss_kind](loss_args)
    reducer = dp.GradReducer(model, world) if (world > 1 and a.mode == "train") else None
    B, L = a.batch, a.list_len
    spec = synthetic.BatchSpec(batch_size=B, max_len=L, min_len=L)
    # weak scaling: every rank owns its own shard of the session stream (different seeds)
    resident = [synthetic.make_batch(spec_corpus, spec, seed=1000 * rank + i, device=dev) for i in range(a.resident_batches)]
    single = [baselines.SingleSort(choose_list=n) for n in ("pCTR", "pCVR", "pFVR")]      # script/baselines.sh:1-20
    borda, fusion = baselines.Borda(), baselines.RandomFusion()

    # keep: a dict that receives what a caller of the step gets back (model outputs, losses, gradients, NDCG sums)
    def train_step(batch, keep=None):
        for p in model.parameters():
            p.grad = None
        out = model(batch)
        loss, ens_l, int_l = crit(out, batch)
        loss.backward()
        if reducer is not None:
            reducer.allreduce()
        if keep is not None:
            keep.update(out, loss=loss, ensemble_loss=ens_l, intent_loss=int_l)
            keep.update({"grad." + n: p.grad for n, p in model.named_parameters() if p.grad is not None})
        return loss

    def ndcg(ens, b):
        return evaluate.ndcg_sums(ens, b["ranking"], b["session_len"], b["c_paynum_i"], b["c_favnum_i"], b["c_clicknum_i"],
                                  max(L, max(TOPK)), TOPK)[0]

    def eval_step(b, keep=None):
        with torch.no_grad():
            out = model(b)
        s = ndcg(out["ens_score"], b)
        if keep is not None:
            keep.update(out, ndcg_sums=s)
        return s

    def baselines_step(b, keep=None):
        s = None
        for name, m in zip(("single_sort_pCTR", "single_sort_pCVR", "single_sort_pFVR", "borda", "random_fusion"),
                           single + [borda, fusion]):
            out = m(b)
            r = ndcg(out["ens_score"], b)
            s = r if s is None else s + r
            if keep is not None:
                keep.update({f"{name}.{k}": v for k, v in out.items()})
        if keep is not None:
            keep["ndcg_sums"] = s
        return s

    step_fn = {"train": train_step, "eval": eval_step, "baselines": baselines_step}[a.mode]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # the step creates a few thousand short-lived Python objects (ctypes structs, autograd nodes); a full
    # gen-2 collection over torch's object graph costs 50-100 ms and would land inside the timed region at random
    import gc
    gc.collect()
    gc.freeze()
    if a.mode != "train":
        model.eval()
    # ---- warm-up, then the timed region (inputs resident in HBM) ----
    for i in range(a.warmup if a.profile_mode else max(a.warmup, 3)):
        step_fn(resident[i % len(resident)])
    sampler = ClockSampler(local) if rank == 0 else None
    last = {} if a.dump_outputs else None
    ms_total = timed(lambda i: step_fn(resident[i % len(resident)], last if i == a.steps - 1 else None), a.steps)
    clocks = sampler.stop() if sampler else None
    if last is not None:
        if rank == 0:
            dump_outputs(last, a.dump_outputs)
        last.clear()
    ms_step = ms_total / a.steps
    value = world * B / (ms_step * 1e-3)
    if a.profile_mode:
        if rank == 0:
            print(json.dumps({"profile_mode": True, "ms_per_step_under_profiler": ms_step}))
        return

    # ---- launch count + live per-kernel timing (CUDA events around every launch; separate pass) ----
    def profile(fn, n=3):
        _lib.profile(True)
        for i in range(n):
            fn(resident[i % len(resident)])
        prof = _lib.profile_report()
        _lib.profile(False)
        if "dense_rows_fwd" in prof:
            # the library books every history row of the dense float64 inputs; the kernel skips the padding rows behind
            # history_len / history_item_len, so only the live share of those bytes is actually streamed
            live = [float(b[k].double().mean()) / b[t].shape[1] for b in resident[:n]
                    for k, t in (("history_len", "his_intents"), ("history_item_len", "his_item_int"))]
            prof["dense_rows_fwd"]["bytes"] *= sum(live) / len(live)
        return prof
    prof_steps = 3
    prof = profile(step_fn, prof_steps)
    gpu_launches = int(sum(v["launches"] for v in prof.values()) / prof_steps * a.steps)
    traffic = {}
    for f in ("r02_traffic.json", "r01_traffic.json"):     # dram bytes per launch from the committed ncu --set full captures
        try:
            for k, v in json.load(open(os.path.join(ROOT, "profiles", f))).items():
                traffic.setdefault(k, v)
        except Exception:
            pass
    roofline = roofline_of(prof, prof_steps, traffic)
    # the eval step runs the same kernels in inference mode (nothing saved): their captures are filed under "<kernel>@eval"
    eval_traffic = dict(traffic)
    eval_traffic.update({k[:-5]: v for k, v in traffic.items() if k.endswith("@eval")})

    # ---- eval rate of the train configs (BASELINE metric: "train fwd+bwd and eval"), with the roofline of its own kernels ----
    eval_rate = roofline_eval = None
    if a.mode == "train":
        model.eval()
        for i in range(2):
            eval_step(resident[i % len(resident)])
        ms_eval = timed(lambda i: eval_step(resident[i % len(resident)]), a.eval_steps) / a.eval_steps
        eval_rate = world * B / (ms_eval * 1e-3)
        eprof = profile(eval_step, prof_steps)
        roofline_eval = {"step": "forward (no_grad) + intel_ndcg_topk", "ms_per_step": ms_eval,
                         "dominant": {k: v for k, v in roofline_of(eprof, prof_steps, eval_traffic).items() if k != "per_kernel"}}
        if "ndcg" in eprof:
            roofline_eval["ndcg_kernel"] = {k: v for k, v in roofline_of(eprof, prof_steps, eval_traffic, pick="ndcg").items() if k != "per_kernel"}
        model.train()

    # ---- end to end: host indices -> H2D -> device batch builder -> step -> result D2H, every step ----
    e2e = e2e_dense = None
    if not a.no_e2e:
        n_corpus = a.corpus_batches * B
        cols, shared, nz = corpus_mod.synthetic_columns(n_corpus, L, a.n_item, 357, a.n_user, a.n_ctx, a.model_num, a.intent_num,
                                                        max_his=20, seed=77 + rank)
        dc = corpus_mod.DeviceCorpus(cols, shared, a.model_num, a.intent_num, 20, nz, dev)
        del cols, shared
        order = np.random.default_rng(5 + rank).permutation(n_corpus)
        result_host = torch.zeros(len(TOPK) * 7 if a.mode != "train" else 1, dtype=torch.float64).pin_memory()

        def e2e_step(i):
            rows = order[(i % a.corpus_batches) * B:(i % a.corpus_batches + 1) * B]       # what a sampler hands to the loader
            r = step_fn(dc.batch(rows))
            result_host.copy_(r.detach().reshape(-1)[:result_host.numel()], non_blocking=True)
        for i in range(3):
            e2e_step(i)
        n_e2e = max(5, min(a.steps, 10))
        passes = sorted(timed(e2e_step, n_e2e) / n_e2e for _ in range(3))
        ms = passes[1]
        e2e = {"value": world * B / (ms * 1e-3), "unit": "sessions/s", "h2d_bytes_per_step": B * 8, "d2h_bytes_per_step": result_host.numel() * 8,
               "ms_per_step": ms, "passes_ms": passes, "reported": "median of 3 passes",
               "input_path": "host session indices (pinned) -> H2D -> intel_batch_build from the device-resident columnar corpus "
                             f"({n_corpus} sessions) -> step -> result D2H"}
        del dc
        if a.e2e_dense_api and a.mode == "train":
            host = [{k: (v.cpu().pin_memory() if torch.is_tensor(v) else v) for k, v in b.items()} for b in resident[:2]]
            pf = loader.DevicePrefetcher(iter(host[:1]), dev, pack_history=True)
            h2d = batch_bytes(next(iter(pf)))
            torch.cuda.synchronize()
            loss_host = torch.zeros(1, dtype=torch.float64).pin_memory()

            def dense_pass(_):
                for b in loader.DevicePrefetcher((host[i % len(host)] for i in range(n_e2e)), dev, pack_history=True):
                    loss_host.copy_(train_step(b).detach().reshape(1), non_blocking=True)
            timed(dense_pass, 1)
            ms_d = statistics.median(timed(dense_pass, 1) / n_e2e for _ in range(3))
            e2e_dense = {"value": world * B / (ms_d * 1e-3), "unit": "sessions/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 8,
                         "ms_per_step": ms_d, "input_path": "pinned host batches in the reference's dense float64 layout, history tensors "
                                                            "packed by host threads, H2D of step i+1 on a copy stream (round-1 e2e)"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    line = {
        "metric": metric_name(a.mode), "value": value, "unit": "sessions/s", "n_gpus": world,
        "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(a, cfg, loss_kind, B), "clocks": clocks, "gpu_launches": gpu_launches, "roofline": roofline,
    }
    if eval_rate is not None:
        line["eval_sessions_per_s"] = eval_rate
        line["roofline_eval"] = roofline_eval
    if e2e is not None:
        line["e2e"] = e2e
    if e2e_dense is not None:
        line["e2e_dense_api"] = e2e_dense
    if not a.no_cpu_baseline and world == 1:
        rate, ms, ncores, kind, sample = cpu_reference_rate(a, spec_corpus, cfg, loss_kind, loss_args, 40, 2)     # ~10 s of CPU work
        line["cpu_baseline"] = {"value": rate, "unit": "sessions/s", "cores": ncores, "kind": kind, "sample": sample}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)
