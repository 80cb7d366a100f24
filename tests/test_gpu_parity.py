"""Parity gate on the B200: host layer -> C ABI -> sm_100a kernels against the golden vectors of the
unmodified reference and the CPU oracle (bit-exact for index work, 1e-5 relative for fp32, NDCG to 1e-6)."""
import pytest
import torch

import parity_checks as P
from conftest import MODEL_CASES

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(scope="module", autouse=True)
def real_lib():
    from intel_sigir2023_b200 import _lib
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    lib = _lib.load()
    assert not _lib._allow_host_tensors
    assert lib._name.endswith("libintel_b200.so")
    yield


def test_cpu_tensors_are_rejected():
    from intel_sigir2023_b200 import _lib
    with pytest.raises(RuntimeError):
        _lib.ptr(torch.zeros(3))


def test_linear():
    P.check_linear(DEV)


def test_linear_grads():
    P.check_linear_grads(DEV)


def test_mha_blocks():
    P.check_mha(DEV)


def test_gather_scatter():
    P.check_gather_scatter(DEV)


@pytest.mark.parametrize("name", MODEL_CASES)
def test_forward(name):
    P.check_forward(name, DEV)


@pytest.mark.parametrize("name", MODEL_CASES)
@pytest.mark.parametrize("kind", ["list", "bpr", "mse"])
def test_backward(name, kind):
    P.check_backward(name, kind, DEV)


def test_loss_edge_cases():
    P.check_loss_edge_cases(DEV)


def test_gru_prep_index_kernels():
    P.check_gru_prep(DEV)


def test_bert_fused_vs_staged():
    P.check_bert_fused_vs_staged(DEV)


def test_bert_fused_token_tiles():
    P.check_bert_fused_token_tiles(DEV, B=37)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["script_pl_gru", "default_bert"])
def test_phased_backward_equals_single_call(name):
    P.check_phased_backward(DEV, name)


def test_list_loss_bucket_and_pair_forms():
    P.check_list_loss_forms(DEV)


@pytest.mark.parametrize("tag", ["A", "B", "C"])
def test_evaluate(tag):
    P.check_evaluate(tag, DEV)


def test_evaluate_ties():
    P.check_evaluate_ties(DEV)


def test_evaluate_intents():
    P.check_evaluate_intents(DEV)


def test_baselines():
    P.check_baselines(DEV)


@pytest.mark.parametrize("cfg", [
    dict(B=70, L=21, encoder="GRU4Rec", num_heads=2, num_layers=2, context_emb_size=32, intent_emb_size=32),
    dict(B=37, L=100, min_len=40, encoder="BERT4Rec", num_heads=1, num_layers=1),
    dict(B=9, L=130, min_len=90, kind="bpr", encoder="GRU4Rec", num_heads=2, num_layers=1, cross_attn_qsize=64),
    dict(B=33, L=50, min_len=50, kind="mse", encoder="BERT4Rec", cross_attention=0, num_heads=2,
         corpus_kw=dict(model_num=4, intent_num=120, history_max=20)),
])
def test_against_oracle(cfg):
    P.check_against_oracle(DEV, **cfg)


def test_compact_layout_matches_dense():
    P.check_compact_layout(DEV)


def test_linear_large_tcgen05_vs_mma_sync():
    P.check_linear_large(DEV)


def test_rows_gemm_persistent_tcgen05():
    P.check_rows_gemm(DEV)


def test_fused_stack_matches_staged():
    P.check_fused_vs_staged(DEV)


def test_awelv_matches_reference_golden():
    P.check_awelv(DEV)


def test_fused_adam_matches_torch():
    P.check_adam(DEV)


def test_fused_stack_shapes():
    P.check_fused_shapes(DEV)


def test_tcgen05_stack_matches_mma_sync_stack():
    P.check_tc_stack(DEV)


def test_tcgen05_gru_matches_mma_sync_gru():
    P.check_gru_tc(DEV)


def test_tcgen05_gru_matches_mma_sync_gru_long_histories():
    P.check_gru_tc(DEV, history_max=70)


def test_dropout():
    P.check_dropout(DEV)
