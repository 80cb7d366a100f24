"""Kernel logic + host orchestration on the CUDA emulator (tests/emu/cuda_emu.h): the same .cu sources
compiled for CPU fibers.  This is a debugger for the build container (no GPU here); the parity gate
proper is tests/test_gpu_parity.py."""
import os
import sys

import pytest

import parity_checks as P
from conftest import MODEL_CASES

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "emu"))


@pytest.fixture(scope="module", autouse=True)
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


def test_linear():
    P.check_linear("cpu")


def test_linear_grads():
    P.check_linear_grads("cpu")


def test_mha_blocks():
    P.check_mha("cpu", shapes=((3, 12, 32, 2), (1, 70, 32, 2), (1, 130, 48, 2)))


def test_gather_scatter():
    P.check_gather_scatter("cpu")


@pytest.mark.parametrize("name", MODEL_CASES)
def test_forward(name):
    P.check_forward(name, "cpu")


@pytest.mark.parametrize("name", MODEL_CASES)
@pytest.mark.parametrize("kind", ["list", "bpr", "mse"])
def test_backward(name, kind):
    if name == "wide_intent_bert_full" and kind != "list":
        pytest.skip("emulator time: covered on the GPU")
    P.check_backward(name, kind, "cpu")


def test_loss_edge_cases():
    P.check_loss_edge_cases("cpu")


def test_list_loss_bucket_and_pair_forms():
    P.check_list_loss_forms("cpu")


@pytest.mark.parametrize("tag", ["A", "B", "C"])
def test_evaluate(tag):
    P.check_evaluate(tag, "cpu")


def test_evaluate_ties():
    P.check_evaluate_ties("cpu")


def test_evaluate_intents():
    P.check_evaluate_intents("cpu")


def test_baselines():
    P.check_baselines("cpu")


def test_against_oracle_multi_tile():
    P.check_against_oracle("cpu", B=35, L=9, encoder="GRU4Rec", num_heads=2, num_layers=1,
                           corpus_kw=dict(history_max=4, intent_num=24))


def test_against_oracle_six_basic_models():
    """model_num = 6: the general instances of the list-loss kernel (bucket sums bounded at 16 models) and of the score
    embedding kernels, and the staged weight head (the folded one covers K = 2..4)"""
    P.check_against_oracle("cpu", seed=4, B=11, L=10, encoder="GRU4Rec", num_heads=2, num_layers=1,
                           corpus_kw=dict(model_num=6, history_max=4, intent_num=24))


def test_against_oracle_wide_score_embedding():
    """s_emb_size = 48: the two-channels-per-lane instance of the score embedding backward and the scalar forward"""
    P.check_against_oracle("cpu", seed=6, B=7, L=8, encoder="GRU4Rec", num_heads=2, num_layers=1, s_emb_size=48,
                           corpus_kw=dict(model_num=5, history_max=4, intent_num=24))


def test_list_loss_forms_seven_models():
    P.check_list_loss_forms("cpu", B=13, L=19, K=7, seed=9)


@pytest.mark.parametrize("intent_num", [12, 2048])
def test_config3_shapes_against_the_oracle(intent_num):
    P.check_config3_shapes("cpu", intent_num)


def test_compact_layout_matches_dense():
    P.check_compact_layout("cpu")


def test_fused_stack_matches_staged():
    P.check_fused_vs_staged("cpu")


def test_awelv_matches_reference_golden():
    P.check_awelv("cpu")


@pytest.mark.parametrize("name", ["gru", "bert"])
def test_awelv_int_matches_reference_golden(name):
    P.check_awelv_int("cpu", name)


@pytest.mark.parametrize("name", ["gru", "bert"])
def test_awelv_intel_matches_reference_golden(name):
    P.check_awelv_intel("cpu", name)


@pytest.mark.parametrize("name", ["h32", "h24_8"])
def test_lambdarank_scorer_matches_reference_golden(name):
    P.check_lambdarank_model("cpu", name)


def test_lambdarank_matches_reference_golden():
    P.check_lambdarank("cpu")


def test_fused_adam_matches_torch():
    P.check_adam("cpu")


def test_fused_stack_shapes():
    P.check_fused_shapes("cpu")


def test_dropout():
    P.check_dropout("cpu")


def test_phased_backward_equals_single_call():
    P.check_phased_backward("cpu")


def test_gru_prep_index_kernels():
    P.check_gru_prep("cpu")


def test_gru_hidden_other_than_128_is_rejected():
    """GRU4Rec runs at hidden size 128 only, the size the reference fixes (IntEL.py:105-106); BERT4Rec ignores gru_hidden"""
    import ctypes
    from intel_sigir2023_b200 import _lib
    from intel_sigir2023_b200.config import IntelConfig
    lib = _lib.load()
    for encoder in ("GRU4Rec", "BERT4Rec"):
        cfg = IntelConfig(item_rows=50, class_rows=7, user_rows=5, ctx_rows=5, intent_num=12, encoder=encoder, gru_hidden=64)
        dims = _lib.make_dims(cfg, B=4, L=6, H1=3, H2=3)
        nbytes = lib.intel_intent_workspace_bytes(ctypes.byref(dims))
        status = lib.intel_intent_fwd(ctypes.byref(dims), None, None, None, None, 0, None)
        if encoder == "GRU4Rec":
            assert nbytes == 0
            assert status == 4, status                  # INTEL_ERR_UNSUPPORTED
            assert b"gru_hidden = 128" in lib.intel_last_error()
        else:
            assert nbytes > 0
            assert status == 1, status                  # INTEL_ERR_ARG: the dims pass, the null tensors do not


def test_bert_fused_vs_staged():
    P.check_bert_fused_vs_staged("cpu", names=("default_bert",))


def test_bert_fused_token_tiles():
    P.check_bert_fused_token_tiles("cpu", B=6)
