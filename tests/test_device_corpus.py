"""Columnar reader + device-side batch construction (SURVEY.md 8f-2 / 8f-3) against the UNMODIFIED reference pipeline on
the bundled Tmall toy sample: `SeqReader` -> `IntEL.Dataset._get_feed_dict` -> `collate_batch`
(helpers/SeqReader.py, models/BaseModel.py:121-197, models/GeneralSeq.py:35-54, models/IntEL/IntEL.py:220-239).

The batch builder kernel runs on the GPU where there is one (`-m gpu`) and on the CPU kernel emulator otherwise, so the
comparison is exercised in the build container as well.  The per-session list shuffle of the reference draws from numpy's
global RNG; the test replays the same draws and hands the permutation to the builder.
"""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
from oracle import ref_run  # noqa: E402

needs_ref = pytest.mark.skipif(not ref_run.available(), reason="no reference tree (oracle/_ref or /root/reference)")


@pytest.fixture(scope="module")
def device():
    from intel_sigir2023_b200 import _lib
    if torch.cuda.is_available():
        yield torch.device("cuda")
        return
    from build_emu import build_emu
    old = (_lib._lib, _lib._allow_host_tensors)
    _lib._lib = None
    _lib.load(build_emu())
    _lib._allow_host_tensors = True
    yield torch.device("cpu")
    _lib._lib, _lib._allow_host_tensors = old


@pytest.fixture(scope="module")
def wired(tmp_path_factory):
    return ref_run.wire("IntEL", "IntListloss", "BaseRunner", ref_run.SCRIPT_FLAGS["pl"], torch.device("cpu"),
                        str(tmp_path_factory.mktemp("ref")))


@pytest.fixture(scope="module")
def columnar(wired):
    from intel_sigir2023_b200.corpus import ColumnarCorpus
    a = wired.args
    return ColumnarCorpus(a.datapath, a.dataset, max_session_len=a.max_session_len, intent_note=a.intent_note,
                          history_max=a.history_max, model_num=a.model_num)


@needs_ref
def test_reader_reports_the_reference_corpus_sizes(wired, columnar):
    ref = wired.corpus
    assert (columnar.max_uid, columnar.max_iid) == (ref.max_uid, ref.max_iid)
    assert columnar.itemfnum == ref.itemfnum and columnar.contextfnum == ref.contextfnum and columnar.userfnum == ref.userfnum
    assert len(columnar.zero_int) == len(ref.zero_int)
    for p in ("train", "dev", "test"):
        d = ref.interactions[p]
        assert np.array_equal(columnar.phase[p]["c_id_c"], d["c_id_c"])
        assert np.array_equal(columnar.phase[p]["position"], d["position"])
        assert np.array_equal(columnar.phase[p]["item_position"], d["item_position"])
    from intel_sigir2023_b200.config import IntelConfig
    assert IntelConfig.from_args(wired.args, columnar) == IntelConfig.from_args(wired.args, ref)


def _dense(idx, val, I):
    out = torch.zeros(*idx.shape[:2], I, dtype=torch.float64)
    out.scatter_add_(2, idx.long(), val.double())
    return out


@needs_ref
@pytest.mark.parametrize("phase,rows", [("train", list(range(40, 104))), ("train", [0, 1, 2, 700, 1105]), ("dev", list(range(0, 48))),
                                        ("test", list(range(400, 512)))])
def test_device_built_batch_equals_collate_batch(wired, columnar, device, phase, rows):
    from intel_sigir2023_b200.corpus import DeviceCorpus
    ds = wired.data[phase]
    # the reference batch; every _get_feed_dict draws its list permutation with np.random.choice (BaseModel.py:194-196)
    np.random.seed(123)
    if phase == "train":
        feed = [ds._get_feed_dict(i) for i in rows]
    else:
        feed = [ds[i] for i in rows]          # dev / test are buffered at prepare() time: compare un-permuted content below
    ref = ds.collate_batch(feed)
    dc = DeviceCorpus.from_columnar(columnar, phase, device)
    L, H1, H2 = dc.shape_of(np.asarray(rows))
    assert (L, H1, H2) == (ref["i_id_s"].shape[1], ref["his_context_mh"].shape[1], ref["his_item_id"].shape[1])
    # recover the permutation the reference applied: replay the draws for train, match item ids for the buffered phases
    perm = np.zeros((len(rows), L), dtype=np.int32)
    if phase == "train":
        np.random.seed(123)
        for b, i in enumerate(rows):
            n = int(columnar.phase[phase]["session_len"][i])
            perm[b, :n] = np.random.choice(np.arange(n), n, replace=False)
    else:
        col = columnar.phase[phase]
        for b, i in enumerate(rows):
            n = int(col["session_len"][i])
            stored = col["item_id"][col["item_off"][i]:col["item_off"][i] + n]
            sc = col["scores"][col["item_off"][i]:col["item_off"][i] + n, 0]
            got_id, got_sc = ref["i_id_s"][b, :n].numpy(), ref["scores"][b, :n, 0].numpy()
            used = np.zeros(n, dtype=bool)
            for l in range(n):                     # items can repeat inside a list: match on (id, first score)
                cand = np.nonzero((stored == got_id[l]) & (sc == got_sc[l]) & ~used)[0]
                assert len(cand), (b, l)
                perm[b, l] = cand[0]
                used[cand[0]] = True
    out = dc.batch(np.asarray(rows), perm=torch.from_numpy(perm).to(device))
    out = {k: (v.cpu() if torch.is_tensor(v) else v) for k, v in out.items()}
    for k in ("u_id_c", "c_id_c", "context_mh", "user_mh", "c_paynum_i", "c_favnum_i", "c_clicknum_i", "session_len", "position",
              "history_len", "history_item_len", "i_id_s", "i_class_c", "ranking", "his_context_mh", "his_item_id"):
        assert out[k].dtype == ref[k].dtype == torch.int64, k
        assert torch.equal(out[k], ref[k]), k
    assert out["scores"].dtype == torch.float64 and torch.equal(out["scores"], ref["scores"])       # bit exact
    assert torch.equal(out["intents"], ref["intents"])
    assert torch.equal(_dense(out["his_intents_idx"], out["his_intents_val"], columnar.intent_num).float(), ref["his_intents"].float())
    assert torch.equal(_dense(out["his_item_int_idx"], out["his_item_int_val"], columnar.intent_num), ref["his_item_int"])
    assert out["batch_size"] == ref["batch_size"] and out["phase"] == ref["phase"]


def _ragged(cols, seed=0):
    """the synthetic corpus with every list cut to a random length in 1..L"""
    L = int(cols["session_len"][0])
    n = np.random.default_rng(seed).integers(1, L + 1, len(cols["session_len"]))
    keep = (np.arange(L)[None, :] < n[:, None]).reshape(-1)
    out = dict(cols, session_len=n.astype(np.int64), item_off=np.concatenate([[0], np.cumsum(n)]).astype(np.int64))
    for k in ("item_id", "item_class", "ranking", "scores"):
        out[k] = np.ascontiguousarray(cols[k][keep])
    return out


def test_default_shuffle_is_a_permutation_of_every_list(device):
    from intel_sigir2023_b200.corpus import DeviceCorpus, synthetic_columns
    cols, shared, nz = synthetic_columns(256, 40, 5000, 17, 30, 31, 3, 60, max_his=8, seed=1)
    dc = DeviceCorpus(_ragged(cols), shared, 3, 60, 8, nz, device)
    rows = np.arange(100, 164)
    a = dc.batch(rows, shuffle=False)
    b = dc.batch(rows)
    n = a["session_len"].cpu().numpy()
    ia, ib = a["i_id_s"].cpu().numpy(), b["i_id_s"].cpu().numpy()
    sa, sb = a["scores"].cpu().numpy(), b["scores"].cpu().numpy()
    moved = 0
    for r in range(len(rows)):
        assert sorted(ia[r, :n[r]]) == sorted(ib[r, :n[r]]) and not ib[r, n[r]:].any()
        assert np.allclose(np.sort(sa[r, :n[r], 0]), np.sort(sb[r, :n[r], 0]), rtol=0, atol=0)
        moved += int((ia[r, :n[r]] != ib[r, :n[r]]).any())
    assert moved > len(rows) // 2
