"""Host side of candidate ranking (no GPU): the item -> category table, the ordering / rank / metric helpers against a literal
restatement, and argument checks of the C ABI and the Python layers."""
import ctypes as C
import math
import pickle

import numpy as np
import pytest

from pamrec_b200 import deeprec_utils as DU
from pamrec_b200 import sequential_iterator as IT


def _iterator(tmp_path, n_items=12):
    d = tmp_path / "wechat"
    d.mkdir()
    for name, voc in (("user_vocab.pkl", {"default_uid": 0, "u1": 1}), ("item_vocab.pkl", {"default_mid": 0, **{f"i{i}": i for i in range(1, n_items)}}),
                      ("category_vocab.pkl", {"default_cat": 0, **{f"c{i}": i for i in range(1, 6)}})):
        pickle.dump(voc, open(d / name, "wb"))
    (d / "wechat_business_recommenders.csv").write_text("1\t1\t10.0\n")
    hp = DU.prepare_hparams(None, model_type="mmoe", dataset="wechat", bucket_num=10, batch_size=10, max_seq_length=8,
                            noise_train_hist=0, noise_train_listwise=0, noise_only_predict=0, user_vocab=str(d / "user_vocab.pkl"),
                            item_vocab=str(d / "item_vocab.pkl"), cate_vocab=str(d / "category_vocab.pkl"))
    return IT.SequentialIterator(hp, None), d


def _eval_line(tgt, tcat, hist, hcat):
    n = len(hist)
    return "\t".join(["1", "12000", "u1", tgt, tcat, "10.0", ",".join(hist), ",".join(hcat), ",".join(["10.0"] * n), ",".join(["1"] * n),
                      ",".join(["12000"] * n)])


@pytest.mark.parametrize("python_parser", [False, True])
def test_item_categories_first_occurrence_wins(tmp_path, monkeypatch, python_parser):
    if python_parser:
        monkeypatch.setenv("PAMREC_PY_TOKENIZER", "1")
    it, d = _iterator(tmp_path)
    # line 1: target i3/c1 comes before its history (i3/c2 there); i5 first seen in a history with c4
    (d / "valid_data").write_text(_eval_line("i3", "c1", ["i5", "i3", "i7"], ["c4", "c2", "c3"]) + "\n" +
                                  _eval_line("i5", "c5", ["i7", "unknown"], ["c5", "c2"]) + "\n")
    # a training file (history columns only) read after it: it may add items, never change the ones already seen
    (d / "train_data").write_text("\t".join(["u1", "i7,i9,i3", "c1,c2,c3", "10.0,10.0,10.0", "1,1,1", "12000,12000,12000"]) + "\n")
    table = it.item_categories([str(d / "valid_data"), str(d / "train_data")])
    assert table.dtype == np.int32 and table.shape == (12,)
    want = np.full(12, -1)
    want[3], want[5], want[7], want[9] = 1, 4, 3, 2
    np.testing.assert_array_equal(table, want)              # item 0 (the unknown token's id) is never a candidate
    only_train = it.item_categories([str(d / "train_data")])
    assert only_train[7] == 1 and only_train[9] == 2 and only_train[3] == 3 and only_train[5] == -1


def _literal_order(scores, ids, k, keep):
    """The ordering restated with Python's sort over (-score, id) tuples."""
    out = []
    for r in range(scores.shape[0]):
        rows = sorted((-float(scores[r, j]), int(ids[j])) for j in range(len(ids)) if keep[r, j])[:k]
        out.append([i for _, i in rows] + [-1] * (k - len(rows)))
    return np.asarray(out)


def test_rank_topk_and_own_rank_match_a_literal_restatement():
    rng = np.random.default_rng(3)
    ids = rng.permutation(np.arange(1, 41))[:25]
    scores = rng.integers(0, 6, size=(6, ids.size)).astype(np.float32) / 4         # many ties
    keep = rng.random((6, ids.size)) > 0.3
    for k in (1, 5, 25, 40):                                                       # K larger than the candidate count too
        got_ids, got_sc = DU.rank_topk(scores, ids, k, keep)
        want = _literal_order(scores, ids, k, keep)
        np.testing.assert_array_equal(got_ids, want)
        for r in range(6):
            n = int((want[r] >= 0).sum())
            np.testing.assert_array_equal(got_sc[r, :n], [scores[r, list(ids).index(i)] for i in want[r, :n]])
            assert np.all(np.isneginf(got_sc[r, n:]))
    own = np.array([ids[0], ids[3], 999, ids[7], ids[24], ids[10]])               # 999 is not a candidate
    keep[:, [0, 3, 7, 24, 10]] = True                                              # the own item is never excluded
    ranks = DU.own_rank(scores, ids, own, keep)
    full = _literal_order(scores, ids, ids.size, keep)
    for r in range(6):
        assert ranks[r] == (-1 if own[r] == 999 else list(full[r]).index(own[r]) + 1)


def test_full_ranking_metrics_match_a_literal_restatement():
    ranks = np.array([1, 3, 12, -1, 2, 7, 1, 30])
    labels = np.array([1, 1, 1, 1, 0, 1, 0, 1])          # label-0 lines do not count; rank -1 (not a candidate) is a miss
    got = DU.full_ranking_metrics(ranks, labels, ks=(1, 5, 10))
    pos = [1, 3, 12, None, 7, 30]
    mean = lambda v: round(sum(v) / len(v), 4)
    for k in (1, 5, 10):
        assert got[f"hit@{k}"] == mean([1.0 if r and r <= k else 0.0 for r in pos])
        assert got[f"ndcg@{k}"] == mean([1.0 / math.log2(r + 1) if r and r <= k else 0.0 for r in pos])
    assert got["mrr"] == mean([1.0 / r if r else 0.0 for r in pos])
    assert DU.full_ranking_metrics([], [], ks=(10,)) == {"hit@10": 0.0, "ndcg@10": 0.0, "mrr": 0.0}


def test_candidate_ids_checks():
    from pamrec_b200.models import candidate_ids
    table = np.array([3, 1, -1, 2, 0, -1])               # item 0 has a category entry but is padding
    np.testing.assert_array_equal(candidate_ids(table, None, 6), [1, 3, 4])
    np.testing.assert_array_equal(candidate_ids(table, [4, 1], 6), [4, 1])
    for bad in ([], [1, 1], [0], [6], [2], [1.5]):
        with pytest.raises(ValueError):
            candidate_ids(table, bad, 6)
    with pytest.raises(ValueError):
        candidate_ids(np.full(4, -1), None, 4)


def test_rank_abi_argument_checks(lib_built):
    from pamrec_b200 import _lib as L
    from pamrec_b200.engine import Engine, PamrecError
    eng = Engine(n_users=11, n_items=50, n_cates=7, max_seq_len=8, max_batch=16)
    lib = eng.lib
    for k in (0, L.RANK_MAX_K + 1):
        assert lib.pamrec_rank_scratch_bytes(eng.handle, k) == -1
        assert b"top_k" in lib.pamrec_last_error(eng.handle)
    assert lib.pamrec_rank_scratch_bytes(eng.handle, 1) == lib.pamrec_rank_scratch_bytes(eng.handle, L.RANK_MAX_K) > 50 * 4
    b = L.PamrecBatch(batch=1)
    assert lib.pamrec_rank_candidates(eng.handle, C.byref(b), None, None, 1, 1, 0, None, 0, None, None, None, None) != 0
    assert b"bind" in lib.pamrec_last_error(eng.handle)           # before any device work
    with pytest.raises(PamrecError):
        eng.rank_candidates(None, [1], [1], 0)
    sharded = Engine(n_users=11, n_items=50, n_cates=7, max_seq_len=8, max_batch=16, tables="sharded")
    assert sharded.lib.pamrec_rank_candidates(sharded.handle, C.byref(b), None, None, 1, 1, 0, None, 0, None, None, None, None) != 0
    assert b"one GPU" in sharded.lib.pamrec_last_error(sharded.handle)
    with pytest.raises(PamrecError):
        sharded.rank_candidates(None, [1], [1], 5)
