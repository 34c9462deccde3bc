"""Host logic pinned against the reference: batches of pamrec_b200.SequentialIterator are BIT-EXACT with the
reference's SequentialIterator (golden fixtures made by oracle/gen_golden.py from the unmodified reference run
under a stub tensorflow), bucket ids and metrics likewise."""
import json
import os
import tempfile

import numpy as np
import pytest

from oracle import gen_golden as G
from pamrec_b200 import deeprec_utils as DU
from pamrec_b200 import sequential_iterator as IT

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _ours(case, data_dir):
    hp = G.hparams_for(case, data_dir)
    return G.run_iterator(lambda: IT.SequentialIterator(hp, None), data_dir)


@pytest.mark.parametrize("case", list(G.CASES))
def test_iterator_matches_golden(case):
    z = np.load(os.path.join(GOLDEN, f"iterator_{case}.npz"))
    with tempfile.TemporaryDirectory() as tmp:
        data_dir = G.synth_case(case, tmp)
        res = _ours(case, data_dir)
    for split in ("train", "valid"):
        want = z[f"{split}_digests"].tolist()
        got = [G.batch_digest(b) for b in res[split]]
        assert len(got) == len(want), (split, len(got), len(want))
        bad = [i for i, (a, b) in enumerate(zip(got, want)) if a != b]
        assert not bad, f"{split}: first differing batch {bad[0]} of {len(want)}"
    for tag, b in (("train_first", res["train"][0]), ("train_last", res["train"][-1]), ("valid_first", res["valid"][0]),
                   ("valid_last", res["valid"][-1])):
        for name in G.FEED_NAMES:
            ref = z[f"{tag}.{name}"]
            assert b[name].dtype == ref.dtype and b[name].shape == ref.shape, (tag, name)
            assert np.array_equal(b[name], ref, equal_nan=True), (tag, name)
    # structure the kernels rely on: train batches are groups of 5 rows sharing one history
    tb = res["train"][0]
    assert tb["items"].shape[0] % 5 == 0
    for k in ("item_history", "item_cate_history", "mask", "item_loop_times_history", "users"):
        a = tb[k].reshape(-1, 5, *tb[k].shape[1:])
        assert (a == a[:, :1]).all(), k


@pytest.mark.parametrize("case", list(G.CASES))
def test_iterator_matches_reference_live(case):
    """A run of one epoch, then the valid pass, against the reference's batches as oracle/gen_golden.py recorded them (a digest
    of the name, dtype, shape and bytes of every array of every batch): the first epoch of the recorded two-epoch run is this
    run, and the valid pass does not depend on how many epochs came before it."""
    z = np.load(os.path.join(GOLDEN, f"iterator_{case}.npz"))
    with tempfile.TemporaryDirectory() as tmp:
        data_dir = G.synth_case(case, tmp)
        hp = G.hparams_for(case, data_dir)
        got = G.run_iterator(lambda: IT.SequentialIterator(hp, None), data_dir, epochs=1)
    first_epoch = {"wechat_small": 134, "takatak_small": 370}[case]         # of the 269 / 739 recorded train batches
    ref = {"train": z["train_digests"].tolist()[:first_epoch], "valid": z["valid_digests"].tolist()}
    for split in ("train", "valid"):
        assert len(got[split]) == len(ref[split]) > 0, split
        for i, (b, want) in enumerate(zip(got[split], ref[split])):
            assert G.batch_digest(b) == want, (split, i)


def test_lisan_known_answers():
    kat = json.load(open(os.path.join(GOLDEN, "lisan.json")))
    xs = np.asarray(kat["x"], dtype=np.float64)
    for key, (ds, num) in {"wechat": ("wechat", 10), "takatak10": ("takatak", 10), "takatak8": ("takatak", 8),
                           "takatak6": ("takatak", 6)}.items():
        assert IT.lisan_array(xs, ds, num).tolist() == kat[key], key
        assert [IT.lisan(float(x), ds, num) for x in xs[:5]] == kat[key][:5]
    assert IT.lisan(float("nan"), "wechat") == 9            # bisect walks right on NaN
    with pytest.raises(Exception):
        IT.lisan(1.0, "taobao")


def test_metrics_match_reference():
    want = json.load(open(os.path.join(GOLDEN, "metrics.json")))
    users, preds, labels, g_labels, g_preds = G.metric_inputs()
    u, p, l = DU.filter_single_class_users(users, preds, labels)
    assert 3 not in u and 4 not in u
    point = DU.cal_metric(l, p, G.POINT_METRICS)
    group = DU.cal_metric(g_labels, g_preds, G.GROUP_METRICS)
    weighted = DU.cal_weighted_metric(u, p, l, G.WEIGHTED_METRICS)
    for got, ref in ((point, want["point"]), (group, want["group"]), (weighted, want["weighted"])):
        assert set(got) == set(ref)
        for k in ref:
            assert abs(float(got[k]) - ref[k]) < 1e-12, (k, got[k], ref[k])
    with pytest.raises(ValueError):
        DU.cal_metric([1, 0], [0.2, 0.3], ["nope"])
    with pytest.raises(ValueError):
        DU.cal_weighted_metric([1, 1], [0.2, 0.3], [1, 0], ["nope"])
    assert DU.cal_metric([1], [0.5], []) == {}


def test_hparams_yaml_and_errors(tmp_path):
    yml = os.path.join(os.path.dirname(GOLDEN), "..", "pamrec_b200", "config", "mmoe.yaml")
    hp = DU.prepare_hparams(yml, dataset="wechat", batch_size=500, max_seq_length=100, embed_l2=1e-6)
    assert hp.expert_num == 5 and hp.gate_layer_sizes == [64, 5] and hp.max_seq_length == 100 and hp.batch_size == 500
    assert hp.time_unit == "s" and hp.max_grad_norm == 2 and hp.embed_l2 == 1e-6 and hp.enable_BN is True
    with pytest.raises(TypeError):
        DU.prepare_hparams(yml, batch_size="500")
    with pytest.raises(TypeError):
        DU.prepare_hparams(yml, learning_rate=1)
    with pytest.raises(ValueError):
        DU.prepare_hparams(yml, weird={"a": 1})
    with pytest.raises(FileNotFoundError):
        DU.prepare_hparams(str(tmp_path / "missing.yaml"))
    bad = tmp_path / "bad.yaml"
    bad.write_text("a: [1, 2\n")
    with pytest.raises(IOError):
        DU.load_yaml(str(bad))


def test_iterator_edge_cases(tmp_path):
    """empty / ragged inputs: users with < 2 satisfied items are skipped, unknown tokens map to id 0, histories
    longer than T keep the most recent T, the tail batch is smaller, negatives in-batch are refused."""
    d = tmp_path / "wechat"
    d.mkdir()
    import pickle
    for name, voc in (("user_vocab.pkl", {"default_uid": 0, "u1": 1, "u2": 2}), ("item_vocab.pkl", {"default_mid": 0, **{str(i): i for i in range(1, 50)}}),
                      ("category_vocab.pkl", {"default_cat": 0, "c1": 1})):
        pickle.dump(voc, open(d / name, "wb"))
    (d / "wechat_business_recommenders.csv").write_text("1\t1\t10.0\n")
    n = 30
    items = ",".join(str(1 + i % 49) for i in range(n))
    line = lambda u, sats: "\t".join([u, items, ",".join(["c1"] * n), ",".join(["10.0"] * n), ",".join(sats), ",".join(["12000"] * n)])
    (d / "train_data").write_text(line("u1", ["1"] * n) + "\n" + line("u2", ["0"] * (n - 1) + ["1"]) + "\n" + line("zzz", ["1", "0"] * (n // 2)) + "\n")
    ev = "\t".join(["1", "12000", "u1", "999", "c1", "10.0", items, ",".join(["c1"] * n), ",".join(["10.0"] * n), ",".join(["1"] * n), ",".join(["12000"] * n)])
    (d / "valid_data").write_text((ev + "\n") * 7)
    hp = DU.prepare_hparams(None, model_type="mmoe", dataset="wechat", bucket_num=10, batch_size=10, max_seq_length=8,
                            noise_train_hist=0, noise_train_listwise=0, noise_only_predict=0, user_vocab=str(d / "user_vocab.pkl"),
                            item_vocab=str(d / "item_vocab.pkl"), cate_vocab=str(d / "category_vocab.pkl"))
    import random
    random.seed(8)
    it = IT.SequentialIterator(hp, None)
    tr = list(it.load_data_from_file(str(d / "train_data")))
    assert all(b["items"].shape[0] % 5 == 0 for b in tr)
    users = np.concatenate([b["users"] for b in tr])
    assert set(users.tolist()) <= {0.0, 1.0}          # u2 has a single satisfied item -> skipped; zzz -> id 0
    assert tr[0]["item_history"].shape == (10, 8)
    va = list(it.load_data_from_file(str(d / "valid_data")))
    assert [b["items"].shape[0] for b in va] == [7]
    assert va[0]["items"][0] == 0                     # unknown item token
    assert (va[0]["mask"].sum(1) == 8).all()          # truncated to the last T
    assert va[0]["item_history"][0].tolist() == [1 + i % 49 for i in range(n - 8, n)]
    assert va[0]["labels_play"][0, 0] == 1.0 and va[0]["plays"][0, 0] == 12.0
    with pytest.raises(NotImplementedError):
        next(it.load_data_from_file(str(d / "valid_data"), batch_num_ngs=4))      # negatives are sampled for the train file only
    assert list(it.load_data_from_file(str(d / "valid_data"), min_seq_length=1000)) == []


@pytest.mark.parametrize("case", list(G.CASES))
def test_native_batcher_equals_python_batcher(case, monkeypatch):
    """csrc/batcher.cu against the pure-Python batcher of the same module: every array of every batch, two epochs
    (the RNG state carries over) and the eval pass; then zero-duration / unsatisfied-eviction / long-history lines."""
    with tempfile.TemporaryDirectory() as tmp:
        data_dir = G.synth_case(case, tmp)
        hp = G.hparams_for(case, data_dir)
        monkeypatch.setenv("PAMREC_PY_ITERATOR", "1")
        py = G.run_iterator(lambda: IT.SequentialIterator(hp, None), data_dir)
        monkeypatch.setenv("PAMREC_PY_ITERATOR", "0")
        it_holder = {}

        def make():
            it_holder["it"] = IT.SequentialIterator(hp, None)
            return it_holder["it"]
        nat = G.run_iterator(make, data_dir)
        assert it_holder["it"].__dict__.get("_native_cache"), "the native batcher was not used"
        assert all(v is not None for v in it_holder["it"]._native_cache.values())
    for split in ("train", "valid"):
        assert len(py[split]) == len(nat[split]) > 0
        for i, (a, b) in enumerate(zip(py[split], nat[split])):
            assert list(a) == list(b)
            for k in a:
                assert a[k].dtype == b[k].dtype and a[k].shape == b[k].shape, (split, i, k)
                assert np.array_equal(a[k], b[k], equal_nan=True), (split, i, k)


def test_native_batcher_hard_lines(tmp_path, monkeypatch):
    """Lines built to hit the branches of add_a_item_to_hist (IT:479-522): > 100 kept items with and without
    unsatisfied entries to evict, plays under 8 s that are dropped, zero durations (inf / NaN ratios)."""
    import pickle
    import random
    d = tmp_path / "takatak"
    d.mkdir()
    rng = np.random.default_rng(5)
    pickle.dump({"default_uid": 0, **{f"u{i}": i for i in range(1, 40)}}, open(d / "user_vocab.pkl", "wb"))
    pickle.dump({"default_mid": 0, **{str(i): i for i in range(1, 500)}}, open(d / "item_vocab.pkl", "wb"))
    pickle.dump({"default_cat": 0, **{f"c{i}": i for i in range(1, 9)}}, open(d / "category_vocab.pkl", "wb"))
    (d / "takatak_business_recommenders.csv").write_text("1\t1\t10.0\n")
    tr, ev = [], []
    for u in range(1, 40):
        n = int(rng.integers(8, 400))
        items = rng.integers(1, 520, size=n)                       # some unknown tokens (>= 500)
        cates = rng.integers(1, 9, size=n)
        durs = rng.choice([0.0, 5.0, 12.5, 30.0], size=n, p=[0.05, 0.3, 0.35, 0.3])
        p_sat = [0.0, 0.2, 0.6, 1.0][u % 4]                        # users with none / few / many / all satisfied
        sats = (rng.random(n) < p_sat).astype(int)
        plays = (rng.choice([500, 3000, 7999, 8000, 20000, 90000], size=n)).astype(int)
        j = lambda a: ",".join(str(x) for x in a)
        tr.append("\t".join([f"u{u}", j(items), j(f"c{c}" for c in cates), j(durs), j(sats), j(plays)]))
        ev.append("\t".join([str(sats[-1]), str(plays[-1]), f"u{u}", str(items[-1]), f"c{cates[-1]}", str(durs[-1]), j(items[:-1]),
                             j(f"c{c}" for c in cates[:-1]), j(durs[:-1]), j(sats[:-1]), j(plays[:-1])]))
    (d / "train_data").write_text("\n".join(tr) + "\n")
    (d / "valid_data").write_text("\n".join(ev) + "\n")
    hp = DU.prepare_hparams(None, model_type="mmoe", dataset="takatak", bucket_num=10, batch_size=35, max_seq_length=50,
                            noise_train_hist=0, noise_train_listwise=0, noise_only_predict=0, user_vocab=str(d / "user_vocab.pkl"),
                            item_vocab=str(d / "item_vocab.pkl"), cate_vocab=str(d / "category_vocab.pkl"))
    out = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("PAMREC_PY_ITERATOR", mode)
        random.seed(8)
        it = IT.SequentialIterator(hp, None)
        out[mode] = [list(it.load_data_from_file(str(d / "train_data"))) for _ in range(2)] + \
                    [list(it.load_data_from_file(str(d / "valid_data"), min_seq_length=20))]
    for pa, na in zip(out["1"], out["0"]):
        assert len(pa) == len(na) > 0
        for a, b in zip(pa, na):
            for k in a:
                assert a[k].dtype == b[k].dtype and np.array_equal(a[k], b[k], equal_nan=True), k


def test_in_batch_negative_sampler_follows_the_disabled_reference_block():
    """IT:801-1007 is a comment ending in exit(-1): there is no behaviour to pin, only statements to follow."""
    import random
    with tempfile.TemporaryDirectory() as tmp:
        data_dir = G.synth_case("wechat_small", tmp) if "wechat_small" in G.CASES else G.synth_case(list(G.CASES)[0], tmp)
        hp = G.hparams_for(list(G.CASES)[0], data_dir)
        train = os.path.join(data_dir, "train_data")
        random.seed(8)
        base = list(IT.SequentialIterator(hp, None).load_data_from_file(train, batch_num_ngs=0))
        random.seed(8)
        it = IT.SequentialIterator(hp, None)
        neg = list(it.load_data_from_file(train, batch_num_ngs=4))
    assert len(neg) == len(base)
    b0, n0 = base[0], neg[0]
    n = b0["items"].shape[0]
    assert n0["items"].shape[0] == 5 * n and n0["item_history"].shape == (5 * n, b0["item_history"].shape[1])
    assert list(n0) == list(b0)                                         # same 19 feed keys
    pos = np.arange(0, 5 * n, 5)
    for k in ("items", "cates", "durations", "labels_satisfied", "labels_play", "plays"):
        assert np.array_equal(n0[k][pos], b0[k]), k                      # row 0 of every group of 5 is the positive
    neg_rows = np.setdiff1d(np.arange(5 * n), pos)
    for k in ("labels_satisfied", "labels_play", "plays"):
        assert not n0[k][neg_rows].any(), k
    for k in ("item_history", "item_cate_history", "mask", "item_loop_times_history", "users"):
        a = n0[k].reshape(n, 5, *n0[k].shape[1:])
        assert (a == a[:, :1]).all() and np.array_equal(a[:, 0], b0[k]), k   # negatives share the positive's history
    items = b0["items"].tolist()
    pair = {(int(i), int(c), float(d)) for i, c, d in zip(b0["items"], b0["cates"], b0["durations"])}
    for i in range(n):
        group = items[i // 5: i // 5 + 5]
        for j in range(1, 5):
            r = 5 * i + j
            assert int(n0["items"][r]) not in group                     # the rejection rule of IT:949-951, slice as written
            assert (int(n0["items"][r]), int(n0["cates"][r]), float(n0["durations"][r])) in pair
    # a batch in which every target is in the positive's slice admits no negative (the block would spin forever): it is dropped,
    # like the batch of fewer than 5 rows the block itself returns None for
    lone = {k: v[:5] for k, v in b0.items()}
    assert it._with_negatives(lone, 4) == {} and it._with_negatives({k: v[:3] for k, v in b0.items()}, 4) == {}


def test_memoised_group_auc_is_sklearn_bit_for_bit():
    """_group_auc sends every (labels in score order, tie structure) pattern to sklearn once: same float64 as a direct call for
    every group, ties and unsorted input included; single-class groups raise what sklearn raises."""
    from sklearn.metrics import roc_auc_score
    rng = np.random.default_rng(4)
    DU._AUC_CACHE.clear()
    n_groups = 0
    for _ in range(3000):
        n = int(rng.integers(2, 12))
        y = rng.integers(0, 2, n).astype(np.float64)
        if y.min() == y.max():
            y[0] = 1 - y[0]
        p = np.round(rng.random(n), int(rng.integers(1, 4)))          # coarse rounding -> many ties
        want = roc_auc_score(y, p)
        assert DU._group_auc(y, p) == want
        assert DU._group_auc(y.tolist(), (p * 0.5 + 0.25).tolist()) == want      # same pattern, other scores: served from the cache
        n_groups += 1
    assert 0 < len(DU._AUC_CACHE) < n_groups
    def outcome(f):                                                  # sklearn < 1.5 raises for one class, later versions warn + nan
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            try:
                return repr(f(np.asarray([1.0, 1.0]), np.asarray([0.2, 0.3])))
            except ValueError as e:
                return "ValueError " + str(e)
    assert outcome(DU._group_auc) == outcome(roc_auc_score) == outcome(DU._group_auc)
    big_y, big_p = rng.integers(0, 2, 500).astype(np.float64), rng.random(500)
    assert DU._group_auc(big_y, big_p) == roc_auc_score(big_y, big_p)            # large inputs bypass the cache
    # and through the public functions
    users = np.repeat(np.arange(400), 3)
    labels = np.tile([1.0, 0.0, 0.0], 400)
    preds = np.round(rng.random(1200), 2)
    direct = sum(3 / 1200 * roc_auc_score(labels[users == u], preds[users == u]) for u in range(400))
    assert DU.cal_weighted_metric(users, preds, labels, ["wauc"])["wauc"] == round(direct, 4)
    groups_l, groups_p = list(labels.reshape(-1, 3)), list(preds.reshape(-1, 3))
    assert DU.cal_metric(groups_l, groups_p, ["group_auc"])["group_auc"] == round(np.mean([roc_auc_score(l, p) for l, p in zip(groups_l, groups_p)]), 4)


def test_pairwise_metrics_over_all_groups_equal_the_per_group_functions():
    """cal_metric's fast path for rectangular groups (every impression has num_ngs + 1 rows): mrr / ndcg@k / hit@k evaluated on the
    rows of one 2-D array are bit-identical to the reference's per-group functions (DU:665-747), ties and k > group included, and
    cal_metric returns the same dict whether the groups come as a list of arrays, a list of lists or one array."""
    from pamrec_b200 import deeprec_utils as D
    rng = np.random.default_rng(0)
    for trial in range(60):
        G, n = int(rng.integers(1, 30)), int(rng.integers(1, 110))
        P = rng.random((G, n)).astype(np.float32)
        if trial % 3 == 0:
            P = np.round(P, 1)                                   # many ties
        L = (rng.random((G, n)) < 0.1).astype(np.float32)
        L[np.arange(G), rng.integers(0, n, G)] = 1
        for k in (1, 2, 10, 200):
            assert np.array_equal([D.ndcg_score(l, p, k) for l, p in zip(L, P)], D._dcg_rows(L, P, k) / D._dcg_rows(L, L, k))
            assert np.array_equal([D.hit_score(l, p, k) for l, p in zip(L, P)], D._hit_rows(L, P, k))
        assert np.array_equal([D.mrr_score(l, p) for l, p in zip(L, P)], D._mrr_rows(L, P))
        metrics = ["mean_mrr", "ndcg@2;10", "hit@1;10", "group_auc"] if (L.sum(1) < n).all() else ["mean_mrr", "ndcg@2;10", "hit@1;10"]
        a = D.cal_metric(L, P, metrics)
        b = D.cal_metric([l for l in L], [p for p in P], metrics)
        c = D.cal_metric([l.tolist() for l in L], [p.tolist() for p in P], metrics)
        assert a == b, (a, b)
        for key in a:                                            # python floats instead of float32 rows: same to the 4 decimals reported
            assert abs(a[key] - c[key]) <= 1.001e-4, (key, a[key], c[key])
    # ragged groups take the per-group path
    r = D.cal_metric([np.array([1., 0.]), np.array([0., 1., 0.])], [np.array([.3, .2]), np.array([.1, .5, .4])], ["mean_mrr", "hit@1"])
    assert r == {"mean_mrr": 1.0, "hit@1": 1.0}
    # log loss: the clipping list comprehension of DU:769 as np.clip
    y, p = np.array([1., 0., 1., 0.]), np.array([1.0, 0.0, 0.7, 0.2], np.float32)
    from sklearn.metrics import log_loss
    want = round(log_loss(y, np.asarray([max(min(v, 1.0 - 10e-12), 10e-12) for v in p])), 4)
    assert D.cal_metric(y, p, ["logloss"])["logloss"] == want
