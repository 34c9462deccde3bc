"""TEST INFRASTRUCTURE.  Pins the integer / host half of the path against the REFERENCE ITSELF.

Runs the reference's own ``io/sequential_iterator.py`` and the metric functions of ``deeprec_utils.py``
(imported from /root/reference, unmodified) under a stub ``tensorflow`` module that only provides
``placeholder`` / dtypes / ``disable_v2_behavior``, on seeded synthetic data written by
``pamrec_b200.synth`` and writes the results as small fixtures under tests/golden/:

  iterator_<case>.npz   for every batch: a SHA-256 over all 19 feed arrays, plus the first and last
                        batches in full
  metrics.json          cal_metric / cal_weighted_metric outputs on seeded random labels / scores

The reference is not part of this repository, so the fixtures are committed, and
tests/test_iterator_and_metrics.py compares with them.

    python -m oracle.gen_golden            # regenerate tests/golden/*
"""
import hashlib
import json
import os
import random
import sys
import tempfile
import types

import numpy as np

REF = os.environ.get("PAMREC_REFERENCE", "/root/reference")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

FEED_NAMES = ["labels_satisfied", "labels_play", "plays", "users", "items", "cates", "durations", "item_history",
              "item_cate_history", "item_duration_history", "mask", "item_satisfied_value_history",
              "item_play_value_history", "item_loop_times_history", "satisfied_item_history", "satisfied_cate_history",
              "satisfied_duration_history", "satisfied_play_history", "satisfied_mask"]

CASES = {
    # name: (dataset, synth kwargs, batch_size, max_seq_length, bucket_num)
    "wechat_small": ("wechat", dict(n_users=120, n_items=900, n_cates=30, mean_len=60, seed=7), 50, 100, 10),
    "takatak_small": ("takatak", dict(n_users=90, n_items=500, n_cates=12, mean_len=140, seed=9, max_len=400), 35, 50, 10),
}


class _Placeholder:
    def __init__(self, dtype, shape=None, name=None):
        self.dtype, self.shape, self.name = dtype, shape, name

    def __hash__(self):
        return id(self)


def install_tf_stub():
    """A ``tensorflow`` that is just enough for the reference's iterator + metric modules to import."""
    if "tensorflow" in sys.modules and not getattr(sys.modules["tensorflow"], "_pamrec_stub", False):
        return
    tf = types.ModuleType("tensorflow")
    tf._pamrec_stub = True
    compat = types.ModuleType("tensorflow.compat")
    v1 = types.ModuleType("tensorflow.compat.v1")
    for m in (tf, v1):
        m.float32, m.int32, m.bool = "float32", "int32", "bool"
        m.placeholder = lambda dtype, shape=None, name=None: _Placeholder(dtype, shape, name)
        m.disable_v2_behavior = lambda: None
    tf.compat, compat.v1 = compat, v1
    tf.keras = types.ModuleType("tensorflow.keras")
    sys.modules.update({"tensorflow": tf, "tensorflow.compat": compat, "tensorflow.compat.v1": v1,
                        "tensorflow.keras": tf.keras})


class _Graph:
    class _Ctx:
        def __enter__(self):
            return self

        def __exit__(self, *a):
            return False

    def as_default(self):
        return _Graph._Ctx()


def reference_modules():
    install_tf_stub()
    if REF not in sys.path:
        sys.path.insert(0, REF)
    from reco_utils.recommender.deeprec import deeprec_utils as DU
    from reco_utils.recommender.deeprec.io import sequential_iterator as IT
    return DU, IT


def hparams_for(case, data_dir):
    from pamrec_b200.deeprec_utils import prepare_hparams
    dataset, _, batch, T, buckets = CASES[case]
    return prepare_hparams(None, model_type="mmoe", dataset=dataset, bucket_num=buckets, batch_size=batch,
                           max_seq_length=T, noise_train_hist=0, noise_train_listwise=0, noise_only_predict=0,
                           user_vocab=os.path.join(data_dir, "user_vocab.pkl"), item_vocab=os.path.join(data_dir, "item_vocab.pkl"),
                           cate_vocab=os.path.join(data_dir, "category_vocab.pkl"))


def batch_digest(arrays):
    h = hashlib.sha256()
    for name in FEED_NAMES:
        a = np.ascontiguousarray(arrays[name])
        h.update(name.encode()); h.update(str(a.dtype).encode()); h.update(str(a.shape).encode()); h.update(a.tobytes())
    return h.hexdigest()


def by_name(feed):
    """reference feed dict (placeholder -> array) or ours (name -> array) -> name -> array"""
    return {(k.name if isinstance(k, _Placeholder) else k): np.asarray(v) for k, v in feed.items()}


def run_iterator(make_iter, data_dir, epochs=2, seed=8):
    """Replays what fit_step does to the RNGs (base_model.py:30-33): seed once, then iterate epochs of train_data,
    then one pass of valid_data."""
    np.random.seed(seed)
    random.seed(seed)
    it = make_iter()
    out = {"train": [], "valid": []}
    for _ in range(epochs):
        for feed in it.load_data_from_file(os.path.join(data_dir, "train_data"), min_seq_length=1, batch_num_ngs=0):
            out["train"].append(by_name(feed))
    for feed in it.load_data_from_file(os.path.join(data_dir, "valid_data"), min_seq_length=1, batch_num_ngs=0):
        out["valid"].append(by_name(feed))
    return out


def synth_case(case, root):
    from pamrec_b200 import synth
    dataset, kw, *_ = CASES[case]
    return synth.generate(root, dataset, **kw)


def metric_inputs(seed=5):
    rng = np.random.default_rng(seed)
    n = 600
    users = rng.integers(0, 40, size=n)
    preds = rng.random(n)
    labels = (rng.random(n) < 0.35).astype(np.float32)
    labels[users == 3] = 1.0            # a single-class user
    labels[users == 4] = 0.0
    g_labels = [(rng.random(8) < 0.4).astype(np.float32) for _ in range(50)]
    for g in g_labels:
        g[rng.integers(0, 8)] = 1.0
    g_preds = [rng.random(8) for _ in range(50)]
    return users, preds, labels, g_labels, g_preds


POINT_METRICS = ["auc", "logloss", "rmse", "acc", "f1"]
GROUP_METRICS = ["mean_mrr", "ndcg@2;4;6;10", "hit@2;4;6", "group_auc"]
WEIGHTED_METRICS = ["wauc", "wmrr", "wndcg@2;4;6;8;10", "whit@2;4;6;8;10", "wmrr@10"]


def reference_weighted(DU, users, preds, labels):
    """cal_weighted_metric of the reference (deeprec_utils.py:831-971).  Its pandas glue (groupby.apply handing a
    Series to np.take) raises under the pandas 3 of this image, so the reference's own per-user numpy functions
    (mrr_score / ndcg_score / hit_score, sklearn's roc_auc_score) are called per user and weighted by the user's
    share of rows exactly as cal_wauc / cal_wmrr / cal_wmrr_k / cal_whit / cal_wndcg do.  Metrics whose reference glue
    still runs are taken from the reference call itself."""
    from sklearn.metrics import roc_auc_score
    res = {}
    try:
        res.update(DU.cal_weighted_metric(users.tolist(), preds.tolist(), labels.tolist(), ["wauc"]))
    except Exception:
        pass
    uniq = np.unique(users)
    w = {u: float((users == u).sum()) / len(users) for u in uniq}
    per = lambda fn: sum(w[u] * fn(labels[users == u].astype(np.float64), preds[users == u]) for u in uniq)

    def sub_mrr(y, s, k):
        order = np.argsort(s)[::-1][:k]
        yy = np.take(y, order)
        return np.sum(yy / (np.arange(len(yy)) + 1))
    res.setdefault("wauc", round(per(lambda y, s: roc_auc_score(y, s)), 4))
    res["wmrr"] = round(per(DU.mrr_score), 4)
    res["wmrr@10"] = round(per(lambda y, s: sub_mrr(y, s, 10)), 4)
    for k in (2, 4, 6, 8, 10):
        res[f"wndcg@{k}"] = round(per(lambda y, s, k=k: DU.ndcg_score(y, s, k)), 4)
        res[f"whit@{k}"] = round(per(lambda y, s, k=k: DU.hit_score(y, s, k)), 4)
    return res


def main():
    DU, IT = reference_modules()
    os.makedirs(GOLDEN, exist_ok=True)
    for case in CASES:
        with tempfile.TemporaryDirectory() as tmp:
            data_dir = synth_case(case, tmp)
            hp = hparams_for(case, data_dir)
            res = run_iterator(lambda: IT.SequentialIterator(hp, _Graph()), data_dir)
        save = {"train_digests": np.array([batch_digest(b) for b in res["train"]]),
                "valid_digests": np.array([batch_digest(b) for b in res["valid"]])}
        for tag, b in (("train_first", res["train"][0]), ("train_last", res["train"][-1]), ("valid_first", res["valid"][0]),
                       ("valid_last", res["valid"][-1])):
            for name in FEED_NAMES:
                save[f"{tag}.{name}"] = b[name]
        np.savez_compressed(os.path.join(GOLDEN, f"iterator_{case}.npz"), **save)
        print(case, "train batches", len(res["train"]), "valid batches", len(res["valid"]))
    users, preds, labels, g_labels, g_preds = metric_inputs()
    # the single-class users are removed first, as run_weighted_eval does (sequential_base_model.py:466-479)
    mixed = [u for u in np.unique(users) if 0 < labels[users == u].sum() < (users == u).sum()]
    keep = np.isin(users, mixed)
    out = {"point": DU.cal_metric(labels[keep].tolist(), preds[keep].tolist(), POINT_METRICS),
           "group": DU.cal_metric(g_labels, g_preds, GROUP_METRICS),
           "weighted": reference_weighted(DU, users[keep], preds[keep], labels[keep])}
    out = {k: {m: float(v) for m, v in d.items()} for k, d in out.items()}
    with open(os.path.join(GOLDEN, "metrics.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    # lisan known answers on the borders and around them
    xs = np.concatenate([np.asarray(IT.bar_border_list), np.asarray(IT.takatak_bar_border_list_dict[10]),
                         np.linspace(-1, 6, 57), [np.inf, 142.5, 5000.0]])
    kat = {"x": xs.tolist(),
           "wechat": [IT.lisan(x, "wechat", 10) for x in xs],
           "takatak10": [IT.lisan(x, "takatak", 10) for x in xs],
           "takatak8": [IT.lisan(x, "takatak", 8) for x in xs],
           "takatak6": [IT.lisan(x, "takatak", 6) for x in xs]}
    with open(os.path.join(GOLDEN, "lisan.json"), "w") as f:
        json.dump(kat, f)
    print("metrics", out)


if __name__ == "__main__":
    main()
