"""Host-side mirror of the reference's ``reco_utils/recommender/deeprec/deeprec_utils.py`` for the PAMRec
path: the two-level hparams YAML -> flat ``HParams`` object, and the ranking metrics used by
``run_eval`` / ``run_weighted_eval``.  Same function names, arguments and error behaviour as the
reference (citations: DU = deeprec_utils.py in the reference tree); no TensorFlow.
"""
import pickle

import numpy as np
import yaml
from sklearn.metrics import accuracy_score, f1_score, log_loss, mean_squared_error, roc_auc_score

__all__ = ["prepare_hparams", "create_hparams", "HParams", "load_yaml", "flat_config", "check_type", "check_nn_config",
           "cal_metric", "cal_weighted_metric", "mrr_score", "ndcg_score", "dcg_score", "hit_score", "load_dict",
           "filter_single_class_users"]


# ----------------------------------------------------------------------------- configuration
def flat_config(config):
    """DU:27-41: {section: {key: value}} -> {key: value} (later sections win)."""
    flat = {}
    for section in config.values():
        flat.update(section)
    return flat


_INT_KEYS = ("epochs", "batch_size", "show_step", "save_epoch", "item_embedding_dim", "cate_embedding_dim",
             "user_embedding_dim", "max_seq_length", "hidden_size", "min_seq_length", "attention_size", "train_num_ngs")
_FLOAT_KEYS = ("init_value", "learning_rate", "embed_l2", "embed_l1", "layer_l2", "layer_l1")
_STR_KEYS = ("method", "loss", "optimizer", "init_method", "user_vocab", "item_vocab", "cate_vocab")
_LIST_KEYS = ("layer_sizes", "activation", "dropout", "att_fcn_layer_sizes")


def check_type(config):
    """DU:44-137: TypeError with the reference's message when a known key has the wrong type."""
    for keys, typ, word in ((_INT_KEYS, int, "int"), (_FLOAT_KEYS, float, "float"), (_STR_KEYS, str, "str"),
                            (_LIST_KEYS, list, "list")):
        for k in keys:
            if k in config and not isinstance(config[k], typ):
                raise TypeError("Parameters {0} must be {1}".format(k, word))


def check_nn_config(f_config):
    """DU:140-297.  ``model_type: mmoe`` (what PAMRec loads, config/mmoe.yaml:11) has no required-key list
    in the reference, so only the type check applies; a missing model_type is a KeyError as there."""
    f_config["model_type"]
    check_type(f_config)


def load_yaml(filename):
    """DU:310-326."""
    try:
        with open(filename, "r") as f:
            return yaml.load(f, yaml.SafeLoader)
    except FileNotFoundError:
        raise
    except Exception:
        raise IOError("load {0} error!".format(filename))


class HParams:
    """DU:329-363: attribute access over a dict whose values must be int / float / str / list."""

    def __init__(self, hparams_dict):
        for val in hparams_dict.values():
            if not isinstance(val, (int, float, str, list)):
                raise ValueError("Hyperparameter value {} should be integer, float, string or list.".format(val))
        self._values = hparams_dict
        for k, v in hparams_dict.items():
            setattr(self, k, v)

    def __repr__(self):
        return "HParams object with values {}".format(self._values.__repr__())

    def values(self):
        return self._values


# defaults that the PAMRec path can observe (DU:375-445); keys of other model families are not carried.
_DEFAULTS = {
    "user_dropout": False, "dropout": [0.0], "load_saved_model": False,
    "init_method": "tnormal", "init_value": 0.01,
    "embed_l2": 0.0, "embed_l1": 0.0, "layer_l2": 0.0, "layer_l1": 0.0, "cross_l2": 0.0, "cross_l1": 0.0,
    "attn_loss_weight": 0.0, "contrastive_loss": "bpr", "triplet_margin": 1.0, "discrepancy_loss_weight": 0.0,
    "contrastive_loss_weight": 0.0, "contrastive_length_threshold": 1, "contrastive_recent_k": 3,
    "learning_rate": 0.001, "max_grad_norm": 2, "is_clip_norm": 0, "manual_alpha": False, "manual_alpha_value": 0.5,
    "interest_evolve": True, "predict_long_short": True, "dtype": 32, "optimizer": "adam", "epochs": 10, "batch_size": 1,
    "enable_BN": False, "show_step": 1, "save_model": True, "save_epoch": 5, "write_tfevents": False,
    "train_num_ngs": 4, "need_sample": True, "embedding_dropout": 0.3, "EARLY_STOP": 100, "min_seq_length": 1,
    "sequential_model": "time4lstm", "time_unit": "s",
}


def create_hparams(flags):
    """DU:366-446."""
    d = dict(_DEFAULTS)
    d.update(flags)
    return HParams(d)


def prepare_hparams(yaml_file=None, **kwargs):
    """DU:625-645: YAML (optional) overridden by keyword arguments, type-checked, defaults merged."""
    config = flat_config(load_yaml(yaml_file)) if yaml_file is not None else {}
    config.update(kwargs)
    check_nn_config(config)
    return create_hparams(config)


def load_dict(filename):
    """DU:985-997: vocabulary pickle."""
    with open(filename, "rb") as f:
        return pickle.load(f)


# ----------------------------------------------------------------------------- metrics
def mrr_score(y_true, y_score):
    """DU:665-678."""
    order = np.argsort(y_score)[::-1]
    y_true = np.take(y_true, order)
    return np.sum(y_true / (np.arange(len(y_true)) + 1)) / np.sum(y_true)


def dcg_score(y_true, y_score, k=10):
    """DU:732-747: gain 2^y - 1, log2 discount."""
    k = min(np.shape(y_true)[-1], k)
    order = np.argsort(y_score)[::-1]
    y_true = np.take(y_true, order[:k])
    return np.sum((2 ** y_true - 1) / np.log2(np.arange(len(y_true)) + 2))


def ndcg_score(y_true, y_score, k=10):
    """DU:681-694."""
    return dcg_score(y_true, y_score, k) / dcg_score(y_true, y_true, k)


def hit_score(y_true, y_score, k=10):
    """DU:713-729: fraction of the top-k that are positives (hits / len(top-k), not 0/1)."""
    positives = set(np.where(np.asarray(y_true) == 1)[0].tolist())
    top = np.argsort(y_score)[::-1][:k]
    return sum(1 for i in top if i in positives) / len(top)


_AUC_CACHE = {}


def _group_auc(y_true, y_score):
    """sklearn.metrics.roc_auc_score for the small groups of group_auc / wauc (DU:808-814, DU:873-881), memoised.

    roc_auc_score sorts by score (stable, descending), merges equal scores into one threshold and works on the cumulative
    positive / negative COUNTS from there on, so its float64 result is a function of the labels in score order and of where
    the ties are - nothing else.  Thousands of two-to-ten-row user groups share a handful of such patterns; each pattern is
    sent to sklearn once and its exact value reused (the per-call overhead of sklearn's input validation, ~2 ms, is what
    made the reference's user-weighted metrics the slowest part of an evaluation pass)."""
    y_true = np.asarray(y_true, dtype=np.float64)
    y_score = np.asarray(y_score, dtype=np.float64)
    n = y_true.shape[0]
    if y_true.ndim != 1 or y_score.shape != y_true.shape or n > 128 or not np.isfinite(y_score).all():
        return roc_auc_score(y_true, y_score)
    order = np.argsort(y_score, kind="mergesort")[::-1]
    s = y_score[order]
    key = (y_true[order].tobytes(), (s[1:] != s[:-1]).tobytes())
    val = _AUC_CACHE.get(key)
    if val is None:
        val = roc_auc_score(y_true, y_score)               # raises for a single-class group exactly like the reference
        if len(_AUC_CACHE) < 200_000:
            _AUC_CACHE[key] = val
    return val


def _rect(groups):
    """The groups as one [n_groups, group] array when they all have the same length (every evaluation file does: num_ngs + 1 rows
    per impression, SBM:437), else None.  Element dtype is kept: the row functions below must see what the per-group ones see."""
    if isinstance(groups, np.ndarray):
        return groups if groups.ndim == 2 and groups.shape[1] > 0 else None
    if len(groups) == 0:
        return None
    n = len(groups[0])
    if n == 0 or any(len(g) != n for g in groups):
        return None
    a = np.asarray(groups)
    return a if a.ndim == 2 else None


# mrr_score / dcg_score / hit_score over all groups at once: the same numpy operations on the rows of a 2-D array (argsort along
# the last axis runs the 1-D sort per row, sums over the last axis the 1-D pairwise sum), so the values are bit-identical to the
# per-group loop - tests/test_iterator_and_metrics.py compares them, ties included.  100-row groups x 600 impressions: 150 -> 6 ms.
def _mrr_rows(L, P):
    yt = np.take_along_axis(L, np.argsort(P, axis=1)[:, ::-1], 1)
    return np.sum(yt / (np.arange(L.shape[1]) + 1), axis=1) / np.sum(yt, axis=1)


def _dcg_rows(L, P, k):
    k = min(L.shape[1], k)
    yt = np.take_along_axis(L, np.argsort(P, axis=1)[:, ::-1][:, :k], 1)
    return np.sum((2 ** yt - 1) / np.log2(np.arange(k) + 2), axis=1)


def _hit_rows(L, P, k):
    top = np.argsort(P, axis=1)[:, ::-1][:, :k]
    return np.sum(np.take_along_axis(L, top, 1) == 1, axis=1) / top.shape[1]


def _ks(metric, default):
    parts = metric.split("@")
    return [int(t) for t in parts[1].split(";")] if len(parts) > 1 else default


def cal_metric(labels, preds, metrics):
    """DU:750-828.  Point metrics take flat lists; mean_mrr / ndcg@ / hit@ / group_auc take lists of groups."""
    res = {}
    if not metrics:
        return res
    rect = None
    if any(m == "mean_mrr" or m.startswith(("ndcg", "hit")) for m in metrics):
        L, P = _rect(labels), _rect(preds)
        if L is not None and P is not None and L.shape == P.shape:
            rect = (L, P)
    for metric in metrics:
        if metric == "auc":
            res["auc"] = round(roc_auc_score(np.asarray(labels), np.asarray(preds)), 4)
        elif metric == "rmse":
            res["rmse"] = np.sqrt(round(mean_squared_error(np.asarray(labels), np.asarray(preds)), 4))
        elif metric == "logloss":
            preds = np.clip(np.asarray(preds, dtype=np.float64), 10e-12, 1.0 - 10e-12)      # [max(min(p, 1 - 10e-12), 10e-12) for p in preds]
            res["logloss"] = round(log_loss(np.asarray(labels), preds), 4)
        elif metric == "acc":
            res["acc"] = round(accuracy_score(np.asarray(labels), (np.asarray(preds) >= 0.5).astype(np.float64)), 4)
        elif metric == "f1":
            res["f1"] = round(f1_score(np.asarray(labels), (np.asarray(preds) >= 0.5).astype(np.float64)), 4)
        elif metric == "mean_mrr":
            res["mean_mrr"] = round(np.mean(_mrr_rows(*rect) if rect else [mrr_score(l, p) for l, p in zip(labels, preds)]), 4)
        elif metric.startswith("ndcg"):
            for k in _ks(metric, [1, 2]):
                vals = _dcg_rows(rect[0], rect[1], k) / _dcg_rows(rect[0], rect[0], k) if rect else [ndcg_score(l, p, k) for l, p in zip(labels, preds)]
                res["ndcg@{0}".format(k)] = round(np.mean(vals), 4)
        elif metric.startswith("hit"):
            for k in _ks(metric, [1, 2]):
                res["hit@{0}".format(k)] = round(np.mean(_hit_rows(rect[0], rect[1], k) if rect else [hit_score(l, p, k) for l, p in zip(labels, preds)]), 4)
        elif metric == "group_auc":
            res["group_auc"] = round(np.mean([_group_auc(l, p) for l, p in zip(labels, preds)]), 4)
        else:
            raise ValueError("not define this metric {0}".format(metric))
    return res


def rank_topk(scores, ids, top_k, keep=None):
    """Top ``top_k`` of each row of scores [n, c] over the candidate ids [c], in the order of pamrec_rank_candidates: score
    descending, then id ascending.  keep [n, c] (optional) marks the candidates a row may rank.  Returns (ids [n, top_k] with -1
    past the last kept candidate, scores [n, top_k] with -inf there)."""
    scores = np.asarray(scores, np.float32)
    ids = np.asarray(ids, np.int64)
    n = scores.shape[0]
    out_ids = np.full((n, top_k), -1, np.int32)
    out_sc = np.full((n, top_k), -np.inf, np.float32)
    for r in range(n):
        sel = np.arange(ids.size) if keep is None else np.flatnonzero(keep[r])
        order = sel[np.lexsort((ids[sel], -scores[r, sel].astype(np.float64)))][:top_k]
        out_ids[r, :order.size] = ids[order]
        out_sc[r, :order.size] = scores[r, order]
    return out_ids, out_sc


def own_rank(scores, ids, own, keep=None):
    """Rank of each row's own item among the candidates it may rank: 1 + the candidates ordered before it (score descending, then
    id ascending); -1 when the own item is not a candidate.  scores [n, c], ids [c], own [n], keep [n, c] as in rank_topk."""
    scores = np.asarray(scores, np.float32)
    ids = np.asarray(ids, np.int64)
    out = np.full(len(own), -1, np.int64)
    for r, item in enumerate(np.asarray(own, np.int64)):
        j = np.flatnonzero(ids == item)
        if j.size == 0:
            continue
        s = scores[r]
        before = (s > s[j[0]]) | ((s == s[j[0]]) & (ids < item))
        if keep is not None:
            before &= np.asarray(keep[r], bool)
        out[r] = 1 + int(before.sum())
    return out


def attention_topk(weights, live, top_k):
    """The ``top_k`` largest weights of each row of weights [n, T] among its live positions (live [n, T] true), ordered by weight
    descending, then position ascending.  Returns (positions [n, top_k] int64 with -1 past the last live position, weights
    [n, top_k] float32 with 0 there)."""
    w = np.asarray(weights, np.float32)
    live = np.asarray(live, bool)
    n, T = w.shape
    pos = np.broadcast_to(np.arange(T), (n, T))
    key = np.where(live, -w.astype(np.float64), np.inf)               # dead positions sort last
    order = np.lexsort((pos, key), axis=-1)[:, :top_k]
    ok = np.take_along_axis(live, order, -1)
    return np.where(ok, order, -1).astype(np.int64), np.where(ok, np.take_along_axis(w, order, -1), 0.0).astype(np.float32)


def full_ranking_metrics(ranks, labels, ks=(10,)):
    """Full-catalogue ranking metrics over the lines with label 1: hit@k (rank <= k), ndcg@k (1 / log2(rank + 1) when rank <= k,
    else 0) and mrr (1 / rank).  A rank < 1 (the positive is not a candidate) counts as a miss in every metric.  Rounded to 4
    decimals like cal_metric; an empty set of positives gives 0."""
    ranks = np.asarray(ranks, np.float64).reshape(-1)
    pos = np.asarray(labels).reshape(-1) == 1
    r = ranks[pos]
    hit_any = r >= 1
    safe = np.where(hit_any, r, 1.0)
    mean = lambda v: round(float(np.mean(v)), 4) if v.size else 0.0
    res = {}
    for k in ks:
        inside = hit_any & (r <= k)
        res["hit@{0}".format(k)] = mean(inside.astype(np.float64))
        res["ndcg@{0}".format(k)] = mean(np.where(inside, 1.0 / np.log2(safe + 1.0), 0.0))
    res["mrr"] = mean(np.where(hit_any, 1.0 / safe, 0.0))
    return res


def _user_groups(users, preds, labels):
    """Rows of each user in first-to-last order, users sorted ascending (pandas groupby order)."""
    users = np.asarray(users)
    preds = np.asarray(preds, dtype=np.float64)
    labels = np.asarray(labels, dtype=np.float64)
    order = np.argsort(users, kind="stable")
    su = users[order]
    cuts = np.flatnonzero(su[1:] != su[:-1]) + 1
    return [(labels[idx], preds[idx]) for idx in np.split(order, cuts)] if len(users) else []


def cal_weighted_metric(users, preds, labels, metrics):
    """DU:831-971: per-user metric weighted by the user's share of rows (wauc, wmrr, wmrr@k, whit@k, wndcg@k)."""
    res = {}
    if not metrics:
        return res
    groups = _user_groups(users, preds, labels)
    total = float(sum(len(l) for l, _ in groups))
    weights = [len(l) / total for l, _ in groups]

    def wsum(fn):
        return sum(w * fn(l, p) for w, (l, p) in zip(weights, groups))

    def sub_mrr(y_true, y_score, k):                      # DU:925-931
        order = np.argsort(y_score)[::-1][:k]
        y = np.take(y_true, order)
        return np.sum(y / (np.arange(len(y)) + 1))

    for metric in metrics:
        if metric == "wauc":
            res["wauc"] = round(wsum(_group_auc), 4)
        elif metric == "wmrr":
            res["wmrr"] = round(wsum(mrr_score), 4)
        elif metric.startswith("wmrr"):
            for k in _ks(metric, [10]):
                res["wmrr@{0}".format(k)] = round(wsum(lambda l, p, k=k: sub_mrr(l, p, k)), 4)
        elif metric.startswith("whit"):
            for k in _ks(metric, [1, 2]):
                res["whit@{0}".format(k)] = round(wsum(lambda l, p, k=k: hit_score(l, p, k)), 4)
        elif metric.startswith("wndcg"):
            for k in _ks(metric, [1, 2]):
                res["wndcg@{0}".format(k)] = round(wsum(lambda l, p, k=k: ndcg_score(l, p, k)), 4)
        else:
            raise ValueError("not define this metric {0}".format(metric))
    return res


def filter_single_class_users(users, preds, labels, as_arrays=False):
    """sequential_base_model.py:466-486: drop every user whose labels are all 0 or all 1.  The reference does it with a
    groupby.apply + inner merge on the left frame, which keeps the surviving rows in their original order."""
    users = np.asarray(users)
    preds = np.asarray(preds)
    labels = np.asarray(labels)
    if len(users) == 0:
        return ([], [], []) if not as_arrays else (users, preds, labels)
    uniq, inv = np.unique(users, return_inverse=True)
    n_rows = np.bincount(inv, minlength=len(uniq))
    n_zero = np.bincount(inv, weights=(labels == 0).astype(np.float64), minlength=len(uniq))
    mixed = (n_zero != 0) & (n_zero != n_rows)
    keep = mixed[inv]
    if as_arrays:
        return users[keep], preds[keep], labels[keep]
    return users[keep].tolist(), preds[keep].tolist(), labels[keep].tolist()
