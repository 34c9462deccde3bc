"""Candidate ranking on the device (pamrec_rank_candidates) for all five models.  Reference: every (line, candidate) row
materialised on the host and scored by the existing scoring path (Engine.forward, what predict runs), then ordered by numpy
(deeprec_utils.rank_topk / own_rank).  Inference is row-local and the same kernels run, so scores, top K and ranks must be
bit-identical."""
import os
import types

import numpy as np
import pytest

from pamrec_b200 import deeprec_utils as DU

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NU, NI, NC, T = 40, 300, 20, 20
N_LINES = 9
CONFIGS = [("pamrec", (16, 4, 20)), ("mmoe", (16, 4, 20)), ("ple", (16, 4, 20)), ("sharebottom", (16, 4, 20)), ("sasrec", (16, 4, 20)),
           ("mmoe", (32, 8, 40)), ("ple", (32, 8, 40)), ("sharebottom", (32, 8, 40)), ("sasrec", (32, 8, 16))]


def _variables(model, dims, seed=4):
    from oracle import pamrec_oracle as O
    from pamrec_b200.engine import Engine
    from pamrec_b200.models import initial_variables
    shapes = Engine(NU, NI, NC, T, 8, model=model, emb_dims=dims).variable_shapes()
    v = initial_variables(shapes, types.SimpleNamespace(init_method="tnormal", init_value=0.3), seed)
    params = {n: __import__("torch").from_numpy(a) for n, a in v.items()}
    bn = {n: params.pop(n) for n in list(params) if n.endswith(("moving_mean", "moving_variance"))}
    O.perturb_params(params, bn, seed=seed)
    return {n: t.numpy() for n, t in {**params, **bn}.items()}


def _engine(model, dims, max_batch, variables, **kw):
    from pamrec_b200.engine import Engine
    eng = Engine(NU, NI, NC, T, max_batch, model=model, emb_dims=dims, **kw).allocate("cuda:0")
    eng.set_variables(variables)
    return eng


def _lines(seed=11):
    """Scoring lines: line 0 has an empty history; line 1's own item sits in its history; line 2's own item is no candidate."""
    from oracle import pamrec_oracle as O
    from oracle import siblings_oracle as S
    b = S.add_satisfied_fields(O.make_batch(seed, N_LINES, T, NU, NI, NC, grouped=False), seed=seed)
    for k in ("item_history", "item_cate_history", "item_loop_times_history", "mask", "satisfied_item_history", "satisfied_cate_history",
              "satisfied_mask"):
        b[k][0] = 0
    b["items"][1] = b["item_history"][1][0]
    b["items"][2] = 7
    return b


def _candidates(seed=12, n=150):
    rng = np.random.default_rng(seed)
    ids = rng.permutation(np.arange(1, NI))[:n]
    ids = ids[ids != 7]
    lines = _lines()
    ids = np.unique(np.concatenate([ids, lines["items"][[0, 1, 3, 4]], lines["item_history"][3][:3]]))   # own items and history items
    ids = ids[(ids > 0) & (ids != 7)]
    return ids.astype(np.int32), rng.integers(0, NC, size=ids.size).astype(np.int32)


def _row_scores(eng, lines, ids, cates):
    """scores [lines, candidates] through Engine.forward on host-materialised rows; own [lines]: the own item with its candidate
    category (the line's own category when it is no candidate)."""
    n, c = len(lines["items"]), ids.size
    rows = {k: np.repeat(np.asarray(v), c, axis=0) for k, v in lines.items()}
    rows["items"] = np.tile(ids, n)
    rows["cates"] = np.tile(cates, n)
    cap = eng.dims[4]
    out = []
    for s in range(0, n * c, cap):
        part = {k: v[s:s + cap] for k, v in rows.items()}
        out.append(eng.forward(eng.upload(part, training=False), training=False).cpu().numpy())
    return np.concatenate(out).reshape(n, c)


def _keep(lines, ids, exclude):
    keep = np.ones((len(lines["items"]), ids.size), bool)
    if exclude:
        for r in range(keep.shape[0]):
            hist = set(np.asarray(lines["item_history"][r])[np.asarray(lines["mask"][r]) > 0].tolist())
            keep[r] = [(i not in hist) or i == lines["items"][r] for i in ids]
    return keep


def _check(got, scores, lines, ids, k, exclude):
    items, sc, rank = got
    keep = _keep(lines, ids, exclude)
    want_ids, want_sc = DU.rank_topk(scores, ids, k, keep)
    np.testing.assert_array_equal(items, want_ids)
    np.testing.assert_array_equal(sc, want_sc)
    np.testing.assert_array_equal(rank, DU.own_rank(scores, ids, lines["items"], keep))


@pytest.fixture(scope="module", params=CONFIGS, ids=[f"{m}-{d[0]}-{d[1]}-{d[2]}" for m, d in CONFIGS])
def setup(request):
    model, dims = request.param
    var = _variables(model, dims)
    small = _engine(model, dims, 64, var)              # 9 lines x ~150 candidates: about 22 chunks, none aligned to a line
    lines, (ids, cates) = _lines(), _candidates()
    scores = _row_scores(small, lines, ids, cates)
    yield types.SimpleNamespace(model=model, dims=dims, var=var, eng=small, lines=lines, ids=ids, cates=cates, scores=scores)
    small.close()


@pytest.mark.parametrize("k,exclude", [(1, False), (10, False), (10, True), (1024, False), (1024, True)])
def test_rank_equals_brute_force(setup, k, exclude):
    s = setup
    assert s.ids.size < 1024 and np.isin(s.lines["items"][1], s.lines["item_history"][1]) and not np.isin(7, s.ids)
    db = s.eng.upload(s.lines, training=False)
    got = s.eng.rank_candidates(db, s.ids, s.cates, k, exclude, want_rank=True).result()
    _check(got, s.scores, s.lines, s.ids, k, exclude)
    assert got[2][2] == -1 and got[2][1] >= 1


def test_chunking_does_not_change_the_result(setup):
    """One chunk for everything (max_batch above lines x candidates) against the 64-row chunks; the candidate count (not a
    divisor of 64) is odd on purpose."""
    s = setup
    big = _engine(s.model, s.dims, 2048, s.var)
    try:
        for k, exclude in ((5, True), (300, False)):
            a = s.eng.rank_candidates(s.eng.upload(s.lines, training=False), s.ids[:-1], s.cates[:-1], k, exclude, True).result()
            b = big.rank_candidates(big.upload(s.lines, training=False), s.ids[:-1], s.cates[:-1], k, exclude, True).result()
            for x, y in zip(a, b):
                np.testing.assert_array_equal(x, y)
            _check(b, s.scores[:, :-1], s.lines, s.ids[:-1], k, exclude)
    finally:
        big.close()


def test_sasrec_tower_path_equals_expansion_path(setup):
    s = setup
    if s.model != "sasrec":
        pytest.skip("the tower-only path is SASRec's")
    from pamrec_b200 import _lib as L
    db = s.eng.upload(s.lines, training=False)
    tower = s.eng.rank_candidates(db, s.ids, s.cates, 50, True, True).result()
    s.eng.set_debug(L.DEBUG_RANK_EXPAND)
    try:
        expand = s.eng.rank_candidates(db, s.ids, s.cates, 50, True, True).result()
    finally:
        s.eng.set_debug(0)
    for x, y in zip(tower, expand):
        np.testing.assert_array_equal(x, y)


def test_ties_follow_item_ids(setup):
    """With the output layers' weights at zero every candidate of a line gets the same score: the order is item id ascending."""
    s = setup
    var = dict(s.var)
    for n in var:
        if n.endswith("logit_fcn/nn_part/w_nn_output"):
            var[n] = np.zeros_like(var[n])
    eng = _engine(s.model, s.dims, 64, var)
    try:
        items, sc, rank = eng.rank_candidates(eng.upload(s.lines, training=False), s.ids, s.cates, 40, False, True).result()
        np.testing.assert_array_equal(items, np.tile(np.sort(s.ids)[:40], (N_LINES, 1)))
        assert (sc == sc[:, :1]).all()
        for r in range(N_LINES):
            own = s.lines["items"][r]
            assert rank[r] == (int(np.searchsorted(np.sort(s.ids), own)) + 1 if own in s.ids else -1)
    finally:
        eng.close()


def test_bad_candidates_are_refused(setup):
    from pamrec_b200.engine import PamrecError
    s = setup
    db = s.eng.upload(s.lines, training=False)
    for ids, cates, what in (([3, 3], [1, 1], "twice"), ([0, 3], [1, 1], "item id"), ([NI, 3], [1, 1], "item id"), ([3], [NC], "category")):
        with pytest.raises(PamrecError, match=what):
            s.eng.rank_candidates(db, ids, cates, 5)


@pytest.mark.parametrize("model,graph", [("pamrec", True), ("pamrec", False), ("mmoe", False), ("sasrec", False)])
def test_train_step_after_ranking_is_unchanged(model, graph):
    """rank_candidates between train steps leaves the following steps' losses as they are without it (CUDA-graph replay on and
    off).  Not bit for bit: the weight-gradient kernels (k_dense_dw, the encoder's and the persistent head's) sum their partial
    products with atomicAdd, so two engines that run the same steps already differ in the last bits of a loss (measured: 1.2e-7,
    one float32 ulp); a disturbed BN statistic, Adam slot or parameter would move them by orders of magnitude more."""
    from oracle import pamrec_oracle as O
    from oracle import siblings_oracle as S
    dims = (16, 4, 20)
    var = _variables(model, dims, seed=5)
    batch = S.add_satisfied_fields(O.make_batch(3, 20, T, NU, NI, NC), seed=3)
    ids, cates = _candidates()
    losses = []
    for rank in (False, True):
        eng = _engine(model, dims, 64, var, graph=graph)
        db, lines = eng.upload(batch), eng.upload(_lines(), training=False)
        steps = []
        for i in range(4):                   # with graph replay: step 2 is captured, steps 3 and 4 replay it
            if rank and i:
                eng.rank_candidates(lines, ids, cates, 10, True, True).result()
            steps.append(eng.train_step(db).cpu().numpy().copy())
        losses.append(steps)
        eng.close()
    for a, b in zip(*losses):
        np.testing.assert_allclose(a, b, rtol=1e-6, atol=1e-7)


@pytest.fixture(scope="module")
def data_root(tmp_path_factory):
    from pamrec_b200 import synth
    root = tmp_path_factory.mktemp("rank")
    synth.generate(str(root), "wechat", n_users=60, n_items=400, n_cates=15, mean_len=30, seed=21, eval_per_user=2)
    return str(root)


@pytest.mark.parametrize("cls_name,yaml_name", [("PAMRECModel", "mmoe.yaml"), ("SASRecModel", "sasrec.yaml")])
def test_recommend_and_full_ranking_eval_end_to_end(data_root, tmp_path, cls_name, yaml_name):
    from pamrec_b200 import models as M
    from pamrec_b200.deeprec_utils import prepare_hparams
    from pamrec_b200.sequential_iterator import SequentialIterator
    d = os.path.join(data_root, "wechat")
    hp = prepare_hparams(os.path.join(ROOT, "pamrec_b200", "config", yaml_name), dataset="wechat", bucket_num=10, add_feature=False,
                         embed_l2=1e-6, layer_l2=1e-6, learning_rate=0.001, epochs=1, EARLY_STOP=5, is_clip_norm=1, batch_size=50,
                         show_step=10 ** 9, MODEL_DIR=str(tmp_path / "m") + "/", SUMMARIES_DIR=str(tmp_path / "s") + "/",
                         user_vocab=os.path.join(d, "user_vocab.pkl"), item_vocab=os.path.join(d, "item_vocab.pkl"),
                         cate_vocab=os.path.join(d, "category_vocab.pkl"), train_num_ngs=0, max_seq_length=30, pairwise_metrics=[],
                         weighted_metrics=["wauc"], eval_step=4, write_tfevents=False, noise_train_hist=0, noise_train_listwise=0,
                         noise_only_predict=0)
    model = getattr(M, cls_name)(hp, SequentialIterator, seed=3)
    test = os.path.join(d, "test_data")
    out = str(tmp_path / "rec.tsv")
    rec = model.recommend(test, out, top_k=7, exclude_history=True)
    table = model.iterator.item_categories([test])
    ids = np.flatnonzero(table >= 0)
    ids = ids[ids > 0].astype(np.int32)
    cates = table[ids].astype(np.int32)
    eng = model.engine
    as_lines = lambda f: {k: (np.asarray(v).reshape(-1) if np.asarray(v).ndim == 2 and np.asarray(v).shape[1] == 1 else np.asarray(v))
                          for k, v in f.items()}
    want_items, ranks, labels = [], [], []
    for f in model.iterator.load_data_from_file(test, batch_num_ngs=0):
        lines = as_lines(f)
        want_items.append(DU.rank_topk(_row_scores(eng, lines, ids, cates), ids, 7, _keep(lines, ids, True))[0])
    for f in model.iterator.load_data_from_file(test, batch_num_ngs=0, min_seq_length=model.min_seq_length):
        lines = as_lines(f)
        ranks.append(DU.own_rank(_row_scores(eng, lines, ids, cates), ids, lines["items"].astype(np.int64)))
        labels.append(lines["labels_satisfied"])
    want_items = np.concatenate(want_items)
    np.testing.assert_array_equal(rec["items"], want_items)
    text = open(out).read().splitlines()
    assert len(text) == want_items.shape[0]
    inv = {v: k for k, v in model.iterator.itemdict.items()}
    first = text[0].split("\t")
    assert first[1].split(",") == [inv[int(i)] for i in want_items[0] if i >= 0]
    np.testing.assert_array_equal(np.asarray(first[2].split(","), np.float32), rec["scores"][0][rec["items"][0] >= 0])
    got = model.run_full_ranking_eval(test, ks=(1, 10, 50))
    assert got == DU.full_ranking_metrics(np.concatenate(ranks), np.concatenate(labels), ks=(1, 10, 50))
    with pytest.raises(ValueError):
        model.recommend(test, out, top_k=0)
    with pytest.raises(ValueError):
        model.run_full_ranking_eval(test, candidates=[int(ids[0]), int(ids[0])])
