"""GPU parity of the sibling baselines at the reference's own embedding widths (item / cate / user = 32 / 8 / 40 for MMoE, PLE and
share-bottom, 32 / 8 / 16 for SASRec) against oracle/siblings_oracle.py at the same widths: gather bit-exact, every forward stage
(the attention MLP's first layer contracts over 4 * 40 = 160 > kKMax columns, the chunked path of the dense forward kernel),
activation gradients, dense and merged sparse gradients, clip norms and losses; five optimisation steps and scoring; the file-driven
flow with checkpoints.  Widths are derived from the set under test, tolerances are those of tests/test_gpu_siblings.py."""
import os

import numpy as np
import pytest
import torch

from oracle import pamrec_oracle as O
import siblings_oracle_dims as D
from test_gpu_siblings import (EMB, FAILS, ROOT, _batch, _branches, _close, _expect, _on, expert_scopes, satisfied_edge_rows,
                               sibling_relu_masks)

pytestmark = pytest.mark.gpu

DIN_DIMS = (32, 8, 40)
SAS_DIMS = (32, 8, 16)


def _setup(model, nu, ni, nc, T, B, seed, dims):
    from pamrec_b200.engine import Engine
    om = D.SiblingOracleModel(model, nu, ni, nc, T, seed=seed, dims=dims)
    O.perturb_params(om.params, om.bn_state, seed=seed + 1)
    eng = Engine(nu, ni, nc, T, B, model=model, emb_dims=dims).allocate()
    eng.set_variables({n: t.numpy() for n, t in om.params.items()})
    eng.set_variables({n: t.numpy() for n, t in om.bn_state.items()})
    return om, eng


def _dense_grads(eng, om, ref, rep, L):
    l2 = om.hp["layer_l2"]
    gmax = max(float(ref["grads"][n].abs().max()) for n in eng.info[L.POOL_DENSE])
    bad = []
    for name, d in eng.info[L.POOL_DENSE].items():
        g = eng.dense(name, "dense_grad").cpu().numpy().astype(np.float64)
        if d["flags"] & L.SEG_L2:
            g = g + l2 * eng.dense(name).cpu().numpy().astype(np.float64)
        gr = ref["grads"][name].numpy().reshape(g.shape)
        err = np.abs(g - gr).max()
        lim = 1e-4 * np.abs(gr).max() + 2e-6 * gmax + (1e-5 * gmax if "/b_nn_layer" in name else 0.0)
        if "/b_nn_layer" not in name:
            rep.append(("grad " + name, err / max(np.abs(gr).max(), 1e-30)))
        if not (np.isfinite(g).all() and err <= lim):
            bad.append((name, err, np.abs(gr).max()))
    _expect(not bad, f"dense gradients, gmax={gmax:.3e}: " + "; ".join(f"{n}: err {e:.3e} max|ref| {m:.3e}" for n, e, m in bad))
    return gmax


def _sparse_and_norms(eng, om, ref, batch, tables0, rep, gmax, L, norm_slots):
    """merged sparse gradients (tables0: the tables before the update) and the clip norms of every variable"""
    nun = eng.ws("sp.nuniq").cpu().numpy()
    has0 = eng.ws("sib.has0").cpu().numpy()
    el2 = om.hp["embed_l2"]
    for tab, idx, name in (("item", 0, EMB + "item_embedding"), ("cate", 1, EMB + "cate_embedding")):
        n = int(nun[idx])
        uk = eng.ws(f"sp.{tab}.ukeys").cpu().numpy()[:n]
        acc = eng.ws(f"sp.{tab}.accum").cpu().numpy()[:n].astype(np.float64)
        gref = ref["grads"][name].numpy()
        hk, sk, tk = (("item_history", "satisfied_item_history", "items") if tab == "item" else ("item_cate_history", "satisfied_cate_history", "cates"))
        involved = np.unique(np.concatenate([batch[hk].reshape(-1), batch[tk].reshape(-1)]))
        touched = np.unique(np.concatenate([involved, batch[sk].reshape(-1)]))
        if not np.array_equal(uk, touched):
            FAILS.append(f"{tab}: unique ids differ")
            continue
        _expect(int(has0[idx]) == int(0 in involved), f"has0[{tab}]")
        g = acc + el2 * np.isin(uk, involved).astype(np.float64)[:, None] * tables0[tab][uk]
        _close(f"sparse grad {tab}", g, gref[uk], rtol=1e-4, report=rep)
    spn = eng.ws("sp_normsq").cpu().numpy()
    for i, name in norm_slots:
        want_sq = ref["sqnorms"][EMB + name]
        _expect(abs(spn[i] - want_sq) <= 2e-4 * want_sq + 1e-30, ("clip norm", name, spn[i], want_sq))
    segn = eng.ws("seg_normsq").cpu().numpy()
    for s_, (name, d) in enumerate(eng.info[L.POOL_DENSE].items()):
        want_sq = ref["sqnorms"][name]
        floor = (1e-5 if "/b_nn_layer" in name else 2e-6) * gmax
        _expect(abs(segn[s_] - want_sq) <= 2e-4 * want_sq + d["numel"] * floor ** 2, ("clip norm", name, segn[s_], want_sq))


DIN_CASES = [
    # model, nu, ni, nc, T, B, min_len
    ("mmoe", 50, 300, 20, 12, 20, 1),
    ("ple", 50, 300, 20, 12, 20, 1),
    ("sharebottom", 50, 300, 20, 12, 20, 1),
    ("ple", 400, 5000, 60, 50, 130, 50),           # full-length histories: id 0 only through the satisfied-only padding (no L2 on row 0)
    ("sharebottom", 100, 1000, 30, 200, 10, 1),    # T = 200
    ("mmoe", 50000, 30000, 50, 50, 1025, 1),       # the takatak bench shape
]


@pytest.mark.parametrize("model,nu,ni,nc,T,B,min_len", DIN_CASES)
def test_sibling_step_stagewise_reference_dims(model, nu, ni, nc, T, B, min_len):
    from pamrec_b200 import _lib as L
    dims = DIN_DIMS
    I, E = dims[0], dims[0] + dims[1]
    F = 4 * E                                                   # one branch's feature row = attention MLP input
    om, eng = _setup(model, nu, ni, nc, T, B, 11, dims)
    batch = _batch(5, B, T, nu, ni, nc, min_len=min_len)
    N = B * T
    FAILS.clear()
    db = eng.upload(batch)
    eng.forward(db, training=True, want_pred=False)
    torch.cuda.synchronize()
    masks = sibling_relu_masks(eng, model, B, T)
    ref = om.train_step(batch, apply=False, keep=("x", "logits"), relu_masks=masks)
    n_units = sum(int(np.prod(m.shape)) for m in masks.values())
    print(f"\n[{model},{dims},{nu},{ni},{nc},T={T},B={B}] ReLU units {n_units}, on opposite sides in fp32 / fp64: {ref['relu_forced']}")
    _expect(ref["relu_forced"] <= max(4, n_units // 40000), "the two forward passes disagree on far more ReLU units than rounding explains")
    t = ref["t"]
    rep = []
    item_w, cate_w = om.params[EMB + "item_embedding"].numpy(), om.params[EMB + "cate_embedding"].numpy()
    _expect(item_w.shape[1] == I and eng.pool["item_w"].shape[1] == I, "item table width")
    h = _branches(eng, "sib.h", N, E)
    want = [np.concatenate([item_w[batch["satisfied_item_history"].reshape(-1)], cate_w[batch["satisfied_cate_history"].reshape(-1)]], 1),
            np.concatenate([item_w[batch["item_history"].reshape(-1)], cate_w[batch["item_cate_history"].reshape(-1)]], 1)]
    _expect(np.array_equal(h[0], want[0]) and np.array_equal(h[1], want[1]), "gather is not bit-exact")
    tg = np.concatenate([item_w[batch["items"]], cate_w[batch["cates"]]], 1)
    _expect(np.array_equal(eng.ws("tgt", B).cpu().numpy(), tg), "target gather is not bit-exact")
    feat = eng.ws("sib.feat", N).cpu().numpy()
    z1, z2 = eng.ws("z1", N).cpu().numpy(), eng.ws("z2", N).cpu().numpy()
    score = eng.ws("sib.score", N).cpu().numpy()
    aw = eng.ws("sib.aw").reshape(-1)[:2 * N].view(2, N).cpu().numpy()
    for r in range(2):
        _close(f"att{r}.feat", feat[:, F * r:F * r + F], t[f"att{r}.feat"].detach().numpy(), report=rep)
        _close(f"att{r}.z0 (K = {F})", z1[:, 80 * r:80 * r + 80], t[f"att{r}.z0"].detach().numpy(), report=rep)
        _close(f"att{r}.z1", z2[:, 40 * r:40 * r + 40], t[f"att{r}.z1"].detach().numpy(), report=rep)
        _close(f"att{r}.score", score[:, r], t[f"att{r}.score"].detach().numpy(), report=rep)
        _close(f"att{r}.w", aw[r], t[f"att{r}.w"].detach().numpy(), report=rep)
    _close("x", eng.ws("x", B).cpu().numpy(), t["x"].detach().numpy(), report=rep)
    ex = expert_scopes(model)
    if ex:
        nE, TI = len(ex), 64 + E
        _close("ze0", eng.ws("ze0", B).cpu().numpy(), np.concatenate([t[f"expert{j}.z0"].detach().numpy() for j in range(nE)], 1), report=rep)
        _close("ze1", eng.ws("ze1", B).cpu().numpy(), np.concatenate([t[f"expert{j}.z1"].detach().numpy() for j in range(nE)], 1), report=rep)
        _close("zg1", eng.ws("zg1", B).cpu().numpy(), np.concatenate([t[f"gate{k}.z1"].detach().numpy() for k in range(2)], 1), report=rep)
        u = eng.ws("u", B).cpu().numpy()
        _close("main", u[:, :64], t["main"].detach().numpy(), report=rep)
        _close("sub", u[:, TI:TI + 64], t["sub"].detach().numpy(), report=rep)
        _expect(np.array_equal(u[:, 64:TI], tg) and np.array_equal(u[:, TI + 64:], tg), "target columns of the tower inputs")
    _close("zt1", eng.ws("zt1", B).cpu().numpy(), np.concatenate([t[f"tower{k}.z1"].detach().numpy() for k in range(2)], 1), report=rep)
    _close("logits", eng.ws("logits", B).cpu().numpy(), t["logits"].detach().numpy(), report=rep)
    eng.backward(db)
    torch.cuda.synchronize()
    _close("d_logits", eng.ws("d_logits", B).cpu().numpy(), t["logits"].grad.numpy(), rtol=2e-5, report=rep)
    _close("d_x", eng.ws("d_x", B).cpu().numpy(), t["x"].grad.numpy(), rtol=5e-5, report=rep)
    gmax = _dense_grads(eng, om, ref, rep, L)
    tables0 = {k: eng.pool[k + "_w"].cpu().numpy() for k in ("item", "cate", "ulong", "ushort")}
    losses = eng.apply_gradients(db).cpu().numpy()
    torch.cuda.synchronize()
    lr = ref["losses"]
    for i, k in enumerate(("loss", "data_loss", "regular_loss", "auxiliary_data_loss")):
        _expect(abs(losses[i] - lr[k]) <= 1e-5 * max(abs(lr[k]), 1e-3), (k, losses[i], lr[k]))
    _sparse_and_norms(eng, om, ref, batch, tables0, rep, gmax, L,
                      enumerate(("item_embedding", "cate_embedding", "user_long_embedding", "user_short_embedding")))
    if min_len == T:
        has0 = eng.ws("sib.has0").cpu().numpy()
        _expect(has0[0] == 0 and has0[1] == 0, "this case is meant to exercise the row-0-without-L2 path")
    for tab in ("item", "cate", "ulong", "ushort"):
        w0 = tables0[tab]; w1 = eng.pool[tab + "_w"].cpu().numpy()
        _expect(np.isfinite(w1).all() and (w0 != w1).any(), f"table {tab} after Adam")
    _expect(eng.pool["ulong_w"].shape[1] == dims[2], "user table width")
    print("\n".join(f"  {n:80s} {e:.2e}" for n, e in sorted(rep, key=lambda x: -x[1])[:10]))
    eng.close()
    assert not FAILS, "\n".join(FAILS)


SAS_CASES = [
    # nu, ni, nc, T, B, min_len
    (50, 300, 20, 12, 20, 1),
    (400, 5000, 60, 50, 130, 50),
    (100, 1000, 30, 200, 10, 1),
    (50000, 30000, 50, 50, 1025, 1),
    (60, 2000, 30, 256, 10, 1),                      # T = 256: 81 / 83 KB of shared memory per attention CTA (the opt-in at bind)
    (100, 1000, 30, 129, 10, 1),                     # T = 129: a thread's second query row (kernels_sasrec.cu) at model width 40
]


@pytest.mark.parametrize("nu,ni,nc,T,B,min_len", SAS_CASES)
def test_sasrec_step_stagewise_reference_dims(nu, ni, nc, T, B, min_len):
    from pamrec_b200 import _lib as L
    dims = SAS_DIMS
    Sw = dims[0] + dims[1]                                   # model width
    om, eng = _setup("sasrec", nu, ni, nc, T, B, 11, dims)
    batch = _batch(5, B, T, nu, ni, nc, min_len=min_len)
    satisfied_edge_rows(batch)                             # none, a single one at the last position, all satisfied
    N = B * T
    FAILS.clear()
    db = eng.upload(batch)
    eng.forward(db, training=True, want_pred=False)
    torch.cuda.synchronize()
    tw = "sequential/logit_fcn/nn_part/batch_normalization"
    masks = {f"blk{k}.ffn": (eng.ws(f"blk{k}.hpre", N).cpu().numpy() > 0).reshape(B, T, Sw) for k in range(2)}
    for zbuf, bn, scope in (("zt0", "t0", tw), ("zt1", "t1", tw + "_1")):
        masks[scope] = _on(eng.ws(zbuf, B).cpu().numpy(), eng.ws(f"bn.{bn}.stat").cpu().numpy(), eng.dense(scope + "/gamma").cpu().numpy(),
                           eng.dense(scope + "/beta").cpu().numpy())
    ref = om.train_step(batch, apply=False, keep=("x0", "logits"), relu_masks=masks)
    n_units = sum(int(np.prod(m.shape)) for m in masks.values())
    print(f"\n[sasrec,{dims},{nu},{ni},{nc},T={T},B={B}] ReLU units {n_units}, on opposite sides in fp32 / fp64: {ref['relu_forced']}")
    _expect(ref["relu_forced"] <= max(4, n_units // 40000), "the two forward passes disagree on far more ReLU units than rounding explains")
    t = ref["t"]
    rep = []
    _close("x0", eng.ws("x0", N).cpu().numpy(), t["x0"].detach().numpy(), rtol=1e-6, report=rep)
    for k in range(2):
        xq, qkv = eng.ws(f"blk{k}.xq", N).cpu().numpy(), eng.ws(f"blk{k}.qkv", N).cpu().numpy()
        _close(f"blk{k}.qin", xq[:, :Sw], t[f"blk{k}.qin"].detach().numpy(), report=rep)
        for j, nm in enumerate("QKV"):
            _close(f"blk{k}.{nm}", qkv[:, Sw * j:Sw * j + Sw], t[f"blk{k}.{nm}"].detach().numpy(), report=rep)
        for nm in ("y", "f", "out"):
            _close(f"blk{k}.{nm}", eng.ws(f"blk{k}.{nm}", N).cpu().numpy(), t[f"blk{k}.{nm}"].detach().numpy(), report=rep)
    u = eng.ws("u", B).cpu().numpy()
    _close("final_state", u[:, :Sw], t["final_state"].detach().numpy(), report=rep)
    _expect(not u[3, :Sw].any(), "read-out of the row without a satisfied item")
    _close("zt1", eng.ws("zt1", B).cpu().numpy(), t["tower0.z1"].detach().numpy(), report=rep)
    _close("logits", eng.ws("logits", B).cpu().numpy(), t["logits"].detach().numpy(), report=rep)
    eng.backward(db)
    torch.cuda.synchronize()
    _close("d_logits", eng.ws("d_logits", B).cpu().numpy(), t["logits"].grad.numpy(), rtol=2e-5, report=rep)
    _close("d_x0", _branches(eng, "sib.dh", N, Sw)[0], t["x0"].grad.numpy(), rtol=1e-4, report=rep)
    gmax = _dense_grads(eng, om, ref, rep, L)
    tables0 = {k: eng.pool[k + "_w"].cpu().numpy() for k in ("item", "cate")}
    losses = eng.apply_gradients(db).cpu().numpy()
    torch.cuda.synchronize()
    lr = ref["losses"]
    for i, k in enumerate(("loss", "data_loss", "regular_loss")):
        _expect(abs(losses[i] - lr[k]) <= 1e-5 * max(abs(lr[k]), 1e-3), (k, losses[i], lr[k]))
    _sparse_and_norms(eng, om, ref, batch, tables0, rep, gmax, L, ((0, "item_embedding"), (1, "cate_embedding"), (4, "position_embedding")))
    print("\n".join(f"  {n:80s} {e:.2e}" for n, e in sorted(rep, key=lambda x: -x[1])[:10]))
    eng.close()
    assert not FAILS, "\n".join(FAILS)


@pytest.mark.parametrize("model", ["mmoe", "ple", "sharebottom", "sasrec"])
def test_sibling_multi_step_and_eval_reference_dims(model):
    """Five optimisation steps at the reference's widths (the losses follow the oracle's), then a scoring pass."""
    nu, ni, nc, T, B = 300, 3000, 50, 50, 100
    dims = SAS_DIMS if model == "sasrec" else DIN_DIMS
    om, eng = _setup(model, nu, ni, nc, T, B, 3, dims)
    for step in range(5):
        batch = _batch(100 + step, B, T, nu, ni, nc, min_len=(T if step == 2 else 1))
        ref = om.train_step(batch)
        got = eng.train_step(eng.upload(batch)).cpu().numpy()
        for i, k in enumerate(("loss", "data_loss", "regular_loss", "auxiliary_data_loss")):
            if k not in ref["losses"]:
                assert model == "sasrec" and got[i] == 0.0
                continue
            r = ref["losses"][k]
            assert abs(got[i] - r) <= (1e-5 if step == 0 else 1e-4 * step) * max(abs(r), 1e-3), (step, k, got[i], r)
    got_vars = eng.get_variables()
    lr = om.hp["learning_rate"]
    for name in (EMB + "item_embedding", EMB + "cate_embedding", EMB + ("position_embedding" if model == "sasrec" else "user_long_embedding")):
        d = np.abs(got_vars[name] - om.params[name].numpy())
        assert d.max() <= 2 * lr * 5 * 1.01 and d.mean() <= 0.05 * lr, (name, float(d.max()), float(d.mean()))
    for name, tval in om.bn_state.items():
        tol = 5 * lr * 0.25 if name.endswith("moving_mean") else 2e-4
        assert np.allclose(got_vars[name], tval.numpy(), rtol=2e-4, atol=tol), name
    ev = _batch(999, 77, T, nu, ni, nc, grouped=False)
    pred = eng.forward(eng.upload(ev, training=False), training=False).cpu().numpy()
    want = om.eval_forward(ev).t["pred"].numpy().reshape(-1)
    assert np.abs(pred - want).max() <= 1e-4, float(np.abs(pred - want).max())
    eng.close()


# ----------------------------------------------------------------------------- the reference's driver flow at its widths
@pytest.fixture(scope="module")
def data_root(tmp_path_factory):
    from pamrec_b200 import synth
    root = tmp_path_factory.mktemp("siblings_ref")
    synth.generate(str(root), "wechat", n_users=300, n_items=2000, n_cates=30, mean_len=50, seed=9, eval_per_user=2)
    return str(root)


def _compat():
    import sys
    if os.path.join(ROOT, "compat") not in sys.path:
        sys.path.insert(0, os.path.join(ROOT, "compat"))


def _hparams(data_root, tmp_path, yaml_name, **kw):
    _compat()
    from reco_utils.recommender.deeprec.deeprec_utils import prepare_hparams
    d = os.path.join(data_root, "wechat")
    return prepare_hparams(os.path.join(ROOT, "compat", "reco_utils", "recommender", "deeprec", "config", yaml_name), dataset="wechat",
                           bucket_num=10, add_feature=False, embed_l2=1e-6, layer_l2=1e-6, learning_rate=0.001, epochs=1, EARLY_STOP=5,
                           is_clip_norm=1, batch_size=100, show_step=10 ** 9, MODEL_DIR=str(tmp_path / "model") + "/",
                           SUMMARIES_DIR=str(tmp_path / "s") + "/", user_vocab=os.path.join(d, "user_vocab.pkl"),
                           item_vocab=os.path.join(d, "item_vocab.pkl"), cate_vocab=os.path.join(d, "category_vocab.pkl"), train_num_ngs=0,
                           max_seq_length=50, pairwise_metrics=[], weighted_metrics=["wauc", "wmrr"], eval_step=4, write_tfevents=False,
                           noise_train_hist=0, noise_train_listwise=0, noise_only_predict=0, **kw)


@pytest.mark.parametrize("cls_name,yaml_name,kind,fmt", [("MMoEModel_original", "mmoe.yaml", "mmoe", "safetensors"),
                                                         ("PLEModel", "ple.yaml", "ple", "tf"),
                                                         ("ShareBottomModel", "sharebottom.yaml", "sharebottom", "safetensors"),
                                                         ("SASRecModel", "sasrec.yaml", "sasrec", "tf")])
def test_sibling_fit_checkpoint_eval_reference_dims(data_root, tmp_path, cls_name, yaml_name, kind, fmt):
    """prepare_hparams(..., item_embedding_dim=32, cate_embedding_dim=8, user_embedding_dim=40 (16 for SASRec)) -> fit_step ->
    checkpoint -> load_model -> run_weighted_eval; the fp64 oracle at the same widths re-scores the impressions from the checkpoint.
    A checkpoint written at 16 / 4 / 20 does not load into this model."""
    import importlib
    import tensorflow.compat.v1 as tf                      # compat shim: latest_checkpoint only
    dims = SAS_DIMS if kind == "sasrec" else DIN_DIMS
    _compat()
    from reco_utils.recommender.deeprec.io.sequential_iterator import SequentialIterator as it
    cls = getattr(importlib.import_module("reco_utils.recommender.deeprec.models.sequential." + kind), cls_name)
    hp = _hparams(data_root, tmp_path, yaml_name, item_embedding_dim=dims[0], cate_embedding_dim=dims[1], user_embedding_dim=dims[2],
                  checkpoint_format=fmt)
    d = os.path.join(data_root, "wechat")
    model = cls(hp, it, seed=8)
    assert model.engine.emb_dims == dims
    assert model.fit_step(os.path.join(d, "train_data"), os.path.join(d, "valid_data"), valid_num_ngs=0, eval_metric="auc") is model
    ckpt = tf.train.latest_checkpoint(str(tmp_path / "model") + "/")
    assert ckpt
    fresh = cls(hp, it, seed=123)
    fresh.load_model(ckpt)
    test = os.path.join(d, "test_data")
    res = fresh.run_weighted_eval(test, num_ngs=0)
    for k in ("auc", "logloss", "wauc", "wmrr"):
        assert k in res and np.isfinite(res[k]), (k, res)
    var = fresh.engine.get_variables()
    nu, ni, nc, T, _ = fresh.engine.dims
    om = D.SiblingOracleModel(kind, nu, ni, nc, T, seed=1, dims=dims)
    assert set(om.params) | set(om.bn_state) == set(var)
    for n in om.params:
        assert tuple(var[n].shape) == tuple(om.params[n].shape), n
        om.params[n] = torch.as_tensor(var[n], dtype=om.params[n].dtype)
    for n in om.bn_state:
        om.bn_state[n] = torch.as_tensor(var[n], dtype=om.bn_state[n].dtype).reshape(om.bn_state[n].shape)
    got, want = [], []
    for feed in fresh.iterator.load_data_from_file(test, min_seq_length=fresh.min_seq_length, batch_num_ngs=0):
        if not feed:
            continue
        got.append(fresh.eval(None, feed)[0].reshape(-1))
        f2 = {k: np.asarray(v) for k, v in feed.items()}
        for k in ("mask", "satisfied_mask", "users"):
            f2[k] = f2[k].astype(np.int32)
        want.append(om.eval_forward(f2).t["pred"].numpy().reshape(-1))
    got, want = np.concatenate(got), np.concatenate(want)
    assert got.shape == want.shape and np.abs(got - want).max() <= 1e-4, float(np.abs(got - want).max())
    # a checkpoint of the same model at 16 / 4 / 20 carries the same names with narrower shapes: refused, not loaded
    narrow = cls(_hparams(data_root, tmp_path / "narrow", yaml_name, checkpoint_format=fmt), it, seed=8)
    path = narrow.saver.save(save_path=str(tmp_path / "narrow_ckpt" / "step_0"))
    with pytest.raises(ValueError, match="has shape"):
        fresh.saver.restore(None, path)
    with pytest.raises(IOError):
        fresh.load_model(path)
