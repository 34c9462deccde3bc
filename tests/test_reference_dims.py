"""The sibling baselines at the reference's own embedding widths (item / cate / user = 32 / 8 / 40 in ple.yaml and sharebottom.yaml,
32 / 8 / 16 in sasrec.yaml), without a GPU: the C ABI's validation of the widths, the TF-name inventory against the oracle's at those
widths, model construction through the public classes, and the oracle's own consistency at the wider tokens."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import pamrec_oracle as O
from oracle import siblings_oracle as S
import siblings_oracle_dims as D
from test_host_loops import StubEngine
from test_siblings_oracle import NC, NI, NU, T, _batch, _randomise

REFERENCE = {"mmoe": (32, 8, 40), "ple": (32, 8, 40), "sharebottom": (32, 8, 40), "sasrec": (32, 8, 16)}
MIXED = (32, 8, 20)


def _oracle_shapes(model, nu, ni, nc, T_, dims):
    if model == "sasrec":
        spec, bn = D.sasrec_param_spec(nu, ni, nc, T_, dims=dims)
    else:
        spec, bn = D.param_spec(model, nu, ni, nc, dims=dims)
    shapes = {n: tuple(s) for n, s, _, _ in spec}
    for scope, c in bn:
        shapes[scope + "/moving_mean"] = shapes[scope + "/moving_variance"] = (c,)
    return shapes


@pytest.mark.parametrize("dims", ["reference", "mixed"])
@pytest.mark.parametrize("model", ["mmoe", "ple", "sharebottom", "sasrec"])
def test_inventory_matches_oracle(lib_built, model, dims):
    from pamrec_b200.engine import Engine
    d = REFERENCE[model] if dims == "reference" else MIXED
    eng = Engine(NU, NI, NC, T, 20, model=model, emb_dims=d)
    got = {n: tuple(int(x) for x in s) for n, s in eng.variable_shapes().items()}
    assert got == _oracle_shapes(model, NU, NI, NC, T, d)
    E = d[0] + d[1]
    assert got["sequential/embedding/item_embedding"] == (NI, d[0]) and got["sequential/embedding/user_embedding"] == (NU, d[2])
    if model == "sasrec":
        assert got["sequential/logit_fcn/nn_part/w_nn_layer0"] == (2 * E, 100)
        assert eng.info[2]["blk0.qkv"]["shape"][1] == 3 * E
    else:
        assert got["sequential/clsr/long_term/attention_fcn/att_fcn/nn_part/w_nn_layer0"] == (4 * E, 80)
        assert got["sequential/logit_fcn/nn_part/w_nn_layer0"] == ((3 * E, 100) if model == "sharebottom" else (64 + E, 100))
        assert eng.info[2]["sib.feat"]["shape"][1] == 8 * E and eng.info[2]["x"]["shape"][1] == 3 * E
    assert eng.info[2]["sp.item.accum"]["shape"][1] == d[0] and eng.info[2]["sp.cate.accum"]["shape"][1] == d[1]
    eng.close()


def test_create_validates_widths(lib_built):
    from pamrec_b200 import _lib as L
    lib = L.load()
    base = dict(n_users=10, n_items=20, n_cates=5, max_seq_len=8, max_batch=10, learning_rate=1e-3, beta1=0.9, beta2=0.999, epsilon=1e-8,
                max_grad_norm=2.0, is_clip_norm=1, fuzhu_weight=0.5, order_weight=0.1, world_size=1, rank=0)

    def create(model, dims):
        cfg = L.PamrecConfig(**base, model_kind=model, item_dim=dims[0], cate_dim=dims[1], user_dim=dims[2])
        h = C.c_void_p()
        rc = lib.pamrec_create(C.byref(cfg), C.byref(h))
        if rc == 0:
            lib.pamrec_destroy(h)
        else:
            assert not h.value
        return rc
    siblings = (L.MODEL_MMOE, L.MODEL_PLE, L.MODEL_SHAREBOTTOM, L.MODEL_SASREC)
    for m in (L.MODEL_PAMREC,) + siblings:
        assert create(m, (0, 0, 0)) == 0
        assert create(m, (16, 4, 20)) == 0
        for bad in ((24, 8, 40), (32, 8, 12), (16, 8, 20), (32, 4, 20), (8, 2, 20)):
            assert create(m, bad) == -10, (m, bad)
    for m in siblings:
        for good in ((32, 8, 40), (32, 8, 16), (32, 8, 20), (16, 4, 40), (16, 4, 16)):
            assert create(m, good) == 0, (m, good)
    for other in ((32, 8, 40), (16, 4, 40), (16, 4, 16)):
        assert create(L.MODEL_PAMREC, other) == -10


class WidthStubEngine(StubEngine):
    """StubEngine whose host tables follow the engine's embedding widths."""

    def allocate(self, device="cpu"):
        super().allocate(device)
        nu, ni, nc, _, _ = self.dims
        di, dc, du = self.emb_dims
        for pre, rows, w in (("item", ni, di), ("cate", nc, dc), ("ulong", nu, du), ("ushort", nu, du)):
            for s in ("w", "m", "v"):
                self.pool[f"{pre}_{s}"] = torch.zeros(self.table_rows(rows), w)
        return self


@pytest.fixture()
def make_model(tmp_path, monkeypatch, lib_built):
    from pamrec_b200 import deeprec_utils as DU
    from pamrec_b200 import models as M
    from pamrec_b200 import synth
    from pamrec_b200.sequential_iterator import SequentialIterator
    monkeypatch.setattr(M, "Engine", WidthStubEngine)
    d = synth.generate(str(tmp_path), "wechat", n_users=40, n_items=200, n_cates=12, mean_len=20, seed=3)

    def make(cls_name, **kw):
        base = dict(model_type="ple", dataset="wechat", bucket_num=10, method="classification", loss="cross_entropy_loss", optimizer="adam",
                    item_embedding_dim=32, cate_embedding_dim=8, user_embedding_dim=40, layer_sizes=[100, 64], expert_layer_sizes=[100, 64],
                    gate_layer_sizes=[64, 5], expert_num=5, share_expert_num=3, independent_expert_num=2, activation=["relu", "relu"],
                    enable_BN=True, dropout=[0.0, 0.0], embedding_dropout=0.0, hidden_size=40, attention_size=40, att_fcn_layer_sizes=[80, 40],
                    batch_size=50, max_seq_length=20, epochs=1, eval_step=10, EARLY_STOP=2, show_step=10 ** 9, train_num_ngs=0,
                    need_sample=False, metrics=["auc"], pairwise_metrics=[], weighted_metrics=["wauc"], noise_train_hist=0,
                    noise_train_listwise=0, noise_only_predict=0,
                    MODEL_DIR=str(tmp_path / "model") + "/", SUMMARIES_DIR=str(tmp_path / "sum") + "/",
                    user_vocab=os.path.join(d, "user_vocab.pkl"), item_vocab=os.path.join(d, "item_vocab.pkl"),
                    cate_vocab=os.path.join(d, "category_vocab.pkl"))
        base.update(kw)
        return getattr(M, cls_name)(DU.prepare_hparams(None, **base), SequentialIterator, seed=8)
    return make


@pytest.mark.parametrize("cls_name,kind", [("PLEModel", "ple"), ("SASRecModel", "sasrec")])
def test_models_build_at_reference_widths(make_model, cls_name, kind):
    dims = REFERENCE[kind]
    m = make_model(cls_name, user_embedding_dim=dims[2])
    eng = m.engine
    assert eng.emb_dims == dims
    shapes = eng.variable_shapes()
    assert tuple(shapes["sequential/embedding/item_embedding"])[1] == 32 and tuple(shapes["sequential/embedding/cate_embedding"])[1] == 8
    assert tuple(shapes["sequential/embedding/user_embedding"])[1] == dims[2]
    var = eng.get_variables()
    assert all(tuple(var[n].shape) == tuple(s) for n, s in shapes.items())
    assert eng.pool["item_w"].shape[1] == 32 and eng.pool["ulong_w"].shape[1] == dims[2]


def test_unsupported_widths_are_refused(make_model):
    with pytest.raises(ValueError, match="embedding dims must be 16 / 4 / 20"):
        make_model("PAMRECModel", model_type="pamrec")
    with pytest.raises(ValueError, match="16 / 4 or 32 / 8, with user 16, 20 or 40"):
        make_model("PLEModel", item_embedding_dim=24)
    with pytest.raises(ValueError, match="16 / 4 or 32 / 8, with user 16, 20 or 40"):
        make_model("ShareBottomModel", user_embedding_dim=12)


# ---- the oracle at the reference's widths: the checks of tests/test_siblings_oracle.py, re-run on 40-wide tokens
DIMS = (32, 8, 40)


def test_oracle_ple_with_only_shared_experts_is_mmoe_at_reference_widths():
    a = D.SiblingOracle("mmoe", NU, NI, NC, dims=DIMS, expert_num=5)
    b = D.SiblingOracle("ple", NU, NI, NC, dims=DIMS, share_expert_num=5, independent_expert_num=0)
    _randomise(a, 2)
    for n in a.params:
        m = n.replace("/clsr/expert_", "/clsr/share_expert_")
        assert m in b.params, m
        b.params[m] = a.params[n].clone()
    for n in a.bn_state:
        b.bn_state[n.replace("/clsr/expert_", "/clsr/share_expert_")] = a.bn_state[n].clone()
    batch = _batch(5)
    la, _, ca = a.loss_and_grads(batch)
    lb, _, cb = b.loss_and_grads(batch)
    assert ca.t["x"].shape == (20, 120)
    assert torch.equal(ca.t["logits"], cb.t["logits"]) and la == lb
    assert torch.equal(a.eval_forward(batch).t["pred"], b.eval_forward(batch).t["pred"])


@pytest.mark.parametrize("model", S.MODELS)
def test_oracle_gradients_match_finite_differences_at_reference_widths(model):
    m = D.SiblingOracle(model, NU, NI, NC, dims=DIMS)
    _randomise(m, 7)
    batch = _batch(8)
    _, grads, _ = m.loss_and_grads(batch)
    for name, idx in (("sequential/clsr/short_term/attention_fcn/attention_mat", (31, 37)),
                      ("sequential/clsr/long_term/attention_fcn/att_fcn/nn_part/w_nn_layer0", (150, 7)),
                      ("sequential/valid_logit_fcn/nn_part/w_nn_layer1", (10, 3)),
                      ("sequential/embedding/item_embedding", (int(batch["items"][0]), 30)),
                      ("sequential/embedding/cate_embedding", (int(batch["cates"][0]), 6))):
        base = m.params[name].clone()
        vals = []
        for sgn in (+1, -1):
            m.params[name] = base.clone().double()
            m.params[name][idx] += sgn * 1e-6
            vals.append(m.loss_and_grads(batch)[0]["loss"])
        m.params[name] = base
        fd = (vals[0] - vals[1]) / 2e-6
        assert abs(fd - float(grads[name][idx])) <= 1e-5 * max(abs(fd), 1e-5), (name, fd, float(grads[name][idx]))


def test_oracle_sasrec_at_reference_widths():
    dims = REFERENCE["sasrec"]
    spec, bn = D.sasrec_param_spec(NU, NI, NC, T, dims=dims)
    params, bn_state = S.sasrec_init(spec, bn, seed=3)
    assert params["sequential/sasrec/num_blocks_1/self_attention/dense_2/kernel"].shape == (40, 40)
    assert params["sequential/embedding/user_embedding"].shape == (NU, 16)
    g = torch.Generator().manual_seed(5)
    params = {n: t + 0.1 * torch.randn(t.shape, generator=g) for n, t in params.items()}
    batch = _batch(9)
    hp = dict(embed_l2=1e-4, layer_l2=1e-4)
    p = {n: t.double().requires_grad_(True) for n, t in params.items()}
    ctx = D.sasrec_forward(p, bn_state, batch, True)
    S.sasrec_losses(ctx, spec, batch, hp)["loss"].backward()
    assert ctx.t["final_state"].shape == (20, 40)
    for name, idx in (("sequential/sasrec/num_blocks_0/self_attention/dense_1/kernel", (33, 7)),
                      ("sequential/sasrec/num_blocks_1/multihead_attention/conv1d/kernel", (0, 38, 21))):
        vals = []
        for sgn in (+1, -1):
            q = {n: t.double().clone() for n, t in params.items()}
            q[name][idx] += sgn * 1e-6
            with torch.no_grad():
                vals.append(float(S.sasrec_losses(D.sasrec_forward(q, bn_state, batch, True), spec, batch, hp)["loss"]))
        fd = (vals[0] - vals[1]) / 2e-6
        assert abs(fd - float(p[name].grad[idx])) <= 1e-5 * max(abs(fd), 1e-5), (name, fd)


@pytest.mark.parametrize("model", S.MODELS + ("sasrec",))
def test_oracle_train_step_at_reference_widths(model):
    """SiblingOracleModel at the reference's widths: the per-lookup sparse gradients equal autograd through the tables, and a step
    moves every live variable."""
    hp = dict(embed_l2=1e-4, layer_l2=1e-4)
    dims = REFERENCE[model]
    m = D.SiblingOracleModel(model, NU, NI, NC, T, hp=hp, seed=4, dims=dims)
    O.perturb_params(m.params, m.bn_state, seed=5)
    batch = _batch(11)
    ref = m.train_step(batch, apply=False)
    p = {n: t.double().clone().requires_grad_(True) for n, t in m.params.items()}
    if model == "sasrec":
        want = S.sasrec_losses(D.sasrec_forward(p, m.bn_state, batch, True), m.spec, batch, hp)
    else:
        want = S.losses(S.forward(model, p, m.bn_state, batch, True), m.spec, batch, hp)
    want["loss"].backward()
    for k, v in want.items():
        assert abs(float(v.detach()) - ref["losses"][k]) < 1e-12, k
    for n, g in ref["grads"].items():
        assert torch.allclose(g, p[n].grad, rtol=1e-10, atol=1e-14), n
    before = {n: t.clone() for n, t in m.params.items()}
    m.train_step(batch)
    for n, _, _, grp in m.spec:
        assert bool((m.params[n] != before[n]).any()) == (grp != "frozen"), (n, grp)
    assert np.array_equal(m.params["sequential/embedding/item_embedding"].shape, (NI, 32))


@pytest.mark.parametrize("model", S.MODELS + ("sasrec",))
def test_width_helper_equals_the_oracle_at_its_own_widths(model):
    """tests/siblings_oracle_dims.py restates the oracle's inventories at any widths: at 16 / 4 / 20 they are the oracle's, and its
    SASRec forward pass is the oracle's (the attention scale it sets for the call is put back afterwards)."""
    if model == "sasrec":
        assert D.sasrec_param_spec(NU, NI, NC, T) == S.sasrec_param_spec(NU, NI, NC, T)
        spec, bn = S.sasrec_param_spec(NU, NI, NC, T)
        params, bn_state = S.sasrec_init(spec, bn, seed=3)
        p = {n: t.double() for n, t in params.items()}
        batch = _batch(9)
        a = D.sasrec_forward(p, bn_state, batch, False).t["logits"]
        assert torch.equal(a, S.sasrec_forward(p, bn_state, batch, False).t["logits"]) and S.SAS_D == 20
        wide, _ = D.sasrec_param_spec(NU, NI, NC, T, dims=(32, 8, 16))
        wp, wbn = S.sasrec_init(wide, bn, seed=3)
        ctx = D.sasrec_forward({n: t.double() for n, t in wp.items()}, wbn, batch, False)
        q, k = ctx.t["blk0.Q"], ctx.t["blk0.K"]
        assert ctx.t["blk0.Q"].shape[-1] == 40 and S.SAS_D == 20
        # the attention weights of block 0 at width 40 use 1 / sqrt(40): recompute them from Q and K
        s = q @ k.transpose(1, 2) / 40 ** 0.5
        mask = torch.as_tensor(np.asarray(batch["satisfied_mask"])).long()
        s = torch.where(mask[:, None, :] == 0, torch.full_like(s, float(-(2 ** 32) + 1)), s)
        y = torch.softmax(s, -1) @ ctx.t["blk0.V"] + ctx.t["blk0.qin"]
        assert torch.allclose(y, ctx.t["blk0.y"], rtol=1e-12, atol=1e-12)
    else:
        assert D.param_spec(model, NU, NI, NC) == S.param_spec(model, NU, NI, NC)
