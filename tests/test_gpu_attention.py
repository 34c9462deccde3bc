"""The attention weights behind each score (pamrec_attention / Engine.attention / explain) for all five models, against the float64
oracles and against the engine's own forward pass: the pooling weights are the ones the forward multiplied with, the encoder maps
reproduce the blocks' outputs, the predictions are bit-identical to forward(training=False), and a train step after the call is
unchanged."""
import ctypes
import os
import types

import numpy as np
import pytest
import torch

from oracle import pamrec_oracle as O
from oracle import siblings_oracle as S
import siblings_oracle_dims as D
from pamrec_b200 import deeprec_utils as DU

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NU, NI, NC = 40, 300, 20
MASK_NEG = -4294967295.0
TOL = 1e-5


def _masks(batch, keys=("mask",), seed=0):
    """Line 0 without any live key, line 1 with holes (a non-prefix mask), line 2 live at its last position only."""
    rng = np.random.default_rng(seed)
    T = batch["mask"].shape[1]
    for k in keys:
        m = np.asarray(batch[k]).copy()
        m[0] = 0
        if T > 1:
            m[1] = (rng.random(T) > 0.4).astype(np.int32)
            m[1, 0] = 1
            m[2] = 0
            m[2, T - 1] = 1
        batch[k] = m
    return batch


def _softmax_ref(Q, K, mask, scale):
    """softmax(mask ? Q K^T * scale : -(2^32)+1) in float64, [B, T, T]"""
    s = torch.einsum("btd,bsd->bts", Q, K) * scale
    s = torch.where(torch.as_tensor(mask)[:, None, :] == 0, torch.full_like(s, MASK_NEG), s)
    return torch.softmax(s, -1).numpy()


def _check_rows(w, live):
    """rows sum to 1; a masked key is exactly 0 in a line with a live key, every weight is 1 / T in a line without"""
    T = w.shape[-1]
    np.testing.assert_allclose(w.astype(np.float64).sum(-1), 1.0, rtol=0, atol=TOL)
    for b in range(w.shape[0]):
        if live[b].any():
            assert (w[b][..., ~live[b]] == 0).all(), f"line {b}: a masked key has a non-zero weight"
        else:
            assert (w[b] == np.float32(1.0 / T)).all(), f"line {b}: no live key, but the weights are not 1 / T"


def _pamrec(T, B, legacy, monkeypatch, cap):
    from pamrec_b200.engine import Engine
    if legacy:
        monkeypatch.setenv("PAMREC_HEAD_LEGACY", "1")
    else:
        monkeypatch.delenv("PAMREC_HEAD_LEGACY", raising=False)
    om = O.OracleModel(NU, NI, NC, T, seed=11)
    O.perturb_params(om.params, om.bn_state, seed=12)
    eng = Engine(NU, NI, NC, T, cap).allocate()
    eng.set_variables({n: t.numpy() for n, t in om.params.items()})
    eng.set_variables({n: t.numpy() for n, t in om.bn_state.items()})
    return om, eng


@pytest.mark.parametrize("legacy", [False, True], ids=["head2", "standalone"])
@pytest.mark.parametrize("T", [1, 7, 50, 128, 129, 200, 256])
def test_pamrec_against_the_oracle(T, legacy, monkeypatch):
    """max_batch above the batch at every other T: the copies out of the workspace must use the batch's own rows"""
    B = 6
    om, eng = _pamrec(T, B, legacy, monkeypatch, cap=B + 5 if T in (7, 128, 200) else B)
    batch = _masks(O.make_batch(3 + T, B, T, NU, NI, NC, grouped=False), seed=T)
    mask = np.asarray(batch["mask"])
    live = mask != 0
    db = eng.upload(batch, training=False)
    got = eng.attention(db, maps=True).result()
    torch.cuda.synchronize()
    ws = lambda n, *shape: eng.ws(n, B).reshape(B, *shape).cpu().numpy().astype(np.float64)
    new_long, h = ws("new_long", 40), ws("blk1.out", T, 40)
    blk = {k: {n: ws(f"blk{k}.{n}", T, 40) for n in ("V", "qin", "y")} for k in range(2)}
    ml = [eng.ws(f"blk{k}.ml", B).reshape(B, T, 2).cpu().numpy() for k in range(2)]
    pred = eng.forward(db, training=False).cpu().numpy()
    eng.close()
    ctx = om.eval_forward(batch)
    pool, maps = got["pool"], got["maps"]
    assert pool.shape == (B, 1, T) and maps.shape == (B, 2, T, T) and pool.dtype == maps.dtype == np.float32
    np.testing.assert_array_equal(got["pred"], pred)
    np.testing.assert_allclose(pool[:, 0], ctx.t["att"].numpy(), rtol=0, atol=TOL)
    _check_rows(pool[:, 0], live)
    for k in range(2):
        ref = _softmax_ref(ctx.t[f"blk{k}.Q"], ctx.t[f"blk{k}.K"], mask, 1.0 / np.sqrt(40.0))
        np.testing.assert_allclose(maps[:, k], ref, rtol=0, atol=TOL)
        _check_rows(maps[:, k], live[:, None, :].repeat(T, 1))
        if T <= 128:
            # the forward's tensor-core scores, recomputed bit for bit: the largest weight of a row is exp(m - m) / l = 1 / l exactly
            rows = live.any(1)
            np.testing.assert_array_equal(maps[rows, k].max(-1), np.float32(1) / ml[k][rows, :, 1])
        # the maps are the forward's own: P V + qin reproduces the block's output
        y = np.einsum("bts,bsd->btd", maps[:, k].astype(np.float64), blk[k]["V"]) + blk[k]["qin"]
        np.testing.assert_allclose(y, blk[k]["y"], rtol=0, atol=TOL * np.abs(blk[k]["y"]).max())
    # the pooling weights are the forward's own: sum_t a_t h_t is the engine's new_long
    nl = np.einsum("bt,btd->bd", pool[:, 0].astype(np.float64), h)
    np.testing.assert_allclose(nl, new_long, rtol=0, atol=1e-6 * np.abs(new_long).max())


SIB_DIMS = {16: (16, 4, 20), 32: (32, 8, 40)}
SAS_DIMS = {16: (16, 4, 20), 32: (32, 8, 16)}


def _sibling(model, T, B, dims, cap=None):
    from pamrec_b200.engine import Engine
    om = D.SiblingOracleModel(model, NU, NI, NC, T, seed=11, dims=dims)
    O.perturb_params(om.params, om.bn_state, seed=12)
    eng = Engine(NU, NI, NC, T, cap or B, model=model, emb_dims=dims).allocate()
    eng.set_variables({n: t.numpy() for n, t in om.params.items()})
    eng.set_variables({n: t.numpy() for n, t in om.bn_state.items()})
    return om, eng


def _sib_batch(seed, B, T):
    b = S.add_satisfied_fields(O.make_batch(seed, B, T, NU, NI, NC, grouped=False), seed=seed + 1)
    return _masks(b, ("mask", "satisfied_mask"), seed=seed)


@pytest.mark.parametrize("width", [16, 32], ids=["e20", "e40"])
@pytest.mark.parametrize("model", ["mmoe", "ple", "sharebottom"])
def test_sibling_branches_against_the_oracle(model, width):
    from pamrec_b200.engine import PamrecError
    B, T = 9, 20
    om, eng = _sibling(model, T, B, SIB_DIMS[width], cap=B + 7 if width == 16 else B)
    batch = _sib_batch(7, B, T)
    db = eng.upload(batch, training=False)
    got = eng.attention(db).result()
    torch.cuda.synchronize()
    aw = eng.ws("sib.aw").reshape(-1)[:2 * B * T].view(2, B, T).cpu().numpy()
    with pytest.raises(PamrecError, match="self-attention"):
        eng.attention(db, maps=True)
    maps_buf = torch.empty(B * 2 * T * T, device=eng.device)
    rc = eng.lib.pamrec_attention(eng.handle, ctypes.byref(db.struct), None, None, ctypes.c_void_p(maps_buf.data_ptr()), eng._stream())
    assert rc != 0 and b"maps_out" in eng.lib.pamrec_last_error(eng.handle)
    pred = eng.forward(db, training=False).cpu().numpy()
    eng.close()
    pool = got["pool"]
    assert pool.shape == (B, 2, T) and got["maps"] is None
    np.testing.assert_array_equal(got["pred"], pred)
    np.testing.assert_array_equal(pool.transpose(1, 0, 2), aw)              # the forward's own weights
    ctx = om.eval_forward(batch)
    for slot, (tag, mk) in enumerate((("att0", "satisfied_mask"), ("att1", "mask"))):
        np.testing.assert_allclose(pool[:, slot], ctx.t[tag + ".w"].numpy(), rtol=0, atol=TOL)
        _check_rows(pool[:, slot], np.asarray(batch[mk]) == 1)


@pytest.mark.parametrize("width", [16, 32], ids=["e20", "e40"])
@pytest.mark.parametrize("T", [1, 20, 129])
def test_sasrec_maps_against_the_oracle(width, T):
    B = 7
    om, eng = _sibling("sasrec", T, B, SAS_DIMS[width], cap=B + 3 if T == 20 else B)
    batch = _sib_batch(9, B, T)
    db = eng.upload(batch, training=False)
    got = eng.attention(db, maps=True).result()
    pool_only = eng.attention(db).result()
    pred = eng.forward(db, training=False).cpu().numpy()
    eng.close()
    E = sum(SAS_DIMS[width][:2])
    mask = np.asarray(batch["satisfied_mask"])
    live = mask == 1
    ctx = om.eval_forward(batch)
    maps = got["maps"]
    assert maps.shape == (B, 2, T, T) and got["pool"].shape == (B, 1, T)
    for k in range(2):
        ref = _softmax_ref(ctx.t[f"blk{k}.Q"], ctx.t[f"blk{k}.K"], mask, 1.0 / np.sqrt(E))
        np.testing.assert_allclose(maps[:, k], ref, rtol=0, atol=TOL)
        _check_rows(maps[:, k], live[:, None, :].repeat(T, 1))
    rsel = np.maximum(live.sum(1) - 1, 0)
    readout = maps[np.arange(B), 1, rsel]
    np.testing.assert_array_equal(got["pool"][:, 0], readout)
    np.testing.assert_array_equal(pool_only["pool"], got["pool"])
    for r in (got, pool_only):
        np.testing.assert_array_equal(r["pred"], pred)


@pytest.mark.parametrize("model,graph", [("pamrec", True), ("pamrec", False), ("mmoe", False), ("sasrec", False)])
def test_train_step_after_attention_is_unchanged(model, graph):
    """attention() between train steps leaves the following steps' losses as they are without it (CUDA-graph replay on and off),
    within the last-bit spread of the atomic weight-gradient sums (test_gpu_rank.py:test_train_step_after_ranking_is_unchanged)."""
    from pamrec_b200.engine import Engine
    from pamrec_b200.models import initial_variables
    T, dims = 20, (16, 4, 20)
    shapes = Engine(NU, NI, NC, T, 8, model=model, emb_dims=dims).variable_shapes()
    var = initial_variables(shapes, types.SimpleNamespace(init_method="tnormal", init_value=0.3), 5)
    # perturbed as in test_gpu_rank.py: with the initial batch-norm state some gradients are rounding noise, which Adam's first
    # steps scale up to full-size updates and two identical runs already part by far more than one ulp
    params = {n: torch.from_numpy(a) for n, a in var.items()}
    bn = {n: params.pop(n) for n in list(params) if n.endswith(("moving_mean", "moving_variance"))}
    O.perturb_params(params, bn, seed=5)
    var = {n: t.numpy() for n, t in {**params, **bn}.items()}
    batch = S.add_satisfied_fields(O.make_batch(3, 20, T, NU, NI, NC), seed=3)
    lines = _sib_batch(11, 9, T)
    losses = []
    for explain in (False, True):
        eng = Engine(NU, NI, NC, T, 64, model=model, emb_dims=dims, graph=graph).allocate("cuda:0")
        eng.set_variables(var)
        db, ldb = eng.upload(batch), eng.upload(lines, training=False)
        steps = []
        for i in range(4):                   # with graph replay: step 2 is captured, steps 3 and 4 replay it
            if explain and i:
                eng.attention(ldb, maps=model != "mmoe").result()
            steps.append(eng.train_step(db).cpu().numpy().copy())
        losses.append(steps)
        eng.close()
    for a, b in zip(*losses):
        np.testing.assert_allclose(a, b, rtol=1e-6, atol=1e-7)


@pytest.fixture(scope="module")
def data_root(tmp_path_factory):
    from pamrec_b200 import synth
    root = tmp_path_factory.mktemp("attention")
    synth.generate(str(root), "wechat", n_users=60, n_items=400, n_cates=15, mean_len=30, seed=21, eval_per_user=2)
    return str(root)


@pytest.mark.parametrize("cls_name,yaml_name", [("PAMRECModel", "mmoe.yaml"), ("MMoEModel_original", "mmoe.yaml"),
                                                ("SASRecModel", "sasrec.yaml")])
def test_explain_end_to_end(data_root, tmp_path, cls_name, yaml_name):
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
    K, T = 4, 30
    maps = cls_name != "MMoEModel_original"
    out, pred_file = str(tmp_path / "explain.tsv"), str(tmp_path / "pred.txt")
    got = model.explain(test, out, top_k=K, maps=maps)
    model.predict(test, pred_file)
    pred_lines = open(pred_file).read().splitlines()
    text = open(out).read().splitlines()
    N, P = got["pred"].shape[0], len(model.ATTENTION_SLOTS)
    assert len(text) == len(pred_lines) == N > 50
    assert got["pool"].shape == (N, P, T) and got["positions"].shape == (N, P, K)
    assert (got["maps"] is not None) == maps and (not maps or got["maps"].shape == (N, 2, T, T))
    feeds = list(model.iterator.load_data_from_file(test, batch_num_ngs=0))
    hist = {k: np.concatenate([np.asarray(f[k]).reshape(-1, T) for f in feeds]) for s in model.ATTENTION_SLOTS for k in s}
    users = np.concatenate([np.asarray(f["users"]).reshape(-1) for f in feeds])
    np.testing.assert_array_equal(got["users"], users)
    inv_u = {v: k for k, v in model.iterator.userdict.items()}
    inv_i = {v: k for k, v in model.iterator.itemdict.items()}
    n_tied = 0
    for r in range(N):
        cols = text[r].split("\t")
        assert cols[0] == inv_u[int(users[r])] and cols[1] == pred_lines[r] == str(got["pred"][r])
        assert len(cols) == 2 + P
        for s, (hk, mk) in enumerate(model.ATTENTION_SLOTS):
            live = hist[mk][r] > 0
            pos, w = got["positions"][r, s], got["weights"][r, s]
            want = DU.attention_topk(got["pool"][r:r + 1, s], live[None], K)[0][0]
            np.testing.assert_array_equal(pos, want)
            n = int((pos >= 0).sum())
            assert n == min(K, int(live.sum()))
            ws_ = got["pool"][r, s, pos[:n]]
            np.testing.assert_array_equal(w[:n], ws_)
            assert all(ws_[i] > ws_[i + 1] or (ws_[i] == ws_[i + 1] and pos[i] < pos[i + 1]) for i in range(n - 1))
            n_tied += int(np.sum(ws_[:-1] == ws_[1:])) if n > 1 else 0
            np.testing.assert_array_equal(got["items"][r, s, :n], hist[hk][r][pos[:n]])
            entries = [e.rsplit(":", 1) for e in cols[2 + s].split(",")] if cols[2 + s] else []
            assert [e[0] for e in entries] == [inv_i.get(int(i), str(int(i))) for i in got["items"][r, s, :n]]
            np.testing.assert_array_equal(np.asarray([e[1] for e in entries], np.float32), w[:n])
    with pytest.raises(ValueError):
        model.explain(test, out, top_k=0)
    with pytest.raises(ValueError):
        model.explain(test, out, top_k=T + 1)
