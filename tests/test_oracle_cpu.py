"""The floating-point oracle checked against what CAN be pinned without TensorFlow: hand-computed values and closed forms of
the formulas it restates (ApproxNDCG of TF-Ranking 0.3.x, tf.nn.sigmoid_cross_entropy_with_logits, tf.train.AdamOptimizer's
first step, tf.clip_by_norm, non-fused batch norm), gradient self-consistency, and the structure of the reference graph the
tests rely on.  These do not replace a run of the reference (parity of the float path stays "unpinned", see the oracle's
header); they pin the restatement against transcription errors."""
import math

import numpy as np
import torch

from oracle import pamrec_oracle as O


def test_approx_ndcg_hand_values():
    # one list, scores far apart: approx ranks -> exact ranks 1..5, so the loss is -DCG/IDCG of that ordering
    labels = torch.tensor([[3.0, 0.0, 1.0, 2.0, 0.0]], dtype=torch.float64)
    scores = torch.tensor([[5.0, 1.0, 3.0, 4.0, 2.0]], dtype=torch.float64) * 10       # order: item0, item3, item2, item4, item1
    got = float(O.approx_ndcg_loss(labels, scores))
    gains = 2.0 ** np.array([3.0, 2.0, 1.0, 0.0, 0.0]) - 1
    disc = 1 / np.log1p(np.arange(1, 6))
    ideal = float((gains * disc).sum())
    assert abs(got - (-1.0)) < 1e-6                                                      # perfectly ordered list: NDCG = 1
    # reversed scores: ranks of (item0..4) = 5, 1, 3, 4, 2
    got = float(O.approx_ndcg_loss(labels, -scores))
    ranks = np.array([5, 1, 3, 4, 2], dtype=np.float64)
    dcg = float(((2.0 ** labels.numpy()[0] - 1) / np.log1p(ranks)).sum())
    assert abs(got + dcg / ideal) < 1e-6
    # the smooth rank itself: rank_i = 0.5 + sum_j sigmoid(alpha (s_j - s_i)), alpha = 10, j includes i
    s = torch.tensor([[0.1, 0.3]], dtype=torch.float64)
    y = torch.tensor([[1.0, 0.0]], dtype=torch.float64)
    r0 = 0.5 + 0.5 + 1 / (1 + math.exp(-10 * 0.2))
    r1 = 0.5 + 0.5 + 1 / (1 + math.exp(+10 * 0.2))
    want = -((2 ** 1 - 1) / math.log1p(r0) + 0.0 / math.log1p(r1)) / ((2 ** 1 - 1) / math.log1p(1.0))
    assert abs(float(O.approx_ndcg_loss(y, s)) - want) < 1e-12


def test_approx_ndcg_zero_label_lists_have_weight_zero():
    labels = torch.tensor([[0.0] * 5, [1.0, 0, 0, 0, 2.0], [0.0] * 5], dtype=torch.float64)
    scores = torch.randn(3, 5, dtype=torch.float64, generator=torch.Generator().manual_seed(0))
    full = float(O.approx_ndcg_loss(labels, scores))
    only = float(O.approx_ndcg_loss(labels[1:2], scores[1:2]))
    assert abs(full - only) < 1e-12                     # MEAN over lists with a non-zero label sum only
    assert float(O.approx_ndcg_loss(labels[:1], scores[:1])) == 0.0
    # permuting a list permutes nothing in the loss
    perm = torch.tensor([3, 1, 4, 0, 2])
    assert abs(float(O.approx_ndcg_loss(labels[1:2][:, perm], scores[1:2][:, perm])) - only) < 1e-12


def test_sigmoid_xent_is_the_tf_formula():
    x = torch.tensor([-30.0, -2.0, 0.0, 0.5, 40.0], dtype=torch.float64)
    y = torch.tensor([0.0, 1.0, 1.0, 0.0, 1.0], dtype=torch.float64)
    want = torch.clamp(x, min=0) - x * y + torch.log1p(torch.exp(-x.abs()))           # tf.nn.sigmoid_cross_entropy_with_logits
    assert torch.allclose(O._sigmoid_xent(x, y), want, atol=0, rtol=1e-15)
    direct = -(y * torch.log(torch.sigmoid(x)) + (1 - y) * torch.log(1 - torch.sigmoid(x)))
    assert torch.allclose(want[1:4], direct[1:4], rtol=1e-12)


def test_batch_norm_is_the_non_fused_keras_layer():
    ctx = O._Ctx({"s/gamma": torch.tensor([2.0, 1.0], dtype=torch.float64), "s/beta": torch.tensor([0.5, -1.0], dtype=torch.float64)},
                 {}, True, torch.float64)
    z = torch.tensor([[1.0, 2.0], [3.0, 2.0], [5.0, 8.0]], dtype=torch.float64)
    y = O._bn(ctx, z, "s")
    mean = z.mean(0)
    var = z.var(0, unbiased=False)                                                     # biased variance, eps = 1e-4
    assert torch.allclose(y, torch.tensor([2.0, 1.0]) * (z - mean) / torch.sqrt(var + 1e-4) + torch.tensor([0.5, -1.0]))
    m, v = ctx.new_bn["s"]
    assert torch.allclose(m, mean) and torch.allclose(v, var)
    assert ctx.kink_margin == float(y.abs().min())


def _small():
    om = O.OracleModel(40, 200, 12, 10, seed=1)
    O.perturb_params(om.params, om.bn_state, seed=2)
    return om, O.make_batch(3, 20, 10, 40, 200, 12)


def test_first_adam_step_closed_form_and_clip():
    om, batch = _small()
    p0 = {n: t.clone() for n, t in om.params.items()}
    ref = om.train_step(batch)
    b1, b2, eps, lr = np.float32(0.9), np.float32(0.999), np.float32(1e-8), np.float32(1e-3)
    lr_t = float(lr) * math.sqrt(1 - float(b2)) / (1 - float(b1))
    for name in ("sequential/logit_fcn/nn_part/w_nn_output", "sequential/embedding/item_embedding",
                 "sequential/pamrec/num_blocks_0/self_attention/Q_timeaware_embedding"):
        g = ref["grads"][name].double() * ref["scales"][name]
        m = (1 - float(b1)) * g
        v = (1 - float(b2)) * g * g
        want = p0[name].double() - lr_t * m / (v.sqrt() + float(eps))
        assert torch.allclose(om.params[name].double(), want, rtol=0, atol=1e-7), name       # fp32 storage of the result
        # tf.clip_by_norm: scale = clip / max(norm, clip)
        norm = math.sqrt(ref["sqnorms"][name])
        assert abs(ref["scales"][name] - 2.0 / max(norm, 2.0)) < 1e-15
    # every row of a sparse table moves only if it was looked up in step 1 (m = v = 0 elsewhere) ...
    touched = np.unique(np.concatenate([batch["item_history"].reshape(-1), batch["items"]]))
    moved = (om.params["sequential/embedding/item_embedding"] != p0["sequential/embedding/item_embedding"]).any(1).numpy()
    assert set(np.nonzero(moved)[0]) <= set(touched.tolist())
    # ... and keeps moving afterwards without being looked up again (tf.train.AdamOptimizer is not lazy)
    other = O.make_batch(4, 20, 10, 40, 200, 12)
    before = om.params["sequential/embedding/item_embedding"].clone()
    om.train_step(other)
    touched2 = np.unique(np.concatenate([other["item_history"].reshape(-1), other["items"]]))
    only_first = np.setdiff1d(touched, touched2)
    assert only_first.size and (om.params["sequential/embedding/item_embedding"][only_first] != before[only_first]).any()


def test_loss_is_the_sum_of_its_four_terms_and_l2_groups():
    om, batch = _small()
    ref = om.train_step(batch, apply=False)
    L = ref["losses"]
    assert abs(L["loss"] - (L["data_loss"] + L["regular_loss"] + L["auxiliary_data_loss"] + L["order_loss"])) < 1e-12
    assert L["order_loss"] <= 0 and L["data_loss"] > 0 and L["auxiliary_data_loss"] > 0
    # variables outside every loss term get no gradient entry or a zero one; dead-branch weights get exactly the L2 gradient
    name = "sequential/pamrec/long_term/attention_fcn/attention_mat"
    assert torch.allclose(ref["grads"][name], om.hp["layer_l2"] * om.params[name].double(), rtol=1e-12, atol=0)
    x = "xilidu_logit_fcn/nn_part/w_nn_output"                                          # trained, but not in the L2 set
    p = om.cast_params(True)
    g_wo_l2 = ref["grads"][x]
    assert not torch.allclose(g_wo_l2, torch.zeros_like(g_wo_l2))
    reg = sum(0.5 * om.hp["layer_l2"] * float((p[n].detach() ** 2).sum()) for n, _, _, grp in om.spec if grp == "layer")
    assert reg < L["regular_loss"] < reg + 1e-3                                          # + the embedding rows of the batch


def test_gradients_match_finite_differences():
    om, batch = _small()
    ref = om.train_step(batch, apply=False)
    name = "sequential/logit_fcn/nn_part/w_nn_layer1"
    idx = (3, 5)
    h = 1e-6
    base = om.params[name].clone()
    vals = []
    for sgn in (+1, -1):
        om.params[name] = base.clone().double()
        om.params[name][idx] += sgn * h
        vals.append(om.train_step(batch, apply=False)["losses"]["loss"])
    om.params[name] = base
    fd = (vals[0] - vals[1]) / (2 * h)
    assert abs(fd - float(ref["grads"][name][idx])) <= 1e-5 * max(abs(fd), 1e-6)


def test_softmax_loss_hand_values():
    """hparams.loss == "softmax" (BM:222-242): -group * mean(log(where(y == 1, softmax, 1)))."""
    g = 5
    x = torch.zeros(10, dtype=torch.float64)
    y = torch.tensor([1.0, 0, 0, 0, 0, 0, 0, 1.0, 0, 0], dtype=torch.float64)
    assert abs(float(O.softmax_pos_loss(x, y, g)) - math.log(5)) < 1e-12          # one positive per group, uniform softmax
    y2 = torch.tensor([1.0, 1.0, 0, 0, 0, 0, 0, 0, 0, 0], dtype=torch.float64)    # two positives in one group, none in the other
    assert abs(float(O.softmax_pos_loss(x, y2, g)) - math.log(5)) < 1e-12         # -5 * (2 * -ln 5) / 10
    x3 = torch.tensor([2.0, 0.0, 0.0, 0.0, 0.0], dtype=torch.float64)
    y3 = torch.tensor([1.0, 0, 0, 0, 0], dtype=torch.float64)
    want = -(2.0 - math.log(math.exp(2.0) + 4.0))
    assert abs(float(O.softmax_pos_loss(x3, y3, g)) - want) < 1e-12
    assert float(O.softmax_pos_loss(x3, torch.zeros(5, dtype=torch.float64), g)) == 0.0
    # through the model: only the two softmax terms differ from the cross-entropy configuration
    om_x = O.OracleModel(40, 200, 12, 10, seed=1)
    om_s = O.OracleModel(40, 200, 12, 10, seed=1, hp=dict(loss="softmax", softmax_group=5))
    batch = O.make_batch(3, 20, 10, 40, 200, 12)
    lx, ls = om_x.train_step(batch, apply=False)["losses"], om_s.train_step(batch, apply=False)["losses"]
    assert lx["order_loss"] == ls["order_loss"] and lx["regular_loss"] == ls["regular_loss"]
    assert lx["data_loss"] != ls["data_loss"] and lx["auxiliary_data_loss"] != ls["auxiliary_data_loss"]


def test_forced_relu_masks_and_grouped_projection():
    """The two options the large-batch GPU parity tests rely on: (1) differentiating on a supplied ReLU pattern is the identity
    when the pattern is the pass's own, and flips exactly the supplied units otherwise; (2) the bucket-grouped time-aware
    projection equals the reference-shaped [B,T,40,40] gather formulation (PAM:714-728)."""
    nu, ni, nc, T, B = 60, 400, 20, 14, 20
    om = O.OracleModel(nu, ni, nc, T, seed=5)
    O.perturb_params(om.params, om.bn_state, seed=6)
    batch = O.make_batch(3, B, T, nu, ni, nc)
    base = om.train_step(batch, apply=False, keep=("x0",))
    om.proj = "grouped"
    grp = om.train_step(batch, apply=False, keep=("x0",))
    assert abs(base["losses"]["loss"] - grp["losses"]["loss"]) < 1e-14
    assert float((base["t"]["x0"].grad - grp["t"]["x0"].grad).abs().max()) < 1e-15
    for n in base["grads"]:
        assert float((base["grads"][n] - grp["grads"][n]).abs().max()) < 1e-14, n
    # own pattern -> identical step
    ctx = om._forward(om.cast_params(False), batch, True)
    sp = "sequential/pamrec/new_long/score_1/nn_part/"
    scope = "sequential/pamrec/expert_2/nn_part/batch_normalization"
    z = ctx.t["expert2.z0"]
    mean, var = ctx.new_bn[scope]
    y = om.params[scope + "/gamma"].double() * ((z - mean) / (var + O.BN_EPS) ** 0.5) + om.params[scope + "/beta"].double()
    own = (y > 0).numpy()
    same = om.train_step(batch, apply=False, relu_masks={scope: own})
    assert same["relu_forced"] == 0 and same["losses"]["loss"] == grp["losses"]["loss"]
    for n in grp["grads"]:
        assert torch.equal(same["grads"][n], grp["grads"][n]), n
    # flip the unit closest to its kink: the forward value moves by at most that margin, the gradient of its weights changes
    i, j = np.unravel_index(np.abs(y.numpy()).argmin(), y.shape)
    flipped = own.copy()
    flipped[i, j] = ~flipped[i, j]
    other = om.train_step(batch, apply=False, relu_masks={scope: flipped})
    assert other["relu_forced"] == 1
    assert abs(other["losses"]["loss"] - grp["losses"]["loss"]) <= 10 * abs(float(y[i, j]))
    w = "sequential/pamrec/expert_2/nn_part/w_nn_layer0"
    assert float((other["grads"][w] - grp["grads"][w]).abs().max()) > 0
    assert sp  # (score scopes use the same mechanism; exercised on the GPU by tests/relu_masks.py)


def test_out_of_range_bucket_reads_a_zero_matrix():
    """lisan gives bucket 10 - one past the [10, 1600] time-aware tables - for a play / duration ratio beyond its last border and
    for a zero duration.  tf.gather on the GPU returns a zero row for that index: the token's Q, K and V are 0, its qin still goes
    through the LayerNorm into the attention residual, and no table row gets a gradient from it.  Both projection forms agree."""
    nu, ni, nc, T, B = 60, 400, 20, 14, 20
    om = O.OracleModel(nu, ni, nc, T, seed=5)
    O.perturb_params(om.params, om.bn_state, seed=6)
    batch = O.make_batch(3, B, T, nu, ni, nc)
    lt = batch["item_loop_times_history"]
    lt[:, 3] = 10.0                                  # one position of every history
    lt[:5, :] = 10.0                                 # one listwise group entirely out of range
    lt[10:15, 5] = 12.5
    lt[10:15, 6] = -1.0
    lt[10:15, 7] = 9.99                              # truncates to 9: in range
    lt[10:15, 8] = -0.5                              # truncates to 0: in range
    want = np.where((lt > -1) & (lt < 10), np.trunc(np.where((lt > -1) & (lt < 10), lt, 0)), 10).astype(np.int64)
    assert np.array_equal(O.bucket_ids(lt).numpy(), want)
    out = (want == 10) & (batch["mask"] == 1)
    assert out.sum() > 5 and (want == 9).any() and (want == 0).any()
    keep = ("blk0.Q", "blk0.K", "blk0.V", "blk1.Q", "blk1.K", "blk1.V", "blk0.qin", "blk0.y")
    base = om.train_step(batch, apply=False, keep=keep)
    om.proj = "grouped"
    grp = om.train_step(batch, apply=False, keep=keep)
    assert abs(base["losses"]["loss"] - grp["losses"]["loss"]) < 1e-14
    for n in base["grads"]:
        assert float((base["grads"][n] - grp["grads"][n]).abs().max()) < 1e-14, n
    z = torch.as_tensor(want == 10)
    t = grp["t"]
    for k in keep[:6]:
        assert float(t[k].detach()[z].abs().max()) == 0.0, k      # padded positions included: they take the same path
    # tokens in range: qin (Q) or x0 (K, V) times their bucket's matrix; out of range: qin = LN(x0) as for any token
    qin, x0, b = t["blk0.qin"].detach(), t["x0"].detach(), O.bucket_ids(lt)
    assert float(qin[z].abs().max()) > 0
    for m, a in (("Q", qin), ("K", x0), ("V", x0)):
        W = om.params[f"sequential/pamrec/num_blocks_0/self_attention/{m}_timeaware_embedding"].double()[b[~z]].reshape(-1, O.D, O.D)
        assert torch.allclose(t["blk0." + m].detach()[~z], torch.einsum("ni,nij->nj", a[~z], W), rtol=0, atol=1e-14), m
    # a table row that only out-of-range tokens would select gets the L2 gradient alone
    lt2 = batch["item_loop_times_history"].copy()
    lt2[lt2 == 4] = 10.0
    g2 = om.train_step(dict(batch, item_loop_times_history=lt2), apply=False)["grads"]
    for m in "QKV":
        name = f"sequential/pamrec/num_blocks_1/self_attention/{m}_timeaware_embedding"
        l2 = om.hp["layer_l2"] * om.params[name].double()
        assert torch.allclose(g2[name][4], l2[4], rtol=1e-12, atol=0), name
        assert float((g2[name][3] - l2[3]).abs().max()) > 0, name
