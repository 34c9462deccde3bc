"""CPU oracle for the PAMRec train / score step.

TEST INFRASTRUCTURE ONLY.  Nothing under ``pamrec_b200/`` may import this file;
only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline``
/ ``--impl reference`` legs do, and there only as the checker / timed CPU arm.

PARITY UNPINNED for the floating-point model: the reference is a TensorFlow 2.4
graph (plus ``tensorflow_ranking``'s ApproxNDCG) and neither package can be
installed in this image, the reference ships no golden vectors, and no test of
the reference pins any tensor on this path.  This file restates the reference's
arithmetic from its source (citations below, relative to /root/reference) and
from the published TF 2.4 / TF-Ranking 0.3.x semantics of the few third-party
ops it calls.  The integer half of the path (batching, bucket ids, metrics) IS
pinned: see ``oracle/gen_golden.py`` which runs the reference's own
``sequential_iterator.py`` / ``deeprec_utils.py`` under a stub ``tensorflow``.

Math follows (PAM = reco_utils/recommender/deeprec/models/sequential/pamrec.py,
SBM = .../sequential_base_model.py, BM = .../models/base_model.py):

* embeddings / lookups            SBM:562-712, PAM:119-190
* encoder input                   PAM:251-257
* time-aware SASRec block         PAM:516-543, 638-664 (LN), 666-811 (attention), 545-582 (FFN)
* attention pooling               PAM:272-282, MLP+BN PAM:320-382
* MMoE                            PAM:26-50
* towers                          BM:634-715, PAM:212-215, PAM:71
* losses                          BM:195-205, PAM:81-106, PAM:70-79, BM:122-134, BM:247-254, PAM:54-68
* L2 parameter groups             SBM:640-664, PAM:173-182, SBM:714-721
* clip + Adam                     BM:288-304, BM:256-286 (+ TF 2.4 ``AdamOptimizer`` dense/sparse apply)
"""
import math

import numpy as np
import torch

I_DIM = 16          # item_embedding_dim   (config/mmoe.yaml:22)
C_DIM = 4           # cate_embedding_dim   (config/mmoe.yaml:23)
U_DIM = 20          # user_embedding_dim   (config/mmoe.yaml:24)
E_DIM = I_DIM + C_DIM
D = 2 * E_DIM       # PAM:144, PAM:523
NB = 10             # rows of the time-aware tables, PAM:699-713
GROUP = 5           # PAM:73-75, IT:98
MASK_NEG = float(-(2 ** 32) + 1)   # PAM:276, PAM:780
LN_EPS = 1e-8       # PAM:639
BN_EPS = 1e-4       # PAM:370, BM:684
BN_MOMENTUM = 0.95  # PAM:369, BM:683

EXPERT_NUM = 5
EXPERT_SIZES = (100, 64)
GATE_SIZES = (64, 5)
TOWER_SIZES = (100, 64)
ATT_FCN_SIZES = (80, 40)

TOWERS = ("sequential/logit_fcn", "sequential/valid_logit_fcn", "xilidu_logit_fcn")
DEAD = (("new_distill", 40), ("long_term", 20), ("short_term", 20))


# --------------------------------------------------------------------------- parameters
def _mlp_spec(prefix, in_dim, sizes, out=False, group="layer"):
    """Variables of _fcn_transform_net (PAM:320-382) / _fcn_net (BM:634-715)."""
    spec, bn = [], []
    last = in_dim
    for i, n in enumerate(sizes):
        spec.append((f"{prefix}/nn_part/w_nn_layer{i}", (last, n), "tn", group))
        spec.append((f"{prefix}/nn_part/b_nn_layer{i}", (n,), "zeros", group))
        bname = "batch_normalization" if i == 0 else f"batch_normalization_{i}"
        spec.append((f"{prefix}/nn_part/{bname}/gamma", (n,), "ones", group))
        spec.append((f"{prefix}/nn_part/{bname}/beta", (n,), "zeros", group))
        bn.append((f"{prefix}/nn_part/{bname}", n))
        last = n
    if out:
        spec.append((f"{prefix}/nn_part/w_nn_output", (last, 1), "tn", group))
        spec.append((f"{prefix}/nn_part/b_nn_output", (1,), "zeros", group))
    return spec, bn


def param_spec(n_users, n_items, n_cates, T):
    """TF variable inventory (SURVEY Appendix B).  Returns (params, bn_layers).

    params: list of (name, shape, init, group); group in
      frozen | embed | embed_l2only | pos | layer | layer_nol2
    bn_layers: list of (scope, channels) for moving_mean / moving_variance.
    """
    P, BN = [], []
    emb = "sequential/embedding/"
    P += [
        (emb + "user_embedding", (n_users, U_DIM), "tn", "frozen"),
        (emb + "item_embedding", (n_items, I_DIM), "tn", "embed"),
        (emb + "cate_embedding", (n_cates, C_DIM), "tn", "embed"),
        (emb + "looptimes_embedding", (10, C_DIM), "tn", "frozen"),
        (emb + "user_long_embedding", (n_users, U_DIM), "tn", "embed_l2only"),
        (emb + "user_short_embedding", (n_users, U_DIM), "tn", "embed_l2only"),
        (emb + "play_lookup", (10, 40), "tn", "frozen"),
        (emb + "position_embedding", (T, D), "tn", "pos"),
    ]
    for b in range(2):
        pre = f"sequential/pamrec/num_blocks_{b}/"
        P += [
            (pre + "ln/Variable", (D,), "zeros", "layer"),       # beta  PAM:660
            (pre + "ln/Variable_1", (D,), "ones", "layer"),      # gamma PAM:661
            (pre + "self_attention/Q_timeaware_embedding", (NB, D * D), "glorot", "layer"),
            (pre + "self_attention/K_timeaware_embedding", (NB, D * D), "glorot", "layer"),
            (pre + "self_attention/V_timeaware_embedding", (NB, D * D), "glorot", "layer"),
            (pre + "multihead_attention/conv1d/kernel", (1, D, D), "glorot", "layer"),
            (pre + "multihead_attention/conv1d/bias", (D,), "zeros", "layer"),
            (pre + "multihead_attention/conv1d_1/kernel", (1, D, D), "glorot", "layer"),
            (pre + "multihead_attention/conv1d_1/bias", (D,), "zeros", "layer"),
            (pre + "ln_1/Variable", (D,), "zeros", "layer"),
            (pre + "ln_1/Variable_1", (D,), "ones", "layer"),
        ]
    s, b = _mlp_spec("sequential/pamrec/new_long/score_1", D, (20, 1))
    P += s; BN += b
    for name, q in DEAD:
        pre = f"sequential/pamrec/{name}/attention_fcn"
        P.append((pre + "/attention_mat", (D, q), "tn", "layer"))
        s, b = _mlp_spec(pre + "/att_fcn", 4 * q, ATT_FCN_SIZES, out=True)
        P += s; BN += b
    for j in range(EXPERT_NUM):
        s, b = _mlp_spec(f"sequential/pamrec/expert_{j}", D, EXPERT_SIZES)
        P += s; BN += b
    for g in ("gate_main", "gate_sub"):
        s, b = _mlp_spec(f"sequential/pamrec/{g}", D, GATE_SIZES)
        P += s; BN += b
    for tw in TOWERS:
        grp = "layer_nol2" if tw.startswith("xilidu") else "layer"
        s, b = _mlp_spec(tw, 64 + E_DIM, TOWER_SIZES, out=True, group=grp)
        P += s; BN += b
    return P, BN


def init_params(n_users, n_items, n_cates, T, seed=8, init_value=0.01):
    """Random weights with the reference's initializer *families* (BM:165-193; TF default
    glorot_uniform where no initializer is in scope).  TF's Philox streams cannot be
    reproduced; parity is defined on injected identical weights."""
    g = torch.Generator().manual_seed(seed)
    spec, bn = param_spec(n_users, n_items, n_cates, T)
    params = {}
    for name, shape, init, _ in spec:
        if init == "tn":
            t = torch.empty(shape, dtype=torch.float32)
            torch.nn.init.trunc_normal_(t, mean=0.0, std=init_value, a=-2 * init_value, b=2 * init_value, generator=g)
        elif init == "glorot":
            if len(shape) == 3:
                fan_in, fan_out = shape[0] * shape[1], shape[0] * shape[2]
            else:
                fan_in, fan_out = shape
            lim = math.sqrt(6.0 / (fan_in + fan_out))
            t = (torch.rand(shape, generator=g, dtype=torch.float32) * 2 - 1) * lim
        elif init == "zeros":
            t = torch.zeros(shape, dtype=torch.float32)
        elif init == "ones":
            t = torch.ones(shape, dtype=torch.float32)
        else:
            raise ValueError(init)
        params[name] = t
    bn_state = {}
    for scope, n in bn:
        bn_state[scope + "/moving_mean"] = torch.zeros(n, dtype=torch.float32)
        bn_state[scope + "/moving_variance"] = torch.ones(n, dtype=torch.float32)
    return params, bn_state


def perturb_params(params, bn_state, seed=123, scale=0.05):
    """Move zeros/ones-initialised variables (biases, LN/BN gamma+beta, moving stats) off
    their trivial values so parity tests exercise every term."""
    g = torch.Generator().manual_seed(seed)
    for name, t in params.items():
        if name.endswith(("beta", "bias", "/Variable")) or "/b_nn_" in name:
            t.add_(torch.randn(t.shape, generator=g) * scale)
        elif name.endswith(("gamma", "/Variable_1")):
            t.add_(torch.randn(t.shape, generator=g) * scale)
    for name, t in bn_state.items():
        if name.endswith("moving_mean"):
            t.add_(torch.randn(t.shape, generator=g) * scale)
        else:
            t.mul_(torch.rand(t.shape, generator=g) * 0.5 + 0.75)


# --------------------------------------------------------------------------- synthetic batches
def make_batch(seed, B, T, n_users, n_items, n_cates, grouped=True, min_len=1, zipf_a=1.1):
    """Array-level synthetic batch in the layout of IT:1111-1135 (only the live keys).

    grouped=True reproduces the train layout: GROUP consecutive rows share one history
    (IT:645-684).  ids follow a Zipf popularity; index 0 is the padding / OOV id.
    """
    rng = np.random.default_rng(seed)
    assert not grouped or B % GROUP == 0
    n_hist = B // GROUP if grouped else B

    def zipf_ids(size, n):
        r = rng.zipf(zipf_a, size=size).astype(np.int64)
        return (1 + (r - 1) % max(n - 1, 1)).astype(np.int32)

    lens = rng.integers(min_len, T + 1, size=n_hist)
    ih = np.zeros((n_hist, T), np.int32)
    ch = np.zeros((n_hist, T), np.int32)
    bk = np.zeros((n_hist, T), np.float32)
    mask = np.zeros((n_hist, T), np.int32)
    for r in range(n_hist):
        L = int(lens[r])
        ih[r, :L] = zipf_ids(L, n_items)
        ch[r, :L] = zipf_ids(L, n_cates)
        bk[r, :L] = rng.integers(0, NB, size=L)
        mask[r, :L] = 1
    rep = GROUP if grouped else 1
    batch = {
        "item_history": np.repeat(ih, rep, axis=0),
        "item_cate_history": np.repeat(ch, rep, axis=0),
        "item_loop_times_history": np.repeat(bk, rep, axis=0),
        "mask": np.repeat(mask, rep, axis=0),
        "users": np.repeat(rng.integers(1, n_users, size=n_hist).astype(np.int32), rep),
        "items": zipf_ids(B, n_items),
        "cates": zipf_ids(B, n_cates),
        "labels_satisfied": rng.integers(0, 2, size=(B, 1)).astype(np.float32),
        "labels_play": rng.integers(0, 2, size=(B, 1)).astype(np.float32),
        "plays": rng.integers(0, NB, size=(B, 1)).astype(np.float32),
    }
    if grouped and B >= 2 * GROUP:           # one all-zero-label group: weight-0 path of ApproxNDCG
        batch["plays"][GROUP:2 * GROUP] = 0.0
    return batch


# --------------------------------------------------------------------------- forward
def _ln(x, beta, gamma):
    """PAM:638-664: population variance, eps inside the sqrt."""
    mean = x.mean(-1, keepdim=True)
    var = ((x - mean) ** 2).mean(-1, keepdim=True)
    return gamma * ((x - mean) / (var + LN_EPS) ** 0.5) + beta


class _Ctx:
    def __init__(self, p, bn_state, training, dtype, relu_masks=None):
        self.p, self.bn_state, self.training, self.dtype = p, bn_state, training, dtype
        self.new_bn = {}
        self.t = {}          # named intermediates
        self.kink_margin = float("inf")   # smallest |BN output| in front of a ReLU over the [B, C] head layers (see _bn)
        self.relu_masks = relu_masks or {}
        self.relu_forced = 0              # units whose forced state differs from this forward pass's own sign


def _act(ctx, y, key):
    """ReLU, or - when the caller supplies the activation pattern of another forward pass under `key` - that pattern.

    ReLU is not differentiable at 0.  Of the ~10^6 pre-activations of a step a few always lie inside the fp32 rounding of the
    forward pass, so an fp32 implementation and this fp64 one can land on different sides; that unit's gradient then differs
    at O(1) and, through the batch-norm statistics, every row's a little.  Neither is wrong: the gradient is only defined once
    the side is fixed.  Parity tests therefore hand the implementation's own masks in (``relu_masks``: key -> bool array shaped
    like y) and the gradient is taken of  y * mask,  the same piecewise-linear function on the same piece.  Forward values
    change by at most the magnitude of the disputed pre-activations (~1e-7)."""
    m = ctx.relu_masks.get(key)
    if m is None:
        return torch.relu(y)
    m = torch.as_tensor(m).reshape(y.shape)
    ctx.relu_forced += int((m != (y.detach() > 0)).sum())
    return y * m.to(y.dtype)


def _bn(ctx, z, scope):
    """tf.layers.batch_normalization, non-fused (PAM:366-372, BM:680-686): biased variance
    over every leading axis for normalisation and for the moving average."""
    gamma, beta = ctx.p[scope + "/gamma"], ctx.p[scope + "/beta"]
    if ctx.training:
        flat = z.reshape(-1, z.shape[-1])
        mean = flat.mean(0)
        var = ((flat - mean) ** 2).mean(0)
        ctx.new_bn[scope] = (mean.detach(), var.detach())
    else:
        mean = ctx.bn_state[scope + "/moving_mean"].to(ctx.dtype)
        var = ctx.bn_state[scope + "/moving_variance"].to(ctx.dtype)
    y = gamma * ((z - mean) / (var + BN_EPS) ** 0.5) + beta
    if z.dim() == 2:
        # ReLU is not differentiable at 0: an fp32 implementation whose y differs from this one in the last bits can land on
        # the other side, and through the batch statistics that one unit changes the gradient of every row.  Tests use the
        # margin to pick inputs whose gradients are well defined at fp32 resolution.
        ctx.kink_margin = min(ctx.kink_margin, float(y.detach().abs().min()))
    return y


def _mlp(ctx, x, prefix, sizes, out=False, tag=None):
    h = x
    for i in range(len(sizes)):
        z = h @ ctx.p[f"{prefix}/nn_part/w_nn_layer{i}"] + ctx.p[f"{prefix}/nn_part/b_nn_layer{i}"]
        if tag:
            ctx.t[f"{tag}.z{i}"] = z
        bname = "batch_normalization" if i == 0 else f"batch_normalization_{i}"
        h = _act(ctx, _bn(ctx, z, f"{prefix}/nn_part/{bname}"), f"{prefix}/nn_part/{bname}")
    if out:
        h = h @ ctx.p[f"{prefix}/nn_part/w_nn_output"] + ctx.p[f"{prefix}/nn_part/b_nn_output"]
    return h


def gather(p, batch):
    """Every embedding_lookup on the live path as its own tensor, so that the per-lookup
    (un-deduplicated) gradients of BM:297-303 can be observed.  SBM:598-668, PAM:155-182."""
    ih = torch.as_tensor(batch["item_history"]).long()
    ch = torch.as_tensor(batch["item_cate_history"]).long()
    items = torch.as_tensor(batch["items"]).long()
    cates = torch.as_tensor(batch["cates"]).long()
    users = torch.as_tensor(batch["users"]).long()
    B, T = ih.shape
    inv_items = torch.unique(torch.cat([ih.reshape(-1), items]))
    inv_cates = torch.unique(torch.cat([ch.reshape(-1), cates]))
    inv_users = torch.unique(users)
    emb = "sequential/embedding/"
    g = {
        "hist_item": (emb + "item_embedding", ih),
        "hist_cate": (emb + "cate_embedding", ch),
        "tgt_item": (emb + "item_embedding", items),
        "tgt_cate": (emb + "cate_embedding", cates),
        "inv_item": (emb + "item_embedding", inv_items),
        "inv_cate": (emb + "cate_embedding", inv_cates),
        "inv_ulong": (emb + "user_long_embedding", inv_users),
        "inv_ushort": (emb + "user_short_embedding", inv_users),
        "pos": (emb + "position_embedding", torch.arange(T)[None, :].expand(B, T)),
    }
    rows = {k: p[name][idx] for k, (name, idx) in g.items()}
    return g, rows


def bucket_ids(loop_times):
    """Row of the time-aware tables for each token: tf.cast(float -> int32) truncates (PAM:716).  An id outside 0..NB-1 (lisan
    returns NB for a play / duration ratio beyond its last border and for a zero duration) maps to the extra row NB, which
    _timeaware reads as a zero matrix: tf.gather on the GPU returns zeros for an out-of-range index (it raises on the CPU)."""
    lt = torch.as_tensor(loop_times).to(torch.float64)
    ok = (lt > -1) & (lt < NB)                                                   # NaN is out of range too
    return torch.where(ok, torch.where(ok, lt, 0.0).long(), torch.full_like(lt, NB, dtype=torch.long))


def _timeaware(x, table, bucket, proj):
    """x[b,t,:] @ reshape(table[bucket[b,t]], (D, D))  (PAM:714-728); bucket NB (see bucket_ids) selects a zero matrix, so such a
    token's product is 0 and it adds nothing to the table's gradient.  proj="gather" materialises the [B,T,D,D] gather like the
    reference's graph does (the CPU baseline keeps that cost shape); proj="grouped" multiplies the tokens of one bucket by
    that bucket's matrix - the same sums, 1600 x less memory, which is what lets the fp64 check run at B = 4095, T = 200."""
    B, T, _ = x.shape
    table = torch.cat([table, torch.zeros_like(table[:1])], 0)                  # row NB: the GPU gather's zeros
    if proj == "gather":
        return torch.einsum("bti,btij->btj", x, table[bucket].reshape(B, T, D, D))
    xf, bf = x.reshape(-1, D), bucket.reshape(-1)
    order = torch.argsort(bf, stable=True)
    counts = torch.bincount(bf, minlength=NB + 1).tolist()
    W = table.reshape(NB + 1, D, D)
    parts = [seg @ W[k] for k, seg in enumerate(torch.split(xf[order], counts)) if seg.shape[0]]
    inv = torch.empty_like(order)
    inv[order] = torch.arange(order.numel())
    return torch.cat(parts, 0)[inv].reshape(B, T, D)


def forward(p, bn_state, batch, training, rows=None, dtype=torch.float64, relu_masks=None, proj="gather"):
    """Returns ctx with .t = named intermediates (x0, blk{i}.{qin,Q,K,V,y,out}, h, z1, z2, att,
    new_long, logits [B,3] = (logit, valid_logit, xilidu_logit), pred).  relu_masks: see _act."""
    ctx = _Ctx(p, bn_state, training, dtype, relu_masks)
    if rows is None:
        _, rows = gather(p, batch)
    mask = torch.as_tensor(batch["mask"]).long()
    bucket = bucket_ids(batch["item_loop_times_history"])                # tf.cast(float, int32) PAM:716
    B, T = mask.shape
    t = ctx.t

    tgt = torch.cat([rows["tgt_item"], rows["tgt_cate"]], -1)                          # SBM:666-668
    x = torch.cat([rows["hist_item"], rows["hist_cate"], tgt[:, None, :].expand(B, T, E_DIM)], 2)  # PAM:251-256
    x = x + rows["pos"]                                                                # PAM:257
    t["tgt"], t["x0"] = tgt, x
    for b in range(2):                                                                 # PAM:516-543
        pre = f"sequential/pamrec/num_blocks_{b}/"
        qin = _ln(x, p[pre + "ln/Variable"], p[pre + "ln/Variable_1"])
        Q = _timeaware(qin, p[pre + "self_attention/Q_timeaware_embedding"], bucket, proj)   # PAM:714-717,726
        K = _timeaware(x, p[pre + "self_attention/K_timeaware_embedding"], bucket, proj)     # PAM:727 (keys = un-normalised x)
        V = _timeaware(x, p[pre + "self_attention/V_timeaware_embedding"], bucket, proj)
        S = Q @ K.transpose(1, 2) / (D ** 0.5)                                         # PAM:768-772
        S = torch.where(mask[:, None, :] == 0, torch.full_like(S, MASK_NEG), S)        # PAM:776-781
        Pm = torch.softmax(S, -1)                                                      # PAM:793
        y = Pm @ V + qin                                                               # PAM:804-810
        f = _ln(y, p[pre + "ln_1/Variable"], p[pre + "ln_1/Variable_1"])
        hid = _act(ctx, f @ p[pre + "multihead_attention/conv1d/kernel"][0] + p[pre + "multihead_attention/conv1d/bias"], f"blk{b}.ffn")
        out = hid @ p[pre + "multihead_attention/conv1d_1/kernel"][0] + p[pre + "multihead_attention/conv1d_1/bias"] + f  # PAM:565-577
        for k_, v_ in (("qin", qin), ("Q", Q), ("K", K), ("V", V), ("y", y), ("out", out)):
            t[f"blk{b}.{k_}"] = v_
        x = out
    h = x
    t["h"] = h
    # attention pooling PAM:272-282
    sp = "sequential/pamrec/new_long/score_1"
    z1 = h @ p[sp + "/nn_part/w_nn_layer0"] + p[sp + "/nn_part/b_nn_layer0"]
    a1 = _act(ctx, _bn(ctx, z1, sp + "/nn_part/batch_normalization"), sp + "/nn_part/batch_normalization")
    z2 = a1 @ p[sp + "/nn_part/w_nn_layer1"] + p[sp + "/nn_part/b_nn_layer1"]
    s = _act(ctx, _bn(ctx, z2, sp + "/nn_part/batch_normalization_1"), sp + "/nn_part/batch_normalization_1").squeeze(-1)
    att = torch.softmax(torch.where(mask == 1, s, torch.full_like(s, MASK_NEG)), -1)
    new_long = (h * att[..., None]).sum(1)
    t["z1"], t["z2"], t["att"], t["new_long"] = z1, z2.squeeze(-1), att, new_long
    # MMoE PAM:26-50 (gates end in BN+ReLU, not softmax)
    experts = torch.stack([_mlp(ctx, new_long, f"sequential/pamrec/expert_{j}", EXPERT_SIZES, tag=f"expert{j}")
                           for j in range(EXPERT_NUM)], 1)
    g_main = _mlp(ctx, new_long, "sequential/pamrec/gate_main", GATE_SIZES, tag="gate_main")
    g_sub = _mlp(ctx, new_long, "sequential/pamrec/gate_sub", GATE_SIZES, tag="gate_sub")
    main = torch.einsum("bj,bjc->bc", g_main, experts)
    sub = torch.einsum("bj,bjc->bc", g_sub, experts)
    model_output = torch.cat([main, tgt], 1)                                           # PAM:315
    valid_output = torch.cat([sub, tgt], 1)                                            # PAM:316
    t["main"], t["sub"] = main, sub
    logit = _mlp(ctx, model_output, TOWERS[0], TOWER_SIZES, out=True, tag="tower0")    # PAM:215
    valid_logit = _mlp(ctx, valid_output, TOWERS[1], TOWER_SIZES, out=True, tag="tower1")  # PAM:212
    xilidu = _mlp(ctx, model_output, TOWERS[2], TOWER_SIZES, out=True, tag="tower2")   # PAM:71
    t["logits"] = torch.cat([logit, valid_logit, xilidu], 1)
    t["pred"] = torch.sigmoid(logit)                                                   # BM:106
    return ctx


# --------------------------------------------------------------------------- losses
def _sigmoid_xent(logits, labels):
    """tf.nn.sigmoid_cross_entropy_with_logits: max(x,0) - x*z + log1p(exp(-|x|))."""
    return torch.clamp(logits, min=0) - logits * labels + torch.log1p(torch.exp(-logits.abs()))


def approx_ndcg_loss(labels, scores, alpha=10.0):
    """tfr.losses._approx_ndcg_loss(labels, logits, reduction=MEAN) as called at PAM:76.

    Restated from TensorFlow-Ranking 0.3.x (un-vendored, un-pinned dependency of the
    reference: ``import tensorflow_ranking as tfr`` PAM:17):
      losses_impl.ApproxNDCGLoss.compute_unreduced_loss, utils.approx_ranks,
      utils.ndcg, utils.inverse_max_dcg, tf.compat.v1.losses.compute_weighted_loss(MEAN).
    labels, scores: [G, list_size].  PARITY UNPINNED (no golden vector exists).
    """
    label_sum = labels.sum(1, keepdim=True)
    nonzero = (label_sum > 0).to(scores.dtype)                       # per-list weight
    labels = torch.where(label_sum > 0, labels, torch.full_like(labels, 1e-10))
    # approx_ranks: rank_i = 0.5 + sum_j sigmoid(alpha * (s_j - s_i))
    pairs = torch.sigmoid(alpha * (scores[:, None, :] - scores[:, :, None]))
    ranks = pairs.sum(-1) + 0.5
    gains = torch.pow(torch.full_like(labels, 2.0), labels) - 1.0
    dcg = (gains / torch.log1p(ranks)).sum(1, keepdim=True)
    ideal, _ = torch.sort(labels, dim=1, descending=True)
    r = torch.arange(1, labels.shape[1] + 1, dtype=scores.dtype)
    idcg = ((torch.pow(torch.full_like(ideal, 2.0), ideal) - 1.0) / torch.log1p(r)).sum(1, keepdim=True)
    inv = torch.where(idcg > 0, 1.0 / idcg, torch.zeros_like(idcg))
    losses = -(dcg * inv)
    den = nonzero.sum()
    if den.item() == 0:
        return (losses * nonzero).sum() * 0.0
    return (losses * nonzero).sum() / den


def softmax_pos_loss(logits, labels, group):
    """hparams.loss == "softmax" (BM:222-242 for the satisfied head, PAM:97-105 for the play head):
    -group * mean(log(where(labels == 1, softmax(logits reshaped [-1, group]), 1)))."""
    x, y = logits.reshape(-1, group), labels.reshape(-1, group)
    sm = torch.softmax(x, dim=-1)
    pos = torch.where(y == 1, sm, torch.ones_like(sm))
    return -group * torch.log(pos).mean()


def compute_losses(ctx, batch, rows, hp):
    p, dtype = ctx.p, ctx.dtype
    logits = ctx.t["logits"]
    y_sat = torch.as_tensor(batch["labels_satisfied"]).to(dtype).reshape(-1)
    y_play = torch.as_tensor(batch["labels_play"]).to(dtype).reshape(-1)
    plays = torch.as_tensor(batch["plays"]).to(dtype).reshape(-1, GROUP)
    if hp.get("loss", "cross_entropy_loss") == "softmax":
        data_loss = softmax_pos_loss(logits[:, 0], y_sat, int(hp["softmax_group"]))         # BM:222-242
        aux = hp["fuzhu_weight"] * softmax_pos_loss(logits[:, 1], y_play, int(hp["softmax_group"]))   # PAM:97-106
    else:
        data_loss = _sigmoid_xent(logits[:, 0], y_sat).mean()                             # BM:196-205
        aux = hp["fuzhu_weight"] * _sigmoid_xent(logits[:, 1], y_play).mean()             # PAM:82-88,106
    order = hp["discrepancy_loss_weight"] * approx_ndcg_loss(plays, torch.sigmoid(logits[:, 2]).reshape(-1, GROUP))  # PAM:70-79
    reg = torch.zeros((), dtype=dtype)
    for k in ("inv_item", "inv_cate", "inv_ulong", "inv_ushort"):                         # SBM:651,664  PAM:178,182
        reg = reg + hp["embed_l2"] * 0.5 * (rows[k] ** 2).sum()
    spec = hp["_spec"]
    for name, _, _, grp in spec:                                                          # SBM:714-721
        if grp == "layer":
            reg = reg + hp["layer_l2"] * 0.5 * (p[name] ** 2).sum()
    total = data_loss + reg + aux + order                                                 # PAM:67
    return {"loss": total, "data_loss": data_loss, "regular_loss": reg, "auxiliary_data_loss": aux, "order_loss": order}


DEFAULT_HP = dict(learning_rate=1e-3, beta1=0.9, beta2=0.999, epsilon=1e-8, embed_l2=1e-6, layer_l2=1e-6,
                  max_grad_norm=2.0, is_clip_norm=1, fuzhu_weight=0.5, discrepancy_loss_weight=0.1)


# --------------------------------------------------------------------------- train step
class OracleModel:
    """Holds fp32 master weights, BN moving stats and TF-style Adam slots."""

    def __init__(self, n_users, n_items, n_cates, T, hp=None, seed=8, dtype=torch.float64):
        self.dims = (n_users, n_items, n_cates, T)
        self.hp = dict(DEFAULT_HP)
        if hp:
            self.hp.update(hp)
        self.spec, self.bn_spec = self._spec()
        self.hp["_spec"] = self.spec
        self.group_of = {n: g for n, _, _, g in self.spec}
        self.params, self.bn_state = self._init(seed)
        self.dtype = dtype
        self.proj = "gather"             # "grouped": same sums without the [B,T,D,D] gather (see _timeaware)
        self.step = 0
        self.m = {n: torch.zeros_like(t, dtype=dtype) for n, t in self.params.items()}
        self.v = {n: torch.zeros_like(t, dtype=dtype) for n, t in self.params.items()}

    # ---- what a model family defines (the sibling baselines override these four, oracle/siblings_oracle.py)
    def _spec(self):
        return param_spec(*self.dims)

    def _init(self, seed):
        return init_params(*self.dims, seed=seed)

    def _gather(self, p, batch):
        return gather(p, batch)

    def _forward(self, p, batch, training, rows=None, relu_masks=None):
        return forward(p, self.bn_state, batch, training, rows=rows, dtype=self.dtype, relu_masks=relu_masks, proj=self.proj)

    def _losses(self, ctx, batch, rows):
        return compute_losses(ctx, batch, rows, self.hp)

    def cast_params(self, requires_grad):
        out = {}
        for n, t in self.params.items():
            c = t.to(self.dtype).clone()
            if requires_grad and self.group_of[n] in ("layer", "layer_nol2"):
                c.requires_grad_(True)
            out[n] = c
        return out

    def eval_forward(self, batch):
        with torch.no_grad():
            p = self.cast_params(False)
            return self._forward(p, batch, False)

    def train_step(self, batch, apply=True, keep=(), relu_masks=None):
        """One optimisation step (PAM:426-453).  Returns dict with losses, intermediates,
        raw gradients (pre-clip) and the clip scales.  relu_masks: activation pattern to differentiate on (see _act)."""
        hp, dtype = self.hp, self.dtype
        p = self.cast_params(True)
        g_idx, rows = self._gather(p, batch)
        rows = {k: v.detach().clone().requires_grad_(True) for k, v in rows.items()}
        ctx = self._forward(p, batch, True, rows=rows, relu_masks=relu_masks) if relu_masks else self._forward(p, batch, True, rows=rows)
        for k in keep:
            ctx.t[k].retain_grad()
        losses = self._losses(ctx, batch, rows)
        losses["loss"].backward()

        clip = float(hp["max_grad_norm"])

        def clip_scale(sq):                       # tf.clip_by_norm: g * clip / max(norm, clip)
            if not hp["is_clip_norm"]:
                return 1.0
            return clip / max(math.sqrt(sq), clip)

        grads, scales, sqnorms = {}, {}, {}
        # dense variables (time-aware tables included: IndexedSlices + dense L2 term -> dense)
        for n, _, _, grp in self.spec:
            if grp in ("layer", "layer_nol2"):
                g = p[n].grad if p[n].grad is not None else torch.zeros_like(p[n])
                grads[n] = g
                sqnorms[n] = float((g * g).sum())
                scales[n] = clip_scale(sqnorms[n])
        # sparse variables: concat of every lookup's values (un-deduplicated) BM:297-303
        by_var = {}
        for k, (name, idx) in g_idx.items():
            if rows[k].grad is None:
                continue
            by_var.setdefault(name, []).append((idx.reshape(-1), rows[k].grad.reshape(-1, rows[k].shape[-1])))
        for name, parts in by_var.items():
            sq = sum(float((v * v).sum()) for _, v in parts)
            sc = clip_scale(sq)
            sqnorms[name] = sq
            dense = torch.zeros_like(p[name])
            for idx, v in parts:
                dense.index_add_(0, idx, v)
            grads[name] = dense
            scales[name] = sc

        result = {"losses": {k: float(v.detach()) for k, v in losses.items()}, "t": ctx.t, "grads": grads, "scales": scales, "sqnorms": sqnorms,
                  "new_bn": ctx.new_bn, "kink_margin": ctx.kink_margin, "relu_forced": ctx.relu_forced}
        if not apply:
            return result

        # Adam (tf.train.AdamOptimizer, TF 2.4 adam.py): beta powers start at beta -> t = step+1
        self.step += 1
        t = self.step
        # TF holds lr / beta1 / beta2 / epsilon and the beta powers as float32 tensors: round them the same way
        f32 = lambda x: float(np.float32(x))
        b1, b2, eps = f32(hp["beta1"]), f32(hp["beta2"]), f32(hp["epsilon"])
        lr_t = f32(hp["learning_rate"]) * math.sqrt(1 - b2 ** t) / (1 - b1 ** t)
        for n, g in grads.items():
            g = g * scales[n]
            grp = self.group_of[n]
            m, v = self.m[n], self.v[n]
            if grp in ("layer", "layer_nol2"):          # ApplyAdam kernel form
                m += (g - m) * (1 - b1)
                v += (g * g - v) * (1 - b2)
            else:                                       # _apply_sparse_shared: decay ALL rows, scatter_add touched
                m.mul_(b1).add_(g * (1 - b1))
                v.mul_(b2).add_((g * g) * (1 - b2))
            new = p[n].detach() - lr_t * m / (v.sqrt() + eps)
            self.params[n] = new.to(torch.float32)
        for scope, (mean, var) in ctx.new_bn.items():   # assign_moving_average, decay = 1 - momentum
            mm, mv = self.bn_state[scope + "/moving_mean"], self.bn_state[scope + "/moving_variance"]
            mm.sub_((mm - mean.to(torch.float32)) * (1 - BN_MOMENTUM))
            mv.sub_((mv - var.to(torch.float32)) * (1 - BN_MOMENTUM))
        return result
