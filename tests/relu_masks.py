"""The ReLU activation pattern of an engine forward pass, read back through the workspace and keyed like the oracle's
``relu_masks`` (oracle/pamrec_oracle.py:_act).

Why: the gradient of a ReLU network is only defined once the side of every kink is fixed.  A step has ~10^6 batch-normalised
pre-activations and a few always lie inside the fp32 rounding of the forward pass; when the fp32 engine and the fp64 oracle land
on different sides of one, that unit's gradient differs at O(1) and - through the batch statistics - every row's a little.
Round 1 detected such batches and retried on other seeds, which cannot work beyond B ~ 200.  Here the oracle differentiates on
the ENGINE's pattern instead, so gradient parity is defined at any batch size.

The head masks are recomputed from the stored pre-activations with the kernels' own fp32 expression
``fmaf(gamma, (z - mean) * invstd, beta) > 0`` (kernels_head.cu:bn_relu; the sign of an fma equals the sign of the exact value,
which float64 reproduces because a product of two float32 is exact in float64).  The point-wise FFN's pattern comes from the
PAMREC_DEBUG_SAVE_FFN_HIDDEN hook (its pre-activation is never stored)."""
from typing import NamedTuple

import numpy as np

P_ = "sequential/pamrec/"
TOWERS = ("sequential/logit_fcn", "sequential/valid_logit_fcn", "xilidu_logit_fcn")
CLSR = "sequential/clsr/"


class Mlp(NamedTuple):
    """One batch-norm MLP of a head (layout.h: MlpOff, bound like api.cu:MlpBind): G members in -> h0 -> h1 (-> 1 when out)."""
    scopes: tuple         # TF scope of each member
    k: int                # input columns per member
    h0: int
    h1: int
    out: bool             # a linear output layer follows the second batch norm
    x: str                # workspace buffer of the input, its row width, first input column of each member
    ldx: int
    x_col: tuple
    z: tuple              # per layer: pre-activations (the output layer's logits), all members side by side
    dz: tuple             # per layer: the gradient buffer of that layer
    dx: str               # gradient of the input (members reading the same columns add up)
    bn: tuple             # batch-norm sets of layers 0 and 1 ("bn.<set>.*")
    tokens: bool          # rows are B * T tokens (else B samples)

    def layers(self):
        return 3 if self.out else 2

    def k_of(self, l):
        return (self.k, self.h0, self.h1)[l]

    def n_of(self, l):
        return (self.h0, self.h1, 1)[l]

    def bn_scope(self, m, l):
        return self.scopes[m] + "/nn_part/batch_normalization" + ("_1" if l else "")


# PAMRec (api.cu:head_mlps): the attention-pooling score, experts and gates on new_long, towers on main | target, sub | target, main | target
HEAD_MLPS = {
    "score": Mlp((P_ + "new_long/score_1",), 40, 20, 1, False, "blk1.out", 40, (0,), ("z1", "z2"), ("d_a1", "d_z2"), "g_a",
                 ("s0", "s1"), True),
    "expert": Mlp(tuple(f"{P_}expert_{j}" for j in range(5)), 40, 100, 64, False, "new_long", 40, (0,) * 5, ("ze0", "ze1"),
                  ("d_e0", "d_e1"), "d_new_long", ("e0", "e1"), False),
    "gate": Mlp((P_ + "gate_main", P_ + "gate_sub"), 40, 64, 5, False, "new_long", 40, (0, 0), ("zg0", "zg1"), ("d_g0", "d_g1"),
                "d_new_long", ("g0", "g1"), False),
    "tower": Mlp(TOWERS, 84, 100, 64, True, "u", 168, (0, 84, 0), ("zt0", "zt1", "logits"), ("d_t0", "d_t1", "d_logits"), "d_u",
                 ("t0", "t1"), False),
}


def expert_scopes(model):
    if model == "mmoe":
        return [f"{CLSR}expert_{j}" for j in range(5)]
    if model == "ple":
        return [f"{CLSR}share_expert_{j}" for j in range(3)] + [f"{CLSR}main_expert_{j}" for j in range(2)] + [f"{CLSR}sub_expert_{j}" for j in range(2)]
    return []


def sibling_mlps(model, E):
    """MMoE / PLE / share-bottom at token width E = item + cate (api_sibling.inl:sib_mlps): att_fcn of both DIN branches on their
    feature rows, experts and gates on x = long | short | target, the towers on main | target, sub | target (share-bottom: x, x)."""
    towers = ("sequential/logit_fcn", "sequential/valid_logit_fcn")
    att = tuple(f"{CLSR}{b}/attention_fcn/att_fcn" for b in ("long_term", "short_term"))
    out = {"att": Mlp(att, 4 * E, 80, 40, True, "sib.feat", 8 * E, (0, 4 * E), ("z1", "z2", "sib.score"),
                      ("sib.d_a0", "sib.d_a1", "sib.d_score"), "sib.d_feat", ("s0", "s1"), True)}
    ex = tuple(expert_scopes(model))
    if ex:
        out["expert"] = Mlp(ex, 3 * E, 100, 64, False, "x", 3 * E, (0,) * len(ex), ("ze0", "ze1"), ("d_e0", "d_e1"), "d_x", ("e0", "e1"), False)
        out["gate"] = Mlp((CLSR + "gate_main", CLSR + "gate_sub"), 3 * E, 64, 5, False, "x", 3 * E, (0, 0), ("zg0", "zg1"), ("d_g0", "d_g1"),
                          "d_x", ("g0", "g1"), False)
        ti = 64 + E
        out["tower"] = Mlp(towers, ti, 100, 64, True, "u", 2 * ti, (0, ti), ("zt0", "zt1", "logits"), ("d_t0", "d_t1", "d_logits"), "d_u",
                           ("t0", "t1"), False)
    else:
        out["tower"] = Mlp(towers, 3 * E, 100, 64, True, "x", 3 * E, (0, 0), ("zt0", "zt1", "logits"), ("d_t0", "d_t1", "d_logits"), "d_x",
                           ("t0", "t1"), False)
    return out


def sas_mlps(E):
    """SASRec's tower on final state | target (api_sibling.inl:sas_tower)."""
    return {"tower": Mlp(("sequential/logit_fcn",), 2 * E, 100, 64, True, "u", 2 * E, (0,), ("zt0", "zt1", "logits"),
                         ("d_t0", "d_t1", "d_logits"), "d_u", ("t0", "t1"), False)}


def bn_layers(mlps):
    """(pre-activation buffer, BN set, columns per member, member BN scopes, rows are tokens) of every batch norm of `mlps`."""
    return [(m.z[l], m.bn[l], m.n_of(l), [m.bn_scope(i, l) for i in range(len(m.scopes))], m.tokens)
            for m in mlps.values() for l in (0, 1)]


# engine pre-activation buffer, BN set, columns per member, member scopes (oracle key = scope)
HEAD_BN = [b[:4] for b in bn_layers(HEAD_MLPS)]


def _on(z, stat, gamma, beta):
    xh = (z.astype(np.float32) - stat[:, 0].astype(np.float32)) * stat[:, 1].astype(np.float32)      # two fp32 roundings, as on the device
    return gamma.astype(np.float64) * xh.astype(np.float64) + beta.astype(np.float64) > 0


def engine_relu_masks(eng, rows, ffn=True):
    """Masks of the last ``eng.forward(db, training=True)`` over its first `rows` rows: key -> bool array.
    ffn=True needs ``eng.set_debug(DEBUG_SAVE_FFN_HIDDEN)`` before that forward call."""
    out = {}
    if rows == 0:
        return out
    for zbuf, bn, width, scopes in HEAD_BN:
        z = eng.ws(zbuf, rows).cpu().numpy()
        st = eng.ws(f"bn.{bn}.stat").cpu().numpy()
        lead = z.shape[:-1] if zbuf != "z2" else z.shape
        z = z.reshape(-1, len(scopes) * width)
        for m, scope in enumerate(scopes):
            sl = slice(m * width, (m + 1) * width)
            g, b = eng.dense(scope + "/gamma").cpu().numpy(), eng.dense(scope + "/beta").cpu().numpy()
            out[scope] = _on(z[:, sl], st[sl], g, b).reshape(tuple(lead) + (width,))
    if ffn:
        out["blk0.ffn"] = eng.ws("d_Q", rows).cpu().numpy() > 0
        out["blk1.ffn"] = eng.ws("d_K", rows).cpu().numpy() > 0
    return out


def gather_masks(local, rows_of_rank, n_global, dist, device):
    """All ranks' masks assembled into global-batch order.  local: this rank's masks (may be {} for an empty share);
    rows_of_rank: global row indices of this rank's rows; every rank must call with the same keys known: the key list and the
    trailing shapes are taken from rank-independent metadata (HEAD_BN + the FFN keys)."""
    import torch
    out = {}
    T = None
    for k, v in local.items():
        if k.endswith(".ffn"):
            T = v.shape[1]
    t_box = torch.tensor([T or 0], device=device)
    dist.all_reduce(t_box, op=dist.ReduceOp.MAX)
    T = int(t_box.item())
    keys = [(scope, (T, width) if zbuf in ("z1", "z2") else (width,)) for zbuf, _, width, scopes in HEAD_BN for scope in scopes]
    keys += [("blk0.ffn", (T, 40)), ("blk1.ffn", (T, 40))]
    for k, tail in keys:
        full = torch.zeros((n_global,) + tail, dtype=torch.int32, device=device)
        if len(rows_of_rank):
            full[torch.as_tensor(np.asarray(rows_of_rank), device=device)] = torch.as_tensor(local[k].reshape((len(rows_of_rank),) + tail).astype(np.int32), device=device)
        dist.all_reduce(full)
        out[k] = full.cpu().numpy() > 0
    return out
