"""oracle/siblings_oracle.py at other embedding widths (test infrastructure, imported by the tests of the reference's widths).

The oracle states the sibling models at config/mmoe.yaml's item / cate / user widths 16 / 4 / 20.  Its forward passes, losses and
update rule read every width from the tensors they are given, with two exceptions: the variable inventories (`param_spec`,
`sasrec_param_spec`) and SASRec's attention scale 1 / sqrt(SAS_D).  This module restates the two inventories at any (item, cate,
user), runs the oracle's SASRec forward pass with SAS_D set to the model width for the duration of the call, and builds the oracle's
two classes on top of those.  With dims = (16, 4, 20) everything here equals the oracle's own results."""
import contextlib

from oracle import pamrec_oracle as O
from oracle import siblings_oracle as S

DEFAULT = (O.I_DIM, O.C_DIM, O.U_DIM)


def param_spec(model, n_users, n_items, n_cates, dims=DEFAULT, expert_num=5, share_expert_num=3, independent_expert_num=2,
               expert_sizes=(100, 64), gate_sizes=(64, 5), tower_sizes=(100, 64)):
    """siblings_oracle.param_spec with the widths of `dims`: a history / target token is item + cate wide."""
    assert model in S.MODELS
    i_dim, c_dim, u_dim = dims
    e_dim = i_dim + c_dim
    emb = "sequential/embedding/"
    P = [(emb + "user_embedding", (n_users, u_dim), "tn", "frozen"),
         (emb + "item_embedding", (n_items, i_dim), "tn", "embed"),
         (emb + "cate_embedding", (n_cates, c_dim), "tn", "embed"),
         (emb + "looptimes_embedding", (10, c_dim), "tn", "frozen"),
         (emb + "user_long_embedding", (n_users, u_dim), "tn", "embed_l2only"),
         (emb + "user_short_embedding", (n_users, u_dim), "tn", "embed_l2only"),
         (emb + "play_lookup", (10, 40), "tn", "frozen")]                               # a literal width, whatever the dims
    BN = []

    def mlp(prefix, in_dim, sizes, out=False):
        s, b = O._mlp_spec(prefix, in_dim, sizes, out=out)
        P.extend(s)
        BN.extend(b)
    for branch in ("long_term", "short_term"):
        pre = f"sequential/clsr/{branch}/attention_fcn"
        P.append((pre + "/attention_mat", (e_dim, e_dim), "tn", "layer"))
        mlp(pre + "/att_fcn", 4 * e_dim, S.ATT_SIZES, out=True)
    x_dim = 3 * e_dim
    if model == "mmoe":
        for j in range(expert_num):
            mlp(f"sequential/clsr/expert_{j}", x_dim, expert_sizes)
        for g in ("gate_main", "gate_sub"):
            mlp(f"sequential/clsr/{g}", x_dim, gate_sizes)
        tower_in = expert_sizes[-1] + e_dim
    elif model == "ple":
        for j in range(share_expert_num):
            mlp(f"sequential/clsr/share_expert_{j}", x_dim, expert_sizes)
        for task in ("main", "sub"):
            for j in range(independent_expert_num):
                mlp(f"sequential/clsr/{task}_expert_{j}", x_dim, expert_sizes)
        for task in ("main", "sub"):
            mlp(f"sequential/clsr/gate_{task}", x_dim, gate_sizes)
        tower_in = expert_sizes[-1] + e_dim
    else:
        tower_in = x_dim
    for tw in ("sequential/valid_logit_fcn", "sequential/logit_fcn"):
        mlp(tw, tower_in, tower_sizes, out=True)
    return P, BN


def sasrec_param_spec(n_users, n_items, n_cates, T, dims=DEFAULT, tower_sizes=(100, 64)):
    """siblings_oracle.sasrec_param_spec with the widths of `dims`: the model width is item + cate."""
    i_dim, c_dim, u_dim = dims
    d = i_dim + c_dim
    emb = "sequential/embedding/"
    P = [(emb + "user_embedding", (n_users, u_dim), "tn", "frozen"),
         (emb + "item_embedding", (n_items, i_dim), "tn", "embed"),
         (emb + "cate_embedding", (n_cates, c_dim), "tn", "embed"),
         (emb + "looptimes_embedding", (10, c_dim), "tn", "frozen"),
         (emb + "position_embedding", (T, d), "tn", "pos")]
    for b in range(2):
        pre = f"sequential/sasrec/num_blocks_{b}/"
        P += [(pre + "ln/Variable", (d,), "zeros", "layer"), (pre + "ln/Variable_1", (d,), "ones", "layer")]
        for name in ("dense", "dense_1", "dense_2"):
            P += [(pre + f"self_attention/{name}/kernel", (d, d), "glorot", "layer"),
                  (pre + f"self_attention/{name}/bias", (d,), "zeros", "layer")]
        P += [(pre + "ln_1/Variable", (d,), "zeros", "layer"), (pre + "ln_1/Variable_1", (d,), "ones", "layer")]
        for name in ("conv1d", "conv1d_1"):
            P += [(pre + f"multihead_attention/{name}/kernel", (1, d, d), "glorot", "layer"),
                  (pre + f"multihead_attention/{name}/bias", (d,), "zeros", "layer")]
    s, BN = O._mlp_spec("sequential/logit_fcn", 2 * d, tower_sizes, out=True)
    return P + s, BN


@contextlib.contextmanager
def _sas_width(d):
    """siblings_oracle.sasrec_forward scales the attention logits by 1 / sqrt(SAS_D), read when it runs"""
    old = S.SAS_D
    S.SAS_D = d
    try:
        yield
    finally:
        S.SAS_D = old


def sasrec_forward(p, bn_state, batch, training, **kw):
    """siblings_oracle.sasrec_forward at the width of the given tables (sasrec.py:281-284: scale 1 / sqrt(model width))."""
    d = p["sequential/embedding/position_embedding"].shape[-1]
    with _sas_width(d):
        return S.sasrec_forward(p, bn_state, batch, training, **kw)


class SiblingOracle(S.SiblingOracle):
    """siblings_oracle.SiblingOracle with the inventory at `dims`."""

    def __init__(self, model, n_users, n_items, n_cates, hp=None, seed=8, dims=DEFAULT, **sizes):
        super().__init__(model, n_users, n_items, n_cates, hp=hp, seed=seed, **sizes)
        self.spec, self.bn_spec = param_spec(model, n_users, n_items, n_cates, dims=dims,
                                             **{k: v for k, v in sizes.items() if k in ("expert_num", "share_expert_num",
                                                                                       "independent_expert_num", "expert_sizes",
                                                                                       "gate_sizes", "tower_sizes")})
        self.params, self.bn_state = S.init_params(self.spec, self.bn_spec, seed=seed)


class SiblingOracleModel(S.SiblingOracleModel):
    """siblings_oracle.SiblingOracleModel (per-lookup sparse gradients, clip, TF Adam, BN moving averages) at `dims`."""

    def __init__(self, model, n_users, n_items, n_cates, T, hp=None, seed=8, dims=DEFAULT, **sizes):
        self.emb_dims = tuple(dims)
        super().__init__(model, n_users, n_items, n_cates, T, hp=hp, seed=seed, **sizes)

    def _spec(self):
        nu, ni, nc, T = self.dims
        if self.model == "sasrec":
            return sasrec_param_spec(nu, ni, nc, T, dims=self.emb_dims, **{k: v for k, v in self.sizes.items() if k == "tower_sizes"})
        return param_spec(self.model, nu, ni, nc, dims=self.emb_dims, **self.sizes)

    def _forward(self, p, batch, training, rows=None, relu_masks=None):
        if self.model == "sasrec":
            return sasrec_forward(p, self.bn_state, batch, training, dtype=self.dtype, rows=rows, relu_masks=relu_masks, **self.sizes)
        return super()._forward(p, batch, training, rows=rows, relu_masks=relu_masks)
