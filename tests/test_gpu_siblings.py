"""GPU parity of the sibling multi-task baselines (SURVEY.md section 8(f) row N3: MMoEModel_original, PLEModel, ShareBottomModel)
against oracle/siblings_oracle.py, through the C ABI: gather bit-exact, every forward stage, activation gradients, all dense
gradients, merged sparse gradients, clip norms, the four losses, several optimisation steps and inference predictions.
The fp64 oracle differentiates on the engine's ReLU pattern (see tests/relu_masks.py for why)."""
import numpy as np
import pytest
import torch

from oracle import pamrec_oracle as O
from oracle import siblings_oracle as S
from relu_masks import bn_layers, expert_scopes, sibling_mlps

pytestmark = pytest.mark.gpu

EMB = "sequential/embedding/"
CLSR = "sequential/clsr/"
RTOL = 1e-5


FAILS = []          # every stage is checked before the test fails: one GPU run localises every disagreement


def _close(name, got, ref, rtol=RTOL, report=None):
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64).reshape(got.shape)
    scale = max(np.abs(ref).max(), 1e-30)
    err = np.abs(got - ref).max() / scale
    if report is not None:
        report.append((name, err))
    if not np.isfinite(got).all():
        FAILS.append(f"{name}: non-finite values")
    elif not err <= rtol:
        FAILS.append(f"{name}: max err / max|ref| = {err:.3e} > {rtol:.1e}")


def _expect(cond, msg):
    if not cond:
        FAILS.append(str(msg))


def _setup(model, nu, ni, nc, T, B, seed):
    from pamrec_b200.engine import Engine
    om = S.SiblingOracleModel(model, nu, ni, nc, T, seed=seed)
    O.perturb_params(om.params, om.bn_state, seed=seed + 1)
    eng = Engine(nu, ni, nc, T, B, model=model).allocate()
    eng.set_variables({n: t.numpy() for n, t in om.params.items()})
    eng.set_variables({n: t.numpy() for n, t in om.bn_state.items()})
    return om, eng


def _batch(seed, B, T, nu, ni, nc, min_len=1, grouped=True):
    return S.add_satisfied_fields(O.make_batch(seed, B, T, nu, ni, nc, min_len=min_len, grouped=grouped), seed=seed + 1)


def satisfied_edge_rows(batch):
    """Rows 3, 4 and 6 of a batch of at least 7 rows: no satisfied item (read-out = zeros, uniform attention), a single one at the
    last position, every position satisfied."""
    for k in ("satisfied_mask", "satisfied_item_history", "satisfied_cate_history"):
        batch[k][3] = 0
        batch[k][4] = 0
    batch["satisfied_mask"][4, -1] = 1
    batch["satisfied_item_history"][4, -1] = max(int(batch["item_history"][4, 0]), 1)
    batch["satisfied_cate_history"][4, -1] = max(int(batch["item_cate_history"][4, 0]), 1)
    batch["satisfied_mask"][6] = 1
    batch["satisfied_item_history"][6] = np.maximum(batch["item_history"][6], 1)
    batch["satisfied_cate_history"][6] = np.maximum(batch["item_cate_history"][6], 1)
    return batch


def _on(z, stat, gamma, beta):
    xh = (z.astype(np.float32) - stat[:, 0].astype(np.float32)) * stat[:, 1].astype(np.float32)
    return gamma.astype(np.float64) * xh.astype(np.float64) + beta.astype(np.float64) > 0


def sibling_relu_masks(eng, model, B, T):
    """Masks of the last training forward, keyed by BN scope, for every batch norm of the model's MLPs (relu_masks.sibling_mlps)."""
    out = {}
    for zbuf, bn, width, scopes, tokens in bn_layers(sibling_mlps(model, sum(eng.emb_dims[:2]))):
        rows, lead = (B * T, (B, T)) if tokens else (B, (B,))
        z = eng.ws(zbuf, rows).cpu().numpy().reshape(rows, len(scopes) * width)
        st = eng.ws(f"bn.{bn}.stat").cpu().numpy()
        for m, scope in enumerate(scopes):
            sl = slice(m * width, (m + 1) * width)
            g, b = eng.dense(scope + "/gamma").cpu().numpy(), eng.dense(scope + "/beta").cpu().numpy()
            out[scope] = _on(z[:, sl], st[sl], g, b).reshape(lead + (width,))
    return out


def _branches(eng, name, N, width):
    """[2, N, width] view of a branch-major workspace tensor (branch stride = the batch's own token count)."""
    return eng.ws(name).reshape(-1)[:2 * N * width].view(2, N, width).cpu().numpy()


CASES = [
    # model, nu, ni, nc, T, B, min_len
    ("mmoe", 50, 300, 20, 12, 20, 1),
    ("ple", 50, 300, 20, 12, 20, 1),
    ("sharebottom", 50, 300, 20, 12, 20, 1),
    ("mmoe", 400, 5000, 60, 50, 130, 50),          # full-length histories: id 0 only through the satisfied-only padding (no L2 on row 0)
    ("ple", 200, 2000, 40, 100, 35, 1),            # quick-start T
    ("sharebottom", 100, 1000, 30, 200, 10, 1),    # T = 200
    ("mmoe", 50000, 30000, 50, 50, 1025, 1),       # the takatak bench shape
    ("ple", 20000, 100000, 500, 100, 500, 1),      # the quick-start shape
    # the DIN pooling keeps 8 scores per lane (kernels_sibling.cu): T = 33 is the first with a second one, 256 the last; T = 1
    # (shared by all three DIN models)
    ("mmoe", 50, 300, 20, 1, 20, 1),
    ("mmoe", 100, 1000, 30, 33, 20, 1),
    ("mmoe", 60, 2000, 30, 256, 10, 1),
]


@pytest.mark.parametrize("model,nu,ni,nc,T,B,min_len", CASES)
def test_sibling_step_stagewise(model, nu, ni, nc, T, B, min_len):
    from pamrec_b200 import _lib as L
    om, eng = _setup(model, nu, ni, nc, T, B, seed=11)
    batch = _batch(5, B, T, nu, ni, nc, min_len=min_len)
    N = B * T
    FAILS.clear()
    db = eng.upload(batch)
    eng.forward(db, training=True, want_pred=False)
    torch.cuda.synchronize()
    masks = sibling_relu_masks(eng, model, B, T)
    keep = ("x", "logits")
    ref = om.train_step(batch, apply=False, keep=keep, relu_masks=masks)
    n_units = sum(int(np.prod(m.shape)) for m in masks.values())
    print(f"\n[{model},{nu},{ni},{nc},T={T},B={B}] ReLU units {n_units}, on opposite sides in fp32 / fp64: {ref['relu_forced']}")
    # (the attention MLPs see every padded position - identical rows of one sample - so units near a kink come in bunches)
    _expect(ref["relu_forced"] <= max(4, n_units // 40000), "the two forward passes disagree on far more ReLU units than rounding explains")
    t = ref["t"]
    rep = []
    # ---- gather: bit exact
    item_w, cate_w = om.params[EMB + "item_embedding"].numpy(), om.params[EMB + "cate_embedding"].numpy()
    h = _branches(eng, "sib.h", N, 20)
    want = [np.concatenate([item_w[batch["satisfied_item_history"].reshape(-1)], cate_w[batch["satisfied_cate_history"].reshape(-1)]], 1),
            np.concatenate([item_w[batch["item_history"].reshape(-1)], cate_w[batch["item_cate_history"].reshape(-1)]], 1)]
    _expect(np.array_equal(h[0], want[0]) and np.array_equal(h[1], want[1]), "gather is not bit-exact")
    tg = np.concatenate([item_w[batch["items"]], cate_w[batch["cates"]]], 1)
    _expect(np.array_equal(eng.ws("tgt", B).cpu().numpy(), tg), "target gather is not bit-exact")
    # ---- forward stages
    feat = eng.ws("sib.feat", N).cpu().numpy()
    z1, z2 = eng.ws("z1", N).cpu().numpy(), eng.ws("z2", N).cpu().numpy()
    score = eng.ws("sib.score", N).cpu().numpy()
    aw = eng.ws("sib.aw").reshape(-1)[:2 * N].view(2, N).cpu().numpy()
    for r in range(2):
        _close(f"att{r}.feat", feat[:, 80 * r:80 * r + 80], t[f"att{r}.feat"].detach().numpy(), report=rep)
        _close(f"att{r}.z0", z1[:, 80 * r:80 * r + 80], t[f"att{r}.z0"].detach().numpy(), report=rep)
        _close(f"att{r}.z1", z2[:, 40 * r:40 * r + 40], t[f"att{r}.z1"].detach().numpy(), report=rep)
        _close(f"att{r}.score", score[:, r], t[f"att{r}.score"].detach().numpy(), report=rep)
        _close(f"att{r}.w", aw[r], t[f"att{r}.w"].detach().numpy(), report=rep)
    _close("x", eng.ws("x", B).cpu().numpy(), t["x"].detach().numpy(), report=rep)
    ex = expert_scopes(model)
    if ex:
        nE = len(ex)
        _close("ze0", eng.ws("ze0", B).cpu().numpy(), np.concatenate([t[f"expert{j}.z0"].detach().numpy() for j in range(nE)], 1), report=rep)
        _close("ze1", eng.ws("ze1", B).cpu().numpy(), np.concatenate([t[f"expert{j}.z1"].detach().numpy() for j in range(nE)], 1), report=rep)
        _close("zg1", eng.ws("zg1", B).cpu().numpy(), np.concatenate([t[f"gate{k}.z1"].detach().numpy() for k in range(2)], 1), report=rep)
        u = eng.ws("u", B).cpu().numpy()
        _close("main", u[:, :64], t["main"].detach().numpy(), report=rep)
        _close("sub", u[:, 84:148], t["sub"].detach().numpy(), report=rep)
    _close("zt1", eng.ws("zt1", B).cpu().numpy(), np.concatenate([t[f"tower{k}.z1"].detach().numpy() for k in range(2)], 1), report=rep)
    _close("logits", eng.ws("logits", B).cpu().numpy(), t["logits"].detach().numpy(), report=rep)
    # ---- backward
    eng.backward(db)
    torch.cuda.synchronize()
    _close("d_logits", eng.ws("d_logits", B).cpu().numpy(), t["logits"].grad.numpy(), rtol=2e-5, report=rep)
    _close("d_x", eng.ws("d_x", B).cpu().numpy(), t["x"].grad.numpy(), rtol=5e-5, report=rep)
    l2 = om.hp["layer_l2"]
    gmax = max(float(ref["grads"][n].abs().max()) for n in eng.info[L.POOL_DENSE])
    bad = []
    for name, d in eng.info[L.POOL_DENSE].items():
        g = eng.dense(name, "dense_grad").cpu().numpy().astype(np.float64)
        if d["flags"] & L.SEG_L2:
            g = g + l2 * eng.dense(name).cpu().numpy().astype(np.float64)
        gr = ref["grads"][name].numpy().reshape(g.shape)
        err = np.abs(g - gr).max()
        lim = 1e-4 * np.abs(gr).max() + 2e-6 * gmax
        if "/b_nn_layer" in name:
            lim += 1e-5 * gmax       # a bias in front of a batch norm: the exact gradient is 0, both sides hold rounding noise only
        else:
            rep.append(("grad " + name, err / max(np.abs(gr).max(), 1e-30)))
        if not (np.isfinite(g).all() and err <= lim):
            bad.append((name, err, np.abs(gr).max()))
    _expect(not bad, f"dense gradients, gmax={gmax:.3e}: " + "; ".join(f"{n}: err {e:.3e} max|ref| {m:.3e}" for n, e, m in bad))
    # ---- apply: merged sparse gradients, clip norms, losses
    tables0 = {k: eng.pool[k].clone() for k in ("item_w", "cate_w", "ulong_w", "ushort_w")}
    losses = eng.apply_gradients(db).cpu().numpy()
    torch.cuda.synchronize()
    lr = ref["losses"]
    for i, k in enumerate(("loss", "data_loss", "regular_loss", "auxiliary_data_loss")):
        _expect(abs(losses[i] - lr[k]) <= 1e-5 * max(abs(lr[k]), 1e-3), (k, losses[i], lr[k]))
    _expect(losses[4] == 0.0, "order loss slot")
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
        l2row = np.isin(uk, involved).astype(np.float64)[:, None]
        g = acc + el2 * l2row * tables0[tab + "_w"].cpu().numpy()[uk]
        _close(f"sparse grad {tab}", g, gref[uk], rtol=1e-4, report=rep)
        rest = np.ones(gref.shape[0], bool); rest[uk] = False
        _expect(not gref[rest].any(), f"{tab}: reference gradient outside the unique rows")
    if min_len == T:
        _expect(has0[0] == 0 and has0[1] == 0, "this case is meant to exercise the row-0-without-L2 path")
    spn = eng.ws("sp_normsq").cpu().numpy()
    for i, name in enumerate(("item_embedding", "cate_embedding", "user_long_embedding", "user_short_embedding")):
        want_sq = ref["sqnorms"][EMB + name]
        _expect(abs(spn[i] - want_sq) <= 2e-4 * want_sq + 1e-30, ("clip norm", name, spn[i], want_sq))
    segn = eng.ws("seg_normsq").cpu().numpy()
    for s, (name, d) in enumerate(eng.info[L.POOL_DENSE].items()):
        want_sq = ref["sqnorms"][name]
        floor = (1e-5 if "/b_nn_layer" in name else 2e-6) * gmax
        _expect(abs(segn[s] - want_sq) <= 2e-4 * want_sq + d["numel"] * floor ** 2, ("clip norm", name, segn[s], want_sq))
    for tab in ("item", "cate", "ulong", "ushort"):
        w0 = tables0[tab + "_w"].cpu().numpy(); w1 = eng.pool[tab + "_w"].cpu().numpy()
        _expect(np.isfinite(w1).all() and (w0 != w1).any(), f"table {tab} after Adam")
    print("\n".join(f"  {n:80s} {e:.2e}" for n, e in sorted(rep, key=lambda x: -x[1])[:14]))
    print("  forward / activation-gradient stages:")
    print("\n".join(f"  {n:80s} {e:.2e}" for n, e in rep if not n.startswith("grad ")))
    eng.close()
    assert not FAILS, "\n".join(FAILS)


@pytest.mark.parametrize("model", ["mmoe", "ple", "sharebottom", "sasrec"])
def test_sibling_multi_step_and_eval(model):
    """Five optimisation steps (tables, dense variables, BN moving statistics all move), then a scoring pass."""
    nu, ni, nc, T, B = 300, 3000, 50, 50, 100
    om, eng = _setup(model, nu, ni, nc, T, B, seed=3)
    for step in range(5):
        batch = _batch(100 + step, B, T, nu, ni, nc, min_len=(T if step == 2 else 1))
        ref = om.train_step(batch)
        got = eng.train_step(eng.upload(batch)).cpu().numpy()
        for i, k in enumerate(("loss", "data_loss", "regular_loss", "auxiliary_data_loss")):
            if k not in ref["losses"]:
                assert model == "sasrec" and got[i] == 0.0
                continue
            r = ref["losses"][k]
            # per-step parity is the stage-wise test; over several Adam steps the fp32 and fp64 trajectories drift apart (Adam turns
            # rounding noise on near-zero gradients into steps of size lr, and the batch norms of the attention MLPs amplify by
            # 1 / sqrt(eps) = 100 at init): the gap grows with the number of steps taken - observed up to 8e-5 after four - and is
            # bounded at the north_star's "after equal steps" scale of 1e-4 per step
            assert abs(got[i] - r) <= (1e-5 if step == 0 else 1e-4 * step) * max(abs(r), 1e-3), (step, k, got[i], r)
    got_vars = eng.get_variables()
    lr = om.hp["learning_rate"]
    for name in (EMB + "item_embedding", EMB + "cate_embedding", EMB + ("position_embedding" if model == "sasrec" else "user_long_embedding")):
        d = np.abs(got_vars[name] - om.params[name].numpy())
        # Adam moves a weight by ~lr per step whatever the gradient's size, so an entry whose gradient is rounding noise can walk in
        # opposite directions in fp32 and fp64 (2 * lr per step); the bulk of the table must agree far better than that
        assert d.max() <= 2 * lr * 5 * 1.01 and d.mean() <= 0.05 * lr, (name, float(d.max()), float(d.mean()))
    for name, tval in om.bn_state.items():
        # A moving mean tracks the batch mean of h W + b, and b - a bias in front of a batch norm, exact gradient 0 - random-walks by
        # +-lr per step on rounding noise that Adam normalises (DESIGN.md section 2): means to 5 steps of that walk, variances tightly
        tol = 5 * lr * 0.25 if name.endswith("moving_mean") else 2e-4
        assert np.allclose(got_vars[name], tval.numpy(), rtol=2e-4, atol=tol), name
    ev = _batch(999, 77, T, nu, ni, nc, grouped=False)
    pred = eng.forward(eng.upload(ev, training=False), training=False).cpu().numpy()
    want = om.eval_forward(ev).t["pred"].numpy().reshape(-1)
    assert np.abs(pred - want).max() <= 1e-4, float(np.abs(pred - want).max())
    eng.close()


SAS_CASES = [
    # nu, ni, nc, T, B, min_len
    (50, 300, 20, 12, 20, 1),
    (400, 5000, 60, 50, 130, 50),
    (100, 1000, 30, 200, 10, 1),
    (50000, 30000, 50, 50, 1025, 1),
    # a thread of the attention kernels loops over query rows in steps of 128 (kernels_sasrec.cu): T = 129 is the first T where
    # one thread owns two rows
    (50, 300, 20, 1, 20, 1),
    (100, 1000, 30, 128, 15, 1),
    (100, 1000, 30, 129, 10, 1),
]


@pytest.mark.parametrize("nu,ni,nc,T,B,min_len", SAS_CASES)
def test_sasrec_step_stagewise(nu, ni, nc, T, B, min_len):
    """SASRecModel (sasrec.py:16-96): every block tensor, the read-out, the tower, then gradients, clip norms and losses."""
    from pamrec_b200 import _lib as L
    om, eng = _setup("sasrec", nu, ni, nc, T, B, seed=11)
    batch = _batch(5, B, T, nu, ni, nc, min_len=min_len)
    if B >= 10:
        satisfied_edge_rows(batch)
    N = B * T
    FAILS.clear()
    db = eng.upload(batch)
    eng.forward(db, training=True, want_pred=False)
    torch.cuda.synchronize()
    tw = "sequential/logit_fcn/nn_part/batch_normalization"
    masks = {f"blk{k}.ffn": (eng.ws(f"blk{k}.hpre", N).cpu().numpy() > 0).reshape(B, T, 20) for k in range(2)}
    for zbuf, bn, scope in (("zt0", "t0", tw), ("zt1", "t1", tw + "_1")):
        masks[scope] = _on(eng.ws(zbuf, B).cpu().numpy(), eng.ws(f"bn.{bn}.stat").cpu().numpy(), eng.dense(scope + "/gamma").cpu().numpy(),
                           eng.dense(scope + "/beta").cpu().numpy())
    ref = om.train_step(batch, apply=False, keep=("x0", "logits"), relu_masks=masks)
    n_units = sum(int(np.prod(m.shape)) for m in masks.values())
    print(f"\n[sasrec,{nu},{ni},{nc},T={T},B={B}] ReLU units {n_units}, on opposite sides in fp32 / fp64: {ref['relu_forced']}")
    _expect(ref["relu_forced"] <= max(4, n_units // 40000), "the two forward passes disagree on far more ReLU units than rounding explains")
    t = ref["t"]
    rep = []
    _close("x0", eng.ws("x0", N).cpu().numpy(), t["x0"].detach().numpy(), rtol=1e-6, report=rep)
    for k in range(2):
        xq, qkv = eng.ws(f"blk{k}.xq", N).cpu().numpy(), eng.ws(f"blk{k}.qkv", N).cpu().numpy()
        _close(f"blk{k}.qin", xq[:, :20], t[f"blk{k}.qin"].detach().numpy(), report=rep)
        for j, nm in enumerate("QKV"):
            _close(f"blk{k}.{nm}", qkv[:, 20 * j:20 * j + 20], t[f"blk{k}.{nm}"].detach().numpy(), report=rep)
        for nm in ("y", "f", "out"):
            _close(f"blk{k}.{nm}", eng.ws(f"blk{k}.{nm}", N).cpu().numpy(), t[f"blk{k}.{nm}"].detach().numpy(), report=rep)
    u = eng.ws("u", B).cpu().numpy()
    _close("final_state", u[:, :20], t["final_state"].detach().numpy(), report=rep)
    _close("zt1", eng.ws("zt1", B).cpu().numpy(), t["tower0.z1"].detach().numpy(), report=rep)
    _close("logits", eng.ws("logits", B).cpu().numpy(), t["logits"].detach().numpy(), report=rep)
    eng.backward(db)
    torch.cuda.synchronize()
    _close("d_logits", eng.ws("d_logits", B).cpu().numpy(), t["logits"].grad.numpy(), rtol=2e-5, report=rep)
    _close("d_x0", _branches(eng, "sib.dh", N, 20)[0], t["x0"].grad.numpy(), rtol=1e-4, report=rep)
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
    tables0 = {k: eng.pool[k].clone() for k in ("item_w", "cate_w")}
    losses = eng.apply_gradients(db).cpu().numpy()
    torch.cuda.synchronize()
    lr = ref["losses"]
    for i, k in enumerate(("loss", "data_loss", "regular_loss")):
        _expect(abs(losses[i] - lr[k]) <= 1e-5 * max(abs(lr[k]), 1e-3), (k, losses[i], lr[k]))
    _expect(losses[3] == 0.0 and losses[4] == 0.0, "auxiliary / order loss slots")
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
        g = acc + el2 * np.isin(uk, involved).astype(np.float64)[:, None] * tables0[tab + "_w"].cpu().numpy()[uk]
        _close(f"sparse grad {tab}", g, gref[uk], rtol=1e-4, report=rep)
    spn = eng.ws("sp_normsq").cpu().numpy()
    for i, name in ((0, "item_embedding"), (1, "cate_embedding"), (4, "position_embedding")):
        want_sq = ref["sqnorms"][EMB + name]
        _expect(abs(spn[i] - want_sq) <= 2e-4 * want_sq + 1e-30, ("clip norm", name, spn[i], want_sq))
    segn = eng.ws("seg_normsq").cpu().numpy()
    for s_, (name, d) in enumerate(eng.info[L.POOL_DENSE].items()):
        want_sq = ref["sqnorms"][name]
        floor = (1e-5 if "/b_nn_layer" in name else 2e-6) * gmax
        _expect(abs(segn[s_] - want_sq) <= 2e-4 * want_sq + d["numel"] * floor ** 2, ("clip norm", name, segn[s_], want_sq))
    print("  forward / activation-gradient stages:")
    print("\n".join(f"  {n:80s} {e:.2e}" for n, e in rep if not n.startswith("grad ")))
    print("\n".join(f"  {n:80s} {e:.2e}" for n, e in sorted((x for x in rep if x[0].startswith("grad ")), key=lambda x: -x[1])[:8]))
    eng.close()
    assert not FAILS, "\n".join(FAILS)


# ----------------------------------------------------------------------------- the reference's driver flow, from text files
ROOT = __import__("os").path.dirname(__import__("os").path.dirname(__import__("os").path.abspath(__file__)))


@pytest.fixture(scope="module")
def data_root(tmp_path_factory):
    from pamrec_b200 import synth
    root = tmp_path_factory.mktemp("siblings")
    synth.generate(str(root), "wechat", n_users=300, n_items=2000, n_cates=30, mean_len=50, seed=9, eval_per_user=2)
    return str(root)


@pytest.mark.parametrize("cls_name,yaml_name,kind", [("MMoEModel_original", "mmoe.yaml", "mmoe"), ("PLEModel", "ple.yaml", "ple"),
                                                     ("ShareBottomModel", "sharebottom.yaml", "sharebottom"), ("SASRecModel", "sasrec.yaml", "sasrec")])
def test_sibling_fit_checkpoint_eval_match_oracle(data_root, tmp_path, cls_name, yaml_name, kind):
    """fit_step (iterator -> train steps -> run_weighted_eval -> checkpoint) -> latest_checkpoint -> load_model -> scores, then the
    fp64 oracle re-scores the same impressions from the checkpointed variables (example/00_quick_start/sequential.py:435-522)."""
    import os
    import sys
    sys.path.insert(0, os.path.join(ROOT, "compat"))
    import importlib
    from reco_utils.recommender.deeprec.deeprec_utils import prepare_hparams
    from reco_utils.recommender.deeprec.io.sequential_iterator import SequentialIterator
    import tensorflow.compat.v1 as tf                      # compat shim: latest_checkpoint only
    mod = kind
    cls = getattr(importlib.import_module("reco_utils.recommender.deeprec.models.sequential." + mod), cls_name)
    d = os.path.join(data_root, "wechat")
    model_dir = str(tmp_path / "model") + "/"
    hp = prepare_hparams(os.path.join(ROOT, "compat", "reco_utils", "recommender", "deeprec", "config", yaml_name), dataset="wechat",
                         bucket_num=10, add_feature=False, embed_l2=1e-6, layer_l2=1e-6, learning_rate=0.001, epochs=1, EARLY_STOP=5,
                         is_clip_norm=1, batch_size=100, show_step=10 ** 9, MODEL_DIR=model_dir, SUMMARIES_DIR=str(tmp_path / "s") + "/",
                         user_vocab=os.path.join(d, "user_vocab.pkl"), item_vocab=os.path.join(d, "item_vocab.pkl"),
                         cate_vocab=os.path.join(d, "category_vocab.pkl"), train_num_ngs=0, max_seq_length=50, pairwise_metrics=[],
                         weighted_metrics=["wauc", "wmrr", "wndcg@2;4", "whit@2;4"], eval_step=4, write_tfevents=False,
                         noise_train_hist=0, noise_train_listwise=0, noise_only_predict=0)
    model = cls(hp, SequentialIterator, seed=8)
    test = os.path.join(d, "test_data")
    r = model.train(None, next(f for f in model.iterator.load_data_from_file(os.path.join(d, "train_data"), min_seq_length=1, batch_num_ngs=0) if f))
    if kind == "sasrec":
        assert len(r) == 5 and np.isfinite(r[2]) and r[2] > r[3] > 0                                        # BM:362-371: loss, data_loss
    else:
        assert len(r) == 7 and np.isfinite(r[2]) and abs(r[2] - (r[3] + r[4] + r[5])) <= 1e-5 * abs(r[2])  # MM:360-373: no order loss
    assert model.fit_step(os.path.join(d, "train_data"), os.path.join(d, "valid_data"), valid_num_ngs=0, eval_metric="auc") is model
    ckpt = tf.train.latest_checkpoint(model_dir)
    assert ckpt and os.path.exists(ckpt + ".safetensors")
    fresh = cls(hp, SequentialIterator, seed=123)
    fresh.load_model(ckpt)
    res = fresh.run_weighted_eval(test, num_ngs=0)
    for k in ("auc", "logloss", "wauc", "wmrr", "wndcg@2", "whit@4"):
        assert k in res and np.isfinite(res[k]), (k, res)
    var = fresh.engine.get_variables()
    nu, ni, nc, T, _ = fresh.engine.dims
    om = S.SiblingOracleModel(kind, nu, ni, nc, T, seed=1)
    assert set(om.params) | set(om.bn_state) == set(var), "checkpointed variable list = the reference Saver's var-list"
    for n in om.params:
        om.params[n] = torch.as_tensor(var[n], dtype=om.params[n].dtype).reshape(om.params[n].shape)
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


def test_sibling_driver_runs_as_subprocess(data_root, tmp_path):
    """compat/example/00_quick_start/sequential.py --model PLE (the reference's flag names and model names)."""
    import os
    import subprocess
    import sys
    drv = os.path.join(ROOT, "compat", "example", "00_quick_start", "sequential.py")
    cmd = [sys.executable, drv, "--dataset", "wechat", "--data_path", data_root, "--epochs", "1", "--batch_size", "100", "--model", "PLE",
           "--eval_step", "5", "--show_step", "5", "--save_path", str(tmp_path / "ranking"), "--write_prediction_to_file"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600, cwd=os.path.dirname(drv))
    assert r.returncode == 0, r.stdout[-3000:]
    assert "Time cost for training" in r.stdout and "'auc'" in r.stdout and "wauc" in r.stdout, r.stdout[-2000:]
    preds = np.loadtxt(os.path.join(data_root, "wechat", "output.txt"))
    n_test = sum(1 for _ in open(os.path.join(data_root, "wechat", "test_data")))
    assert preds.shape == (n_test,) and np.isfinite(preds).all() and (preds > 0).all() and (preds < 1).all()
