"""GPU parity: every stage of the CUDA step, called through the C ABI, against the fp64 oracle on the
same injected weights and the same seeded batch.  Tolerance from BASELINE.json north_star:
1e-5 relative for fp32 logits and loss (tensors are compared relative to their max magnitude)."""
import math

import numpy as np
import pytest
import torch

from oracle import pamrec_oracle as O

pytestmark = pytest.mark.gpu

RTOL = 1e-5


def _close(name, got, ref, rtol=RTOL, report=None):
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64).reshape(got.shape)
    scale = max(np.abs(ref).max(), 1e-30)
    err = np.abs(got - ref).max() / scale
    if report is not None:
        report.append((name, err))
    assert np.isfinite(got).all(), f"{name}: non-finite values"
    assert err <= rtol, f"{name}: max err / max|ref| = {err:.3e} > {rtol:.1e}"


def _setup(nu, ni, nc, T, B, seed, hp=None, sparse_adam="dense_exact", max_batch=None):
    """Oracle and engine on the same weights; the engine holds max_batch rows (default B), so batches of B < max_batch run
    like the file-driven loop's last batch and every data-parallel rank's share."""
    from pamrec_b200.engine import Engine
    om = O.OracleModel(nu, ni, nc, T, hp=hp, seed=seed)
    O.perturb_params(om.params, om.bn_state, seed=seed + 1)
    eng = Engine(nu, ni, nc, T, max_batch or B, hp=hp, sparse_adam=sparse_adam).allocate()
    eng.set_variables({n: t.numpy() for n, t in om.params.items()})
    eng.set_variables({n: t.numpy() for n, t in om.bn_state.items()})
    return om, eng


CASES = [
    # nu, ni, nc, T, B
    (50, 300, 20, 12, 20),
    (400, 5000, 60, 50, 130),     # B*T not a multiple of the 128-token tile; T=50 like cfg-B
    (200, 2000, 40, 100, 35),     # quick-start T
    (100, 1000, 30, 200, 10),     # long history (cfg-4 T)
    # the BASELINE.json shapes themselves (bench.py WORKLOADS): multi-wave grids, k_pos_grad grid.y > 1, > 64 K-row dense
    # tiles, the T = 200 shared-memory footprints at full occupancy
    (50000, 30000, 50, 50, 1025),      # configs[1] takatak_b1025_t50
    (20000, 100000, 500, 100, 500),    # configs[0] quick start, wechat_b500_t100
    (50000, 30000, 50, 200, 4095),     # configs[3] long_b4095_t200 (fp64 oracle: ~40 s, 16 GB on 8 host cores)
]


def _case_id(c):
    return "-".join(map(str, c))


# The sequence lengths where the kernels' code paths change: T = 1 (one key, one position row), the last T of the MMA attention
# (128) and the first of the FFMA one (129, five warps with one query row in the last), the largest T (256).  Two of them run with
# fewer rows than the engine holds (nu, ni, nc, T, B, max_batch).
EDGE_CASES = [
    (50, 300, 20, 1, 20, None),
    (100, 1000, 30, 128, 15, 40),
    (100, 1000, 30, 129, 10, None),
    (60, 2000, 30, 256, 10, 25),
]


def _edge_id(c):
    return _case_id(c[:5]) + (f"-cap{c[5]}" if c[5] else "")


# the default head at every shape; the stand-alone head (PAMREC_HEAD_LEGACY=1, kernels_head.cu: the head beyond 8 ranks and
# without peer mailboxes) at the four small ones and the edge cases
STAGEWISE = ([pytest.param(*c, None, False, id=_case_id(c)) for c in CASES] +
             [pytest.param(*c, None, True, id=_case_id(c) + "-legacy_head") for c in CASES[:4]] +
             [pytest.param(*c, False, id=_edge_id(c)) for c in EDGE_CASES] +
             [pytest.param(*c, True, id=_edge_id(c) + "-legacy_head") for c in EDGE_CASES])


@pytest.mark.parametrize("nu,ni,nc,T,B,max_batch,legacy_head", STAGEWISE)
def test_train_step_stagewise(nu, ni, nc, T, B, max_batch, legacy_head, monkeypatch):
    if legacy_head:
        monkeypatch.setenv("PAMREC_HEAD_LEGACY", "1")
    om, eng = _setup(nu, ni, nc, T, B, seed=11, max_batch=max_batch)
    _check_step(om, eng, O.make_batch(5, B, T, nu, ni, nc))


def _check_step(om, eng, batch):
    """One training step of the engine against the oracle stage by stage: gather, every forward stage of the encoder and the
    head, activation and parameter gradients, sparse gradients, clip norms, losses and the optimiser.  Closes the engine."""
    from pamrec_b200 import _lib as L
    from relu_masks import engine_relu_masks
    nu, ni, nc, T = om.dims
    B = len(batch["items"])
    om.proj = "grouped"                     # same sums as the reference's [B,T,40,40] gather without materialising it
    keep = ("x0", "new_long", "blk0.out", "blk1.out", "logits")
    db = eng.upload(batch)
    # The oracle differentiates on the ENGINE's ReLU pattern (tests/relu_masks.py): gradient parity is then defined at any batch
    # size instead of only where no pre-activation happens to fall inside fp32 rounding of a kink.
    eng.set_debug(L.DEBUG_SAVE_FFN_HIDDEN)
    eng.forward(db, training=True, want_pred=False)
    masks = engine_relu_masks(eng, B)
    eng.set_debug(0)
    ref = om.train_step(batch, apply=False, keep=keep, relu_masks=masks)
    n_units = sum(int(np.prod(m.shape)) for m in masks.values())
    print(f"\n[{nu},{ni},{nc},T={T},B={B}] ReLU units {n_units}, on opposite sides in fp32 / fp64: {ref['relu_forced']}")
    assert ref["relu_forced"] <= max(4, n_units // 100000), "the two forward passes disagree on far more units than rounding explains"
    t = ref["t"]
    rep = []
    # ---- gather alone (bit-exact: pure loads + one add)
    x0 = eng.gather(db).cpu().numpy()
    x0_ref32 = (torch.cat([om.params[O_EMB + "item_embedding"][torch.as_tensor(batch["item_history"]).long()],
                           om.params[O_EMB + "cate_embedding"][torch.as_tensor(batch["item_cate_history"]).long()],
                           torch.cat([om.params[O_EMB + "item_embedding"][torch.as_tensor(batch["items"]).long()],
                                      om.params[O_EMB + "cate_embedding"][torch.as_tensor(batch["cates"]).long()]], -1)[:, None, :].expand(B, T, 20)], 2)
                + om.params[O_EMB + "position_embedding"][None]).numpy()
    assert np.array_equal(x0, x0_ref32), "gather is not bit-exact"
    # ---- forward
    eng.forward(db, training=True, want_pred=False)
    torch.cuda.synchronize()
    for k in range(2):
        for nm in ("qin", "Q", "K", "V", "y", "out"):
            _close(f"blk{k}.{nm}", eng.ws(f"blk{k}.{nm}", B).cpu().numpy(), t[f"blk{k}.{nm}"].detach().numpy(), report=rep)
    _close("z1", eng.ws("z1", B).cpu().numpy(), t["z1"].detach().numpy(), report=rep)
    _close("z2", eng.ws("z2", B).cpu().numpy(), t["z2"].detach().numpy(), report=rep)
    _close("new_long", eng.ws("new_long", B).cpu().numpy(), t["new_long"].detach().numpy(), report=rep)
    ze0 = np.concatenate([t[f"expert{j}.z0"].detach().numpy() for j in range(5)], 1)
    ze1 = np.concatenate([t[f"expert{j}.z1"].detach().numpy() for j in range(5)], 1)
    _close("ze0", eng.ws("ze0", B).cpu().numpy(), ze0, report=rep)
    _close("ze1", eng.ws("ze1", B).cpu().numpy(), ze1, report=rep)
    zg1 = np.concatenate([t["gate_main.z1"].detach().numpy(), t["gate_sub.z1"].detach().numpy()], 1)
    _close("zg1", eng.ws("zg1", B).cpu().numpy(), zg1, report=rep)
    u = eng.ws("u", B).cpu().numpy()
    _close("main", u[:, :64], t["main"].detach().numpy(), report=rep)
    _close("sub", u[:, 84:148], t["sub"].detach().numpy(), report=rep)
    zt1 = np.concatenate([t[f"tower{g}.z1"].detach().numpy() for g in range(3)], 1)
    _close("zt1", eng.ws("zt1", B).cpu().numpy(), zt1, report=rep)
    _close("logits", eng.ws("logits", B).cpu().numpy(), t["logits"].detach().numpy(), report=rep)
    # ---- backward
    P0 = eng.pool["dense_param"].clone()
    eng.backward(db)
    torch.cuda.synchronize()
    _close("d_logits", eng.ws("d_logits", B).cpu().numpy(), t["logits"].grad.numpy(), rtol=2e-5, report=rep)
    _close("d_new_long", eng.ws("d_new_long", B).cpu().numpy(), t["new_long"].grad.numpy(), rtol=5e-5, report=rep)
    _close("d_x0", eng.ws("g_a", B).cpu().numpy(), t["x0"].grad.numpy(), rtol=1e-4, report=rep)
    l2 = om.hp["layer_l2"]
    # Parameter gradients are sums over B*T tokens that can cancel almost completely (e.g. a bias in front of a
    # mean-removing BN): the fp32 rounding noise of such a sum scales with the summands, not with the result, so
    # the absolute floor is tied to the largest gradient entry of the whole model.
    gmax = max(float(ref["grads"][n].abs().max()) for n in eng.info[L.POOL_DENSE])
    bad = []
    for name, d in eng.info[L.POOL_DENSE].items():
        g = eng.dense(name, "dense_grad").cpu().numpy().astype(np.float64)
        if d["flags"] & L.SEG_L2:
            g = g + l2 * eng.dense(name).cpu().numpy().astype(np.float64)
        gr = ref["grads"][name].numpy().reshape(g.shape)
        err = np.abs(g - gr).max()
        lim = 1e-4 * np.abs(gr).max() + 2e-6 * gmax
        rep.append(("grad " + name, err / max(np.abs(gr).max(), 1e-30)))
        if not (np.isfinite(g).all() and err <= lim):
            bad.append((name, err, np.abs(gr).max()))
    assert not bad, f"gmax={gmax:.3e} " + "; ".join(f"{n}: err {e:.3e} max|ref| {m:.3e}" for n, e, m in bad)
    # ---- apply: sparse gradients, clip norms, losses
    tables0 = {k: eng.pool[k].clone() for k in ("item_w", "cate_w", "ulong_w", "ushort_w")}
    M0, V0 = eng.pool["dense_m"].clone(), eng.pool["dense_v"].clone()
    G0 = eng.pool["dense_grad"].clone()
    losses = eng.apply_gradients(db).cpu().numpy()
    torch.cuda.synchronize()
    lr = ref["losses"]
    for i, k in enumerate(("loss", "data_loss", "regular_loss", "auxiliary_data_loss", "order_loss")):
        assert abs(losses[i] - lr[k]) <= 1e-5 * max(abs(lr[k]), 1e-3), (k, losses[i], lr[k])
    nun = eng.ws("sp.nuniq").cpu().numpy()
    el2 = om.hp["embed_l2"]
    for tab, idx, name in (("item", 0, O_EMB + "item_embedding"), ("cate", 1, O_EMB + "cate_embedding")):
        n = int(nun[idx])
        uk = eng.ws(f"sp.{tab}.ukeys").cpu().numpy()[:n]
        acc = eng.ws(f"sp.{tab}.accum").cpu().numpy()[:n].astype(np.float64)
        gref = ref["grads"][name].numpy()
        touched = np.unique(np.concatenate([batch["item_history" if tab == "item" else "item_cate_history"].reshape(-1),
                                            batch["items" if tab == "item" else "cates"]]))
        assert np.array_equal(uk, touched), "unique ids differ"        # sortedness + uniqueness, bit exact
        g = acc + el2 * tables0[tab + "_w"].cpu().numpy()[uk]
        _close(f"sparse grad {tab}", g, gref[uk], rtol=1e-4, report=rep)
        mask = np.ones(gref.shape[0], bool); mask[uk] = False
        assert not gref[mask].any()
    spn = eng.ws("sp_normsq").cpu().numpy()
    for i, name in enumerate(("item_embedding", "cate_embedding", "user_long_embedding", "user_short_embedding", "position_embedding")):
        want = ref["sqnorms"][O_EMB + name]
        assert abs(spn[i] - want) <= 2e-4 * want + 1e-30, (name, spn[i], want)
    segn = eng.ws("seg_normsq").cpu().numpy()
    for s, (name, d) in enumerate(eng.info[L.POOL_DENSE].items()):
        want = ref["sqnorms"][name]
        # the gradient bound above, squared: |g + e|^2 - |g|^2 <= 2 |g| |e| + |e|^2 with |e| <= 1e-4 |g| + sqrt(numel) 2e-6 gmax
        floor = math.sqrt(d["numel"]) * 2e-6 * gmax
        assert abs(segn[s] - want) <= 2e-4 * want + 2 * math.sqrt(want) * floor + floor ** 2, (name, segn[s], want)
    # ---- optimiser kernels against the TF formulas applied to the engine's own gradients
    hp = om.hp
    b1, b2, eps = hp["beta1"], hp["beta2"], hp["epsilon"]
    f32 = lambda x: float(np.float32(x))
    lr_t = np.float32(f32(hp["learning_rate"]) * math.sqrt(1 - f32(b2)) / (1 - f32(b1)))
    for s, (name, d) in enumerate(eng.info[L.POOL_DENSE].items()):
        o, n = d["offset"], d["numel"]
        p0 = P0[o:o + n].cpu().numpy(); g = G0[o:o + n].cpu().numpy()
        if d["flags"] & L.SEG_L2:
            g = g + np.float32(l2) * p0
        norm = np.float32(math.sqrt(segn[s]))
        g = g * np.float32(2.0) / max(norm, np.float32(2.0))
        m = (M0[o:o + n].cpu().numpy() + (g - M0[o:o + n].cpu().numpy()) * (np.float32(1) - np.float32(b1))).astype(np.float32)
        v = (V0[o:o + n].cpu().numpy() + (g * g - V0[o:o + n].cpu().numpy()) * (np.float32(1) - np.float32(b2))).astype(np.float32)
        p = p0 - lr_t * m / (np.sqrt(v) + np.float32(eps))
        got = eng.dense(name).cpu().numpy().reshape(-1)
        assert np.allclose(got, p, rtol=1e-6, atol=1e-9), name
    # untouched table rows still decay/move (dense_exact); with zero slots they must stay bit-identical
    for tab in ("item", "cate", "ulong", "ushort"):
        w0 = tables0[tab + "_w"].cpu().numpy(); w1 = eng.pool[tab + "_w"].cpu().numpy()
        assert np.isfinite(w1).all()
        assert (w0 != w1).any()
    print(f"\n[{nu},{ni},{nc},T={T},B={B}] worst relative errors:")
    print("\n".join(f"  {n:70s} {e:.2e}" for n, e in sorted(rep, key=lambda x: -x[1])[:10]))
    print("  forward / activation-gradient stages:")
    print("\n".join(f"  {n:70s} {e:.2e}" for n, e in sorted((x for x in rep if not x[0].startswith("grad ")), key=lambda x: -x[1])[:8]))
    eng.close()


O_EMB = "sequential/embedding/"


def test_multi_step_losses_and_eval():
    """Five optimisation steps then a scoring pass: losses and predictions track the fp64 oracle."""
    nu, ni, nc, T, B = 300, 3000, 50, 50, 100
    om, eng = _setup(nu, ni, nc, T, B, seed=3)
    for step in range(5):
        batch = O.make_batch(100 + step, B, T, nu, ni, nc)
        ref = om.train_step(batch)
        got = eng.train_step(eng.upload(batch)).cpu().numpy()
        for i, k in enumerate(("loss", "data_loss", "regular_loss", "auxiliary_data_loss", "order_loss")):
            r = ref["losses"][k]
            assert abs(got[i] - r) <= 5e-5 * max(abs(r), 1e-3), (step, k, got[i], r)   # trajectories drift: per-step parity is the stagewise test
    ev = O.make_batch(999, 77, T, nu, ni, nc, grouped=False)
    pred = eng.forward(eng.upload(ev, training=False), training=False).cpu().numpy()
    want = om.eval_forward(ev).t["pred"].numpy().reshape(-1)
    assert np.abs(pred - want).max() <= 1e-4
    # A bias in front of a BN layer has a mathematically zero data gradient, so Adam moves it along fp32 rounding
    # noise; moving_mean tracks that bias (and cancels it again at inference), hence the looser absolute floor.
    for name in eng.info[1]:
        got = eng.bn(name).cpu().numpy()
        atol = 2e-4 if name.endswith("moving_mean") else 1e-6
        assert np.allclose(got, om.bn_state[name].numpy(), rtol=1e-4, atol=atol), name
    eng.close()


@pytest.mark.parametrize("group", [5, 1, 2])
def test_softmax_loss_branch(group):
    """hparams.loss == "softmax" (BM:222-242, PAM:97-105) with groups of train_num_ngs + 1 rows: the two softmax terms, their
    gradient at the logits, every dense gradient and three steps of losses against the oracle."""
    nu, ni, nc, T, B = 120, 900, 25, 30, 40
    hp = dict(loss="softmax", softmax_group=group)
    om, eng = _setup(nu, ni, nc, T, B, seed=21, hp=hp)
    batch = O.make_batch(9, B, T, nu, ni, nc)
    if group == 5:                                                   # the in-batch sampler's layout: one positive, four negatives
        for k in ("labels_satisfied", "labels_play"):
            batch[k] = np.tile(np.asarray([1, 0, 0, 0, 0], np.float32), B // 5).reshape(batch[k].shape)
    ref = om.train_step(batch, apply=False, keep=("logits",))
    db = eng.upload(batch)
    eng.forward(db, training=True, want_pred=False)
    eng.backward(db)
    torch.cuda.synchronize()
    _close("d_logits", eng.ws("d_logits", B).cpu().numpy(), ref["t"]["logits"].grad.numpy(), rtol=2e-5)
    from pamrec_b200 import _lib as L
    gmax = max(float(ref["grads"][n].abs().max()) for n in eng.info[L.POOL_DENSE])
    for name, d in eng.info[L.POOL_DENSE].items():
        g = eng.dense(name, "dense_grad").cpu().numpy().astype(np.float64)
        if d["flags"] & L.SEG_L2:
            g = g + om.hp["layer_l2"] * eng.dense(name).cpu().numpy().astype(np.float64)
        gr = ref["grads"][name].numpy().reshape(g.shape)
        assert np.abs(g - gr).max() <= 1e-4 * np.abs(gr).max() + 2e-6 * gmax, name
    eng2 = _setup(nu, ni, nc, T, B, seed=21, hp=hp)[1]
    for step in range(3):
        b = O.make_batch(30 + step, B, T, nu, ni, nc)
        want = om.train_step(b)["losses"]
        got = eng2.train_step(eng2.upload(b)).cpu().numpy()
        for i, k in enumerate(("loss", "data_loss", "regular_loss", "auxiliary_data_loss", "order_loss")):
            assert abs(got[i] - want[k]) <= 1e-4 * max(abs(want[k]), 1e-3), (step, k, got[i], want[k])
    # a batch that is not a multiple of the group is refused like the reference's reshape would
    if group == 2:
        from pamrec_b200.engine import PamrecError
        odd = O.make_batch(1, 15, T, nu, ni, nc)
        with pytest.raises(PamrecError, match="softmax group"):
            eng2.train_step(eng2.upload(odd))
    eng.close(); eng2.close()


def test_lazy_mode_touches_only_looked_up_rows():
    nu, ni, nc, T, B = 100, 4000, 30, 20, 25
    om, eng = _setup(nu, ni, nc, T, B, seed=5, sparse_adam="lazy")
    batch = O.make_batch(1, B, T, nu, ni, nc)
    w0 = eng.pool["item_w"].clone()
    eng.train_step(eng.upload(batch))
    torch.cuda.synchronize()
    changed = (eng.pool["item_w"] != w0).any(1).cpu().numpy()
    touched = np.zeros(ni, bool)
    touched[np.unique(np.concatenate([batch["item_history"].reshape(-1), batch["items"]]))] = True
    assert np.array_equal(changed, touched)
    eng.close()


@pytest.mark.parametrize("shape", [(100, 4000, 30, 20, 25), (300, 900, 7, 50, 400)])
def test_lazy_fused_adam_equals_dense_exact_on_the_first_step(shape):
    """LAZY applies Adam inside the run walk (kernels_sparse2.cu: complete runs directly, runs that cross a warp block through the
    compact accumulator + k_sp2_lazy_finish).  From zero Adam slots one step of DENSE_EXACT leaves untouched rows alone, so after
    the first step both modes must agree on every row of every table and slot (the second shape has few items and long histories:
    hot rows whose runs span many warp blocks, and 7 categories with runs of thousands of positions)."""
    nu, ni, nc, T, B = shape
    om, lazy = _setup(nu, ni, nc, T, B, seed=5, sparse_adam="lazy")
    om2, exact = _setup(nu, ni, nc, T, B, seed=5, sparse_adam="dense_exact")
    batch = O.make_batch(1, B, T, nu, ni, nc)
    la = lazy.train_step(lazy.upload(batch)).cpu().numpy()
    ex = exact.train_step(exact.upload(batch)).cpu().numpy()
    assert np.allclose(la, ex, rtol=1e-6, atol=1e-8), (la, ex)
    for tab in ("item", "cate", "ulong", "ushort"):
        for sfx in ("w", "m", "v"):
            a, b = lazy.pool[f"{tab}_{sfx}"].cpu().numpy(), exact.pool[f"{tab}_{sfx}"].cpu().numpy()
            # summation order of a run that crosses warp blocks is not fixed (atomics): agreement to fp32 rounding of the sum
            assert np.allclose(a, b, rtol=2e-5, atol=1e-9), (tab, sfx, float(np.abs(a - b).max()))
    # second step: rows looked up in both steps keep agreeing only where the first step touched them too; check the lazy rule
    batch2 = O.make_batch(2, B, T, nu, ni, nc)
    m0 = lazy.pool["item_m"].clone()
    lazy.train_step(lazy.upload(batch2))
    torch.cuda.synchronize()
    touched = np.zeros(ni, bool)
    touched[np.unique(np.concatenate([batch2["item_history"].reshape(-1), batch2["items"]]))] = True
    same = (lazy.pool["item_m"] == m0).all(1).cpu().numpy()
    assert same[~touched].all(), "LAZY moved the first moment of a row that was not looked up"
    lazy.close(); exact.close()


def test_error_paths():
    from pamrec_b200.engine import PamrecError
    nu, ni, nc, T, B = 50, 300, 20, 12, 20
    om, eng = _setup(nu, ni, nc, T, B, seed=1)
    bad = O.make_batch(1, 10, T, nu, ni, nc)
    for k in list(bad):
        bad[k] = bad[k][:7]
    with pytest.raises(PamrecError):          # 7 rows: not a multiple of the listwise group
        eng.train_step(eng.upload(bad))
    big = O.make_batch(1, 40, T, nu, ni, nc)
    with pytest.raises(PamrecError):          # larger than max_batch
        eng.forward(eng.upload(big), training=False)
    eng.close()


def _mask_patterns(T, rng):
    """One key mask per listwise group.  The MMA kernels stage the compacted live keys padded to a multiple of 8 (forward) and
    16 (backward), so the live-key counts around 8 and 16 matter, not T; a pattern that needs more keys than T has all keys."""
    def scattered(n):
        m = np.zeros(T, np.int32)
        m[rng.choice(T, n, replace=False) if n <= T else np.arange(T)] = 1
        return m
    last8 = np.zeros(T, np.int32); last8[-8:] = 1
    first, final = np.zeros(T, np.int32), np.zeros(T, np.int32)
    first[0] = 1; final[-1] = 1
    return ([np.zeros(T, np.int32), first, final] + [scattered(n) for n in (7, 8, 9, 15, 16, 17)] +
            [last8, (np.arange(T) % 2 == 0).astype(np.int32), np.ones(T, np.int32), (rng.random(T) < 0.5).astype(np.int32)])


# the attention dispatch (MMA up to T = 128, FFMA beyond), the MMA forward's template ladder (7 / 13 / 25 key tiles up to T = 56 /
# 104 / 128), its grid.y split at 64 query rows, the FFMA kernels' warps of 32 query rows
ATTN_T = [1, 2, 7, 8, 9, 12, 16, 17, 33, 50, 56, 57, 64, 65, 100, 104, 105, 127, 128, 129, 160, 200, 255, 256]


@pytest.mark.parametrize("T", ATTN_T)
def test_attention_matches_oracle(T):
    """The attention kernels against the fp64 oracle on a table of key masks, one listwise group each (_mask_patterns): none,
    the first or the last key alone, 7 / 8 / 9 / 15 / 16 / 17 scattered live keys, the last 8, every other, all, random holes.
    Warp-level 3xTF32 MMAs over the live keys up to T = 128 (kernels_attn_mma.cu), the FFMA kernels of kernels_encoder.cu
    beyond - outputs, saved row statistics and all three gradients."""
    from pamrec_b200 import _lib as L
    from relu_masks import engine_relu_masks
    nu, ni, nc = 200, 2000, 40
    rng = np.random.default_rng(3)
    keys = _mask_patterns(T, rng)
    B = O.GROUP * len(keys)
    om, eng = _setup(nu, ni, nc, T, B, seed=11)
    om.proj = "grouped"
    batch = O.make_batch(21, B, T, nu, ni, nc, min_len=T)               # real ids everywhere; the patterns choose the live keys
    batch["mask"] = np.repeat(np.stack(keys), O.GROUP, axis=0)
    db = eng.upload(batch)
    eng.set_debug(L.DEBUG_SAVE_FFN_HIDDEN)                              # differentiate on the engine's ReLU pattern (tests/relu_masks.py)
    eng.forward(db, training=True, want_pred=False)
    masks = engine_relu_masks(eng, B)
    eng.set_debug(0)
    ref = om.train_step(batch, apply=False, keep=("blk0.Q", "blk0.K", "blk0.V", "blk0.y", "x0"), relu_masks=masks)
    t = ref["t"]
    rep = []
    for k in range(2):
        _close(f"blk{k}.y", eng.ws(f"blk{k}.y", B).cpu().numpy(), t[f"blk{k}.y"].detach().numpy(), report=rep)
        # row maximum and row sum of the scaled, masked scores (a sample without a live key: the padding constant and T)
        Q, K = t[f"blk{k}.Q"].detach(), t[f"blk{k}.K"].detach()
        S = Q @ K.transpose(1, 2) / math.sqrt(Q.shape[-1])
        S = torch.where(torch.as_tensor(batch["mask"])[:, None, :] == 0, torch.full_like(S, O.MASK_NEG), S)
        m = S.max(-1).values
        want = np.stack([m.numpy(), torch.exp(S - m[..., None]).sum(-1).numpy()], -1)
        ml = eng.ws(f"blk{k}.ml", B).cpu().numpy().astype(np.float64).reshape(want.shape)
        assert np.allclose(ml[..., 0], want[..., 0], rtol=1e-5, atol=1e-5), f"blk{k}.ml row max"
        assert np.allclose(ml[..., 1], want[..., 1], rtol=1e-4), f"blk{k}.ml row sum"
    _close("logits", eng.ws("logits", B).cpu().numpy(), t["logits"].detach().numpy(), report=rep)
    eng.backward(db)
    torch.cuda.synchronize()
    for nm in ("Q", "K", "V"):                                          # the workspace holds block 0's after the backward
        got = eng.ws(f"d_{nm}", B).cpu().numpy()
        if T == 1 and nm != "V":
            # a single key: the softmax is constant, dQ = dK = 0 exactly, and what is left is the rounding of dS = P (dY.V - D):
            # bounded by the products that cancel, |dY| |V| |K or Q| / sqrt(40)
            dy, other = t["blk0.y"].grad, t["blk0." + ("K" if nm == "Q" else "Q")].detach()
            scale = float(dy.norm(dim=-1).max() * t["blk0.V"].detach().norm(dim=-1).max() * other.abs().max()) / math.sqrt(40)
            rep.append((f"d_{nm}", float(np.abs(got).max()) / scale))
            assert np.isfinite(got).all() and np.abs(got).max() <= 1e-4 * scale, f"d_{nm}: {np.abs(got).max():.3e} at T = 1"
            continue
        _close(f"d_{nm}", got, t[f"blk0.{nm}"].grad.numpy(), rtol=1e-4, report=rep)
    _close("d_x0", eng.ws("g_a", B).cpu().numpy(), t["x0"].grad.numpy(), rtol=1e-4, report=rep)
    print(f"\n[T={T},B={B}] max err / max|ref|: " + ", ".join(f"{n} {e:.2e}" for n, e in rep))
    eng.close()


@pytest.mark.parametrize("legacy_head", [False, True], ids=["head", "legacy_head"])
@pytest.mark.parametrize("T", [1, 57, 128, 129, 256])
def test_scoring_matches_oracle(T, legacy_head, monkeypatch):
    """Scoring (training=False: the head normalises with the moving statistics, perturbed off their initial values) on an engine
    of 20 rows, at batches of 1, 7 and 20 rows: the encoder's output and the predictions against the fp64 oracle."""
    if legacy_head:
        monkeypatch.setenv("PAMREC_HEAD_LEGACY", "1")
    nu, ni, nc, cap = 200, 2000, 40, 20
    om, eng = _setup(nu, ni, nc, T, cap, seed=13)
    om.proj = "grouped"
    for B in (1, 7, cap):
        ev = O.make_batch(40 + B, B, T, nu, ni, nc, grouped=False)
        pred = eng.forward(eng.upload(ev, training=False), training=False).cpu().numpy()
        ref = om.eval_forward(ev).t
        rep = []
        _close("blk1.out", eng.ws("blk1.out", B).cpu().numpy(), ref["blk1.out"].numpy(), report=rep)
        err = float(np.abs(pred - ref["pred"].numpy().reshape(-1)).max())
        print(f"\n[T={T},B={B}/{cap}] blk1.out max err / max|ref| {rep[0][1]:.2e}, predictions max abs err {err:.2e}")
        assert err <= 1e-5, f"B={B}: predictions differ by {err:.3e}"
    eng.close()


def _bucket_layout(layout, B, T, rng):
    """Play-ratio bucket values of all B * T tokens, padded positions included."""
    n = B * T
    if layout == "all0":
        lt = np.zeros(n)
    elif layout == "all9":
        lt = np.full(n, 9.0)
    elif layout == "sizes":
        # bucket sizes around the 64-token tile; the rest of the tokens fill five whole tiles of bucket 7; buckets 0, 5, 6, 8 empty
        sizes = {9: 1, 1: 63, 2: 64, 3: 65, 4: 127}
        sizes[7] = n - sum(sizes.values())
        lt = rng.permutation(np.repeat(list(sizes), list(sizes.values())).astype(np.float64))
    elif layout == "fractional":
        lt = np.where(rng.random(n) < 0.5, rng.choice([2.7, 9.99], n), np.minimum(rng.uniform(0, 10, n), 9.99))
    else:                                   # "bucket10": lisan's id past the tables, one listwise group entirely
        lt = rng.integers(0, 10, n).astype(np.float64)
        lt[rng.random(n) < 0.3] = 10.0
        lt[:5 * T] = 10.0
    return lt.reshape(B, T).astype(np.float32)


@pytest.mark.parametrize("layout", ["all0", "all9", "sizes", "fractional", "bucket10"])
def test_bucket_tiles_stagewise(layout):
    """The time-aware projection runs over bucket-sorted tiles of at most 64 tokens of one bucket (kernels_encoder.cu:
    k_bucket_plan): a whole step at T = 64 with every token in one bucket, with buckets of 1 / 63 / 64 / 65 / 127 tokens, with
    non-integer values (truncated like tf.cast) and with bucket 10 - lisan's id for a ratio beyond its borders or a zero
    duration - which selects a zero matrix (the reference's tf.gather on the GPU): Q = K = V = 0 and no table gradient."""
    nu, ni, nc, T, B = 100, 1000, 30, 64, 10
    om, eng = _setup(nu, ni, nc, T, B, seed=11)
    batch = O.make_batch(5, B, T, nu, ni, nc)
    batch["item_loop_times_history"] = _bucket_layout(layout, B, T, np.random.default_rng(7))
    if layout == "bucket10":
        assert (O.bucket_ids(batch["item_loop_times_history"]) == O.NB).float().mean() > 0.3
    _check_step(om, eng, batch)
