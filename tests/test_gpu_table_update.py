"""Every embedding-table update - whole tables (kernels_sparse2.cu: COMPACT for DENSE_EXACT, the fused walk for LAZY), row-sharded
tables and the sibling models (kernels_optim.cu) - against float64 Adam on injected gradients whose merged sums are exact.  The
method and the per-element bounds are described in tests/table_update_ref.py.  After every step: the merged gradient equals the
reference wherever it is stored, the clip norms agree to 1e-6, w / m / v of every row of every table lie within their bounds, LAZY
leaves rows that were not looked up bit-identical, sp2.dflag is all zero and sp2.slot marks the current plan's rows only."""
import numpy as np
import pytest
import torch

from oracle import pamrec_oracle as O
from oracle import siblings_oracle as S
from table_update_ref import (CATE_RUNS, EPS32, ITEM_RUNS, SEG_RUNS, UNIT, adam_consts, adam_reference, clip_scale, dyadic,
                              ids_with_runs, longest_run, merged, plan_runs, worst_ratio)

pytestmark = pytest.mark.gpu

MODES = ["dense_exact", "lazy"]


# ----------------------------------------------------------------------------------------------------------------- batches
def _users(rng, nu, B):
    """User ids with a repeat, row 0 and row nu - 1."""
    u = rng.integers(0, nu, B).astype(np.int32)
    u[-1] = u[0]
    if B > 2:
        u[1], u[2] = 0, nu - 1
    return u


def layout_batch(rng, nu, ni, nc, T, B, item_runs=(), cate_runs=(), item_wb=128, cate_wb=512, group=16, lo=0):
    """A training batch whose item and category ids, in sorted order over the table's history and target positions, hold the runs
    [(length, kind)] (plan_runs) and distinct ids or short runs elsewhere.  lo = 1 keeps id 0 out of the history and the targets."""
    n = B * T + B

    def ids(vocab, runs, wb):
        return ids_with_runs(n, vocab, plan_runs(n, list(runs), wb, group), rng, lo=lo)

    it, ct = ids(ni, item_runs, item_wb), ids(nc, cate_runs, cate_wb)
    return dict(item_history=it[:B * T].reshape(B, T), item_cate_history=ct[:B * T].reshape(B, T),
                item_loop_times_history=rng.integers(0, 10, (B, T)).astype(np.float32), mask=np.ones((B, T), np.int32),
                users=_users(rng, nu, B), items=it[B * T:].copy(), cates=ct[B * T:].copy(),
                labels_satisfied=(rng.random(B) < 0.3).astype(np.float32), labels_play=(rng.random(B) < 0.5).astype(np.float32),
                plays=rng.uniform(0.1, 1.0, B).astype(np.float32))


# ----------------------------------------------------------------------------------------------------------------- engine state
def make_engine(dims, B, mode, hp=None, tables="local", model="pamrec", emb_dims=None, graph=False, seed=0):
    """Engine with random dense parameters, tables and Adam slots (a fifth of the rows' slots exactly zero)."""
    from pamrec_b200.engine import DEFAULT_HP, EMB_DIMS, Engine
    nu, ni, nc, T = dims
    h = dict(DEFAULT_HP)
    h.update(hp or {})
    eng = Engine(nu, ni, nc, T, B, hp=h, sparse_adam=mode, tables=tables, model=model, graph=graph,
                 emb_dims=emb_dims or EMB_DIMS).allocate()
    rng = np.random.default_rng(seed)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(eng.device)
    eng.pool["dense_param"].copy_(dev(rng.normal(0, 0.05, eng.dense_numel)))
    eng.pool["bn_moving"].fill_(1.0)
    for tab in table_names(eng):
        shape = tuple(eng.pool[tab + "_w"].shape)
        eng.pool[tab + "_w"].copy_(dev(rng.normal(0, 0.05, shape)))
        m = rng.normal(0, 1e-3, shape)
        v = m * m + rng.uniform(0, 1e-6, shape)
        zero = rng.random(shape[0]) < 0.2
        m[zero], v[zero] = 0.0, 0.0
        eng.pool[tab + "_m"].copy_(dev(m))
        eng.pool[tab + "_v"].copy_(dev(v))
    eng.step = 4                                             # the next step runs at t = 5
    torch.cuda.synchronize()
    return eng


def table_names(eng):
    return [pre for pre, _ in eng.tables_by_name.values()]


def _vocab(eng, tab):
    nu, ni, nc = eng.dims[:3]
    return {"item": ni, "cate": nc, "ulong": nu, "ushort": nu}[tab]


def _dense_reg(eng):
    """0.5 layer_l2 sum |p|^2 over the L2-regularised dense variables (float64 from the fp32 parameters)."""
    from pamrec_b200 import _lib as L
    p = eng.pool["dense_param"].cpu().numpy().astype(np.float64)
    tot = sum(float((p[d["offset"]:d["offset"] + d["numel"]] ** 2).sum()) for d in eng.info[L.POOL_DENSE].values() if d["flags"] & L.SEG_L2)
    return 0.5 * float(np.float32(eng.hp["layer_l2"])) * tot


# ----------------------------------------------------------------------------------------------------------------- one step
class Lookups:
    """The lookups of one gradient-carrying table in the order its sparse plan reads them, the injected rows, the L2 rows."""

    def __init__(self, keys, q, vocab, l2_keys, longest):
        self.keys, self.q, self.vocab = keys, q, vocab
        self.G = merged(keys, q, vocab) * UNIT
        self.looked = np.zeros(vocab, bool)
        self.looked[keys] = True
        self.l2row = np.zeros(vocab, bool)
        self.l2row[l2_keys] = True
        self.nsq_rows = float((q.astype(np.float64) ** 2).sum()) * UNIT * UNIT
        self.longest = longest


def _inject(eng, batch, rng):
    """Overwrite the gradient rows of the sparse update; returns {table: Lookups} (users: keys only, no rows)."""
    B, T = len(batch["items"]), eng.dims[3]
    N = B * T
    di, dc = eng.emb_dims[:2]
    E = di + dc
    ni, nc = eng.dims[1], eng.dims[2]
    out = {}
    if eng.model == "pamrec":
        g_a, dt = eng.ws("g_a", B), eng.ws("d_tgt_total", B)
        for tab, hk, tk, col, w, vocab in (("item", "item_history", "items", 0, di, ni), ("cate", "item_cate_history", "cates", di, dc, nc)):
            keys = np.concatenate([batch[hk].reshape(-1), batch[tk]]).astype(np.int64)
            lr_ = longest_run(keys)
            q = dyadic(rng, (N + B, w), lr_)
            g_a[:, :, col:col + w].copy_(torch.from_numpy((q[:N] * UNIT).reshape(B, T, w).astype(np.float32)))
            dt[:, col:col + w].copy_(torch.from_numpy((q[N:] * UNIT).astype(np.float32)))
            out[tab] = Lookups(keys, q, vocab, np.unique(keys), lr_)
    else:
        sas = eng.model == "sasrec"
        dh = eng.ws("sib.dh").reshape(-1)[:2 * N * E].view(2, N, E)
        dt = eng.ws("d_tgt_total", B)
        for tab, sk, hk, tk, col, w, vocab in (("item", "satisfied_item_history", "item_history", "items", 0, di, ni),
                                               ("cate", "satisfied_cate_history", "item_cate_history", "cates", di, dc, nc)):
            keys = np.concatenate([batch[sk].reshape(-1), batch[hk].reshape(-1), batch[tk]]).astype(np.int64)
            lr_ = longest_run(keys)
            q = dyadic(rng, (2 * N + B, w), lr_)
            if sas:
                q[N:2 * N] = 0                                     # the full-history lookups carry no gradient (L2 rows only)
            dh[:, :, col:col + w].copy_(torch.from_numpy((q[:2 * N] * UNIT).reshape(2, N, w).astype(np.float32)))
            dt[:, col:col + w].copy_(torch.from_numpy((q[2 * N:] * UNIT).astype(np.float32)))
            involved = np.unique(np.concatenate([batch[hk].reshape(-1), batch[tk]]))      # tf.unique(history | targets)
            out[tab] = Lookups(keys, q, vocab, involved, lr_)
    if "ulong" in table_names(eng):
        out["user"] = np.unique(batch["users"]).astype(np.int64)
    return out


def _host(eng, tabs):
    return {t: {s: eng.pool[f"{t}_{s}"].cpu().numpy() for s in "wmv"} for t in tabs}


def run_step(eng, batch, seed, twice=False, label=""):
    """One eager step with injected gradients, checked against the float64 reference.  twice: forward(training=True) twice before
    the backward pass and the update."""
    from pamrec_b200 import _lib as L
    rng = np.random.default_rng(seed)
    lazy = eng.cfg.sparse_adam_mode == L.ADAM_LAZY
    local, sharded, pam = eng.tables == "local", eng.tables == "sharded", eng.model == "pamrec"
    tabs = table_names(eng)
    B = len(batch["items"])
    before = _host(eng, tabs)
    for tab in ("item", "cate"):                              # stale values in the accumulators: every row must be written or zeroed
        eng.ws(f"sp.{tab}.accum").fill_(3.0)
    db = eng.upload(batch)
    eng.forward(db, training=True, want_pred=False)
    if twice:
        eng.forward(db, training=True, want_pred=False)
    eng.backward(db)
    lk = _inject(eng, batch, rng)
    if pam and local:                                         # the backward pass's un-deduplicated norms, of the injected rows
        spn = eng.ws("sp_normsq")
        spn[0] = lk["item"].nsq_rows
        spn[1] = lk["cate"].nsq_rows
    dense_reg = _dense_reg(eng)
    losses = eng.apply_gradients(db).cpu().numpy()
    torch.cuda.synchronize()
    after = _host(eng, tabs)
    c = adam_consts(eng.hp, eng.step)
    fails, report, scales = [], [], {}
    nuniq = eng.ws("sp.nuniq").cpu().numpy()
    spn = eng.ws("sp_normsq").cpu().numpy()
    emb_reg = 0.0
    if not pam:
        has0 = eng.ws("sib.has0").cpu().numpy()
        N = B * eng.dims[3]
        for k, (tab, sk, hk) in enumerate((("item", "satisfied_item_history", "item_history"), ("cate", "satisfied_cate_history", "item_cate_history"))):
            ids = eng.ws(f"sib.ids_{tab}").reshape(-1)[:2 * N].cpu().numpy()
            if not np.array_equal(ids, np.concatenate([batch[sk].reshape(-1), batch[hk].reshape(-1)])):
                fails.append(f"sib.ids_{tab} differ from the batch ids")
            if int(has0[k]) != int(lk[tab].l2row[0]):
                fails.append(f"sib.has0[{tab}] = {has0[k]}, row 0 is {'' if lk[tab].l2row[0] else 'not '}an L2 row")
    # ---- merged gradients, unique lists and slot maps
    slot = eng.ws("sp2.slot").cpu().numpy() if local and pam else None
    for k, tab in enumerate(("item", "cate")):
        x = lk[tab]
        uk_ref = np.flatnonzero(x.looked)
        uk = eng.ws(f"sp.{tab}.ukeys").cpu().numpy()[:int(nuniq[k])]
        if not np.array_equal(uk, uk_ref):
            fails.append(f"sp.{tab}.ukeys differ from the unique ids of the batch")
            continue
        if local and pam:
            sl = slot[(0 if k == 0 else eng.dims[1]):][:x.vocab]
            if not lazy:
                acc = eng.ws(f"sp.{tab}.accum").cpu().numpy()[sl[uk]]
                if not np.array_equal(acc.astype(np.float64), x.G[uk]):
                    bad = np.argwhere(acc != x.G[uk])[0]
                    fails.append(f"{tab}: merged gradient of row {uk[bad[0]]} col {bad[1]}: {acc[tuple(bad)]!r} != {x.G[uk][tuple(bad)]!r}")
        else:
            acc = eng.ws(f"sp.{tab}.accum").cpu().numpy()[:uk.size]
            if not np.array_equal(acc.astype(np.float64), x.G[uk]):
                fails.append(f"sp.{tab}.accum: merged gradient differs in {int((acc != x.G[uk]).any(1).sum())} rows")
            if sharded:
                n_own = int(nuniq[4 + k])
                if not np.array_equal(eng.ws(f"so.{tab}.ukeys").cpu().numpy()[:n_own], uk_ref):
                    fails.append(f"so.{tab}.ukeys differ from the unique ids of the batch")
                elif not np.array_equal(eng.ws(f"so.{tab}.accum").cpu().numpy()[:n_own].astype(np.float64), x.G[uk]):
                    fails.append(f"so.{tab}.accum: the owner's merged gradient differs")
    if local and pam:
        want = np.full(slot.shape, -1, np.int64)
        if not lazy:
            bases = (0, eng.dims[1], eng.dims[1] + eng.dims[2])
            keys = (np.flatnonzero(lk["item"].looked), np.flatnonzero(lk["cate"].looked), lk["user"])
            for b, kk in zip(bases, keys):
                want[b + kk] = np.arange(kk.size)
        if not np.array_equal(slot, want):
            fails.append(f"sp2.slot: {int((slot != want).sum())} entries differ from the current plan's rows")
        dflag = eng.ws("sp2.dflag").cpu().numpy()
        if dflag.any():
            fails.append(f"sp2.dflag: {int((dflag != 0).sum())} flags left set")
    # ---- clip norms, Adam, regular loss
    for t_i, tab in enumerate(tabs):
        w0, m0, v0 = (before[tab][s] for s in "wmv")
        vocab = _vocab(eng, tab)
        if tab in ("item", "cate"):
            x = lk[tab]
            G, looked, l2row, nsq_rows = x.G, x.looked, x.l2row, x.nsq_rows
        else:
            G = np.zeros((vocab, w0.shape[1]))
            looked = np.zeros(vocab, bool); looked[lk["user"]] = True
            l2row, nsq_rows = looked, 0.0
        w0, m0, v0 = w0[:vocab], m0[:vocab], v0[:vocab]
        l2sq = float((w0[l2row].astype(np.float64) ** 2).sum())
        emb_reg += 0.5 * c["l2"] * l2sq
        s, ds, nsq = clip_scale(nsq_rows, l2sq, c)
        if abs(spn[t_i] - nsq) > 1e-6 * nsq:
            fails.append(f"sp_normsq[{t_i}] ({tab}) = {spn[t_i]!r}, reference {nsq!r}")
        (w, m, v), (bw, bm, bv) = adam_reference(w0, m0, v0, G, looked, l2row, c, s, ds)
        line = []
        for nm, ref, bd in (("w", w, bw), ("m", m, bm), ("v", v, bv)):
            got = after[tab][nm][:vocab]
            if lazy:
                if not np.array_equal(got[~looked], before[tab][nm][:vocab][~looked]):
                    fails.append(f"{tab}.{nm}: LAZY moved {int((got[~looked] != before[tab][nm][:vocab][~looked]).any(1).sum())} rows that were not looked up")
                ref, bd, got = ref[looked], bd[looked], got[looked]
            r, ok = worst_ratio(got, ref, bd)
            line.append(f"{nm} {r:.2f}")
            if not ok:
                i = np.unravel_index(int(np.argmax(np.abs(got - ref) - bd)), got.shape)
                fails.append(f"{tab}.{nm}: worst error / bound {r:.3g} at {i}: got {got[i]!r}, reference {ref[i]!r}, bound {bd[i]:.3g}")
        report.append(f"  {tab:7s} scale {s:.6f}  worst error / bound: " + ", ".join(line))
        scales[tab] = s
    want_reg = dense_reg + emb_reg
    if abs(losses[2] - want_reg) > 2 * EPS32 * want_reg + 1e-6 * emb_reg:
        fails.append(f"regular_loss {losses[2]!r}: dense part {dense_reg!r} + embedding part {emb_reg!r} = {want_reg!r}")
    print(f"\n[{label} step {eng.step}, B={B}, {'lazy' if lazy else 'dense_exact'}]\n" + "\n".join(report))
    assert not fails, "\n".join(fails)
    return scales


# ----------------------------------------------------------------------------------------------------------------- PAMRec, whole tables
def _case1(rng, nu=300, ni=5000, nc=700, T=50, B=100):
    return layout_batch(rng, nu, ni, nc, T, B, ITEM_RUNS, CATE_RUNS)


# max_grad_norm 0.45 lies between the norms of the injected item rows (5100 x 16 entries of rms 255 / sqrt(3) 2^-16: 0.64) and
# category rows (0.32); with embed_l2 = 1e-2 the L2 rows' share of every table's norm matters, and every table clips at 0.02
VARIANTS = {
    "default": ({}, None),
    "no_clip": (dict(is_clip_norm=0), None),
    "clip_item_only": (dict(max_grad_norm=0.45), lambda s: s["item"] < 1 and s["cate"] == 1),
    "l2": (dict(embed_l2=1e-2, max_grad_norm=0.02), lambda s: max(s.values()) < 1),
}


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_run_boundaries(variant, mode):
    """Case 1: item and category runs at every boundary of k_sp2_walk, hot rows over many warp blocks, rows 0 and vocab - 1."""
    dims = (300, 5000, 700, 50)
    batch = _case1(np.random.default_rng(11))
    hp, scales_ok = VARIANTS[variant]
    eng = make_engine(dims, 100, mode, hp=hp, seed=1)
    scales = run_step(eng, batch, seed=2, label=f"case 1 {variant}")
    eng.close()
    assert scales_ok is None or scales_ok(scales), scales


@pytest.mark.parametrize("mode", MODES)
def test_one_id_per_table(mode):
    """Case 2: one id per table - one run over every warp block."""
    nu, ni, nc, T, B = 50, 300, 20, 50, 100
    rng = np.random.default_rng(3)
    batch = layout_batch(rng, nu, ni, nc, T, B)
    for k, v in (("item_history", 7), ("items", 7), ("item_cate_history", 3), ("cates", 3), ("users", 5)):
        batch[k] = np.full_like(batch[k], v)
    eng = make_engine((nu, ni, nc, T), B, mode, seed=3)
    run_step(eng, batch, seed=4, label="case 2")
    eng.close()


@pytest.mark.parametrize("mode", MODES)
def test_all_distinct(mode):
    """Case 3: no duplicate id in any table."""
    nu, ni, nc, T, B = 300, 6000, 6000, 50, 100
    rng = np.random.default_rng(5)
    batch = layout_batch(rng, nu, ni, nc, T, B)
    batch["users"] = rng.permutation(nu)[:B].astype(np.int32)
    eng = make_engine((nu, ni, nc, T), B, mode, seed=5)
    run_step(eng, batch, seed=6, label="case 3")
    eng.close()


@pytest.mark.parametrize("mode", MODES)
def test_tiny(mode):
    """Case 4: B 5, T 1, two categories - every table region is smaller than one group."""
    nu, ni, nc, T, B = 7, 9, 2, 1, 5
    batch = layout_batch(np.random.default_rng(7), nu, ni, nc, T, B, [(2, "after")], [(3, "any")])
    eng = make_engine((nu, ni, nc, T), B, mode, seed=7)
    run_step(eng, batch, seed=8, label="case 4")
    eng.close()


@pytest.mark.parametrize("mode", MODES)
def test_large_tables(mode):
    """Case 5: 400 K items, 200 K users, Zipf ids: the one-launch sweep takes proportional CTA shares and its grid-stride loop."""
    nu, ni, nc, T, B = 200000, 400000, 500, 50, 1025
    batch = O.make_batch(9, B, T, nu, ni, nc)
    eng = make_engine((nu, ni, nc, T), B, mode, seed=9)
    run_step(eng, batch, seed=10, label="case 5")
    eng.close()


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("extra", [0, 1], ids=["pow2", "pow2+1"])
def test_radix_bits_edge(extra, mode):
    """Case 6: n_items + n_cates + n_users = 2^13 and 2^13 + 1 (the sort's bit count), vocab - 1 looked up in every table."""
    nu, nc = 300, 700
    ni = 2 ** 13 - nu - nc + extra
    batch = _case1(np.random.default_rng(12), nu=nu, ni=ni, nc=nc)
    eng = make_engine((nu, ni, nc, 50), 100, mode, seed=12)
    run_step(eng, batch, seed=13, label=f"case 6 +{extra}")
    eng.close()


@pytest.mark.parametrize("mode", MODES)
def test_several_steps_one_engine(mode):
    """Case 7: steps of 200 and 100 rows with a scoring pass between them, a step with two training forward passes, then 200 rows
    again; each step's reference starts from the engine's own state before it."""
    nu, ni, nc, T = 300, 5000, 700, 50
    eng = make_engine((nu, ni, nc, T), 200, mode, seed=14)
    rng = np.random.default_rng(15)
    run_step(eng, _case1(rng, B=200, T=T), seed=16, label="case 7")
    ev = O.make_batch(17, 77, T, nu, ni, nc, grouped=False)
    eng.forward(eng.upload(ev, training=False), training=False)
    run_step(eng, _case1(rng, B=100, T=T), seed=18, label="case 7")
    run_step(eng, layout_batch(rng, nu, ni, nc, T, 150, ITEM_RUNS[::2], CATE_RUNS[:4]), seed=19, twice=True, label="case 7 twice")
    run_step(eng, O.make_batch(20, 200, T, nu, ni, nc), seed=21, label="case 7")
    eng.close()


def test_graph_replay():
    """Case 8: train steps replayed from CUDA graphs (two batches alternating).  Nothing can be injected: the merged gradient is
    checked against the float64 sum of the engine's own rows within the summation depth of the walk - 16 in a group, 64 merged
    partials, one partial per warp block the run touches - and the update against float64 Adam applied to that gradient."""
    from pamrec_b200 import _lib as L
    nu, ni, nc, T, B = 300, 5000, 700, 50, 100
    eng = make_engine((nu, ni, nc, T), B, "dense_exact", graph=True, seed=22)
    rng = np.random.default_rng(23)
    dbs = [eng.upload(_case1(rng)), eng.upload(O.make_batch(24, B, T, nu, ni, nc))]
    batches = [{k: v.cpu().numpy() for k, v in db.tensors.items()} for db in dbs]
    fails = []
    tabs = table_names(eng)
    for i in range(6):
        db, batch = dbs[i % 2], batches[i % 2]
        before = _host(eng, tabs)
        eng.train_step(db)
        torch.cuda.synchronize()
        after = _host(eng, tabs)
        c = adam_consts(eng.hp, eng.step)
        slot = eng.ws("sp2.slot").cpu().numpy()
        spn = eng.ws("sp_normsq").cpu().numpy()
        g_a, dt = eng.ws("g_a", B).cpu().numpy().astype(np.float64), eng.ws("d_tgt_total", B).cpu().numpy().astype(np.float64)
        report = []
        for k, tab in enumerate(tabs):
            w0, m0, v0 = (before[tab][s] for s in "wmv")
            vocab = _vocab(eng, tab)
            if k < 2:
                col, w_, wb = (0, 16, 128) if k == 0 else (16, 4, 512)
                hk, tk = ("item_history", "items") if k == 0 else ("item_cate_history", "cates")
                keys = np.concatenate([batch[hk].reshape(-1), batch[tk]]).astype(np.int64)
                rows = np.concatenate([g_a[:, :, col:col + w_].reshape(-1, w_), dt[:, col:col + w_]])
                G64 = np.stack([np.bincount(keys, weights=rows[:, j], minlength=vocab) for j in range(w_)], 1)
                A64 = np.stack([np.bincount(keys, weights=np.abs(rows[:, j]), minlength=vocab) for j in range(w_)], 1)
                cnt = np.bincount(keys, minlength=vocab)
                start = np.concatenate([[0], np.cumsum(cnt)[:-1]])
                looked = cnt > 0
                nblk = np.where(looked, (start + cnt - 1) // wb - start // wb + 1, 0)
                uk = np.flatnonzero(looked)
                acc = eng.ws(f"sp.{tab}.accum").cpu().numpy()[slot[(0 if k == 0 else ni):][:vocab][uk]].astype(np.float64)
                bound = (16 + 64 + nblk[uk, None]) * EPS32 * A64[uk]
                err = np.abs(acc - G64[uk])
                if not (err <= bound).all():
                    fails.append(f"step {eng.step} {tab}: merged gradient off by {float((err / np.maximum(bound, 1e-300)).max()):.3g} bounds")
                G = np.zeros_like(G64)
                G[uk] = acc
                nsq_rows = float((rows ** 2).sum())
                l2row = looked
            else:
                users = np.unique(batch["users"]).astype(np.int64)
                G = np.zeros((vocab, w0.shape[1]))
                looked = np.zeros(vocab, bool); looked[users] = True
                l2row, nsq_rows = looked, 0.0
            l2sq = float((w0[l2row].astype(np.float64) ** 2).sum())
            s, ds, nsq = clip_scale(nsq_rows, l2sq, c)
            if abs(spn[k] - nsq) > 1e-6 * nsq:
                fails.append(f"step {eng.step} sp_normsq[{k}] = {spn[k]!r}, reference {nsq!r}")
            (w, m, v), (bw, bm, bv) = adam_reference(w0, m0, v0, G, looked, l2row, c, s, ds)
            line = []
            for nm, ref, bd in (("w", w, bw), ("m", m, bm), ("v", v, bv)):
                r, ok = worst_ratio(after[tab][nm], ref, bd)
                line.append(f"{nm} {r:.2f}")
                if not ok:
                    fails.append(f"step {eng.step} {tab}.{nm}: worst error / bound {r:.3g}")
            report.append(f"  {tab:7s} worst error / bound: " + ", ".join(line))
        print(f"\n[case 8 graph step {eng.step}]\n" + "\n".join(report))
    assert len(eng._graphs) == 2, "both batches were replayed from their graphs"
    eng.close()
    assert not fails, "\n".join(fails)


# ----------------------------------------------------------------------------------------------------------------- PAMRec, sharded
@pytest.mark.parametrize("mode", MODES)
def test_sharded_seg_reduce_walks(mode):
    """Case 9: runs around k_seg_reduce's 32-position blocks and its walks of two blocks (iters = 2 from 606 208 lookups on)."""
    nu, ni, nc, T, B = 3000, 300000, 5000, 256, 2400
    assert B * T + B >= 2 * 148 * 8 * 8 * 32
    batch = layout_batch(np.random.default_rng(25), nu, ni, nc, T, B, SEG_RUNS, SEG_RUNS, item_wb=64, cate_wb=64, group=32)
    eng = make_engine((nu, ni, nc, T), B, mode, tables="sharded", seed=25)
    run_step(eng, batch, seed=26, label="case 9")
    eng.close()


@pytest.mark.parametrize("mode", MODES)
def test_sharded_run_boundaries(mode):
    """Case 10: case 1's layout through the sharded path."""
    eng = make_engine((300, 5000, 700, 50), 100, mode, tables="sharded", seed=27)
    run_step(eng, _case1(np.random.default_rng(27)), seed=28, label="case 10")
    eng.close()


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("extra", [0, 1], ids=["pow2", "pow2+1"])
def test_sharded_table_rows_edge(extra, mode):
    """Case 11: table rows a power of two and one more, vocab - 1 looked up in every table."""
    nu, ni, nc, T, B = 256 + extra, 4096 + extra, 512 + extra, 20, 100
    batch = layout_batch(np.random.default_rng(29), nu, ni, nc, T, B, ITEM_RUNS[:8], CATE_RUNS[2:4])
    eng = make_engine((nu, ni, nc, T), B, mode, tables="sharded", seed=29)
    run_step(eng, batch, seed=30, label=f"case 11 +{extra}")
    eng.close()


# ----------------------------------------------------------------------------------------------------------------- sibling models
SIBLINGS = [("mmoe", (16, 4, 20)), ("ple", (32, 8, 40)), ("sharebottom", (32, 8, 16)), ("sasrec", (32, 8, 16))]


def sibling_batch(rng, nu, ni, nc, T, B, has0, item_runs=(), cate_runs=(), **blocks):
    """layout_batch over the history and target positions (id 0 among them only when has0) plus the satisfied-only copies of the
    history, whose zero padding looks row 0 up in any case."""
    b = layout_batch(rng, nu, ni, nc, T, B, item_runs, cate_runs, lo=0 if has0 else 1, **blocks)
    b = S.add_satisfied_fields(b, seed=int(rng.integers(1 << 30)))
    assert (b["satisfied_item_history"] == 0).any()
    return b


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("has0", [0, 1], ids=["row0_padding_only", "row0_looked_up"])
@pytest.mark.parametrize("model,emb_dims", SIBLINGS, ids=[m for m, _ in SIBLINGS])
def test_sibling_tables(model, emb_dims, has0, mode):
    """Case 12: the first-generation path at every table width it instantiates, with row 0 looked up only through the
    satisfied-only history's padding (no L2 term on row 0) or among the history / target ids.  The padding-only half runs with
    embed_l2 = 1e-2 and clips, so that an L2 term on row 0 or a lost L2 share of the norm is far outside the bounds."""
    nu, ni, nc, T, B = 200, 3000, 400, 30, 60
    batch = sibling_batch(np.random.default_rng(31 + has0), nu, ni, nc, T, B, has0, ITEM_RUNS[:9], CATE_RUNS[2:5])
    hp = {} if has0 else dict(embed_l2=1e-2, max_grad_norm=0.05)
    eng = make_engine((nu, ni, nc, T), B, mode, hp=hp, model=model, emb_dims=emb_dims, seed=33)
    run_step(eng, batch, seed=34, label=f"case 12 {model} has0={has0}")
    eng.close()


@pytest.mark.parametrize("mode", MODES)
def test_sibling_seg_reduce_walks(mode):
    """Case 13: MMoE with 2 B T + B >= 606 208 lookups per table (k_seg_reduce walks two blocks)."""
    nu, ni, nc, T, B = 3000, 300000, 5000, 128, 2400
    assert 2 * B * T + B >= 2 * 148 * 8 * 8 * 32
    batch = sibling_batch(np.random.default_rng(35), nu, ni, nc, T, B, 1, SEG_RUNS, SEG_RUNS, item_wb=64, cate_wb=64, group=32)
    eng = make_engine((nu, ni, nc, T), B, mode, model="mmoe", seed=35)
    run_step(eng, batch, seed=36, label="case 13")
    eng.close()
