"""CPU checks of tests/table_update_ref.py: the id layouts put runs where asked, the float64 reference restates TF's sparse Adam,
and the per-element bound holds for fp32 arithmetic while a dropped L2 term breaks it."""
import math

import numpy as np
import pytest

from table_update_ref import (CATE_RUNS, ITEM_RUNS, SEG_RUNS, UNIT, adam_consts, adam_reference, clip_scale, dyadic, ids_with_runs, longest_run, merged,
                              plan_runs, worst_ratio)


@pytest.mark.parametrize("n_pos,vocab,wb,group,spec", [
    (5100, 5000, 128, 16, ITEM_RUNS),
    (5100, 700, 512, 16, CATE_RUNS),
    (20000, 20000, 64, 32, SEG_RUNS),
    (5100, 300, 64, 32, SEG_RUNS),
], ids=["item", "cate", "seg", "seg-filled"])
def test_layout_puts_runs_where_asked(n_pos, vocab, wb, group, spec):
    rng = np.random.default_rng(1)
    runs = plan_runs(n_pos, spec, wb, group)
    for (s, _), (_, kind) in zip(runs, spec):
        want = {"group": s % group == 0 and s % wb != 0, "block": s % wb == 0, "before": s % wb == wb - 1, "after": s % wb == 1}[kind]
        assert want, (s, kind)
    ids = ids_with_runs(n_pos, vocab, runs, rng)
    srt = np.sort(ids)
    assert srt[0] == 0 and srt[-1] == vocab - 1
    for s, L in runs:
        assert (srt[s:s + L] == srt[s]).all(), (s, L)
        assert s == 0 or srt[s - 1] != srt[s], (s, L)
        assert s + L == n_pos or srt[s + L] != srt[s], (s, L)
    assert not np.array_equal(ids, srt), "the multiset is scattered over the positions"


def _row_loop_reference(w0, m0, v0, keys, q, l2rows, c, lazy):
    """One row at a time, the way TF's _apply_sparse_shared reads: merged gradient, norm, clip, Adam."""
    rows, width = w0.shape
    G = [[0.0] * width for _ in range(rows)]
    nsq = 0.0
    for k, row in zip(keys, q):
        for j in range(width):
            G[k][j] += row[j] * UNIT
            nsq += (row[j] * UNIT) ** 2
    looked = set(int(k) for k in keys)
    nsq += sum(c["l2"] ** 2 * float(w0[r] @ w0[r]) for r in l2rows)
    s = c["clip"] / max(math.sqrt(nsq), c["clip"]) if c["is_clip"] else 1.0
    w, m, v = w0.copy(), m0.copy(), v0.copy()
    for r in range(rows):
        if lazy and r not in looked:
            continue
        for j in range(width):
            g = s * (G[r][j] + (c["l2"] * w0[r, j] if r in l2rows else 0.0)) if r in looked else 0.0
            m[r, j] = c["b1"] * m0[r, j] + (1 - c["b1"]) * g
            v[r, j] = c["b2"] * v0[r, j] + (1 - c["b2"]) * g * g
            w[r, j] = w0[r, j] - c["lr"] * m[r, j] / (math.sqrt(v[r, j]) + c["eps"])
    return w, m, v, nsq


def _random_slots(rng, shape, zero_frac=0.2):
    m = rng.normal(0, 1e-3, shape)
    v = m * m + rng.uniform(0, 1e-6, shape)
    z = rng.random(shape[0]) < zero_frac
    m[z], v[z] = 0.0, 0.0
    return m, v


@pytest.mark.parametrize("lazy", [False, True])
def test_reference_matches_row_loop(lazy):
    rng = np.random.default_rng(2)
    rows, width, n = 9, 4, 30
    hp = dict(learning_rate=1e-3, beta1=0.9, beta2=0.999, epsilon=1e-8, embed_l2=1e-2, max_grad_norm=0.005, is_clip_norm=1)
    c = adam_consts(hp, 7)
    w0 = rng.normal(0, 0.05, (rows, width))
    m0, v0 = _random_slots(rng, (rows, width))
    keys = rng.integers(1, rows - 2, n)
    keys[:3] = 0                                               # row 0 looked up, but not an L2 row (the siblings' has0 = 0 rule)
    q = dyadic(rng, (n, width), longest_run(keys))
    l2rows = sorted(set(int(k) for k in keys) - {0})
    G = merged(keys, q, rows) * UNIT
    l2sq = float((w0[l2rows] ** 2).sum())
    s, ds, nsq = clip_scale(float((q.astype(np.float64) ** 2).sum()) * UNIT * UNIT, l2sq, c)
    assert s < 1, "the case is meant to clip"
    looked = np.zeros(rows, bool); looked[keys] = True
    l2row = np.zeros(rows, bool); l2row[l2rows] = True
    (w, m, v), _ = adam_reference(w0, m0, v0, G, looked, l2row, c, s, ds)
    if lazy:
        w, m, v = (np.where(looked[:, None], a, b) for a, b in ((w, w0), (m, m0), (v, v0)))
    wl, ml, vl, nsq_l = _row_loop_reference(w0, m0, v0, keys, q, set(l2rows), c, lazy)
    assert abs(nsq - nsq_l) <= 1e-14 * nsq
    for a, b in ((w, wl), (m, ml), (v, vl)):
        assert np.allclose(a, b, rtol=1e-13, atol=1e-18)


def test_bound_holds_for_fp32_adam():
    """The fp32 restatement of the kernels' arithmetic (numpy, no FMA) stays inside the per-element bound on random data, with
    and without clipping; a dropped L2 term does not."""
    rng = np.random.default_rng(3)
    rows, width, n = 4000, 16, 20000
    for l2, clip in ((1e-6, 2.0), (1e-2, 0.05), (1e-2, 100.0)):
        hp = dict(learning_rate=1e-3, beta1=0.9, beta2=0.999, epsilon=1e-8, embed_l2=l2, max_grad_norm=clip, is_clip_norm=1)
        c = adam_consts(hp, 5)
        w0 = rng.normal(0, 0.05, (rows, width)).astype(np.float32)
        m0, v0 = (a.astype(np.float32) for a in _random_slots(rng, (rows, width)))
        keys = rng.integers(0, rows, n)
        q = dyadic(rng, (n, width), longest_run(keys))
        G = merged(keys, q, rows) * UNIT
        looked = np.zeros(rows, bool); looked[keys] = True
        l2sq = float((w0[looked].astype(np.float64) ** 2).sum())
        s, ds, nsq = clip_scale(float((q.astype(np.float64) ** 2).sum()) * UNIT * UNIT, l2sq, c)
        (w, m, v), (bw, bm, bv) = adam_reference(w0, m0, v0, G, looked, looked, c, s, ds)
        F = np.float32
        s32 = F(c["clip"]) / max(F(math.sqrt(nsq)), F(c["clip"]))
        for drop_l2 in (False, True):
            g32 = np.where(looked[:, None], s32 * (G.astype(F) + (F(0) if drop_l2 else F(c["l2"])) * w0), F(0)).astype(F)
            m32 = (m0 * F(c["b1"]) + g32 * (F(1) - F(c["b1"]))).astype(F)
            v32 = (v0 * F(c["b2"]) + (g32 * g32) * (F(1) - F(c["b2"]))).astype(F)
            w32 = (w0 - F(c["lr"]) * m32 / (np.sqrt(v32) + F(c["eps"]))).astype(F)
            oks = [worst_ratio(a, b, bd)[1] for a, b, bd in ((w32, w, bw), (m32, m, bm), (v32, v, bv))]
            if drop_l2:
                assert not all(oks), (l2, clip, "a missing L2 term passes the bound")
            else:
                assert all(oks), (l2, clip, [worst_ratio(a, b, bd)[0] for a, b, bd in ((w32, w, bw), (m32, m, bm), (v32, v, bv))])
