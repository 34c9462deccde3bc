"""Every embedding-table update against float64 Adam, on gradients whose merged sums are exact.

Between the backward pass and apply_gradients the test overwrites the gradient rows that the sparse update reads (PAMRec: columns
0:20 of g_a and d_tgt_total; the sibling models: sib.dh and d_tgt_total) with dyadic values q * 2^-16, |q| <= Q, where
Q = min(255, 2^23 // longest run).  Every partial sum of a row is then a multiple of 2^-16 below 128 in magnitude, exact in fp32 in
any order, so the merged gradient of every row is a known number whatever order the atomics take.  Adam starts from random slots
(some rows exactly zero) at a step t > 1.  The reference is built from the batch ids in float64: merged gradient, L2 rows (the
siblings' row-0 rule), clip norm, TF's sparse-apply Adam, and the embedding share of regular_loss.

The id layouts are designed in sorted order (ids_with_runs): a run of id k starts at the sum of the counts of the ids below k, so
run lengths and start offsets put runs across the walk's groups of 16 positions, its warp blocks of 128 (item) / 512 (category)
positions, k_seg_reduce's 32-position blocks and its multi-block walks.

Comparison: the merged gradient is compared for equality wherever it is stored; w, m and v of every row of every table within a
per-element bound (adam_reference):
  g:  s (G + l2 w0) with s the clip scale; |dg| <= s (|G| + l2 |w0|) (ds + 3 eps), ds the clip scale's relative uncertainty
      (3 eps, plus 10 eps times the share of the norm that comes from fp32 row sums of the L2 rows)
  m:  |dm| <= (1 - b1) |dg| + 3 eps (b1 |m0| + (1 - b1) |g|)
  v:  |dv| <= (1 - b2) (2 |g| |dg| + |dg|^2) + 4 eps (b2 v0 + (1 - b2) g^2)
  w:  |dw| <= lr_t (|dm| + |m| dsqrt(v) / (sqrt(v) + eps)) / (sqrt(v) + eps) + 4 eps |u| + 2 eps (|w0| + |u|), u = lr_t m / (sqrt(v)
      + eps), dsqrt(v) = sqrt(v + |dv|) - sqrt(v)
with eps = 2^-24.  LAZY leaves the rows that were not looked up bit-identical."""
import math

import numpy as np
import pytest

EPS32 = 2.0 ** -24
UNIT = 2.0 ** -16
KINDS = ("group", "block", "before", "after")     # a run starting at a group start, a warp-block start, one before / after one
# k_sp2_walk's run boundaries in one table of 5100 positions: item runs of every length around a group (16) and a warp block (128),
# each length at two kinds of start, and a hot run over more than 8 warp blocks; category runs around a warp block (512), a hot
# run over 3 warp blocks among them
ITEM_LENS = (1, 2, 15, 16, 17, 127, 128, 129, 255, 256, 257)
ITEM_RUNS = ([(L, KINDS[i % 4]) for i, L in enumerate(ITEM_LENS)] + [(1100, "block")] +
             [(L, KINDS[(i + 2) % 4]) for i, L in enumerate(ITEM_LENS)])
CATE_RUNS = [(1023, "block"), (1, "before"), (16, "block"), (17, "group"), (511, "after"), (512, "block"), (513, "after"), (1025, "group")]
# k_seg_reduce: runs around its 32-position blocks and the 64-position walks of two blocks (iters = 2)
SEG_LENS = (1, 31, 32, 33, 63, 64, 65)
SEG_RUNS = [(L, KINDS[i % 4]) for i, L in enumerate(SEG_LENS)] + [(L, KINDS[(i + 2) % 4]) for i, L in enumerate(SEG_LENS)]


# ----------------------------------------------------------------------------------------------------------------- id layouts
def plan_runs(n_pos, runs, wb, group=16):
    """Start offsets in sorted order for runs = [(length, kind)], placed one after the other: kind "group" starts at a multiple of
    `group` that is not a multiple of `wb`, "block" at a multiple of `wb`, "before" / "after" one position before / after one,
    "any" at the cursor.  Returns [(start, length)]."""
    out, p = [], 0
    for length, kind in runs:
        s = p
        if kind == "group":
            s = -(-s // group) * group
            if s % wb == 0:
                s += group
        elif kind == "block":
            s = -(-s // wb) * wb
        elif kind == "before":
            s = -(-(s + 1) // wb) * wb - 1
        elif kind == "after":
            s = -(-(s - 1) // wb) * wb + 1
        elif kind != "any":
            raise ValueError(kind)
        if s + length > n_pos:
            raise ValueError(f"runs do not fit in {n_pos} positions")
        out.append((s, length))
        p = s + length
    return out


def ids_with_runs(n_pos, vocab, runs, rng, lo=0):
    """n_pos ids from [lo, vocab) whose sorted order holds a run of length L at start s for every (s, L) of `runs` (ascending,
    non-overlapping).  The positions in between are filled with runs of `fill` ids (1 while the vocabulary allows: distinct ids).
    The smallest id is lo and the largest vocab - 1.  The multiset is scattered over the positions at random."""
    free = n_pos - sum(length for _, length in runs)
    room = vocab - lo - len(runs)
    # one gap per run at most, so filler runs of `fill` ids need at most free / fill + len(runs) + 1 ids
    fill = 1 if free + len(runs) + 1 <= room else max(1, -(-free // max(room // 2, 1)))
    counts, p = [], 0
    for s, length in list(runs) + [(n_pos, 0)]:
        while p < s:
            c = min(fill, s - p)
            counts.append(c)
            p += c
        if length:
            counts.append(length)
            p += length
    n = len(counts)
    if n > vocab - lo:
        raise ValueError(f"{n} distinct ids do not fit in a vocabulary of {vocab}")
    if n == 1:
        ids = np.asarray([vocab - 1])
    else:
        mid = np.sort(rng.choice(np.arange(lo + 1, vocab - 1), n - 2, replace=False))
        ids = np.concatenate([[lo], mid, [vocab - 1]])
    out = np.empty(n_pos, np.int32)
    out[rng.permutation(n_pos)] = np.repeat(ids, counts)
    return out


def longest_run(ids):
    return int(np.bincount(np.asarray(ids).reshape(-1)).max()) if np.size(ids) else 1


def dyadic(rng, shape, longest):
    """Integers q in [-Q, Q], Q = min(255, 2^23 // longest): the gradient row entries are q * 2^-16."""
    Q = min(255, 2 ** 23 // max(int(longest), 1))
    return rng.integers(-Q, Q + 1, size=shape).astype(np.int64)


def merged(keys, q, vocab):
    """Sum of the rows q[i] over the lookups keys[i], per table row (exact: integer sums in float64)."""
    keys = np.asarray(keys).reshape(-1)
    q = np.asarray(q).reshape(keys.size, -1)
    return np.stack([np.bincount(keys, weights=q[:, c], minlength=vocab) for c in range(q.shape[1])], 1)


# ----------------------------------------------------------------------------------------------------------------- reference
def f32(x):
    return float(np.float32(x))


def adam_consts(hp, step):
    """The fp32 constants the kernels see, in float64, and lr_t with the library's double formula cast to fp32."""
    b1, b2 = f32(hp["beta1"]), f32(hp["beta2"])
    lr = f32(float(np.float32(hp["learning_rate"])) * math.sqrt(1.0 - b2 ** step) / (1.0 - b1 ** step))
    return dict(b1=b1, b2=b2, eps=f32(hp["epsilon"]), l2=f32(hp["embed_l2"]), clip=f32(hp["max_grad_norm"]),
                is_clip=int(hp["is_clip_norm"]), lr=lr)


def clip_scale(nsq_rows, l2sq, c):
    """(s, ds): tf.clip_by_norm's scale for a table whose un-deduplicated rows have squared norm nsq_rows and whose L2 rows have
    squared norm l2sq, and its relative uncertainty in the kernels (fp32 row sums of the L2 rows, fp32 sqrt and division)."""
    nsq = nsq_rows + c["l2"] * c["l2"] * l2sq
    if not c["is_clip"]:
        return 1.0, 0.0, nsq
    s = c["clip"] / max(math.sqrt(nsq), c["clip"])
    frac = c["l2"] * c["l2"] * l2sq / nsq if nsq > 0 else 0.0
    return s, (3.0 + 10.0 * frac) * EPS32, nsq


def adam_reference(w0, m0, v0, G, looked, l2row, c, s, ds):
    """TF's sparse apply in float64 (rows: looked [rows] bool, l2row [rows] bool; G [rows, width]) and the per-element bounds of
    the module docstring.  Returns (w, m, v), (bw, bm, bv)."""
    w0, m0, v0, G = (np.asarray(a, np.float64) for a in (w0, m0, v0, G))
    lk = np.asarray(looked, bool)[:, None]
    l2 = c["l2"] * np.asarray(l2row, bool)[:, None]
    b1, b2, eps, lr = c["b1"], c["b2"], c["eps"], c["lr"]
    g = np.where(lk, s * (G + l2 * w0), 0.0)
    eg = np.where(lk, s * (np.abs(G) + l2 * np.abs(w0)) * (ds + 3 * EPS32), 0.0)
    m = b1 * m0 + (1 - b1) * g
    v = b2 * v0 + (1 - b2) * g * g
    bm = (1 - b1) * eg + 3 * EPS32 * (b1 * np.abs(m0) + (1 - b1) * np.abs(g))
    bv = (1 - b2) * (2 * np.abs(g) * eg + eg * eg) + 4 * EPS32 * (b2 * v0 + (1 - b2) * g * g)
    sq = np.sqrt(v)
    den = sq + eps
    u = lr * m / den
    dsq = np.sqrt(v + bv) - sq
    bw = lr * (bm + np.abs(m) * dsq / den) / den + 4 * EPS32 * np.abs(u) + 2 * EPS32 * (np.abs(w0) + np.abs(u))
    return (w0 - u, m, v), (bw, bm, bv)


def worst_ratio(got, ref, bound):
    """max |got - ref| / bound (0 / 0 counts as 0) and whether every element is within its bound."""
    err = np.abs(np.asarray(got, np.float64) - ref)
    ok = bool(np.isfinite(got).all() and (err <= bound).all())
    r = err / np.maximum(bound, 1e-300)
    return float(np.where(err == 0, 0.0, r).max()) if err.size else 0.0, ok
