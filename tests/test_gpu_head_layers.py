"""Every layer of every head, element by element, against float64 on the engine's own tensors: PAMRec's row-stationary head
(kernels_head2.cu) and its stand-alone head (PAMREC_HEAD_LEGACY=1, kernels_head.cu / head_tiles.cuh), the MMoE / PLE /
share-bottom heads and SASRec's tower (the same tile kernels, api_sibling.inl).

Each reference is layer-local: it is built from the fp32 tensors the step saved at that point (pre-activations, batch statistics,
gradient buffers) and the parameters the step ran with, so errors do not compound and a failure names one layer, one tensor and
one element.  Where an implementation keeps a gradient only in shared memory (head2: dA of the towers, experts, gates and of the
score MLP's first layer, d_u), it is carried in float64 from the nearest stored tensor together with its bound.

The bound of an element is the same expression over absolute values (|x|^T |dz| for dW, sum |dz| for db, |dz| |W|^T for dX, the
batch-norm backward term by term); the error must stay below rel times that.  rel = 2e-5 covers the fp32 chains of up to ~256
serial terms (the worst case of recursive summation, n u, is 1.5e-5 there); a longer chain gets (n + 8) u (rel_chain).  ReLU sides
are the kernels' own fp32 decisions (relu_masks._on), so gradients are defined at every batch size.  There is no floor relative to
the model's largest gradient anywhere."""
import numpy as np
import pytest
import torch

from oracle import pamrec_oracle as O
from oracle import siblings_oracle as S
import siblings_oracle_dims as D
from relu_masks import HEAD_MLPS, _on, sas_mlps, sibling_mlps

pytestmark = pytest.mark.gpu

U = 2.0 ** -24                          # fp32 unit roundoff
REL = 2e-5
EPS = float(np.float32(1e-4))           # kBnEps, added to the variance as a float
DECAY = float(np.float32(0.05))         # kBnDecay
BN_SETS = ("s0", "s1", "e0", "g0", "e1", "g1", "t0", "t1")    # layout.h: BnId order, the row order of bn.bsums
MASK_NEG = -4294967295.0                # kMaskNeg
PLE_SEL = ((0, 1, 2, 3, 4), (0, 1, 2, 5, 6))                  # experts mixed by gate_main / gate_sub (layout.h: gate_sel)
LAYER = ("layer0", "layer1", "output")


def rel_chain(n):
    """rel for sums of n serial fp32 terms (plus the atomics that join the partial sums)."""
    return max(REL, (n + 8) * U)


def dx_chain(*mlps):
    """Serial terms of one input-gradient element of k_dense_dx: every member that reads the column contributes its layer-0 width
    to one accumulator (the gates then add theirs to the experts')."""
    return sum(max(m.x_col.count(c) for c in m.x_col) * m.h0 for m in mlps)


def tiles_dw_chain(M, G, K, N):
    """Serial terms of one k_dense_dw element: the rows of one CTA (head_tiles.cuh:dense_dw_grid, 148 * 6 CTAs) and one atomic per CTA."""
    ny = G * -(-K // 32) * -(-N // 32)
    chunks = max(1, min(-(-888 // ny), -(-M // 32)))
    rpc = -(-(-(-M // chunks)) // 32) * 32
    return rpc + -(-M // rpc)


class Check:
    def __init__(self, tag):
        self.tag, self.bad, self.rep = tag, [], {}

    def close(self, name, got, ref, bound, rel=REL):
        """|got - ref| <= rel * bound element by element; records the worst err / (rel * bound) of the tensor."""
        ref = np.asarray(ref, np.float64)
        got = np.asarray(got, np.float64).reshape(ref.shape)
        bound = np.broadcast_to(np.asarray(bound, np.float64), ref.shape)
        err = np.abs(got - ref)
        q = np.where(err == 0, 0.0, err / np.maximum(rel * bound, 1e-300))
        q = np.where(np.isfinite(got), q, np.inf)
        worst = float(q.max()) if q.size else 0.0
        self.rep[name] = max(self.rep.get(name, 0.0), worst)
        if worst > 1.0:
            i = np.unravel_index(int(np.argmax(q)), q.shape)
            self.bad.append(f"{name} at {tuple(int(v) for v in i)}: got {got[i]:.9g}, ref {ref[i]:.9g}, bound {rel:.1e} x {bound[i]:.3e} "
                            f"(err / allowed {worst:.3e})")

    def done(self):
        print(f"\n[{self.tag}] worst err / allowed per tensor: " + ", ".join(f"{k} {v:.2e}" for k, v in self.rep.items()))
        assert not self.bad, f"[{self.tag}] {len(self.bad)} tensors off: " + "; ".join(self.bad[:10])


class Step:
    """The engine's tensors after one step, as float64.  P: the dense parameters the step ran with; mov0: the moving statistics
    before its forward pass."""

    def __init__(self, eng, P, mov0, B, T):
        from pamrec_b200 import _lib as L
        self.eng, self.B, self.T = eng, B, T
        self.info, self.bn_info = eng.info[L.POOL_DENSE], eng.info[L.POOL_BN]
        self.P, self.mov0 = P.cpu().numpy(), mov0.cpu().numpy()
        self.mov1 = eng.pool["bn_moving"].cpu().numpy()
        self.G = eng.pool["dense_grad"].cpu().numpy()
        self.C = {s: int(eng.info[L.POOL_WORKSPACE][f"bn.{s}.stat"]["shape"][0]) for s in BN_SETS}
        self._ws = {}

    def par(self, name, grad=False):
        d = self.info[name]
        return (self.G if grad else self.P)[d["offset"]:d["offset"] + d["numel"]].astype(np.float64).reshape(d["shape"])

    def mov(self, name, after):
        d = self.bn_info[name]
        return (self.mov1 if after else self.mov0)[d["offset"]:d["offset"] + d["numel"]].astype(np.float64)

    def buf(self, name, rows, width):
        """rows x width leading block of a row-major workspace tensor (rows of a [B, T, .] tensor are its tokens)."""
        key = (name, rows, width)
        if key not in self._ws:
            self._ws[key] = self.eng.ws(name).reshape(-1)[:rows * width].view(rows, width).cpu().numpy().astype(np.float64)
        return self._ws[key]

    def stat(self, s):
        return self.eng.ws(f"bn.{s}.stat").cpu().numpy()

    def bsums(self, s):
        o = sum(self.C[k] for k in BN_SETS[:BN_SETS.index(s)])
        return self.eng.ws("bn.bsums").cpu().numpy()[o:o + self.C[s]]

    def bn_par(self, m, l, leaf):
        """gamma or beta of layer l's batch norm, all members side by side."""
        return np.concatenate([self.par(m.bn_scope(i, l) + "/" + leaf).reshape(-1) for i in range(len(m.scopes))])

    def act(self, m, l, z):
        """relu(bn(z)) of layer l (every member) on the engine's statistics: value, abs-sum of its terms, ReLU side, x-hat."""
        st = self.stat(m.bn[l])
        ga, be = self.bn_par(m, l, "gamma"), self.bn_par(m, l, "beta")
        on = _on(z, st, ga, be)
        xh = (z - st[:, 0].astype(np.float64)) * st[:, 1].astype(np.float64)
        return np.where(on, ga * xh + be, 0.0), np.where(on, np.abs(ga * xh) + np.abs(be), 0.0), on, xh


def _w(m, i, l):
    sc = m.scopes[i] + "/nn_part/"
    return sc + ("w_nn_layer0", "w_nn_layer1", "w_nn_output")[l], sc + ("b_nn_layer0", "b_nn_layer1", "b_nn_output")[l]


def _inputs(s, m, rows):
    """Per layer, the input of every member: (value, abs) lists; layer 0 reads its columns of x."""
    G = len(m.scopes)
    X = s.buf(m.x, rows, m.ldx)
    zs = [s.buf(m.z[l], rows, G * m.n_of(l)) for l in range(m.layers())]
    ins = [[(X[:, c:c + m.k], np.abs(X[:, c:c + m.k])) for c in m.x_col]]
    for l in range(1, m.layers()):
        a, a_abs, _, _ = s.act(m, l - 1, zs[l - 1])
        K = m.k_of(l)
        ins.append([(a[:, i * K:(i + 1) * K], a_abs[:, i * K:(i + 1) * K]) for i in range(G)])
    return zs, ins


def check_forward(ck, s, name, m, rows, training):
    """z of every layer from its input; the batch statistics (training) or the moving ones (scoring); the moving-average update."""
    G = len(m.scopes)
    zs, ins = _inputs(s, m, rows)
    for l in range(m.layers()):
        N = m.n_of(l)
        for i in range(G):
            wn, bn = _w(m, i, l)
            W, b = s.par(wn).reshape(m.k_of(l), N), s.par(bn)
            A, A_abs = ins[l][i]
            ck.close(f"{name}{i} z.{LAYER[l]}", zs[l][:, i * N:(i + 1) * N], A @ W + b, A_abs @ np.abs(W) + np.abs(b))
    for l in range(2):
        st, z = s.stat(m.bn[l]).astype(np.float64), zs[l]
        names = [m.bn_scope(i, l) + "/moving_" for i in range(G)]
        mm0, mv0 = (np.concatenate([s.mov(n + k, False) for n in names]) for k in ("mean", "variance"))
        mm1, mv1 = (np.concatenate([s.mov(n + k, True) for n in names]) for k in ("mean", "variance"))
        tag = f"{name} bn.{m.bn[l]}"
        if not training:
            inv = 1.0 / np.sqrt(mv0 + EPS)
            ck.close(f"{tag} eval mean", st[:, 0], mm0, np.abs(mm0), 0.0)
            ck.close(f"{tag} eval invstd", st[:, 1], inv, 3 * U * inv, 1.0)
            ck.close(f"{tag} moving unchanged", np.concatenate([mm1, mv1]), np.concatenate([mm0, mv0]), 0.0, 0.0)
            continue
        # biased batch statistics over the set's rows; the engine sums z and z^2 in fp64 (exact products of fp32 values, `rows`
        # roundings each) and takes E[z^2] - E[z]^2: the cancellation costs ~ rows * 2^-52 * E[z^2], the rest is one fp32 rounding
        n = float(rows)
        mean = z.sum(0) / n
        var = ((z - mean) ** 2).sum(0) / n
        ez, ez2 = np.abs(z).sum(0) / n, (z * z).sum(0) / n
        dvar = (n + 4) * 2.0 ** -52 * ez2 * 2
        inv = 1.0 / np.sqrt(var + EPS)
        ck.close(f"{tag} mean", st[:, 0], mean, 2 * U * ez, 1.0)
        ck.close(f"{tag} invstd", st[:, 1], inv, 2 * U * inv + 0.5 * inv ** 3 * dvar, 1.0)
        ck.close(f"{tag} moving_mean", mm1, mm0 - (mm0 - mean) * DECAY, 4 * U * (np.abs(mm0) + np.abs(mean)) + DECAY * 2 * U * ez, 1.0)
        ck.close(f"{tag} moving_variance", mv1, mv0 - (mv0 - var) * DECAY, 4 * U * (np.abs(mv0) + var) + DECAY * (2 * U * var + dvar), 1.0)


def check_backward(ck, s, name, m, rows, top, stores, dw_chain):
    """Walk one MLP from its top gradient down.  top: (value, abs) of the top layer's gradient over all members (the logits'
    gradient, or dA of layer 1 for an MLP without output layer).  stores[l]: what the engine's dz[l] buffer holds after the
    backward pass - "dA" (gradient of the post-BN-ReLU activation: the tile kernels form dz while loading), "dz" (head2's stage_dz
    overwrote it) or nothing.  dw_chain(l): serial terms of one dW / db element of layer l.  Returns dX, bound: [rows, ldx]."""
    G = len(m.scopes)
    zs, ins = _inputs(s, m, rows)
    cur, cur_abs = top
    for l in reversed(range(m.layers())):
        K, N = m.k_of(l), m.n_of(l)
        if l < 2:
            # batch-norm backward of layer l: dy = relu' dA;  S1 = sum dy, S2 = sum dy xhat;  dz = gamma inv (dy - S1/n - xhat S2/n)
            _, _, on, xh = s.act(m, l, zs[l])
            st = s.stat(m.bn[l]).astype(np.float64)
            ga = s.bn_par(m, l, "gamma")
            dy, dy_abs = np.where(on, cur, 0.0), np.where(on, cur_abs, 0.0)
            S1, S2 = dy.sum(0), (dy * xh).sum(0)
            S1a, S2a = dy_abs.sum(0), (dy_abs * np.abs(xh)).sum(0)
            bs = s.bsums(m.bn[l])
            tag = f"{name} bn.{m.bn[l]}"
            ck.close(f"{tag} S1", bs[:, 0], S1, S1a)
            ck.close(f"{tag} S2", bs[:, 1], S2, S2a)
            ck.close(f"{tag} dbeta", np.concatenate([s.par(m.bn_scope(i, l) + "/beta", True).reshape(-1) for i in range(G)]), S1, S1a)
            ck.close(f"{tag} dgamma", np.concatenate([s.par(m.bn_scope(i, l) + "/gamma", True).reshape(-1) for i in range(G)]), S2, S2a)
            n = float(rows)
            dz = ga * st[:, 1] * (dy - S1 / n - xh * S2 / n)
            dz_abs = np.abs(ga) * st[:, 1] * (dy_abs + S1a / n + np.abs(xh) * S2a / n)
            if stores.get(l) == "dz":
                e = s.buf(m.dz[l], rows, G * N)
                ck.close(f"{name} dz.{LAYER[l]}", e, dz, dz_abs)
                dz, dz_abs = e, np.abs(e)
        else:
            dz, dz_abs = cur, cur_abs
        rel = rel_chain(dw_chain(l))
        dA = np.zeros((rows, G * K)) if l else np.zeros((rows, m.ldx))
        dA_abs = np.zeros_like(dA)
        for i in range(G):
            wn, bn = _w(m, i, l)
            W = s.par(wn).reshape(K, N)
            A, A_abs = ins[l][i]
            g, g_abs = dz[:, i * N:(i + 1) * N], dz_abs[:, i * N:(i + 1) * N]
            ck.close(f"{name}{i} dW.{LAYER[l]}", s.par(wn, True).reshape(K, N), A.T @ g, A_abs.T @ g_abs, rel)
            ck.close(f"{name}{i} db.{LAYER[l]}", s.par(bn, True), g.sum(0), g_abs.sum(0), rel)
            c = i * K if l else m.x_col[i]
            dA[:, c:c + K] += g @ W.T
            dA_abs[:, c:c + K] += g_abs @ np.abs(W).T
        if l == 0:
            return dA, dA_abs
        cur, cur_abs = dA, dA_abs
        if stores.get(l - 1) == "dA":
            e = s.buf(m.dz[l - 1], rows, G * K)
            ck.close(f"{name} dA.{LAYER[l - 1]}", e, cur, cur_abs)
            cur, cur_abs = e, np.abs(e)


def mix_backward(s, mlps, B, E, sel, du, du_abs):
    """The MMoE / PLE mixing backward (kernels_head.cu:k_combine_bwd, kernels_sibling.cu:k_sib_mix_bwd) from d_u:
    main = sum_j gate_main[j] expert_sel[0][j], sub likewise; u = main | target | sub | target.  Returns dA of experts
    layer 1, dA of gates layer 1 (value, abs) and d_tgt."""
    ex, gt = mlps["expert"], mlps["gate"]
    nE, TI = len(ex.scopes), 64 + E
    e, e_abs, _, _ = s.act(ex, 1, s.buf(ex.z[1], B, 64 * nE))
    g, g_abs, _, _ = s.act(gt, 1, s.buf(gt.z[1], B, 10))
    d_out = [du[:, :64], du[:, TI:TI + 64]]
    d_abs = [du_abs[:, :64], du_abs[:, TI:TI + 64]]
    dE, dE_abs = np.zeros((B, 64 * nE)), np.zeros((B, 64 * nE))
    dG, dG_abs = np.zeros((B, 10)), np.zeros((B, 10))
    for k in range(2):
        for j in range(5):
            x = sel[k][j]
            sl = slice(64 * x, 64 * x + 64)
            dE[:, sl] += g[:, 5 * k + j:5 * k + j + 1] * d_out[k]
            dE_abs[:, sl] += g_abs[:, 5 * k + j:5 * k + j + 1] * d_abs[k]
            dG[:, 5 * k + j] = (e[:, sl] * d_out[k]).sum(1)
            dG_abs[:, 5 * k + j] = (e_abs[:, sl] * d_abs[k]).sum(1)
    d_tgt = du[:, 64:TI] + du[:, TI + 64:]
    return (dE, dE_abs), (dG, dG_abs), (d_tgt, du_abs[:, 64:TI] + du_abs[:, TI + 64:])


def pool_backward(aw, mask, H, d_out, d_out_abs, aw_rel=0.0):
    """Softmax-weighted pooling backward (k_pool_bwd, k_sib_pool_bwd): out = sum_t aw_t h_t  ->  the gradient of the masked logit
    s_t = mask ? aw_t (v_t - sum aw v) : 0, v_t = d_out . h_t.  aw_rel: relative error of weights the engine recomputed itself."""
    v = np.einsum("bte,be->bt", H, d_out)
    v_abs = np.einsum("bte,be->bt", np.abs(H), d_out_abs)
    dot, dot_abs = (aw * v).sum(1, keepdims=True), (aw * v_abs).sum(1, keepdims=True)
    ds = np.where(mask == 1, aw * (v - dot), 0.0)
    bound = np.where(mask == 1, aw * (v_abs + dot_abs) + aw_rel / REL * aw * (np.abs(v) + np.abs(dot)), 0.0)
    return ds, bound


# ================================================================================================ PAMRec
NU, NI, NC = 200, 2000, 40


def _workers():
    return max(torch.cuda.get_device_properties(0).multi_processor_count - 1, 1)


def _pamrec(T, B, legacy, monkeypatch, max_batch=None, graph=False):
    from pamrec_b200.engine import Engine
    if legacy:
        monkeypatch.setenv("PAMREC_HEAD_LEGACY", "1")
    else:
        monkeypatch.delenv("PAMREC_HEAD_LEGACY", raising=False)
    om = O.OracleModel(NU, NI, NC, T, seed=11)
    O.perturb_params(om.params, om.bn_state, seed=12)
    eng = Engine(NU, NI, NC, T, max_batch or B, graph=graph).allocate()
    eng.set_variables({n: t.numpy() for n, t in om.params.items()})
    eng.set_variables({n: t.numpy() for n, t in om.bn_state.items()})
    return eng


def _far_mean(eng, db, chans, rows_of):
    """Move one channel per listed layer to |mean| / std ~ 1e3 through its bias (measured on a training forward of db)."""
    eng.forward(db, training=True, want_pred=False)
    torch.cuda.synchronize()
    for zbuf, width, col, bias in chans:
        z = eng.ws(zbuf).reshape(-1)[:rows_of(zbuf) * width].view(-1, width)[:, col].double()
        b = eng.dense(bias)
        b[col] += float(1e3 * z.std(unbiased=False) - z.mean())


def check_pamrec(eng, P, mov0, B, T, head2, mask, training=True, tag=""):
    s = Step(eng, P, mov0, B, T)
    ck = Check(f"pamrec {'head2' if head2 else 'stand-alone'} B={B} T={T}{tag}")
    M, N = HEAD_MLPS, B * T
    rows = {"score": N, "expert": B, "gate": B, "tower": B}
    for k, m in M.items():
        check_forward(ck, s, k, m, rows[k], training)
    if not training:
        return ck.done()
    W = _workers()
    if head2:
        # k_head2_dw: row splits of ceil(B / 256), at most 64; the score MLP's dW0 sums a CTA's tokens in fp32 (kernels_head2.cu:K7)
        splits = min(64, -(-B // 256))
        chain = lambda k, l: (-(-B // W) * T + W) if k == "score" else (-(-B // splits) + splits)
    else:
        chain = lambda k, l: tiles_dw_chain(rows[k], len(M[k].scopes), M[k].k_of(l), M[k].n_of(l))
    st = {} if head2 else {0: "dA", 1: "dA"}
    st_top = {0: "dz", 1: "dz"} if head2 else st
    dlog = s.buf("d_logits", B, 3)
    du, du_abs = check_backward(ck, s, "tower", M["tower"], B, (dlog, np.abs(dlog)), st_top, lambda l: chain("tower", l))
    if not head2:                                             # head2 keeps d_u in shared memory
        e = s.buf("d_u", B, 168)
        ck.close("d_u", e, du, du_abs, rel_chain(dx_chain(M["tower"])))
        du, du_abs = e, np.abs(e)
    dE, dG, dT = mix_backward(s, M, B, 20, (tuple(range(5)), tuple(range(5))), du, du_abs)
    ck.close("d_tgt", s.buf("d_tgt", B, 20), *dT)
    if not head2:
        for mm, d in (("expert", dE), ("gate", dG)):
            e = s.buf(M[mm].dz[1], B, d[0].shape[1])
            ck.close(f"{mm} dA.layer1", e, *d)
    topE = dE if head2 else (s.buf("d_e1", B, 320), np.abs(s.buf("d_e1", B, 320)))
    topG = dG if head2 else (s.buf("d_g1", B, 10), np.abs(s.buf("d_g1", B, 10)))
    dx1 = check_backward(ck, s, "expert", M["expert"], B, topE, st_top, lambda l: chain("expert", l))
    dx2 = check_backward(ck, s, "gate", M["gate"], B, topG, st_top, lambda l: chain("gate", l))
    dnl = s.buf("d_new_long", B, 40)
    # head2 splits its 628-long contraction over 12 groups of 53 (kernels_head2.cu:K5)
    ck.close("d_new_long", dnl, dx1[0] + dx2[0], dx1[1] + dx2[1], rel_chain(53 + 12 if head2 else dx_chain(M["expert"], M["gate"])))
    # attention pooling (pamrec.py:272-282): aw = softmax_t(mask ? relu(bn(z2)) : -(2^32)+1), recomputed here in float64
    sc = M["score"]
    sv, _, _, _ = s.act(sc, 1, s.buf("z2", N, 1))
    logit = np.where(mask == 1, sv.reshape(B, T), MASK_NEG)
    aw = np.exp(logit - logit.max(1, keepdims=True))
    aw /= aw.sum(1, keepdims=True)
    smax = float(np.abs(np.where(mask == 1, sv.reshape(B, T), 0.0)).max())
    H = s.buf("blk1.out", N, 40).reshape(B, T, 40)
    ds, ds_abs = pool_backward(aw, mask, H, dnl, np.abs(dnl), aw_rel=(2 * smax + 8) * U)
    e = s.buf("d_z2", N, 1)
    ck.close("d_z2 (dA of the score)", e, ds.reshape(N, 1), ds_abs.reshape(N, 1))
    e = (e, np.abs(e))
    chain_s = (lambda l: (-(-B // W) * T + W) if l == 0 else W) if head2 else (lambda l: chain("score", l))
    dx, dx_abs = check_backward(ck, s, "score", sc, N, e, {} if head2 else {0: "dA"}, chain_s)
    share = (aw[:, :, None] * dnl[:, None, :]).reshape(N, 40)
    share_abs = (aw[:, :, None] * np.abs(dnl)[:, None, :]).reshape(N, 40)
    # g_a is the encoder's ping-pong buffer: block 1's backward keeps the head's copy in blk1.d_out (api.cu:pamrec_backward)
    ck.close("g_a (score dX + pooling)", s.buf("blk1.d_out", N, 40), dx + share, dx_abs + share_abs)
    ck.done()




def _pamrec_step(eng, batch, B, T, head2, tag=""):
    """One forward + backward on `batch`, then every check; returns the device batch."""
    db = eng.upload(batch)
    P, mov0 = eng.pool["dense_param"].clone(), eng.pool["bn_moving"].clone()
    eng.forward(db, training=True, want_pred=False)
    eng.backward(db)
    torch.cuda.synchronize()
    check_pamrec(eng, P, mov0, B, T, head2, np.asarray(batch["mask"]), tag=tag)
    return db


def _pamrec_score(eng, B, T, head2, seed=9):
    batch = O.make_batch(seed, B, T, NU, NI, NC, grouped=False)
    db = eng.upload(batch, training=False)
    mov0 = eng.pool["bn_moving"].clone()
    eng.forward(db, training=False, want_pred=True)
    torch.cuda.synchronize()
    check_pamrec(eng, eng.pool["dense_param"].clone(), mov0, B, T, head2, np.asarray(batch["mask"]), training=False, tag=" scoring")


def _head2_shapes():
    """(T, B, max_batch) where the row-stationary head's paths change; the grid is one CTA per SM, CTA 0 owns no rows, a worker
    owns ceil(B / workers) rows in chunks of 8.  Training batches are multiples of 5 (the listwise groups)."""
    w = _workers()
    b8 = 5 * (8 * w // 5)                  # one chunk of at most 8 rows per worker
    return [
        (12, 5, None),                     # B < workers: idle CTAs; k_head2_dw: one round of 5 rows
        (12, 150, None),                   # 2 rows per worker: the last workers own none; 24 tokens per CTA (not a multiple of 25)
        (1, 20, None),                     # T = 1
        (4, b8, None),                     # exactly one chunk per worker
        (4, b8 + 5, 2 * b8),               # a second, partial chunk; max_batch > B
        (3, 60, None), (3, 65, None),      # k_head2_dw: staging rounds of 64 rows
        (3, 255, None), (3, 260, None),    # one split of 255 rows / two splits
        (50, 1025, None),                  # the takatak bench shape: 51 250 score tokens
        (2, 20000, None),                  # 79 splits capped at 64: 313 rows per split
    ]


def _ids(shapes):
    return [f"T{t}-B{b}" + (f"-cap{c}" if c else "") for t, b, c in shapes]


HEAD2_IDS = ["B-below-workers", "last-workers-idle", "T1", "one-chunk", "partial-chunk-cap", "dw60", "dw65", "dw255", "dw260",
             "b1025-t50", "b20000-splits-capped"]


@pytest.mark.parametrize("i", range(len(HEAD2_IDS)), ids=HEAD2_IDS)
def test_pamrec_head2_layers(i, monkeypatch):
    """The row-stationary head at the shapes where its row ownership, staging rounds, row splits and token passes change (read
    from the device's SM count: the ids show the shapes of a 148-SM B200)."""
    T, B, cap = _head2_shapes()[i]
    eng = _pamrec(T, B, False, monkeypatch, max_batch=cap)
    _pamrec_step(eng, O.make_batch(5, B, T, NU, NI, NC), B, T, True)
    eng.close()


LEGACY_SHAPES = [(12, 5, None), (12, 35, None), (1, 30, None), (7, 40, 100), (50, 1025, None)]


@pytest.mark.parametrize("T,B,cap", LEGACY_SHAPES, ids=_ids(LEGACY_SHAPES))
def test_pamrec_standalone_layers(T, B, cap, monkeypatch):
    """The stand-alone head (tile kernels): M = B rows below, at and above a 32-row tile (5, 35; 30 at T = 1, where the score MLP
    has 30 rows too), B * T = 280 score rows, and 51 250 score rows over several row chunks per CTA."""
    eng = _pamrec(T, B, True, monkeypatch, max_batch=cap)
    _pamrec_step(eng, O.make_batch(5, B, T, NU, NI, NC), B, T, False)
    eng.close()


@pytest.mark.parametrize("legacy", [False, True], ids=["head2", "standalone"])
def test_pamrec_two_steps_far_mean_and_scoring(legacy, monkeypatch):
    """Two steps in one engine, the second on fewer rows (the batch-norm sums, their 8 copies in head2, bn.bsums and the
    gamma / beta gradients start from zero every step); one channel of the towers' and of the score MLP's first layer at
    |mean| / std ~ 1e3 (the variance against cancellation); then scoring at B = 1 and B = 150 against the moving statistics."""
    T = 10
    eng = _pamrec(T, 400, legacy, monkeypatch)
    first = O.make_batch(5, 400, T, NU, NI, NC)
    db = eng.upload(first)
    _far_mean(eng, db, [("zt0", 300, 3, "sequential/logit_fcn/nn_part/b_nn_layer0"),
                        ("z1", 20, 2, "sequential/pamrec/new_long/score_1/nn_part/b_nn_layer0")],
              lambda n: 400 * T if n == "z1" else 400)
    _pamrec_step(eng, first, 400, T, not legacy, tag=" far mean")
    _pamrec_step(eng, O.make_batch(6, 145, T, NU, NI, NC), 145, T, not legacy, tag=" second step")
    for B in (1, 150):
        _pamrec_score(eng, B, T, not legacy)
    eng.close()


def test_pamrec_head2_graph_replay(monkeypatch):
    """Steps replayed from a CUDA graph, alternating two batches: each step's head reads and writes that step's tensors."""
    T, B = 20, 300
    eng = _pamrec(T, B, False, monkeypatch, graph=True)
    batches = [O.make_batch(40 + i, B, T, NU, NI, NC) for i in range(2)]
    dbs = [eng.upload(b) for b in batches]
    for step in range(6):                  # steps 3 and 4 are captured, 5 is a plain replay (test_gpu_encoder_wgrad)
        P, mov0 = eng.pool["dense_param"].clone(), eng.pool["bn_moving"].clone()
        eng.train_step(dbs[step % 2])
        torch.cuda.synchronize()
        if step >= 3:
            check_pamrec(eng, P, mov0, B, T, True, np.asarray(batches[step % 2]["mask"]), tag=f" replay step {step}")
    assert len(eng._graphs) == 2
    eng.close()


# ================================================================================================ siblings, SASRec
SIB_NU, SIB_NI, SIB_NC = 50, 300, 20
SIB_DIMS = {16: (16, 4, 20), 32: (32, 8, 40)}
SAS_DIMS = {16: (16, 4, 20), 32: (32, 8, 16)}


def _sibling(model, T, B, dims):
    from pamrec_b200.engine import Engine
    om = D.SiblingOracleModel(model, SIB_NU, SIB_NI, SIB_NC, T, seed=11, dims=dims)
    O.perturb_params(om.params, om.bn_state, seed=12)
    eng = Engine(SIB_NU, SIB_NI, SIB_NC, T, B, model=model, emb_dims=dims).allocate()
    eng.set_variables({n: t.numpy() for n, t in om.params.items()})
    eng.set_variables({n: t.numpy() for n, t in om.bn_state.items()})
    return eng


def _sib_batch(seed, B, T):
    return S.add_satisfied_fields(O.make_batch(seed, B, T, SIB_NU, SIB_NI, SIB_NC, grouped=False), seed=seed + 1)


def check_sibling(eng, model, P, mov0, B, T, batch, training=True, tag=""):
    E = sum(eng.emb_dims[:2])
    s = Step(eng, P, mov0, B, T)
    ck = Check(f"{model} E={E} B={B} T={T}{tag}")
    M = sas_mlps(E) if model == "sasrec" else sibling_mlps(model, E)
    N = B * T
    rows = {k: (N if m.tokens else B) for k, m in M.items()}
    for k, m in M.items():
        check_forward(ck, s, k, m, rows[k], training)
    if not training:
        return ck.done()
    st = {0: "dA", 1: "dA"}

    def chain(k):
        m = M[k]
        return lambda l: tiles_dw_chain(rows[k], len(m.scopes), m.k_of(l), m.n_of(l))

    tw = M["tower"]
    dlog = s.buf("d_logits", B, len(tw.scopes))
    dx, dx_abs = check_backward(ck, s, "tower", tw, B, (dlog, np.abs(dlog)), st, chain("tower"))
    e = s.buf(tw.dx, B, tw.ldx)
    if model == "sasrec":
        ck.close("d_u", e, dx, dx_abs, rel_chain(dx_chain(tw)))
        return ck.done()
    if "expert" in M:
        ck.close("d_u", e, dx, dx_abs, rel_chain(dx_chain(tw)))
        du = e
        sel = PLE_SEL if model == "ple" else (tuple(range(5)), tuple(range(5)))
        dE, dG, dT = mix_backward(s, M, B, E, sel, du, np.abs(du))
        ck.close("d_tgt", s.buf("d_tgt", B, E), *dT)
        tops = {}
        for mm, d in (("expert", dE), ("gate", dG)):
            e = s.buf(M[mm].dz[1], B, d[0].shape[1])
            ck.close(f"{mm} dA.layer1", e, *d)
            tops[mm] = (e, np.abs(e))
        d1 = check_backward(ck, s, "expert", M["expert"], B, tops["expert"], st, chain("expert"))
        d2 = check_backward(ck, s, "gate", M["gate"], B, tops["gate"], st, chain("gate"))
        dx, dx_abs = d1[0] + d2[0], d1[1] + d2[1]
    dxe = s.buf("d_x", B, 3 * E)
    ck.close("d_x", dxe, dx, dx_abs, rel_chain(dx_chain(M["expert"], M["gate"]) if "expert" in M else dx_chain(tw)))
    # DIN pooling of both branches (mmoe.py:330-337) on the engine's saved weights: the attention logits' gradient
    aw = s.buf("sib.aw", 2 * N, 1).reshape(2, B, T)
    h = s.buf("sib.h", 2 * N, E).reshape(2, B, T, E)
    dsc, dsc_abs = np.zeros((N, 2)), np.zeros((N, 2))
    for r, mk in enumerate((batch["satisfied_mask"], batch["mask"])):
        d_out = dxe[:, r * E:(r + 1) * E]
        v, b = pool_backward(aw[r], np.asarray(mk), h[r], d_out, np.abs(d_out))
        dsc[:, r], dsc_abs[:, r] = v.reshape(-1), b.reshape(-1)
    e = s.buf("sib.d_score", N, 2)
    ck.close("sib.d_score", e, dsc, dsc_abs)
    att = M["att"]
    df, df_abs = check_backward(ck, s, "att", att, N, (e, np.abs(e)), st, chain("att"))
    ck.close("sib.d_feat", s.buf("sib.d_feat", N, 8 * E), df, df_abs)
    # attention_mat (bias-free) of each branch: dA = h^T d_att over the branch's N rows, on k_dense_dw
    d_att = s.buf("sib.d_att", 2 * N, E).reshape(2, N, E)
    rel = rel_chain(tiles_dw_chain(N, 1, E, E))
    for r, br in enumerate(("long_term", "short_term")):
        hr = h[r].reshape(N, E)
        ck.close(f"{br} attention_mat dW", s.par(f"sequential/clsr/{br}/attention_fcn/attention_mat", True), hr.T @ d_att[r],
                 np.abs(hr).T @ np.abs(d_att[r]), rel)
    ck.done()


def _sib_step(eng, model, B, T, seed=5, tag=""):
    batch = _sib_batch(seed, B, T)
    db = eng.upload(batch)
    P, mov0 = eng.pool["dense_param"].clone(), eng.pool["bn_moving"].clone()
    eng.forward(db, training=True, want_pred=False)
    eng.backward(db)
    torch.cuda.synchronize()
    check_sibling(eng, model, P, mov0, B, T, batch, tag=tag)


SIB_SHAPES = [(1, 4), (31, 3), (32, 1), (33, 12), (300, 20)]


@pytest.mark.parametrize("B,T", SIB_SHAPES, ids=[f"B{b}-T{t}" for b, t in SIB_SHAPES])
@pytest.mark.parametrize("width", [16, 32], ids=["e20", "e40"])
@pytest.mark.parametrize("model", ["mmoe", "ple", "sharebottom"])
def test_sibling_layers(model, width, B, T):
    """MMoE, PLE and share-bottom at (16, 4) and at the reference's (32, 8, 40), where att_fcn layer 0 contracts over K = 160 >
    kKMax and the towers over K = 104 = kKMax: B = 1 (variance 0, x-hat 0, dz 0), rows around a 32-row tile, and 6 000 tokens."""
    eng = _sibling(model, T, B, SIB_DIMS[width])
    _sib_step(eng, model, B, T)
    eng.close()


@pytest.mark.parametrize("width", [16, 32], ids=["e20", "e40"])
@pytest.mark.parametrize("model", ["mmoe", "ple", "sharebottom"])
def test_sibling_two_steps_and_scoring(model, width):
    """A second step on fewer rows, with one attention-MLP and one tower channel at |mean| / std ~ 1e3; scoring on the moving
    statistics."""
    T = 8
    eng = _sibling(model, T, 120, SIB_DIMS[width])
    E = sum(SIB_DIMS[width][:2])
    _sib_step(eng, model, 120, T, seed=5)
    db = eng.upload(_sib_batch(6, 70, T))
    _far_mean(eng, db, [("zt0", 200, 3, "sequential/logit_fcn/nn_part/b_nn_layer0"),
                        ("z1", 160, 2, "sequential/clsr/long_term/attention_fcn/att_fcn/nn_part/b_nn_layer0")],
              lambda n: 70 * T if n == "z1" else 70)
    _sib_step(eng, model, 70, T, seed=6, tag=" second step, far mean")
    batch = _sib_batch(7, 9, T)
    db = eng.upload(batch, training=False)
    mov0 = eng.pool["bn_moving"].clone()
    eng.forward(db, training=False, want_pred=True)
    torch.cuda.synchronize()
    check_sibling(eng, model, eng.pool["dense_param"].clone(), mov0, 9, T, batch, training=False, tag=" scoring")
    eng.close()
    assert E in (20, 40)


SAS_SHAPES = [(1, 5), (33, 7), (500, 10)]


@pytest.mark.parametrize("B,T", SAS_SHAPES, ids=[f"B{b}-T{t}" for b, t in SAS_SHAPES])
@pytest.mark.parametrize("width", [16, 32], ids=["e20", "e40"])
def test_sasrec_tower_layers(width, B, T):
    """SASRec's tower on final state | target (K = 40 or 80), then scoring on the moving statistics."""
    eng = _sibling("sasrec", T, B, SAS_DIMS[width])
    _sib_step(eng, "sasrec", B, T)
    batch = _sib_batch(7, B, T)
    db = eng.upload(batch, training=False)
    mov0 = eng.pool["bn_moving"].clone()
    eng.forward(db, training=False, want_pred=True)
    torch.cuda.synchronize()
    check_sibling(eng, "sasrec", eng.pool["dense_param"].clone(), mov0, B, T, batch, training=False, tag=" scoring")
    eng.close()
