"""The encoder's weight gradients (kernels_encoder.cu: k_enc_dw on the side stream, the LayerNorm column sums in k_ffn_bwd /
k_proj_bwd) against fp64 products of the engine's own saved tensors: qin, the block inputs, dQ / dK / dV, y, dOUT and the
engine's ReLU pattern.  Each launch of k_enc_dw (the two FFN products, or bucket x {q, k, v}) lays its products end to end and
cuts that list into equal ranges of at least 256 tokens, so the shapes below put run and tile boundaries inside, at and next to buckets:
buckets of 1 / 64 / 65 / 255 / 256 / 257 tokens, every token in one bucket, the zero bin (bucket 10), token counts that are
not a multiple of the run, T = 1, a grid of whole SM waves, and two CUDA-graph replayed steps on two batches in turn."""
import numpy as np
import pytest
import torch

from oracle import pamrec_oracle as O

pytestmark = pytest.mark.gpu

BLK = "sequential/pamrec/num_blocks_{}/"


def _engine(nu, ni, nc, T, B, graph=False):
    from pamrec_b200.engine import Engine
    om = O.OracleModel(nu, ni, nc, T, seed=11)
    O.perturb_params(om.params, om.bn_state, seed=12)
    eng = Engine(nu, ni, nc, T, B, graph=graph).allocate()
    eng.set_variables({n: t.numpy() for n, t in om.params.items()})
    eng.set_variables({n: t.numpy() for n, t in om.bn_state.items()})
    return eng


def _layout(layout, B, T, rng):
    n = B * T
    if layout == "random":
        lt = rng.uniform(0, 10, n)
    elif layout == "all4":
        lt = np.full(n, 4.0)
    elif layout == "sizes":
        # around the 64-token tile and the 256-token run; the remaining tokens spread over buckets 6..9
        sizes = {0: 1, 1: 64, 2: 65, 3: 255, 4: 256, 5: 257}
        rest = n - sum(sizes.values())
        lt = np.concatenate([np.repeat(list(sizes), list(sizes.values())), rng.integers(6, 10, rest)]).astype(np.float64)
        lt = rng.permutation(lt)
    else:                                   # "bucket10": a third of the tokens in the zero bin
        lt = rng.integers(0, 10, n).astype(np.float64)
        lt[rng.random(n) < 0.3] = 10.0
    return lt.reshape(B, T).astype(np.float32)


def _ln(x):
    mu = x.mean(-1, keepdims=True)
    rstd = 1.0 / np.sqrt(((x - mu) ** 2).mean(-1, keepdims=True) + 1e-8)
    return (x - mu) * rstd, rstd


def _check(eng, P, buckets, relu, B):
    """Every encoder weight gradient and both LayerNorm pairs of the last backward pass against fp64 products; P: the dense
    parameters that step ran with, relu: {block: bool [B, T, 40]}, buckets: [B * T] table rows (10 = zero bin)."""
    from pamrec_b200 import _lib as L
    info = eng.info[L.POOL_DENSE]

    def par(name):
        d = info[name]
        return P[d["offset"]:d["offset"] + d["numel"]].view(d["shape"]).cpu().numpy().astype(np.float64)

    def ws(name):
        return eng.ws(name, B).cpu().numpy().astype(np.float64).reshape(-1, 40)

    def grad(name):
        return eng.dense(name, "dense_grad").cpu().numpy().astype(np.float64)

    bad, rep = [], []

    # The bounds are the same products over absolute values, intermediate ones included: the engine's h and dH o relu' are fp32
    # results of 40-term sums that may cancel, so their rounding scales with |f| |W1| and |dOUT| |W2|, not with h or dH.
    def close(name, got, ref, bound, rel):
        got = got.reshape(ref.shape)
        err = np.abs(got - ref)
        worst = float((err / np.maximum(bound, 1e-30)).max())
        rep.append(f"{name} {worst:.2e}")
        if not (np.isfinite(got).all() and (err <= rel * bound + 1e-30).all()):
            bad.append(f"{name}: max err / bound {worst:.3e} > {rel:.0e}")

    for k in range(2):
        p = BLK.format(k)
        x = ws("x0" if k == 0 else "blk0.out")
        qin, y = ws(f"blk{k}.qin"), ws(f"blk{k}.y")
        dQ, dK, dV = (ws(n if k == 0 else "blk1." + n) for n in ("d_Q", "d_K", "d_V"))
        dout = ws("g_b" if k == 0 else "blk1.d_out")
        on = relu[k].reshape(-1, 40)
        W1, b1 = par(p + "multihead_attention/conv1d/kernel").reshape(40, 40), par(p + "multihead_attention/conv1d/bias")
        W2 = par(p + "multihead_attention/conv1d_1/kernel").reshape(40, 40)
        # ---- FFN: h = relu(f W1 + b1) on the engine's pattern, dH o relu'
        fh, rs_b = _ln(y)
        f = par(p + "ln_1/Variable_1") * fh + par(p + "ln_1/Variable")
        h = np.where(on, f @ W1 + b1, 0.0)
        dhr = np.where(on, dout @ W2.T, 0.0)
        h_abs = np.where(on, np.abs(f) @ np.abs(W1) + np.abs(b1), 0.0)
        dhr_abs = np.where(on, np.abs(dout) @ np.abs(W2).T, 0.0)
        close(f"blk{k} dW1", grad(p + "multihead_attention/conv1d/kernel"), f.T @ dhr, np.abs(f).T @ dhr_abs, 2e-5)
        close(f"blk{k} db1", grad(p + "multihead_attention/conv1d/bias"), dhr.sum(0), dhr_abs.sum(0), 2e-5)
        close(f"blk{k} dW2", grad(p + "multihead_attention/conv1d_1/kernel"), h.T @ dout, h_abs.T @ np.abs(dout), 2e-5)
        close(f"blk{k} db2", grad(p + "multihead_attention/conv1d_1/bias"), dout.sum(0), np.abs(dout).sum(0), 2e-5)
        # ---- LN_b: dF = dOUT + (dH o relu') W1^T, then dY through the LayerNorm
        dF = dout + dhr @ W1.T
        dF_abs = np.abs(dout) + dhr_abs @ np.abs(W1).T
        close(f"blk{k} ln_b dbeta", grad(p + "ln_1/Variable"), dF.sum(0), dF_abs.sum(0), 1e-4)
        close(f"blk{k} ln_b dgamma", grad(p + "ln_1/Variable_1"), (dF * fh).sum(0), (dF_abs * np.abs(fh)).sum(0), 1e-4)
        g_b = par(p + "ln_1/Variable_1")
        e, e_abs = dF * g_b, dF_abs * np.abs(g_b)
        dY = rs_b * (e - e.mean(-1, keepdims=True) - fh * (e * fh).mean(-1, keepdims=True))
        dY_abs = rs_b * (e_abs + e_abs.mean(-1, keepdims=True) + np.abs(fh) * (e_abs * np.abs(fh)).mean(-1, keepdims=True))
        # ---- time-aware projection per bucket; the zero bin has a zero matrix and adds nothing
        Wq = par(p + "self_attention/Q_timeaware_embedding").reshape(10, 40, 40)
        dqin, dqin_abs = dY.copy(), dY_abs.copy()
        for nm, A, G in (("Q", qin, dQ), ("K", x, dK), ("V", x, dV)):
            got = grad(p + f"self_attention/{nm}_timeaware_embedding").reshape(10, 40, 40)
            ref, bound = np.zeros((10, 40, 40)), np.zeros((10, 40, 40))
            for b in range(10):
                sel = buckets == b
                ref[b], bound[b] = A[sel].T @ G[sel], np.abs(A[sel]).T @ np.abs(G[sel])
                if nm == "Q":
                    dqin[sel] += dQ[sel] @ Wq[b].T
                    dqin_abs[sel] += np.abs(dQ[sel]) @ np.abs(Wq[b]).T
            close(f"blk{k} dW{nm.lower()}", got, ref, bound, 2e-5)
        xh, _ = _ln(x)
        close(f"blk{k} ln_a dbeta", grad(p + "ln/Variable"), dqin.sum(0), dqin_abs.sum(0), 1e-4)
        close(f"blk{k} ln_a dgamma", grad(p + "ln/Variable_1"), (dqin * xh).sum(0), (dqin_abs * np.abs(xh)).sum(0), 1e-4)
    print("\nmax err / abs-sum bound: " + ", ".join(rep))
    assert not bad, "; ".join(bad)


CASES = [
    # layout, B, T: 2560 tokens are runs of exactly 256: 20 for the two FFN products, 30 for the three projection ones
    pytest.param("sizes", 40, 64, id="sizes-1-64-65-255-256-257"),
    pytest.param("all4", 40, 64, id="one-bucket"),
    pytest.param("bucket10", 40, 64, id="bucket10"),
    pytest.param("random", 15, 43, id="n645"),
    pytest.param("random", 20, 1, id="T1"),
    pytest.param("bucket10", 1025, 50, id="b1025-t50"),
]


@pytest.mark.parametrize("layout,B,T", CASES)
def test_encoder_weight_gradients(layout, B, T):
    from pamrec_b200 import _lib as L
    nu, ni, nc = 200, 2000, 40
    eng = _engine(nu, ni, nc, T, B)
    batch = O.make_batch(5, B, T, nu, ni, nc)
    batch["item_loop_times_history"] = _layout(layout, B, T, np.random.default_rng(7))
    buckets = O.bucket_ids(batch["item_loop_times_history"]).numpy().reshape(-1)
    db = eng.upload(batch)
    eng.set_debug(L.DEBUG_SAVE_FFN_HIDDEN)
    eng.forward(db, training=True, want_pred=False)
    relu = [eng.ws(n, B).cpu().numpy() > 0 for n in ("d_Q", "d_K")]       # the forward's hidden activations (tests/relu_masks.py)
    eng.set_debug(0)
    P = eng.pool["dense_param"].clone()
    eng.forward(db, training=True, want_pred=False)
    eng.backward(db)
    torch.cuda.synchronize()
    for k in range(2):                                                    # the backward's recomputed h has the forward's signs
        assert np.array_equal(eng.ws(f"blk{k}.h", B).cpu().numpy() > 0, relu[k]), f"blk{k}: ReLU pattern differs"
    _check(eng, P, buckets, relu, B)
    eng.close()


def test_encoder_weight_gradients_graph_replay():
    """Steps replayed from a CUDA graph, alternating two batches: the side-stream weight gradients of each step read that step's
    tensors (the ReLU pattern comes from the backward's saved h, which the test above ties to the forward's)."""
    nu, ni, nc, T, B = 300, 3000, 50, 50, 100
    eng = _engine(nu, ni, nc, T, B, graph=True)
    batches = [O.make_batch(40 + i, B, T, nu, ni, nc) for i in range(2)]
    dbs = [eng.upload(b) for b in batches]
    # a batch's first step seeds the device step counter or counts as its first use; its second use is captured and replayed:
    # steps 3 (second batch) and 4 (first batch) are captured, 5 is a plain replay
    for step in range(6):
        P = eng.pool["dense_param"].clone()
        eng.train_step(dbs[step % 2])
        torch.cuda.synchronize()
        if step >= 3:
            buckets = O.bucket_ids(batches[step % 2]["item_loop_times_history"]).numpy().reshape(-1)
            relu = [eng.ws(f"blk{k}.h", B).cpu().numpy() > 0 for k in range(2)]
            _check(eng, P, buckets, relu, B)
    assert len(eng._graphs) == 2
    eng.close()
