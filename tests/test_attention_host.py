"""Host side of the attention read-out (no GPU): the entry order of explain(), its line format, its argument checks, and the argument
checks of pamrec_attention / Engine.attention."""
import ctypes as C
import types

import numpy as np
import pytest

from pamrec_b200 import deeprec_utils as DU


def _literal_topk(w, live, k):
    """The order restated with Python's sort over (-weight, position) tuples of the live positions."""
    out = []
    for r in range(w.shape[0]):
        rows = sorted((-float(w[r, t]), t) for t in range(w.shape[1]) if live[r, t])[:k]
        out.append([t for _, t in rows] + [-1] * (k - len(rows)))
    return np.asarray(out)


def test_attention_topk_matches_a_literal_restatement():
    rng = np.random.default_rng(5)
    T = 12
    w = (rng.integers(0, 4, size=(7, T)) / 8).astype(np.float32)          # many ties
    live = rng.random((7, T)) > 0.35
    live[0] = False                                                        # a line without history
    live[1] = True
    w[2, ~live[2]] = 1.0                                                   # dead positions never enter, whatever their weight
    for k in (1, 3, T):
        pos, got = DU.attention_topk(w, live, k)
        want = _literal_topk(w, live, k)
        np.testing.assert_array_equal(pos, want)
        np.testing.assert_array_equal(got, np.where(want >= 0, np.take_along_axis(w, np.maximum(want, 0), 1), 0.0))
    assert (DU.attention_topk(w, live, 4)[0][0] == -1).all()


def test_attention_line_format():
    from pamrec_b200.models import attention_line
    keys = {3: "i3", 5: "i5", 9: "i9"}
    items = np.array([[5, 3, -1], [9, 77, -1]])
    weights = np.array([[0.5, 0.25, 0.0], [1.0, 0.125, 0.0]], np.float32)
    line = attention_line("u7", np.float32(0.1), items, weights, keys)
    assert line == "u7\t0.1\ti5:0.5,i3:0.25\ti9:1.0,77:0.125"                 # an id without a key is written as the id
    assert attention_line("u7", 0.75, np.full((1, 2), -1), np.zeros((1, 2)), keys) == "u7\t0.75\t"


def _fake_model(cls_name, model, T=8, world=1):
    from pamrec_b200 import models as M
    m = getattr(M, cls_name).__new__(getattr(M, cls_name))
    m.engine = types.SimpleNamespace(dims=(10, 20, 5, T, 16), world=world, model=model)
    return m


@pytest.mark.parametrize("top_k", [0, -1, 9, 2.0, None])
def test_explain_refuses_top_k_outside_the_history(tmp_path, top_k):
    with pytest.raises(ValueError, match="top_k"):
        _fake_model("PAMRECModel", "pamrec").explain("unused", str(tmp_path / "out"), top_k=top_k)


def test_explain_refuses_several_ranks_and_sibling_maps(tmp_path):
    with pytest.raises(ValueError, match="one GPU"):
        _fake_model("PAMRECModel", "pamrec", world=2).explain("unused", str(tmp_path / "out"))
    for cls_name, model in (("MMoEModel_original", "mmoe"), ("PLEModel", "ple"), ("ShareBottomModel", "sharebottom")):
        with pytest.raises(ValueError, match="maps"):
            _fake_model(cls_name, model).explain("unused", str(tmp_path / "out"), maps=True)


def test_attention_abi_argument_checks(lib_built):
    from pamrec_b200.engine import Engine, PamrecError
    b = __import__("pamrec_b200._lib", fromlist=["PamrecBatch"]).PamrecBatch(batch=1)
    eng = Engine(n_users=11, n_items=50, n_cates=7, max_seq_len=8, max_batch=16)
    assert eng.lib.pamrec_attention(eng.handle, C.byref(b), None, None, None, None) != 0
    assert b"bind" in eng.lib.pamrec_last_error(eng.handle)                # before any device work
    sharded = Engine(n_users=11, n_items=50, n_cates=7, max_seq_len=8, max_batch=16, tables="sharded")
    assert sharded.lib.pamrec_attention(sharded.handle, C.byref(b), None, None, None, None) != 0
    assert b"one GPU" in sharded.lib.pamrec_last_error(sharded.handle)
    with pytest.raises(PamrecError, match="one GPU"):
        sharded.attention(None)
    for model in ("mmoe", "ple", "sharebottom"):
        sib = Engine(n_users=11, n_items=50, n_cates=7, max_seq_len=8, max_batch=16, model=model)
        dummy = C.c_void_p(16)                                                # never dereferenced: the call fails first
        assert sib.lib.pamrec_attention(sib.handle, C.byref(b), None, None, dummy, None) != 0
        assert b"maps_out" in sib.lib.pamrec_last_error(sib.handle)
        with pytest.raises(PamrecError, match="self-attention"):
            sib.attention(None, maps=True)
