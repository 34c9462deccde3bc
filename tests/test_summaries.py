"""TensorBoard summaries (write_tfevents): the device histogram against a float64 restatement of TensorFlow's histogram.cc, the event
file format against TensorBoard's own reader, and the summary cadence of the host loops.  GPU tests are marked `gpu`."""
import ctypes as C
import os
import struct
import sys
import types

import numpy as np
import pytest
import torch

from pamrec_b200 import _lib as L
from pamrec_b200 import checkpoint as CK
from pamrec_b200 import summary as SUM

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FLT_MAX = float(np.finfo(np.float32).max)
DBL_MAX = float(np.finfo(np.float64).max)


# ----------------------------------------------------------------------------- restatements of tensorflow/core/lib/histogram/histogram.cc
def tf_default_limits():
    """InitDefaultBuckets."""
    pos, v = [], 1.0e-12
    while v < 1.0e20:
        pos.append(v)
        v *= 1.1
    return np.array(sorted([-DBL_MAX] + [-p for p in pos] + [0.0] + pos + [DBL_MAX]), np.float64)


LIMITS = tf_default_limits()


def tf_encode(counts, limits=LIMITS):
    """EncodeToProto(preserve_zero_buckets = false) -> (bucket_limit, bucket)."""
    lim, cnt, i = [], [], 0
    while i < len(counts):
        end, count, j = limits[i], counts[i], i + 1
        while count <= 0 and j < len(counts) and counts[j] <= 0:
            end, count, j = limits[j], counts[j], j + 1
        lim.append(end)
        cnt.append(count)
        i = j
    if not lim:
        lim, cnt = [DBL_MAX], [0.0]
    return np.array(lim, np.float64), np.array(cnt, np.float64)


def tf_histogram(x):
    """Histogram::Add over the values of x (float32), encoded: the HistogramProto fields."""
    d = np.asarray(x, np.float32).astype(np.float64).reshape(-1)
    counts = np.bincount(np.searchsorted(LIMITS, d, side="right"), minlength=len(LIMITS)).astype(np.float64)
    lim, cnt = tf_encode(counts)
    return dict(min=float(d.min()) if d.size else DBL_MAX, max=float(d.max()) if d.size else -DBL_MAX, num=float(d.size),
                sum=float(d.sum()), sum_squares=float((d * d).sum()), bucket_limit=lim, bucket=cnt)


def assert_same_histogram(got, values, what):
    """Buckets, num, min and max exactly; sum and sum_squares to 1e-12 of the sum of the magnitudes they add up."""
    want = tf_histogram(values)
    assert np.array_equal(got["bucket_limit"], want["bucket_limit"]), what
    assert np.array_equal(got["bucket"], want["bucket"]), what
    assert (got["num"], got["min"], got["max"]) == (want["num"], want["min"], want["max"]), what
    d = np.asarray(values, np.float32).astype(np.float64).reshape(-1)
    assert abs(got["sum"] - want["sum"]) <= 1e-12 * np.abs(d).sum(), (what, got["sum"], want["sum"])
    assert abs(got["sum_squares"] - want["sum_squares"]) <= 1e-12 * want["sum_squares"], (what, got["sum_squares"], want["sum_squares"])


# ----------------------------------------------------------------------------- CPU
@pytest.fixture()
def ea(monkeypatch):
    """TensorBoard's event reader.  compat/ (on sys.path once a test imports the reference's paths) holds a `tensorflow` module
    for the reference's driver; hidden here, so that TensorBoard reads files through its own stub rather than through that shim."""
    mod = pytest.importorskip("tensorboard.backend.event_processing.event_accumulator")
    monkeypatch.setitem(sys.modules, "tensorflow", None)
    return mod


def test_bucket_limits_match_tensorflow_bit_for_bit(lib_built):
    lib = L.load()
    got = np.zeros(L.HIST_BUCKETS, np.float64)
    assert lib.pamrec_histogram_buckets(None, got.ctypes.data, None, None) == 0
    assert len(LIMITS) == L.HIST_BUCKETS == 1551 and (LIMITS > 0).sum() == 775         # 774 below 1e20, then DBL_MAX
    assert got.tobytes() == LIMITS.tobytes()


@pytest.mark.parametrize("case", ["empty", "single", "both_ends", "first_and_last", "random", "dense"])
def test_compaction_matches_encode_to_proto(lib_built, case):
    lib = L.load()
    c = np.zeros(L.HIST_BUCKETS, np.int32)
    if case == "single":
        c[776] = 7
    elif case == "both_ends":
        c[600:610] = 3                                          # empty runs before and after
    elif case == "first_and_last":
        c[0], c[-1], c[775] = 1, 2, 5
    elif case == "random":
        rng = np.random.default_rng(4)
        c[rng.choice(L.HIST_BUCKETS, 90, replace=False)] = rng.integers(1, 1000, 90)
    elif case == "dense":
        c[:] = 1
    pairs = np.zeros(2 * L.HIST_BUCKETS, np.float64)
    n = C.c_int()
    assert lib.pamrec_histogram_buckets(c.ctypes.data, None, pairs.ctypes.data, C.byref(n)) == 0
    lim, cnt = tf_encode(c.astype(np.float64))
    assert np.array_equal(pairs[:2 * n.value:2], lim) and np.array_equal(pairs[1:2 * n.value:2], cnt)


def _read_records(path):
    buf = open(path, "rb").read()
    pos, out = 0, []
    while pos < len(buf):
        n = struct.unpack_from("<Q", buf, pos)[0]
        assert struct.unpack_from("<I", buf, pos + 8)[0] == CK._mask(CK.crc32c(buf[pos:pos + 8]))
        data = buf[pos + 12:pos + 12 + n]
        assert struct.unpack_from("<I", buf, pos + 12 + n)[0] == CK._mask(CK.crc32c(data))
        out.append(data)
        pos += 16 + n
    return out


def test_event_file_reads_back_through_tensorboard(lib_built, tmp_path, ea):
    rng = np.random.default_rng(2)
    hists = {"sequential/a": tf_histogram(rng.normal(0, 0.01, 1000).astype(np.float32)),
             "sequential/b": tf_histogram(np.zeros(0, np.float32)), "sequential/c": tf_histogram(np.float32([-3.5, 0, 2e30]))}
    w = SUM.EventFileWriter(str(tmp_path))
    steps = [2, 4, 6]
    for s in steps:
        w.add_summary(SUM.summary_proto([("loss", np.float32(1.0 / s)), ("data_loss", np.float32(0.25))], hists.items()), s)
        w.flush()
    w.close()
    name = os.path.basename(w.path)
    assert name.startswith("events.out.tfevents.") and os.listdir(tmp_path) == [name]
    records = _read_records(w.path)                             # every CRC checks out
    assert len(records) == 1 + len(steps) and b"brain.Event:2" in records[0]
    acc = ea.EventAccumulator(str(tmp_path), size_guidance={ea.SCALARS: 0, ea.HISTOGRAMS: 0})
    acc.Reload()
    tags = acc.Tags()
    assert sorted(tags["scalars"]) == ["data_loss", "loss"] and sorted(tags["histograms"]) == sorted(hists)
    assert [(e.step, e.value) for e in acc.Scalars("loss")] == [(s, float(np.float32(1.0 / s))) for s in steps]
    for tag, h in hists.items():
        evs = acc.Histograms(tag)
        assert [e.step for e in evs] == steps
        v = evs[-1].histogram_value
        assert (v.min, v.max, v.num, v.sum, v.sum_squares) == (h["min"], h["max"], h["num"], h["sum"], h["sum_squares"])
        assert list(v.bucket_limit) == list(h["bucket_limit"]) and list(v.bucket) == list(h["bucket"])


def test_fit_step_writes_events_every_summary_step(tmp_path, monkeypatch, lib_built):
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_host_loops import StubEngine
    from pamrec_b200 import deeprec_utils as DU
    from pamrec_b200 import models as M
    from pamrec_b200 import synth
    from pamrec_b200.sequential_iterator import SequentialIterator

    class SummaryStub(StubEngine):
        def histograms(self, names):                          # the host restatement in place of the device kernel
            self.summarised = getattr(self, "summarised", []) + [self.step]
            value = {n: dict(tf_histogram(v), nonfinite=0) for n, v in self.get_variables().items() if n in names}
            return types.SimpleNamespace(result=lambda: value)

    monkeypatch.setattr(M, "Engine", SummaryStub)
    d = synth.generate(str(tmp_path), "wechat", n_users=80, n_items=300, n_cates=12, mean_len=40, seed=3, n_neg=3)
    hp = DU.prepare_hparams(
        None, model_type="mmoe", dataset="wechat", method="classification", loss="cross_entropy_loss", optimizer="adam",
        item_embedding_dim=16, cate_embedding_dim=4, user_embedding_dim=20, layer_sizes=[100, 64], expert_layer_sizes=[100, 64],
        gate_layer_sizes=[64, 5], expert_num=5, activation=["relu", "relu"], enable_BN=True, dropout=[0.0, 0.0], embedding_dropout=0.0,
        hidden_size=40, attention_size=40, att_fcn_layer_sizes=[20, 1], fuzhu_weight=0.5, bucket_num=10, noise_train_hist=0,
        noise_train_listwise=0, noise_only_predict=0, batch_size=60, max_seq_length=20, epochs=1, eval_step=7, EARLY_STOP=0, show_step=10 ** 9, train_num_ngs=0, need_sample=False,
        metrics=["auc"], pairwise_metrics=[], weighted_metrics=[], MODEL_DIR=str(tmp_path / "model") + "/",
        SUMMARIES_DIR=str(tmp_path / "sum") + "/", user_vocab=os.path.join(d, "user_vocab.pkl"),
        item_vocab=os.path.join(d, "item_vocab.pkl"), cate_vocab=os.path.join(d, "category_vocab.pkl"), write_tfevents=True,
        summary_step=3, save_model=False)
    m = M.PAMRECModel(hp, SequentialIterator, seed=8)
    results = []
    m.step_train = lambda step, r: results.append((step + 1, r))
    m.fit_step(os.path.join(d, "train_data"), os.path.join(d, "valid_data"), valid_num_ngs=3, eval_metric="auc")
    n = m.engine.calls["train"]
    assert n >= 7
    want = [s for s in range(1, n + 1) if s % 3 == 0]
    assert m.engine.summarised == want
    assert [s for s, r in results if r[7] is not None] == want and all(len(r) == 8 for _, r in results)
    files = os.listdir(tmp_path / "sum")
    assert len(files) == 1
    records = _read_records(str(tmp_path / "sum" / files[0]))
    assert len(records) == 1 + len(want)
    summaries = {s: r[7] for s, r in results if r[7] is not None}
    for rec, s in zip(records[1:], want):
        fields = {num: val for num, _, val in CK._fields(rec)}
        assert fields[2] == s and fields[5] == summaries[s]
    with pytest.raises(ValueError, match="summary_step"):
        M.PAMRECModel(DU.HParams({**hp.values(), "summary_step": 0}), SequentialIterator, seed=8)


# ----------------------------------------------------------------------------- GPU
def _device_histograms(eng, arrays):
    """pamrec_histograms over device copies of `arrays` (one engine, world 1) -> list of HistogramProto dicts + nonfinite."""
    dev = [torch.from_numpy(np.ascontiguousarray(a, np.float32).reshape(-1)).cuda() for a in arrays]
    n = len(dev)
    counts = (C.c_int64 * n)(*[t.numel() for t in dev])
    caps = [min(L.HIST_BUCKETS, 2 * t.numel() + 1) for t in dev]
    offs = np.concatenate([[0], np.cumsum(caps)]).astype(np.int64)
    offs_c = (C.c_int64 * (n + 1))(*offs.tolist())
    need = C.c_int64(0)
    eng._check(eng.lib.pamrec_histograms(eng.handle, None, counts, n, 0, None, None, None, None, C.byref(need), None))
    scratch = torch.empty(need.value, dtype=torch.uint8, device="cuda")
    stats = torch.full((n * 7,), -1.0, dtype=torch.float64, device="cuda")
    out = torch.zeros(int(offs[-1]) * 2, dtype=torch.float64, device="cuda")
    ptrs = (C.c_void_p * n)(*[t.data_ptr() for t in dev])
    eng._check(eng.lib.pamrec_histograms(eng.handle, ptrs, counts, n, 0, offs_c, C.c_void_p(stats.data_ptr()), C.c_void_p(out.data_ptr()),
                                         C.c_void_p(scratch.data_ptr()), C.byref(need), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    st, pairs = stats.cpu().numpy().reshape(n, 7), out.cpu().numpy().reshape(-1, 2)
    res = []
    for s in range(n):
        k = int(st[s, 4])
        assert k <= caps[s]
        res.append(dict(num=st[s, 0], sum=st[s, 1], sum_squares=st[s, 2], nonfinite=int(st[s, 3]), min=st[s, 5], max=st[s, 6],
                        bucket_limit=pairs[offs[s]:offs[s] + k, 0], bucket=pairs[offs[s]:offs[s] + k, 1]))
    return res, (stats, out)


@pytest.fixture(scope="module")
def eng():
    from pamrec_b200.engine import Engine
    e = Engine(50, 200, 10, 8, 10).allocate("cuda:0")
    yield e
    e.close()


def _special_values():
    lim = LIMITS[(np.abs(LIMITS) < 3e38) & (LIMITS != 0)].astype(np.float32)      # limits as float32, and one ulp either side
    on = np.concatenate([lim, np.nextafter(lim, np.float32(np.inf)), np.nextafter(lim, np.float32(-np.inf))])
    exact = LIMITS[(np.abs(LIMITS) < 3e38) & (LIMITS.astype(np.float32).astype(np.float64) == LIMITS)].astype(np.float32)
    den = np.float32([1e-45, -1e-45, 1e-40, -1e-40, 1.1754942e-38, -1.1754942e-38])
    return np.concatenate([on, exact, den, np.float32([0.0, -0.0, FLT_MAX, -FLT_MAX, 1e-12, -1e-12, 1e20, -1e20, 1.0, -1.0])])


@pytest.mark.gpu
def test_histogram_kernel_matches_tensorflow(eng):
    rng = np.random.default_rng(11)
    arrays = [rng.normal(0, 1, n).astype(np.float32) for n in (1, 31, 32, 33, 1 << 16, (1 << 16) + 1, 3 * (1 << 16) + 5)]
    arrays.append(_special_values())
    arrays.append(rng.permutation(np.repeat(_special_values(), 3)))
    arrays.append(np.zeros(1000, np.float32))
    arrays.append((rng.standard_cauchy(30_000_000) * 1e-3).astype(np.float32))
    got, _ = _device_histograms(eng, arrays)
    for i, (g, a) in enumerate(zip(got, arrays)):
        assert g["nonfinite"] == 0
        assert_same_histogram(g, a, f"segment {i} ({a.size} values)")


@pytest.mark.gpu
def test_histogram_kernel_short_and_long_mix_unaligned_and_repeatable(eng):
    rng = np.random.default_rng(12)
    big = rng.normal(0, 0.05, 5_000_003).astype(np.float32)
    arrays = [rng.normal(0, 10.0 ** rng.integers(-6, 4), rng.integers(1, 300)).astype(np.float32) for _ in range(100)]
    arrays.insert(37, big)
    arrays.append(big[1:])                                        # a segment whose start is not 16-byte aligned in memory
    got, raw1 = _device_histograms(eng, arrays)
    for i, (g, a) in enumerate(zip(got, arrays)):
        assert_same_histogram(g, a, f"segment {i} ({a.size} values)")
    _, raw2 = _device_histograms(eng, arrays)
    for x, y in zip(raw1, raw2):
        assert x.cpu().numpy().tobytes() == y.cpu().numpy().tobytes()


@pytest.mark.gpu
def test_histogram_kernel_reports_non_finite_per_segment(eng):
    a = np.linspace(-1, 1, 1000).astype(np.float32)
    b = a.copy()
    b[[3, 500]] = [np.nan, np.inf]
    c = a.copy()
    c[999] = -np.inf
    got, _ = _device_histograms(eng, [a, b, c, a])
    assert [g["nonfinite"] for g in got] == [0, 2, 1, 0]


def _fit_with_summaries(tmp_path, cls_path, yaml_path, **kw):
    """fit_step with write_tfevents = True, summary_step = 2; returns (model, {step: train() result}, {step: variables})."""
    import importlib
    sys.path.insert(0, os.path.join(ROOT, "compat"))
    from pamrec_b200 import synth
    from reco_utils.recommender.deeprec.deeprec_utils import prepare_hparams
    from reco_utils.recommender.deeprec.io.sequential_iterator import SequentialIterator
    mod, cls_name = cls_path.rsplit(".", 1)
    cls = getattr(importlib.import_module(mod), cls_name)
    root = tmp_path / "data"
    synth.generate(str(root), "wechat", n_users=150, n_items=1500, n_cates=20, mean_len=40, seed=5, eval_per_user=2)
    d = os.path.join(str(root), "wechat")
    hp = prepare_hparams(yaml_path, dataset="wechat", bucket_num=10, add_feature=False, embed_l2=1e-6, layer_l2=1e-6,
                         discrepancy_loss_weight=0.1, learning_rate=0.001, epochs=1, EARLY_STOP=5, is_clip_norm=1, batch_size=100,
                         show_step=10 ** 9, MODEL_DIR=str(tmp_path / "model") + "/", SUMMARIES_DIR=str(tmp_path / "sum") + "/",
                         user_vocab=os.path.join(d, "user_vocab.pkl"), item_vocab=os.path.join(d, "item_vocab.pkl"),
                         cate_vocab=os.path.join(d, "category_vocab.pkl"), train_num_ngs=0, max_seq_length=50, pairwise_metrics=[],
                         weighted_metrics=["wauc"], fuzhu_weight=0.5, fine_tune=False, eval_step=5, noise_train_hist=0,
                         noise_train_listwise=0, noise_only_predict=0, write_tfevents=True, summary_step=2, save_model=False, **kw)
    model = cls(hp, SequentialIterator, seed=8)
    eng, results, snaps = model.engine, {}, {}
    real_hist = eng.histograms

    def histograms(names):                                      # the variables right after the summarised step
        snaps[eng.step] = eng.get_variables()
        return real_hist(names)
    eng.histograms = histograms
    model.step_train = lambda step, r: results.__setitem__(step + 1, r)
    model.fit_step(os.path.join(d, "train_data"), os.path.join(d, "valid_data"), valid_num_ngs=0, eval_metric="auc")
    return model, results, snaps


@pytest.mark.gpu
@pytest.mark.parametrize("cls_path,yaml_name,n_scalars", [
    ("pamrec_b200.models.PAMRECModel", "pamrec_b200/config/mmoe.yaml", 5),
    ("reco_utils.recommender.deeprec.models.sequential.mmoe.MMoEModel_original", "compat/reco_utils/recommender/deeprec/config/mmoe.yaml", 4),
    ("reco_utils.recommender.deeprec.models.sequential.sasrec.SASRecModel", "compat/reco_utils/recommender/deeprec/config/sasrec.yaml", 2)])
def test_fit_step_summaries_read_back_through_tensorboard(tmp_path, ea, cls_path, yaml_name, n_scalars):
    model, results, snaps = _fit_with_summaries(tmp_path, cls_path, os.path.join(ROOT, yaml_name))
    n = max(results)
    want_steps = [s for s in range(1, n + 1) if s % 2 == 0]
    assert len(want_steps) >= 2 and sorted(snaps) == want_steps
    assert all((results[s][-1] is not None) == (s % 2 == 0) for s in results)
    acc = ea.EventAccumulator(str(tmp_path / "sum"), size_guidance={ea.SCALARS: 0, ea.HISTOGRAMS: 0})
    acc.Reload()
    names = model.SCALARS
    assert len(names) == n_scalars and sorted(acc.Tags()["scalars"]) == sorted(names)
    for i, tag in enumerate(names):
        assert [(e.step, e.value) for e in acc.Scalars(tag)] == [(s, results[s][2 + i]) for s in want_steps], tag
    last = want_steps[-1]
    variables = snaps[last]
    assert sorted(acc.Tags()["histograms"]) == sorted(variables)
    for name, val in variables.items():
        evs = acc.Histograms(name)
        assert [e.step for e in evs] == want_steps, name
        v = evs[-1].histogram_value
        got = dict(min=v.min, max=v.max, num=v.num, sum=v.sum, sum_squares=v.sum_squares,
                   bucket_limit=np.array(v.bucket_limit), bucket=np.array(v.bucket))
        assert_same_histogram(got, val, name)


@pytest.mark.gpu
def test_non_finite_variable_fails_the_summarised_step(tmp_path):
    from pamrec_b200.engine import PamrecError
    model, _, _ = _fit_with_summaries(tmp_path, "pamrec_b200.models.PAMRECModel", os.path.join(ROOT, "pamrec_b200", "config", "mmoe.yaml"))
    name = "sequential/embedding/user_embedding"                 # a frozen variable: training never overwrites it
    bad = np.zeros(model.engine.variable_shapes()[name], np.float32)
    bad[1, 2] = np.nan
    model.engine.set_variables({name: bad})
    feed = next(f for f in model.iterator.load_data_from_file(os.path.join(str(tmp_path / "data"), "wechat", "train_data"),
                                                              min_seq_length=1, batch_num_ngs=0) if f)
    if model.engine.step % 2 == 0:
        model.train(None, feed)                                  # an odd step: not summarised
    with pytest.raises(PamrecError, match="Nan in summary histogram for: " + name + r" \(step \d+\)"):
        model.train(None, feed)


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_rank_histograms_of_sharded_tables():
    import subprocess
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29631", os.path.join(ROOT, "tests", "dist_summary_worker.py")]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0 and "SUMMARY_DIST_OK" in r.stdout, r.stdout[-6000:]
