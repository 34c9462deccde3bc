#!/usr/bin/env python
"""Headline benchmark of the PAMRec train step (BASELINE.json: train samples/sec; gather/Adam HBM GB/s vs peak).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload NAME] [--dump-outputs DIR]

One "step" = one optimisation step (forward + losses + backward + per-tensor clip + Adam) over one batch of
synthetic MX-TakaTak-shaped input.  Prints ONE JSON line (rank 0).  Keys: see DESIGN.md "Measurement".
--dump-outputs DIR writes what the last of the K timed steps computed (rank 0): the losses and the logits of a training step, the
predictions of a scoring step.  The inputs are seeded, so two builds run with the same arguments can be compared array by array.
Every timed training step starts from the seeded initial model, so the last one computes from the same state on every run.
"""
import argparse
import gc
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # BASELINE.json configs[1]: takatak-shaped, seq_len 50, group of 5 (1 pos + 4), batch 1024 -> 1025 (must be a
    # multiple of 5: io/sequential_iterator.py:684-685), single B200
    "takatak_b1025_t50": dict(dataset="takatak", n_users=50000, n_items=30000, n_cates=50, T=50, B=1025),
    # configs[3]: long history
    "long_b4095_t200": dict(dataset="takatak", n_users=50000, n_items=30000, n_cates=50, T=200, B=4095),
    # configs[0]-shaped quick start
    "wechat_b500_t100": dict(dataset="wechat", n_users=20000, n_items=100000, n_cates=500, T=100, B=500),
    # configs[2]: 10 M items / 100 K categories, tables row-sharded over the ranks (also runs on one GPU)
    "sharded_10m_b1025_t50": dict(dataset="takatak", n_users=50000, n_items=10_000_000, n_cates=100_000, T=50, B=1025,
                                  tables="sharded", zipf=1.05),
    # configs[4]: eval-only scoring of 1 positive + 99 negatives per impression (a "step" = one scoring batch of 40 impressions;
    # e2e = run_weighted_eval over an 11-column text file with group = 100, sequential_base_model.py:437,456)
    "eval_1p99": dict(dataset="takatak", n_users=50000, n_items=30000, n_cates=50, T=50, B=4000, kind="score", group=100,
                      impressions=600),
}
METRIC = "train samples/sec"
METRIC_SCORE = "scored samples/sec"
N_POOL = 8            # distinct resident batches cycled through the timed steps
ATTN_PIPE = "fp32" if os.environ.get("PAMREC_ATTN", "mma") == "ffma" else "tensor"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tensor=d["bf16_tflops"], tensor_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tensor=1590.0, tensor_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def build_model(w, tmp, sparse_adam="dense_exact", **extra):
    from pamrec_b200 import synth
    from pamrec_b200.deeprec_utils import prepare_hparams
    from pamrec_b200.models import PAMRECModel
    from pamrec_b200.sequential_iterator import SequentialIterator
    d = synth.write_vocab_only(tmp, w["dataset"], w["n_users"], w["n_items"], w["n_cates"])
    kw = dict(dataset=w["dataset"], bucket_num=10,
              add_feature=False, embed_l2=1e-6, layer_l2=1e-6, discrepancy_loss_weight=0.1, learning_rate=0.001,
              epochs=1, EARLY_STOP=5, is_clip_norm=1, batch_size=w["B"], show_step=10 ** 9, MODEL_DIR=os.path.join(tmp, "model/"),
              SUMMARIES_DIR=os.path.join(tmp, "summary/"), user_vocab=os.path.join(d, "user_vocab.pkl"),
              item_vocab=os.path.join(d, "item_vocab.pkl"), cate_vocab=os.path.join(d, "category_vocab.pkl"),
              train_num_ngs=0, max_seq_length=w["T"], pairwise_metrics=[], weighted_metrics=["wauc"], fuzhu_weight=0.5,
              fine_tune=False, eval_step=10 ** 9, noise_train_hist=0, noise_train_listwise=0, noise_only_predict=0,
              write_tfevents=False, sparse_adam=sparse_adam)
    kw.update(extra)
    hp = prepare_hparams(os.path.join(ROOT, "pamrec_b200", "config", "mmoe.yaml"), **kw)
    return PAMRECModel(hp, SequentialIterator, seed=8)


def flops_bytes(w):
    """Algorithmic work per STEP of every launcher (DESIGN.md section 4): name -> dict(flop, byte, pipe, launches).
    flop counts 2 per multiply-add of the minimal algorithm; byte = tensors that must be read + written once (fp32).
    pipe: which unit the kernel's arithmetic runs on ("tensor" = 3xTF32 tensor-core MMAs, "fp32" = FFMA, "hbm" = no arithmetic
    to speak of)."""
    B, T = w["B"], w["T"]
    N = B * T
    t = 160 * N                                  # bytes of one [N, 40] fp32 tensor
    score = 2 * (40 * 20 + 20) * N               # attention-pooling MLP 40 -> 20 -> 1 over every position (pamrec.py:272-283)
    mmoe = 2 * (5 * (40 * 100 + 100 * 64) + 2 * (40 * 64 + 64 * 5)) * B
    tower = 2 * 3 * (84 * 100 + 100 * 64 + 64) * B
    head_act = 4 * (N * 21 + B * (500 + 320 + 128 + 10 + 168 + 300 + 192 + 3))            # pre-activations written once
    return {
        # attention: warp-level 3xTF32 MMAs (kernels_attn_mma.cu) unless PAMREC_ATTN=ffma; the T x T count is the reference's (every
        # key, padded or not); the kernels only visit the live keys of a sample
        "attn_fwd": dict(flop=2 * (2 * T * T * 40) * B * 2, byte=2 * 5 * t, pipe=ATTN_PIPE),   # Q K^T, P V ; Q K V qin -> y  (x 2 blocks)
        "attn_bwd": dict(flop=2 * (5 * T * T * 40) * B * 2, byte=2 * 9 * t, pipe=ATTN_PIPE),   # S, dP, dV, dQ, dK
        "proj_fwd": dict(flop=2 * (3 * 1600) * N * 2, byte=2 * 5 * t, pipe="tensor"),
        "proj_bwd": dict(flop=2 * (6 * 1600) * N * 2, byte=2 * 6 * t, pipe="tensor"),
        "ffn_fwd": dict(flop=2 * (2 * 1600) * N * 2, byte=2 * 2 * t, pipe="tensor"),
        "ffn_bwd": dict(flop=2 * (5 * 1600) * N * 2, byte=2 * 3 * t, pipe="tensor"),           # h recomputed + 2 dX + 2 dW GEMMs
        "embed_fwd": dict(flop=0, byte=248 * N + 168 * B, pipe="hbm"),                          # 88 B read + 160 B written per lookup
        "dense_fwd": dict(flop=score + mmoe + tower, byte=t + head_act, pipe="fp32"),
        "dense_dx": dict(flop=score + mmoe + tower, byte=t + 2 * head_act, pipe="fp32"),
        "dense_dw": dict(flop=score + mmoe + tower, byte=t + 2 * head_act, pipe="fp32"),
        "head_fwd": dict(flop=score + mmoe + tower, byte=t + head_act, pipe="fp32"),
        "head_bwd": dict(flop=2 * (score + mmoe + tower), byte=2 * t + 3 * head_act, pipe="fp32"),
        "sparse_walk": dict(flop=0, byte=96 * (N + B), pipe="hbm"),                            # 80 B gradient row + 16 B rank / index per lookup
        "sparse_scatter_adam": dict(flop=0, byte=96 * (N + B), pipe="hbm"),
        "sparse_adam": dict(flop=0, byte=(6 * 64 + 4) * w["n_items"] + (6 * 16 + 4) * w["n_cates"] + 2 * (6 * 80 + 4) * w["n_users"], pipe="hbm"),
    }


def step_work(w):
    """Algorithmic flops and bytes of one whole step (sum of the launchers' minimal work, every tensor once): a training step, or
    the forward pass of a scoring workload."""
    fb = flops_bytes(w)
    names = ("embed_fwd", "proj_fwd", "attn_fwd", "ffn_fwd", "head_fwd")
    if w.get("kind") != "score":
        names += ("head_bwd", "ffn_bwd", "attn_bwd", "proj_bwd", "sparse_scatter_adam", "sparse_adam")
    return sum(fb[n]["flop"] for n in names), sum(fb[n]["byte"] for n in names)


# dram__bytes_read.sum + dram__bytes_write.sum per launch, from the `ncu --set full` capture of this workload
# (profiles/r01e_ncu_encoder_full.csv, takatak_b1025_t50); null for kernels / workloads without a capture
# (profiles/r02z_ncu_step_full.csv)
NCU_TRAFFIC = {"takatak_b1025_t50": {"attn_bwd": 41.67e6 + 0.96e6, "attn_fwd": 24.87e6 + 0.0, "proj_bwd": 41.66e6 + 0.33e6, "ffn_bwd": 16.49e6 + 0.0}}


def hbm_microbench(pk, dev):
    """Stand-alone HBM kernels on the BASELINE configs[2] table shape (10 M items x 16, 100 K categories x 4: far above the
    126 MB L2), the same kernels the step launches: the fused embedding gather and the full-table (dense_exact) Adam sweep."""
    import ctypes as C
    from pamrec_b200.engine import Engine
    out = {}
    ni, nc, T = 10_000_000, 100_000, 50
    eng = Engine(1000, ni, nc, T, 64).allocate(str(dev))
    eng.pool["item_w"].normal_(0, 0.01)
    eng.pool["cate_w"].normal_(0, 0.01)
    rows = 1 << 20                                         # 1 Mi sequences x T lookups
    g = torch.Generator(device="cpu").manual_seed(1)
    ih = torch.randint(0, ni, (rows * T,), generator=g, dtype=torch.int32).to(dev)
    ch = torch.randint(0, nc, (rows * T,), generator=g, dtype=torch.int32).to(dev)
    ti = torch.randint(0, ni, (rows,), generator=g, dtype=torch.int32).to(dev)
    tc = torch.randint(0, nc, (rows,), generator=g, dtype=torch.int32).to(dev)
    outb = torch.empty(rows * T * 40, dtype=torch.float32, device=dev)
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    def timed(call, reps=5):
        for _ in range(3):
            call()
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); call(); b.record(); torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return min(ts)

    ms = timed(lambda: eng._check(eng.lib.pamrec_bench_gather(eng.handle, C.c_void_p(ih.data_ptr()), C.c_void_p(ch.data_ptr()),
                                                              C.c_void_p(ti.data_ptr()), C.c_void_p(tc.data_ptr()), rows, T,
                                                              C.c_void_p(outb.data_ptr()), st)))
    byts = 248 * rows * T + 8 * rows
    out["embed_fwd"] = dict(kernel="k_embed_fwd", lookups=rows * T, table_rows=ni, ms=ms, achieved=byts / ms / 1e6, peak=pk["hbm"],
                            unit="GB/s", frac=byts / ms / 1e6 / pk["hbm"], bytes_per_lookup=248,
                            note="uniform random ids over a 10 M x 16 fp32 item table (640 MB, misses L2) and a 100 K x 4 category "
                                 "table; 88 B read + 160 B written per lookup (SURVEY.md 8d)")
    del ih, ch, outb
    step = [0]

    def adam():
        step[0] += 1
        eng._check(eng.lib.pamrec_bench_table_adam(eng.handle, step[0], st))
    ms = timed(adam)
    byts = ni * (6 * 64 + 4) + nc * (6 * 16 + 4) + 2 * 1000 * (6 * 80 + 4)
    out["table_adam_dense_exact"] = dict(kernel="k_sp2_adam_sweep<SP2_COMPACT>", table_rows=ni, ms=ms, achieved=byts / ms / 1e6,
                                         peak=pk["hbm"], unit="GB/s", frac=byts / ms / 1e6 / pk["hbm"], bytes_per_row=6 * 64 + 4,
                                         note="TF-exact sparse Adam, all four tables in one launch: m, v, w of EVERY row read and written "
                                              "(6 x row bytes) + 4 B slot word")
    eng.close()
    del eng
    torch.cuda.empty_cache()
    # ---- the sparse backward ("scatter") inside a real step at a batch large enough to be bandwidth-bound:
    # 65 535 rows x 50 = 3.3 M lookups per table on the 10 M-item table, per-launcher CUDA events
    from pamrec_b200 import synth
    B2 = 65535
    eng = Engine(50000, ni, nc, T, B2).allocate(str(dev))
    eng.pool["item_w"].normal_(0, 0.01)
    eng.pool["cate_w"].normal_(0, 0.01)
    eng.pool["dense_param"].normal_(0, 0.05)
    n_look = B2 * T + B2
    byts = n_look * ((64 + 8) + (16 + 8))                    # gradient row + sorted rank / source index, per lookup and table
    for mode in ("dense_exact", "lazy"):
        if mode == "lazy":
            eng.close()
            del eng
            torch.cuda.empty_cache()
            eng = Engine(50000, ni, nc, T, B2, sparse_adam="lazy").allocate(str(dev))
            eng.pool["item_w"].normal_(0, 0.01)
            eng.pool["cate_w"].normal_(0, 0.01)
            eng.pool["dense_param"].normal_(0, 0.05)
        for tag, min_len, what in (("sparse_scatter", T, "full histories (every position a real item)"),
                                   ("sparse_scatter_padded", 1, "history lengths uniform in 1..T: half of all positions are the padding id 0")):
            feed = synth.array_batch(77, B2, T, 50000, ni, nc, zipf_a=1.05, min_len=min_len)
            db = eng.upload(feed)
            for _ in range(2):
                eng.train_step(db)
            eng.profile(True)
            reps = 3
            for _ in range(reps):
                eng.train_step(db)
            tab = eng.profile_table()
            eng.profile(False)
            ms = tab["sparse_walk"][0] / reps                    # ONE launch: item (64-byte) and category (16-byte) rows
            uniq = eng.ws("sp.nuniq").cpu().numpy()
            extra = 0
            if mode == "lazy":                                   # + Adam on the touched rows inside the same kernel: w, m, v read and written
                extra = int(uniq[0]) * 6 * 64 + int(uniq[1]) * 6 * 16
            else:                                                # + the compact accumulator rows written for the sweep
                extra = int(uniq[0]) * 64 + int(uniq[1]) * 16
            key = tag + ("_fused_adam" if mode == "lazy" else "_segreduce")
            out[key] = dict(kernel="k_sp2_walk<%s>" % ("SP2_FUSED" if mode == "lazy" else "SP2_COMPACT"), lookups=n_look,
                            unique_rows=[int(uniq[0]), int(uniq[1])], ms=ms, achieved=(byts + extra) / ms / 1e6, peak=pk["hbm"],
                            unit="GB/s", frac=(byts + extra) / ms / 1e6 / pk["hbm"], bytes_per_lookup=96, bytes_unique_rows=extra,
                            plan_ms=tab["sparse_plan"][0] / reps, adam_ms=tab["sparse_adam"][0] / reps,
                            note="inside a full train step at B=65535, T=50, Zipf(1.05) ids over 10 M items, " + what + ": 80 B of "
                                 "gradient row + 16 B of rank / source index per lookup, plus per unique row "
                                 + ("the Adam update applied in the same kernel (w, m, v read and written: 6 x row bytes)" if mode == "lazy"
                                    else "its compact accumulator row (the full-table sweep follows)")
                                 + "; plan_ms = one merged radix sort + scan on the side stream, adam_ms = what is left for the Adam launch")
            if min_len == T and mode == "dense_exact":
                ms = tab["embed_fwd"][0] / reps
                out["embed_fwd_in_step"] = dict(kernel="k_embed_fwd", lookups=B2 * T, ms=ms, achieved=248 * B2 * T / ms / 1e6, peak=pk["hbm"],
                                                unit="GB/s", frac=248 * B2 * T / ms / 1e6 / pk["hbm"], note="same step; Zipf ids, so hot rows hit L2")
            del db
    eng.close()
    return out


def settle_sampler(clocks, dev, world, step):
    """Extra un-timed steps until the clock sampler has delivered three samples (the same number of steps on every rank)."""
    for _ in range(3000):
        have = torch.tensor([1 if len(clocks.rows) >= 3 else 0], device=dev)
        if world > 1:
            torch.distributed.all_reduce(have, op=torch.distributed.ReduceOp.MIN)
        if int(have.item()):
            break
        step()
        torch.cuda.synchronize()


DUMP_ROWS = 65536            # --dump-outputs: an array with more rows than this is written as a fixed sample of its rows
DUMP_LIMIT = 64 << 20        # bytes of all dumped arrays together


def dump_outputs(out_dir, arrays):
    """Writes name -> array as <out_dir>/<name>.npy in float32 (float64 stays float64).  An array of more than DUMP_ROWS rows is
    cut to the same DUMP_ROWS rows on every run (seeded choice, ascending order), so that two builds compare output for output."""
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
        a = a.astype(np.float64 if a.dtype == np.float64 else np.float32, copy=False)
        if a.ndim and a.shape[0] > DUMP_ROWS:
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], DUMP_ROWS, replace=False))]
        total += a.nbytes
        if total > DUMP_LIMIT:
            raise RuntimeError(f"--dump-outputs: more than {DUMP_LIMIT >> 20} MB at {name}")
        np.save(os.path.join(out_dir, name.replace("/", ".") + ".npy"), np.ascontiguousarray(a))


def run_ours(args, w, rank, world):
    from pamrec_b200 import synth
    pk = peaks()
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
    dev = torch.device("cuda", torch.cuda.current_device())
    tmp = tempfile.mkdtemp(prefix="pamrec_bench_")
    # N > 1: weak scaling — every rank trains on its own B rows of a global batch of N*B rows (listwise groups are
    # independent); tables row-sharded over the ranks, BN statistics / clip norms / losses / dense grads all-reduced.
    extra = {"dp_feed": "local"} if world > 1 else {}
    if w.get("tables"):
        extra["tables"] = w["tables"]
    model = build_model(w, tmp, **extra)
    eng = model.engine
    B, T = w["B"], w["T"]
    feeds = [synth.array_batch(1000 + 17 * i + rank, B, T, w["n_users"], w["n_items"], w["n_cates"], zipf_a=w.get("zipf", 1.1))
             for i in range(N_POOL)]
    resident = [eng.upload(f) for f in feeds]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)          # > 126 MB L2
    K, W = args.steps, args.warmup
    # Every timed step starts from the seeded initial model: variables, Adam slots, BN statistics and the device's Adam step, put
    # back before each step's L2 flush.  A step sums with float atomics, and Adam turns that rounding into +-learning_rate moves of
    # some variables (tests/test_gpu_quickstart.py: _worst_difference), so the state after a trajectory of steps differs from run to
    # run; steps from one state compute the same from the same inputs on every run, whatever the warm-up took.
    state = [eng.pool[k] for k in eng.pool if k != "workspace"] + [eng.ws("adam.step")]
    initial = [t.clone() for t in state]

    def restore():
        torch._foreach_copy_(state, initial)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    # ---- value: inputs resident in HBM, device-timed per step, L2 flushed between steps
    clocks = ClockSampler(torch.cuda.current_device()).start()      # sampled from the warm-up on: nvidia-smi needs ~0.2 s to start
    # warm-up: at least W steps, and every resident batch twice - the second use of a batch captures its CUDA graph (engine.py), which
    # must not fall into the timed region
    for i in range(max(W, 2 * N_POOL)):
        eng.train_step(resident[i % N_POOL])
    barrier()
    # A few clock samples before the timed region (every rank takes the same number of extra warm-up steps).  Not just one: the
    # device stalls for several ms once while nvidia-smi attaches (seen as one 4 - 8 ms step right after its first line of output,
    # never later: tools/step_jitter.py), which a 20-step timed region would carry as + 25 %.
    settle_sampler(clocks, dev, world, lambda: eng.train_step(resident[0]))
    # the events exist before the timed region and the collector is off inside it: a host pause between the record of a step's start
    # and its launch would be charged to the device (the stream only runs ahead of the host after the first few steps)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    gc.collect()
    gc.disable()
    barrier()
    t_wall0 = time.perf_counter()
    for i in range(K):
        restore()
        flush.fill_(i & 0xFF)
        a, b = evs[i]
        a.record()
        losses = eng.train_step(resident[i % N_POOL])
        b.record()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    gc.enable()
    # what the last timed step computed from its inputs: the losses and the logits of the heads.  Not the variables it leaves: where a
    # gradient is zero but for rounding (a bias in front of a batch norm), Adam's first step turns that rounding into the value.
    outputs = {"losses": losses.clone(), "logits": eng.ws("logits", B).clone()} if args.dump_outputs else None
    step_ms = [a.elapsed_time(b) for a, b in evs]
    step_sorted = sorted(step_ms)
    launches = eng.launches()
    total_ms = sum(step_ms)
    if world > 1:
        t = torch.tensor([total_ms], device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        total_ms = float(t.item())
    value = B * world * K / (total_ms / 1e3)

    # ---- e2e: the public call (PAMRECModel.train) with HOST feed dicts: pinned staging + one H2D per step, losses D2H
    # (PAMRECModel.train_async, the way fit_step drives it: step i + 1 is staged, copied and queued before the losses of step i
    # are read, so the host packs a feed while the device runs; every step still copies its own inputs in and its losses out)
    def e2e_pass(n):
        pending = None
        for i in range(n):
            queued = model.train_async(None, feeds[i % N_POOL])
            if pending is not None:
                pending.result()
            pending = queued
        if pending is not None:
            pending.result()
    e2e_pass(W)
    barrier()
    t0 = time.perf_counter()
    e2e_pass(K)
    barrier()
    e2e_s = time.perf_counter() - t0
    clk = clocks.stop()
    if world > 1:
        t = torch.tensor([e2e_s], device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        e2e_s = float(t.item())
    h2d = eng.upload(feeds[0], staged=True).h2d_bytes
    e2e = {"value": B * world * K / e2e_s, "unit": "samples/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 20}

    # ---- per-launcher device time over a second pass of the same K steps (CUDA events around every launch)
    eng.profile(True)
    for i in range(K):
        restore()
        flush.fill_(i & 0xFF)
        eng.train_step(resident[i % N_POOL])
    tab = eng.profile_table()
    eng.profile(False)
    tot = sum(ms for ms, _ in tab.values())
    kernels = {k: {"ms_per_step": ms / K, "share": ms / tot, "launches_per_step": n / K} for k, (ms, n) in
               sorted(tab.items(), key=lambda kv: -kv[1][0])}
    roof, roof_step = rooflines(w, tab, K, total_ms / K, pk, clk, args.workload)
    hbm = hbm_microbench(pk, dev) if world == 1 else None

    out = {
        "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "impl": "pamrec_b200",
        "config": {"workload": args.workload, "batch_per_gpu": B, "seq_len": T, "group": 5, "n_items": w["n_items"],
                   "n_cates": w["n_cates"], "n_users": w["n_users"], "sparse_adam": "dense_exact",
                   "global_batch": B * world, "tables": eng.tables,
                   "parallelism": "single GPU" if world == 1 else (
                       f"dp{world}: groups sharded over ranks, " + (
                           "tables row-sharded (id % N) with NCCL all-to-all of rows / row gradients" if eng.tables == "sharded" else
                           "tables replicated (small vocabularies): gradient tables all-reduced with the dense gradients") +
                       ", sync-BN through NVLink peer mailboxes inside the persistent head kernels"),
                   "l2": "flushed between timed steps (256 MiB write); per-step working set also exceeds L2",
                   "state": "every timed step starts from the seeded initial model (variables, Adam slots and step, BN statistics), "
                            "restored before its L2 flush",
                   "warmup_steps_run": max(W, 2 * N_POOL),
                   "launch": "the step is replayed from a CUDA graph (one per resident / staged batch, captured during warm-up)" if eng.graph and world == 1 else "kernel by kernel",
                   "batch_note": "BASELINE batch 1024 rounded to 1025: batches must be multiples of 5",
                   "e2e_note": "PAMRECModel.train_async one step ahead (as fit_step runs): per step one pinned H2D of the feed, "
                               "the step, one D2H of its 5 losses"},
        "e2e": e2e, "gpu_launches": int(launches) * K, "gpu_launches_per_step": int(launches), "clocks": clk, "roofline": roof,
        "roofline_step": roof_step, "roofline_hbm": hbm,
        "kernels": kernels, "wall_s_timed_region": t_wall,
        "ms_per_step_median": step_sorted[len(step_sorted) // 2], "ms_per_step_max": step_sorted[-1],
    }
    return out, model, outputs


def rooflines(w, tab, K, ms_per_step, pk, clk, workload):
    """`roofline` of the dominant launcher and `roofline_step` of the whole step.

    The dominant launcher is the one with the largest share of the per-launcher device time.  It is judged against the unit its
    arithmetic actually runs on: "hbm" kernels against the measured copy bandwidth, "tensor" kernels against the sustained bf16
    dense peak (every algorithmic product costs three TF32 MMAs there, so frac counts useful flops only), FFMA kernels against
    the fp32 FFMA peak (bound = "fp32": such a kernel can not reach either of the other two roofs and labelling it "hbm" hid
    that in round 1)."""
    fb = flops_bytes(w)
    fp32_peak = 148 * 128 * 2 * (clk["sm_max_mhz"] or 1965.0) * 1e6 / 1e12      # FFMA lanes x 2 flop x clock
    order = sorted(tab.items(), key=lambda kv: -kv[1][0])
    dom = next((k for k, _ in order if k in fb), None)
    roof = None
    if dom:
        wk = fb[dom]
        launches_per_step = tab[dom][1] / K
        per_step_s = tab[dom][0] / K / 1e3
        per_launch_s = per_step_s / launches_per_step
        tf, gb = wk["flop"] / per_step_s / 1e12, wk["byte"] / per_step_s / 1e9
        if wk["pipe"] == "hbm":
            roof = {"kernel": dom, "bound": "hbm", "achieved": gb, "peak": pk["hbm"], "unit": "GB/s", "frac": gb / pk["hbm"],
                    "peak_source": pk["source"]}
        elif wk["pipe"] == "tensor":
            roof = {"kernel": dom, "bound": "tensor", "achieved": tf, "peak": pk["tensor_sustained"], "unit": "TFLOP/s",
                    "frac": tf / pk["tensor_sustained"], "peak_source": pk["source"] + ", sustained bf16"}
        else:
            roof = {"kernel": dom, "bound": "fp32", "achieved": tf, "peak": fp32_peak, "unit": "TFLOP/s", "frac": tf / fp32_peak,
                    "peak_source": "148 SMs x 128 FFMA lanes x 2 flop x max SM clock"}
        roof["traffic"] = NCU_TRAFFIC.get(workload, {}).get(dom)
        roof["launch_us"] = per_launch_s * 1e6
        roof["launches_per_step"] = launches_per_step
        roof["algorithmic_bytes_per_launch"] = wk["byte"] / launches_per_step
        roof["algorithmic_flop_per_launch"] = wk["flop"] / launches_per_step
        roof["also"] = {"algorithmic_GB_per_s": gb, "hbm_frac": gb / pk["hbm"], "algorithmic_TFLOP_per_s": tf,
                        "fp32_frac": tf / fp32_peak, "tensor_frac": tf / pk["tensor_sustained"],
                        # an fp32-accurate product costs three TF32 MMAs, and TF32 runs at half the bf16 rate: the roof such a kernel
                        # could reach at best
                        "tf32x3_frac": tf / (pk["tensor_sustained"] / 6.0)}
        if wk["pipe"] == "tensor":
            roof["note"] = ("3xTF32 mma.sync (m16n8k8) kernel at d = 40: latency- and occupancy-bound, not peak-bound; ncu "
                            "sm__pipe_tensor_cycles_active for this launch is in profiles/ (22.8 % for attn_bwd)")
    flop, byte = step_work(w)
    s_ = ms_per_step / 1e3
    roof_step = {"algorithmic_GB_per_step": byte / 1e9, "algorithmic_GFLOP_per_step": flop / 1e9, "GB_per_s": byte / s_ / 1e9,
                 "TFLOP_per_s": flop / s_ / 1e12, "hbm_frac": byte / s_ / 1e9 / pk["hbm"], "fp32_frac": flop / s_ / 1e12 / fp32_peak,
                 "tensor_frac": flop / s_ / 1e12 / pk["tensor_sustained"],
                 "note": "whole step: every tensor of the minimal algorithm read / written once, 2 flop per multiply-add; at this "
                         "batch the step is bound by launch latency and occupancy, not by a roof"}
    return roof, roof_step


def score_batch(seed, w):
    """One scoring batch in the eval layout: `group` consecutive rows (1 positive + group-1 negatives) share a history."""
    from pamrec_b200 import synth
    B, g = w["B"], w["group"]
    a = synth.array_batch(seed, B // g, w["T"], w["n_users"], w["n_items"], w["n_cates"], grouped=False, zipf_a=w.get("zipf", 1.1))
    rng = np.random.default_rng(seed + 1)
    out = {k: np.repeat(a[k], g, axis=0) for k in ("item_history", "item_cate_history", "item_loop_times_history", "mask", "users")}
    out["items"] = rng.integers(1, w["n_items"], size=B).astype(np.int32)
    out["cates"] = rng.integers(1, w["n_cates"], size=B).astype(np.int32)
    lab = np.zeros((B // g, g), np.float32); lab[:, 0] = 1.0
    out["labels_satisfied"] = lab.reshape(B, 1)
    out["labels_play"] = lab.reshape(B, 1).copy()
    out["plays"] = (lab.reshape(B, 1) * 12.0).astype(np.float32)
    return out


def run_score(args, w, rank, world):
    """BASELINE.json configs[4]: eval-only scoring, 1 positive + 99 negatives per impression.  value = forward passes (BN inference
    mode) over resident batches, device-timed; e2e = run_weighted_eval (SBM:420-500) over an 11-column text file, host one batch
    ahead of the device, including batching, H2D / D2H copies and the ranking metrics."""
    from pamrec_b200 import synth
    pk = peaks()
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
    dev = torch.device("cuda", torch.cuda.current_device())
    shared = os.path.join(tempfile.gettempdir(), "pamrec_bench_eval_" + os.environ.get("MASTER_PORT", str(os.getpid())))
    os.makedirs(shared, exist_ok=True)
    B, T, g = w["B"], w["T"], w["group"]
    model = build_model(w, tempfile.mkdtemp(prefix="pamrec_bench_"), batch_size=B * world,
                        pairwise_metrics=["mean_mrr", "ndcg@10", "hit@10", "group_auc"], weighted_metrics=["wauc"])
    eng = model.engine
    resident = [eng.upload(score_batch(1000 + 17 * i + rank, w), training=False) for i in range(N_POOL)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    K, W = args.steps, args.warmup

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    clocks = ClockSampler(torch.cuda.current_device()).start()
    for i in range(W):
        eng.forward(resident[i % N_POOL], training=False)
    barrier()
    settle_sampler(clocks, dev, world, lambda: eng.forward(resident[0], training=False))
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    barrier()
    for i in range(K):
        flush.fill_(i & 0xFF)
        a, b = evs[i]
        a.record()
        pred = eng.forward(resident[i % N_POOL], training=False)
        b.record()
    barrier()
    outputs = {"pred": pred} if args.dump_outputs else None
    launches = eng.launches()
    total_ms = sum(a.elapsed_time(b) for a, b in evs)
    if world > 1:
        t = torch.tensor([total_ms], device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        total_ms = float(t.item())
    value = B * world * K / (total_ms / 1e3)
    # ---- e2e through the public scoring loop
    path = os.path.join(shared, "test_data")
    if rank == 0:
        synth.write_eval_file(path, w["impressions"] * world, g - 1, T, w["n_users"], w["n_items"], w["n_cates"], seed=5)
    barrier()
    rows = w["impressions"] * world * g
    res = model.run_weighted_eval(path, num_ngs=g - 1)           # first pass: tokenises the file (cached per file, IT:366-370)
    barrier()
    reps = max(1, -(-K * B * world // rows))
    t0 = time.perf_counter()
    for _ in range(reps):
        res = model.run_weighted_eval(path, num_ngs=g - 1)
    barrier()
    e2e_s = time.perf_counter() - t0
    clk = clocks.stop()
    if world > 1:
        t = torch.tensor([e2e_s], device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        e2e_s = float(t.item())
    h2d = resident[0].h2d_bytes
    e2e = {"value": rows * reps / e2e_s, "unit": "samples/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4 * B,
           "passes": reps, "rows_per_pass": rows, "metrics_of_last_pass": res}
    eng.profile(True)
    for i in range(K):
        flush.fill_(i & 0xFF)
        eng.forward(resident[i % N_POOL], training=False)
    tab = eng.profile_table()
    eng.profile(False)
    tot = sum(ms for ms, _ in tab.values())
    kernels = {k: {"ms_per_step": ms / K, "share": ms / tot, "launches_per_step": n / K} for k, (ms, n) in
               sorted(tab.items(), key=lambda kv: -kv[1][0])}
    roof, roof_step = rooflines(w, tab, K, total_ms / K, pk, clk, args.workload)
    out = {
        "metric": METRIC_SCORE, "value": value, "unit": "samples/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "impl": "pamrec_b200",
        "config": {"workload": args.workload, "batch_per_gpu": B, "seq_len": T, "group": g, "n_items": w["n_items"],
                   "n_cates": w["n_cates"], "n_users": w["n_users"], "global_batch": B * world, "tables": eng.tables,
                   "parallelism": "single GPU" if world == 1 else f"dp{world}: rows r, r + N, ... of every batch scored by rank r",
                   "l2": "flushed between timed steps (256 MiB write)",
                   "e2e_note": f"run_weighted_eval over a text file of {rows} lines ({w['impressions'] * world} impressions x {g}), batches of "
                               f"{B * world} rows queued one ahead of the host, metrics auc / logloss / mean_mrr / ndcg@10 / hit@10 / group_auc / wauc included"},
        "e2e": e2e, "gpu_launches": int(launches) * K, "gpu_launches_per_step": int(launches), "clocks": clk, "roofline": roof,
        "roofline_step": roof_step, "kernels": kernels,
    }
    return out, model, outputs


def sample_rows(w):
    """Rows per CPU step: the whole batch when it fits the time budget (<= ~52 K tokens), else a bounded sample of whole groups."""
    return w["B"] if w["B"] * w["T"] <= 52000 else max(5, (41000 // w["T"]) // 5 * 5)


def cpu_baseline(w, seconds=20.0, rows=None):
    """The oracle port of the reference step (torch CPU fp32, all host threads) on a bounded sample of the workload."""
    from oracle import pamrec_oracle as O            # CPU baseline arm: the one place bench.py executes oracle/
    from pamrec_b200 import synth
    torch.set_num_threads(os.cpu_count() or 1)
    rows = rows or sample_rows(w)
    score = w.get("kind") == "score"
    om = O.OracleModel(w["n_users"], w["n_items"], w["n_cates"], w["T"], dtype=torch.float32)
    feeds = [synth.array_batch(50 + i, rows, w["T"], w["n_users"], w["n_items"], w["n_cates"], grouped=not score) for i in range(4)]
    for f in feeds:
        f["mask"] = f["mask"].astype(np.int32); f["users"] = f["users"].astype(np.int32)
    step = om.eval_forward if score else om.train_step
    step(feeds[0])
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        step(feeds[n % 4])
        n += 1
    dt = time.perf_counter() - t0
    return {"value": n * rows / dt, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{n} {'scoring' if score else 'training'} steps of {rows} rows (T={w['T']}) of the same synthetic workload, {dt:.1f} s",
            "note": "restated CPU baseline (oracle/pamrec_oracle.py, torch CPU fp32): TF 2.4 is not installable offline"}


def run_reference(args, w, rank):
    """--impl reference: the reference's CPU implementation of the path = the oracle port (TF cannot be installed)."""
    if rank != 0:
        return None
    from oracle import pamrec_oracle as O
    from pamrec_b200 import synth
    torch.set_num_threads(os.cpu_count() or 1)
    rows = sample_rows(w)
    score = w.get("kind") == "score"
    om = O.OracleModel(w["n_users"], w["n_items"], w["n_cates"], w["T"], dtype=torch.float32)
    feeds = [synth.array_batch(50 + i, rows, w["T"], w["n_users"], w["n_items"], w["n_cates"], grouped=not score) for i in range(4)]
    for f in feeds:
        f["mask"] = f["mask"].astype(np.int32); f["users"] = f["users"].astype(np.int32)
    step = om.eval_forward if score else om.train_step
    for i in range(args.warmup):
        step(feeds[i % 4])
    t0 = time.perf_counter()
    for i in range(args.steps):
        last = step(feeds[i % 4])
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"pred": last.t["pred"].reshape(-1)} if score else
                     {"losses": np.array([last["losses"][k] for k in ("loss", "data_loss", "regular_loss", "auxiliary_data_loss",
                                                                      "order_loss")])})
    v = args.steps * rows / dt
    whole = rows == w["B"]
    cb = {"value": v, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
          "sample": (f"each step = the whole {rows}-row batch" if whole else f"each step = {rows} rows (a bounded sample of the {w['B']}-row batch)")
                    + f" of the {args.workload} workload"}
    return {"metric": METRIC_SCORE if score else METRIC, "value": v, "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": args.workload, "batch_per_step": rows, "batch_per_gpu": w["B"], "seq_len": w["T"], "same_rows_as_gpu_arm": whole,
                       "note": "oracle port of the reference TF graph on host cores; TF 2.4 / tensorflow_ranking not installable offline"},
            "cpu_baseline": cb, "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def main():
    # libraries (NCCL's version banner, torch warnings) print to fd 1: keep the real stdout for the ONE JSON line
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="pamrec_b200", choices=["pamrec_b200", "reference"])
    ap.add_argument("--workload", default="takatak_b1025_t50", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    w = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # started as plain `python bench.py --gpus N`: become the torchrun launch the contract describes (one rank per GPU)
        import socket
        with socket.socket() as sock:
            sock.bind(("127.0.0.1", 0))
            port = sock.getsockname()[1]
        os.dup2(real_stdout.fileno(), 1)
        os.execv(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                                  "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__), *sys.argv[1:]])
    if args.impl == "reference":
        out = run_reference(args, w, rank)
        if out is not None:
            print(json.dumps(out), file=real_stdout, flush=True)
        return
    if world > 1:
        local = int(os.environ.get("LOCAL_RANK", rank))
        torch.cuda.set_device(local)
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))
    out, model, outputs = (run_score if w.get("kind") == "score" else run_ours)(args, w, rank, world)
    if rank == 0:
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(w)
        print(json.dumps(out), file=real_stdout, flush=True)
    if world > 1:
        torch.distributed.barrier()
        model.engine.close()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
