#!/usr/bin/env python
"""Cost of TensorBoard summaries (write_tfevents) on one GPU; one JSON line per measurement, each with the GPU's name and power limit.

    python tools/bench_summaries.py [--steps K] [--rounds R] [--out DIR]

1. takatak_b1025_t50 through PAMRECModel.train_async one step ahead (the way fit_step runs), with summaries off, with
   summary_step = 1 and with summary_step = 100, the three alternated R times in one process; event files go to a temporary
   directory and are flushed and closed inside the timed region.  Reports samples/s and bytes of event file per summarised step.
2. The histogram launches alone (pamrec_histograms: bin, finalize, compact) over one fp32 tensor of 160 M values, the item
   table of sharded_10m_b1025_t50 (10 M rows x 16), timed with CUDA events; bytes/s = 640 MB / time, against 7.7 TB/s."""
import argparse
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

HBM_TBS = 7.7


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True)
    name, power, clock = [x.strip() for x in r.stdout.strip().splitlines()[torch.cuda.current_device()].split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


def e2e(model, feeds, steps, summary_dir):
    """samples/s of `steps` pipelined train steps, and the bytes of event file they wrote."""
    if summary_dir:
        model.hparams.SUMMARIES_DIR = summary_dir
        model._open_summaries()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pending = None
    for i in range(steps):
        queued = model.train_async(None, feeds[i % len(feeds)])
        if pending is not None:
            pending.result()
        pending = queued
    pending.result()
    model._close_summaries()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    nbytes = sum(os.path.getsize(os.path.join(summary_dir, f)) for f in os.listdir(summary_dir)) if summary_dir else 0
    return feeds[0]["items"].shape[0] * steps / dt, nbytes


def kernel_time(eng, n_values, reps):
    from pamrec_b200 import _lib as L
    x = torch.randn(n_values, device="cuda") * 0.01
    counts = (C.c_int64 * 1)(n_values)
    offs = (C.c_int64 * 2)(0, L.HIST_BUCKETS)
    need = C.c_int64(0)
    eng._check(eng.lib.pamrec_histograms(eng.handle, None, counts, 1, 0, None, None, None, None, C.byref(need), None))
    scratch = torch.empty(need.value, dtype=torch.uint8, device="cuda")
    stats = torch.empty(7, dtype=torch.float64, device="cuda")
    out = torch.empty(2 * L.HIST_BUCKETS, dtype=torch.float64, device="cuda")
    ptrs = (C.c_void_p * 1)(x.data_ptr())
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def run():
        eng._check(eng.lib.pamrec_histograms(eng.handle, ptrs, counts, 1, 0, offs, C.c_void_p(stats.data_ptr()),
                                             C.c_void_p(out.data_ptr()), C.c_void_p(scratch.data_ptr()), C.byref(need), stream))
    for _ in range(3):
        run()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in evs:                                  # 640 MB per launch: far more than the 126 MB L2, read from HBM every time
        a.record()
        run()
        b.record()
    torch.cuda.synchronize()
    ms = sorted(a.elapsed_time(b) for a, b in evs)
    return ms[len(ms) // 2], ms[0], eng.launches()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON lines to DIR/bench_summaries.jsonl")
    args = ap.parse_args()
    import bench
    from pamrec_b200 import synth
    info = gpu_info()
    lines = []

    def emit(d):
        d = {**info, **d}
        print(json.dumps(d), flush=True)
        lines.append(d)

    w = bench.WORKLOADS["takatak_b1025_t50"]
    tmp = tempfile.mkdtemp(prefix="pamrec_sum_")
    try:
        model = bench.build_model(w, tmp)
        feeds = [synth.array_batch(1000 + 17 * i, w["B"], w["T"], w["n_users"], w["n_items"], w["n_cates"]) for i in range(8)]
        e2e(model, feeds, 20, None)                       # warm-up: CUDA graphs of both staging slots, pinned buffers
        model.hparams.write_tfevents = True
        model.hparams.summary_step = 1
        e2e(model, feeds, 4, os.path.join(tmp, "warm"))   # the histogram buffers of the checkpoint's name list
        for r in range(args.rounds):
            for label, on, every in (("off", False, 1), ("summary_step=1", True, 1), ("summary_step=100", True, 100)):
                model.hparams.write_tfevents, model.hparams.summary_step = on, every
                d = os.path.join(tmp, f"r{r}_{every}_{int(on)}") if on else None
                rate, nbytes = e2e(model, feeds, args.steps, d)
                n_sum = sum(1 for s in range(model.engine.step - args.steps + 1, model.engine.step + 1) if s % every == 0) if on else 0
                emit(dict(measure="takatak_b1025_t50 e2e", round=r, summaries=label, steps=args.steps, samples_per_s=round(rate, 1),
                          summarised_steps=n_sum, event_bytes=nbytes, bytes_per_summarised_step=round(nbytes / n_sum) if n_sum else 0))
        n = 10_000_000 * 16
        med, best, launches = kernel_time(model.engine, n, 20)
        emit(dict(measure="histogram kernels, one 160 M float segment", values=n, launches=launches, median_ms=round(med, 4),
                  best_ms=round(best, 4), gb_per_s=round(4 * n / med / 1e6, 1), share_of_7_7_tb_s=round(4 * n / med / 1e6 / (HBM_TBS * 1e3), 3)))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_summaries.jsonl"), "a") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
