#!/usr/bin/env python
"""Per-barrier timeline of the persistent head kernels on a bench workload (PAMREC_DEBUG_HEAD_TRACE).

    python tools/head_trace.py [--workload takatak_b1025_t50]
Prints, for the forward and the backward head kernel of one training step, the time of every barrier release relative to the
kernel start and the duration of every barrier interval (us), next to the phases the interval runs."""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from pamrec_b200 import _lib as L  # noqa: E402
from pamrec_b200 import synth  # noqa: E402
from pamrec_b200.engine import Engine  # noqa: E402

FWD = ["F1 score layer 0 (tokens)", "F2 score layer 1 (tokens)", "F3 pooling + experts / gates layer 0", "F4 experts / gates layer 1",
       "F5 mixing + towers layer 0", "F6 towers layer 1", "F7 logits (to the end of CTA 0)"]
BWD = ["K0 weight transposes + losses", "K1 dA(t1)", "K2 dz(t1) -> dA(t0)", "K3 dz(t0) -> d_u -> mixing backward", "K4 dz(e1, g1) -> dA(e0, g0)",
       "K5 dz(e0, g0) -> d_new_long -> pooling backward", "K6 dz2 -> sums of BN_S0, score layer 1 gradients",
       "K7 dz1 -> dH, score layer 0 gradients (to the end of CTA 0)"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="takatak_b1025_t50")
    a = ap.parse_args()
    w = bench.WORKLOADS[a.workload]
    eng = Engine(w["n_users"], w["n_items"], w["n_cates"], w["T"], w["B"]).allocate("cuda:0")
    eng.pool["dense_param"].normal_(0, 0.05)
    eng.pool["item_w"].normal_(0, 0.01)
    eng.pool["cate_w"].normal_(0, 0.01)
    db = eng.upload(synth.array_batch(3, w["B"], w["T"], w["n_users"], w["n_items"], w["n_cates"]))
    for _ in range(5):
        eng.train_step(db)
    eng.set_debug(L.DEBUG_HEAD_TRACE)
    acc = {}
    reps = 20
    for _ in range(reps):
        eng.train_step(db)
        torch.cuda.synchronize()
        for name, bwd in (("forward", False), ("backward", True)):
            acc.setdefault(name, []).append(eng.head_trace(bwd))
    for name, labels in (("forward", FWD), ("backward", BWD)):
        t = np.median(np.asarray(acc[name], np.float64), axis=0) / 1e3
        print(f"{name}: {t[-1]:.1f} us from kernel start to the end of CTA 0, {len(t) - 1} barriers")
        prev = 0.0
        for i, x in enumerate(t):
            print(f"  {labels[i] if i < len(labels) else '?':50s} {x - prev:7.1f} us   (released at {x:7.1f})")
            prev = x


if __name__ == "__main__":
    main()
