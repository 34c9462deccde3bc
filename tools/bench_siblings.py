"""Train-step throughput of the sibling baselines (MMoEModel_original / PLEModel / ShareBottomModel / SASRecModel) on the takatak bench
shape (B = 1025, T = 50): one JSON line per model with the device-timed samples/s (8 resident batches, L2 flushed between steps),
the end-to-end number through Model.train_async with host feeds (one step ahead, as fit_step runs) and the per-launcher table.

    python tools/bench_siblings.py [--steps 200] [--warmup 10] [--emb-dims {mmoe,reference}]

--emb-dims mmoe runs every model at config/mmoe.yaml's embedding widths (item / cate / user = 16 / 4 / 20); reference at the
reference's own widths: 32 / 8 / 40 (MMoE, PLE, share-bottom; ple.yaml, sharebottom.yaml) and 32 / 8 / 16 (SASRec, sasrec.yaml).
Every line names the GPU and its power limit: the rates belong to them.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

W = dict(dataset="takatak", n_users=50000, n_items=30000, n_cates=50, T=50, B=1025)
MODELS = (("MMoEModel_original", "mmoe.yaml"), ("PLEModel", "ple.yaml"), ("ShareBottomModel", "sharebottom.yaml"), ("SASRecModel", "sasrec.yaml"))
EMB_DIMS = {"mmoe": {}, "reference": {"SASRecModel": (32, 8, 16), None: (32, 8, 40)}}


def gpu_info():
    """name and power limit of GPU 0, read in the same run as the measurement"""
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=60).stdout.strip()
        name, power, clock = (x.strip() for x in out.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except (OSError, ValueError, subprocess.SubprocessError):
        return {"name": torch.cuda.get_device_name(0), "power_limit": "unknown", "max_sm_clock": "unknown"}


def satisfied_fields(feed, seed):
    """the satisfied-only copy of the history as `_convert_data` builds it (IT:1069-1103): satisfied entries compacted to the left"""
    rng = np.random.default_rng(seed)
    ih, ch, mask = feed["item_history"], feed["item_cate_history"], feed["mask"]
    sat = (rng.random(ih.shape) < 0.5) & (mask == 1)
    order = np.argsort(~sat, axis=1, kind="stable")
    keep = np.arange(ih.shape[1])[None, :] < sat.sum(1)[:, None]
    out = dict(feed)
    out["satisfied_item_history"] = np.where(keep, np.take_along_axis(ih, order, 1), 0).astype(np.int32)
    out["satisfied_cate_history"] = np.where(keep, np.take_along_axis(ch, order, 1), 0).astype(np.int32)
    out["satisfied_mask"] = keep.astype(np.float32)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--emb-dims", choices=sorted(EMB_DIMS), default="mmoe")
    args = ap.parse_args()
    from pamrec_b200 import models as M
    from pamrec_b200 import synth
    from pamrec_b200.deeprec_utils import prepare_hparams
    from pamrec_b200.sequential_iterator import SequentialIterator
    dev = torch.device("cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    B, T = W["B"], W["T"]
    gpu = gpu_info()
    feeds = [satisfied_fields(synth.array_batch(1000 + 17 * i, B, T, W["n_users"], W["n_items"], W["n_cates"]), 5000 + i) for i in range(8)]
    for cls_name, yaml_name in MODELS:
        tmp = tempfile.mkdtemp(prefix="pamrec_sib_")
        d = synth.write_vocab_only(tmp, W["dataset"], W["n_users"], W["n_items"], W["n_cates"])
        table = EMB_DIMS[args.emb_dims]
        dims = table.get(cls_name, table.get(None))
        widths = {} if dims is None else dict(item_embedding_dim=dims[0], cate_embedding_dim=dims[1], user_embedding_dim=dims[2])
        hp = prepare_hparams(os.path.join(ROOT, "pamrec_b200", "config", yaml_name), dataset=W["dataset"], bucket_num=10, add_feature=False,
                             embed_l2=1e-6, layer_l2=1e-6, learning_rate=0.001, epochs=1, EARLY_STOP=5, is_clip_norm=1, batch_size=B,
                             show_step=10 ** 9, MODEL_DIR=os.path.join(tmp, "model/"), SUMMARIES_DIR=os.path.join(tmp, "summary/"),
                             user_vocab=os.path.join(d, "user_vocab.pkl"), item_vocab=os.path.join(d, "item_vocab.pkl"),
                             cate_vocab=os.path.join(d, "category_vocab.pkl"), train_num_ngs=0, max_seq_length=T, pairwise_metrics=[],
                             weighted_metrics=["wauc"], eval_step=10 ** 9, noise_train_hist=0, noise_train_listwise=0, noise_only_predict=0,
                             write_tfevents=False, **widths)
        model = getattr(M, cls_name)(hp, SequentialIterator, seed=8)
        eng = model.engine
        resident = [eng.upload(f) for f in feeds]
        for i in range(args.warmup):
            eng.train_step(resident[i % 8])
        torch.cuda.synchronize()
        evs = []
        for i in range(args.steps):
            flush.fill_(i & 0xFF)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            eng.train_step(resident[i % 8])
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        ms = sum(a.elapsed_time(b) for a, b in evs) / args.steps
        launches = eng.launches()

        def e2e_pass(n):
            pending = None
            for i in range(n):
                queued = model.train_async(None, feeds[i % 8])
                if pending is not None:
                    pending.result()
                pending = queued
            pending.result()
        e2e_pass(args.warmup)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e2e_pass(args.steps)
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        eng.profile(True)
        for i in range(args.steps):
            eng.train_step(resident[i % 8])
        tab = eng.profile_table()
        eng.profile(False)
        print(json.dumps({"metric": "train samples/sec", "model": cls_name, "value": B * 1e3 / ms, "unit": "samples/s", "ms_per_step": ms,
                          "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "dtype": "f32", "data": "synthetic",
                          "config": {"workload": "takatak_b1025_t50", "batch": B, "seq_len": T, "sparse_adam": "dense_exact",
                                     "emb_dims": list(eng.emb_dims)},
                          "gpu": gpu,
                          "e2e": {"value": B * args.steps / e2e_s, "unit": "samples/s",
                                  "h2d_bytes_per_step": int(eng.upload(feeds[0], staged=True).h2d_bytes), "d2h_bytes_per_step": 20},
                          "gpu_launches_per_step": launches,
                          "kernels": {k: {"ms_per_step": v[0] / args.steps, "launches_per_step": v[1] / args.steps}
                                      for k, v in sorted(tab.items(), key=lambda kv: -kv[1][0])}}), flush=True)
        eng.close()
        del model, eng, resident


if __name__ == "__main__":
    main()
