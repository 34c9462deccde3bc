"""Candidate ranking throughput (Engine.rank_candidates, pamrec_rank_candidates) on one GPU, one JSON line per measurement, each
with the GPU's name and power limit.

  full   : every model ranks `--lines` scoring lines against `--cands` candidates at the takatak shape (T = 50): scored
           (line, candidate) rows per second and seconds per 1 000 lines (top 10, history excluded);
  1p99   : 100 candidates per line through rank_candidates against the same 100 rows per line materialised on the host and scored
           batch by batch (upload + forward: the device part of run_weighted_eval's scoring loop, without its metrics), PAMRec.

Usage: python tools/bench_rank.py [--lines 64] [--cands 30000] [--max-batch 8192] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
        return name, power
    except Exception:
        import torch
        return torch.cuda.get_device_name(0), "unknown"


def engine(model, dims, n_users, n_items, n_cates, T, max_batch, seed=1):
    import types
    from pamrec_b200.engine import Engine
    from pamrec_b200.models import initial_variables
    eng = Engine(n_users, n_items, n_cates, T, max_batch, model=model, emb_dims=dims).allocate("cuda:0")
    eng.set_variables(initial_variables(eng.variable_shapes(), types.SimpleNamespace(init_method="tnormal", init_value=0.1), seed))
    return eng


def lines_batch(n, T, n_users, n_items, n_cates, seed):
    from oracle import pamrec_oracle as O
    from oracle import siblings_oracle as S
    return S.add_satisfied_fields(O.make_batch(seed, n, T, n_users, n_items, n_cates, grouped=False, min_len=T // 2), seed=seed)


def timed(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lines", type=int, default=64)
    ap.add_argument("--cands", type=int, default=30000)
    ap.add_argument("--max-batch", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_rank needs a CUDA device")
    name, power = gpu_info()
    nu, ni, nc, T = 20000, a.cands + 1, 500, 50                      # takatak-like vocabulary: every item but 0 is a candidate
    out = open(a.out, "w") if a.out else None

    def emit(rec):
        rec.update(gpu=name, power_limit=power)
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")

    rng = np.random.default_rng(0)
    ids = np.arange(1, ni, dtype=np.int32)
    cates = rng.integers(0, nc, size=ids.size).astype(np.int32)
    batch = lines_batch(a.lines, T, nu, ni, nc, 5)
    for model, dims in (("pamrec", (16, 4, 20)), ("mmoe", (16, 4, 20)), ("ple", (16, 4, 20)), ("sharebottom", (16, 4, 20)),
                        ("sasrec", (16, 4, 20))):
        eng = engine(model, dims, nu, ni, nc, T, a.max_batch)
        db = eng.upload(batch, training=False)
        cand_i, cand_c = torch.from_numpy(ids).cuda(), torch.from_numpy(cates).cuda()
        sec = timed(lambda: eng.rank_candidates(db, cand_i, cand_c, 10, True, True).result(), a.reps)
        rows = a.lines * ids.size
        emit(dict(bench="full", model=model, lines=a.lines, candidates=int(ids.size), T=T, max_batch=a.max_batch, seconds=round(sec, 4),
                  rows_per_s=round(rows / sec), s_per_1000_lines=round(sec / a.lines * 1000, 3)))
        eng.close()
    # 1 + 99: the same 100 candidate rows per line, on the device or materialised on the host
    n1, K1 = 1000, 100
    eng = engine("pamrec", (16, 4, 20), nu, ni, nc, T, 1000)
    lines = lines_batch(n1, T, nu, ni, nc, 6)
    ids100 = rng.permutation(ids)[:K1]
    cat100 = cates[ids100 - 1]
    db = eng.upload(lines, training=False)
    ci, cc = torch.from_numpy(ids100).cuda(), torch.from_numpy(cat100).cuda()
    sec_rank = timed(lambda: eng.rank_candidates(db, ci, cc, 10, False, True).result(), a.reps)
    rows = {k: np.repeat(np.asarray(v), K1, axis=0) for k, v in lines.items()}
    rows["items"], rows["cates"] = np.tile(ids100, n1), np.tile(cat100, n1)

    def host_path():
        for s in range(0, n1 * K1, 1000):
            part = {k: v[s:s + 1000] for k, v in rows.items()}
            eng.to_host_async(eng.forward(eng.upload(part, training=False, staged=True), training=False)).result()
    sec_host = timed(host_path, a.reps)
    for path, sec in (("rank_candidates", sec_rank), ("materialised_rows", sec_host)):
        emit(dict(bench="1p99", model="pamrec", path=path, lines=n1, candidates=K1, T=T, seconds=round(sec, 4),
                  rows_per_s=round(n1 * K1 / sec)))
    eng.close()
    if out:
        out.close()


if __name__ == "__main__":
    main()
