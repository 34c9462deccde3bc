"""Cost of the attention read-out (pamrec_attention) on one GPU, one JSON line per (model, shape), each with the GPU's name and power
limit.  Per shape, device time per call (host clock around calls that end in a synchronise, after a warm-up):

  forward_ms    : pamrec_forward(training = 0), the scoring pass it builds on;
  pool_ms       : pamrec_attention with the pooling weights only;
  maps_ms       : pamrec_attention with the encoder maps as well (device buffers, no host copy);
  maps_host_ms  : Engine.attention(db, maps=True).result(): the same plus the device -> host copy of the maps into pinned memory;
  maps_copy_ms, pinned_alloc_ms: its two host-side parts, the copy into a pinned buffer allocated once and the pinned allocation;
  map_kernel_ms : the maps kernel alone (the library's per-launcher CUDA events), with its store rate against the maps' bytes.

Shapes: the bench workloads takatak_b1025_t50, wechat_b500_t100, long_b4095_t200, for PAMRec and for SASRec (the sibling with an
encoder); the maps are 2 B T^2 floats (1.3 GB at long_b4095_t200), larger than L2, so every pass writes HBM.

Usage: python tools/bench_attention.py [--reps 20] [--out FILE]"""
import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_rank import engine, gpu_info, lines_batch  # noqa: E402

SHAPES = (("takatak_b1025_t50", 1025, 50), ("wechat_b500_t100", 500, 100), ("long_b4095_t200", 4095, 200))
MODELS = (("pamrec", (16, 4, 20)), ("sasrec", (32, 8, 16)))
HBM_BYTES_S = 7.7e12          # HGX B200 data sheet, one GPU


def timed(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps * 1e3


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    name, power = gpu_info()
    out = open(args.out, "w") if args.out else None
    nu, ni, nc = 10000, 100000, 100
    for model, dims in MODELS:
        for shape, B, T in SHAPES:
            eng = engine(model, dims, nu, ni, nc, T, B)
            db = eng.upload(lines_batch(B, T, nu, ni, nc, seed=3), training=False)
            lib, h, st = eng.lib, eng.handle, eng._stream()
            f32 = lambda *s: torch.empty(s, dtype=torch.float32, device=eng.device)
            pred, pool, maps = f32(B), f32(B, 1, T), f32(B, 2, T, T)
            ptr = lambda t: C.c_void_p(t.data_ptr())

            def call(rc):
                if rc != 0:
                    raise RuntimeError(lib.pamrec_last_error(h).decode())
            fwd = lambda: call(lib.pamrec_forward(h, C.byref(db.struct), 0, ptr(pred), st))
            att_pool = lambda: call(lib.pamrec_attention(h, C.byref(db.struct), ptr(pred), ptr(pool), None, st))
            att_maps = lambda: call(lib.pamrec_attention(h, C.byref(db.struct), ptr(pred), ptr(pool), ptr(maps), st))
            row = dict(gpu=name, power_limit=power, model=model, dims=list(dims), shape=shape, B=B, T=T, reps=args.reps)
            # alternate the three calls so that a drift of the clocks or a neighbour's load hits all of them alike
            ms = {"forward_ms": [], "pool_ms": [], "maps_ms": []}
            for _ in range(3):
                for key, fn in (("forward_ms", fwd), ("pool_ms", att_pool), ("maps_ms", att_maps)):
                    ms[key].append(timed(fn, args.reps))
            row.update({k: round(min(v), 4) for k, v in ms.items()})
            row["maps_host_ms"] = round(timed(lambda: eng.attention(db, maps=True).result(), max(3, args.reps // 4)), 3)
            # the split of maps_host_ms: the device -> host copy into a pinned buffer allocated once, and the pinned allocation
            host = torch.empty(maps.shape, dtype=torch.float32, pin_memory=True)
            row["maps_copy_ms"] = round(timed(lambda: host.copy_(maps), max(3, args.reps // 4)), 3)
            row["pinned_alloc_ms"] = round(timed(lambda: torch.empty(maps.shape, dtype=torch.float32, pin_memory=True), 3), 3)
            del host
            eng.profile(True)
            for _ in range(args.reps):
                att_maps()
            prof = eng.profile_table()
            eng.profile(False)
            k_ms, n = prof["attn_maps"]
            k_ms /= max(n, 1)
            nbytes = 2 * B * T * T * 4
            row.update(map_kernel_ms=round(k_ms, 4), maps_bytes=nbytes, map_store_TBps=round(nbytes / (k_ms * 1e-3) / 1e12, 3),
                       map_store_floor_ms=round(nbytes / HBM_BYTES_S * 1e3, 4),
                       map_score_TFLOPs=round(2 * (dims[0] + dims[1] if model == "sasrec" else 40) * B * 2 * T * T / (k_ms * 1e-3) / 1e12, 2),
                       maps_over_forward=round(row["maps_ms"] / row["forward_ms"], 3),
                       pool_over_forward=round(row["pool_ms"] / row["forward_ms"], 3))
            line = json.dumps(row)
            print(line, flush=True)
            if out:
                out.write(line + "\n")
                out.flush()
            eng.close()
            del eng, db, pred, pool, maps
            torch.cuda.empty_cache()
    if out:
        out.close()


if __name__ == "__main__":
    main()
