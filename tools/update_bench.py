"""Throughput of evs_update_rows and its cost inside a serving loop (configs[1] shape).

  python tools/update_bench.py [--out DIR] [--steps K]

1. update throughput: one call of n keys, n in {1024, 65536, 1048576}, keys drawn uniformly over all rows of the 26
   Kaggle-shape tables (33.76 M rows, dim 16), for the configs[1] store (one fp32 tier, backing rows in evs_host_alloc
   memory) and the configs[2] 32/8 two-tier store.  CUDA events around 10 calls after 3 warm-up calls; rows/s and GB/s of
   backing-store bytes written (slab copies not counted).  Beside it, the device-to-host copy rate into pinned memory.
2. serving step: the configs[1] loop (B = 2048, Zipf(1.05), each batch announced with evs_prefetch) with 4096 updated rows
   every 4 batches (keys of the next batch half, random rows the other half), against the same loop without updates.  Each
   arm is timed twice, alternated, over 400 steps after a warm cache.

Prints one JSON line per measurement, with the GPU's name and power limit; --out DIR also writes them to
DIR/update_bench.jsonl.
"""
import argparse
import importlib
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
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return q
    except Exception as e:                       # the numbers stay valid; the line says what is missing
        return f"unknown ({e!r})"


def random_keys(rng, rows, n):
    rows = np.asarray(rows, dtype=np.int64)
    cum = np.cumsum(rows)
    g = (rng.random(n) * cum[-1]).astype(np.int64)
    t = np.searchsorted(cum, g, side="right")
    r = g - np.concatenate([[0], cum[:-1]])[t]
    return t, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="", help="directory for update_bench.jsonl (default: print only)")
    ap.add_argument("--steps", type=int, default=400)
    args = ap.parse_args()
    import torch
    pkg = importlib.import_module("ev-store-dlrm_b200")
    info = gpu_info()
    lines = []

    def emit(d):
        d["gpu"] = info
        print(json.dumps(d), flush=True)
        lines.append(d)

    rows, dim, B = pkg.workload.KAGGLE_ROWS, 16, 2048
    cache_rows = pkg.workload.KAGGLE_CACHE_ROWS
    t0 = time.time()
    tables = [pkg.to_host_rows(t) for t in pkg.workload.make_tables(rows, dim)]
    print(f"# tables built in {time.time() - t0:.1f} s", file=sys.stderr)
    rng = np.random.default_rng(0)

    # D2H copy rate into pinned memory: the host store's write path goes over the same link
    src = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    dst = torch.empty(256 << 20, dtype=torch.uint8, pin_memory=True)
    for _ in range(3):
        dst.copy_(src, non_blocking=True)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(10):
        dst.copy_(src, non_blocking=True)
    b.record()
    torch.cuda.synchronize()
    emit({"what": "d2h_copy_pinned", "GB_per_s": 10 * (256 << 20) / (a.elapsed_time(b) * 1e-3) / 1e9})
    del src, dst

    configs = {"configs1_fp32": dict(n_layers=1, main_precision=32, total_size=cache_rows),
               "configs2_32_8": dict(n_layers=2, main_precision=32, secondary_precision=8, total_size=cache_rows)}
    for name, kw in configs.items():
        stores = None
        if kw["n_layers"] == 2:
            stores = {32: tables, 8: [pkg.to_host_rows(pkg.codecs.encode_table(t, 8)) for t in tables]}
        store = pkg.EvStore(tables, pkg.CacheConfig(max_batch=B, **kw), stores=stores)
        trace = pkg.workload.ZipfTrace(rows, seed=1)
        for _ in range(200):                                   # resident rows, so that slab copies are written too
            store.lookup(torch.from_numpy(trace.batch(B)).cuda())
        row_bytes = dim * 4 + (dim * kw.get("secondary_precision", 0) // 8)
        for n in (1024, 65536, 1048576):
            t, r = random_keys(rng, rows, n)
            tt, rr = torch.from_numpy(t).cuda(), torch.from_numpy(r).cuda()
            v = torch.rand((n, dim), device="cuda") * 1.8 - 0.9
            for _ in range(3):
                store.update_rows(tt, rr, v)
            torch.cuda.synchronize()
            a.record()
            for _ in range(10):
                w = store.update_rows(tt, rr, v)
            b.record()
            torch.cuda.synchronize()
            s = a.elapsed_time(b) * 1e-3 / 10
            n_res = int(((w & 3) != 0).sum())
            emit({"what": "update_rows", "config": name, "n": n, "us_per_call": s * 1e6, "rows_per_s": n / s,
                  "store_GB_per_s": n * row_bytes / s / 1e9, "store_bytes_per_row": row_bytes, "resident_copies": n_res})
        store.close()

    # serving step with and without updates
    store = pkg.EvStore(tables, pkg.CacheConfig(max_batch=B, n_layers=1, main_precision=32, total_size=cache_rows))
    trace = pkg.workload.ZipfTrace(rows, seed=2)
    n_tr = 64
    idx = [torch.from_numpy(trace.batch(B)).cuda() for _ in range(n_tr)]
    host_idx = [x.cpu().numpy() for x in idx]
    for k in range(1500):                                          # warm: the cache is full after ~1000 batches
        store.lookup(idx[k % n_tr])
        store.prefetch(idx[(k + 1) % n_tr])
    torch.cuda.synchronize()
    upd = []
    for k in range(n_tr):
        nxt = host_idx[(k + 1) % n_tr]
        pos = rng.choice(26 * B, size=2048, replace=False)
        tn, rn = pos // B, nxt.reshape(-1)[pos]
        tr_, rr_ = random_keys(rng, rows, 2048)
        t = torch.from_numpy(np.concatenate([tn, tr_])).cuda()
        r = torch.from_numpy(np.concatenate([rn, rr_])).cuda()
        upd.append((t, r, torch.rand((4096, dim), device="cuda") * 1.8 - 0.9))

    def run(with_updates, steps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k in range(steps):
            store.lookup(idx[k % n_tr])
            if with_updates and k % 4 == 3:
                store.update_rows(*upd[k % n_tr])
            store.prefetch(idx[(k + 1) % n_tr])
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / steps

    res = {False: [], True: []}
    for rep in range(2):
        for wu in (False, True):
            res[wu].append(run(wu, args.steps) * 1e6)
    emit({"what": "serving_step", "config": "configs1_fp32", "B": B, "steps": args.steps,
          "us_per_step_no_updates": res[False], "us_per_step_4096_rows_every_4": res[True]})
    store.close()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "update_bench.jsonl"), "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
