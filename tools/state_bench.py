"""Cost of evs_save_state / evs_load_state, and what a restore buys after a restart (configs[1] shape).

  python tools/state_bench.py [--out DIR] [--follow N]

For configs[1] (26 Kaggle-shape tables, 33.76 M rows, dim 16, one fp32 tier of 4 389 135 entries, backing rows in
evs_host_alloc memory, B = 2048, Zipf(1.05)) and the configs[2] 32/8 two-tier leg:
1. warm handle A by bench.py's rule (the batch at which the cache is full, plus 150);
2. save: blob size, device time (CUDA events around the call) and host time (the call synchronises);
3. load into a new handle B: the same two times, and rows loaded per second (every resident key's row is fetched
   zero-copy from the backing store);
4. the same following trace on B (restored) and on a new handle C (cold start, the restart without a snapshot): hit rate
   and mean step time over the first 1 / 16 / 256 batches, each batch announced with evs_prefetch as bench.py does.
   Step time = CUDA events around each batch's lookup, with the batch before it complete.

Prints one JSON line per measurement with the GPU's name and power limit; --out DIR also writes DIR/state_bench.jsonl.
"""
import argparse
import importlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from update_bench import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="", help="directory for state_bench.jsonl (default: print only)")
    ap.add_argument("--follow", type=int, default=256, help="batches after the restart")
    args = ap.parse_args()
    import torch
    import bench
    pkg = importlib.import_module("ev-store-dlrm_b200")
    info = gpu_info()
    lines = []

    def emit(d):
        d["gpu"] = info
        print(json.dumps(d), flush=True)
        lines.append(d)

    rows, dim, B = pkg.workload.KAGGLE_ROWS, 16, 2048
    cap = pkg.workload.KAGGLE_CACHE_ROWS
    tables = [pkg.to_host_rows(t) for t in pkg.workload.make_tables(rows, dim)]
    n_search = 4200
    idx = pkg.workload.ZipfTrace(rows, seed=42).batches(n_search + args.follow + 1, B)
    n_full = bench.batches_until_full(idx[:n_search], rows, cap)
    warm = min(n_search, n_full + 150)
    follow = idx[warm:warm + args.follow + 1]
    legs = [("configs[1]", dict(total_size=cap, max_batch=B)),
            ("configs[2] 32/8", dict(total_size=cap, max_batch=B, n_layers=2, main_precision=32, secondary_precision=8))]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ev0.record()
        r = fn()
        ev1.record()
        torch.cuda.synchronize()
        return r, ev0.elapsed_time(ev1), (time.perf_counter() - t0) * 1e3

    def serve(store, batches):
        """Per batch: (hit positions, step ms); each batch announced ahead with evs_prefetch."""
        d = torch.from_numpy(batches).cuda()
        out = torch.empty((B, 26, dim), dtype=torch.float32, device="cuda")
        hit = torch.empty((B, 26), dtype=torch.uint8, device="cuda")
        res = []
        store.prefetch(d[0])
        for k in range(len(batches) - 1):
            torch.cuda.synchronize()
            ev0.record()
            store.lookup(d[k], out=out, hit=hit)
            ev1.record()
            store.prefetch(d[k + 1])
            torch.cuda.synchronize()
            res.append((int((hit != 0).sum()), ev0.elapsed_time(ev1)))
        return res

    for name, cfg in legs:
        a = pkg.EvStore(tables, pkg.CacheConfig(**cfg))
        d = torch.from_numpy(idx[:warm]).cuda()
        for k in range(warm):
            a.lookup(d[k])
        torch.cuda.synchronize()
        del d
        size = a.stats()["size"]
        blob, dev_ms, host_ms = timed(lambda: a.save_state())
        keys = sum(size)
        emit({"leg": name, "what": "save", "warm_batches": warm, "resident": size, "blob_bytes": int(blob.nbytes),
              "device_ms": round(dev_ms, 3), "host_ms": round(host_ms, 3)})
        a.close()
        b = pkg.EvStore(tables, pkg.CacheConfig(**cfg))
        _, dev_ms, host_ms = timed(lambda: b.load_state(blob))
        emit({"leg": name, "what": "load", "keys": keys, "device_ms": round(dev_ms, 3), "host_ms": round(host_ms, 3),
              "rows_per_s_device": round(keys / (dev_ms * 1e-3)), "rows_per_s_host": round(keys / (host_ms * 1e-3))})
        c = pkg.EvStore(tables, pkg.CacheConfig(**cfg))
        for arm, st in (("restored", b), ("cold", c)):
            r = serve(st, follow)
            for n in (1, 16, args.follow):
                h = sum(x[0] for x in r[:n])
                emit({"leg": name, "what": "after_restart", "arm": arm, "first_batches": n,
                      "hit_rate": round(h / (n * B * 26), 5), "mean_step_ms": round(float(np.mean([x[1] for x in r[:n]])), 4)})
        b.close()
        c.close()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "state_bench.jsonl"), "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
