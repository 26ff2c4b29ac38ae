#!/usr/bin/env python
"""A/B of tuning switches on the bench workload (configs[1]) in ONE process: the tables and the index
trace are built once, then for every variant (a set of EVSTORE_B200_* environment variables, read by
evs_create) a fresh EvStore is created, warmed with the same batches and timed over the same batches.

    python tools/ab_bench.py default "EVSTORE_B200_PDL=0" \
                             "EVSTORE_B200_PDL=0,EVSTORE_B200_EVICT_CTAS=96"

One JSON line per variant on stdout (value = lookups/s, device-resident indices, CUDA events).
"""
import argparse
import importlib
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("variants", nargs="+")
    ap.add_argument("--batch", type=int, default=2048)
    ap.add_argument("--dim", type=int, default=16)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warm", type=int, default=2700)
    ap.add_argument("--repeat", type=int, default=2)
    a = ap.parse_args()
    import torch
    import bench
    pkg = importlib.import_module("ev-store-dlrm_b200")
    rows = pkg.workload.KAGGLE_ROWS
    B, T = a.batch, len(rows)
    n_batches = a.warm + 24 + a.steps * a.repeat
    _, tables, idx = bench.build_workload(a, n_batches, rows, a.dim, B)
    pinned = [torch.from_numpy(t).pin_memory() for t in tables]
    stores_by_mem = {"pinned": {32: [q.numpy() for q in pinned]}}
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    idx_dev = torch.from_numpy(idx).to(dev)
    out = torch.empty((B, T, a.dim), dtype=torch.float32, device=dev)
    hit = torch.empty((B, T), dtype=torch.uint8, device=dev)
    for var in a.variants:
        env = dict(kv.split("=", 1) for kv in var.split(",") if kv and kv != "default")
        pf = env.pop("PF", "1") == "1"               # pseudo-variables: PF=0 no look-ahead announcements, PTR=1 raw-pointer calls
        ptr = env.pop("PTR", "0") == "1"
        many = int(env.pop("MANY", "0"))             # MANY=n: evs_lookup_batches over n batches per call
        mem = env.pop("MEM", "pinned")               # MEM=mapped: backing rows in evs_host_alloc memory (large device pages)
        if mem not in stores_by_mem:
            stores_by_mem[mem] = {32: [pkg.to_host_rows(t) for t in tables]}
        stores = stores_by_mem[mem]
        saved = {k: os.environ.get(k) for k in env}
        os.environ.update(env)
        try:
            cfg = pkg.CacheConfig(n_layers=1, main_precision=32, total_size=pkg.workload.KAGGLE_CACHE_ROWS, max_batch=B, device=0)
            store = pkg.EvStore(tables, cfg, stores=stores)
        finally:
            for k, v in saved.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
        for k in range(a.warm + 10):
            store.lookup(idx_dev[k], out=out, hit=hit)
            if pf:
                store.prefetch(idx_dev[k + 1])
        store.sync()
        store.stats(reset=True)
        store.phase_times()
        best = None
        for r in range(a.repeat):
            base = a.warm + 10 + r * a.steps
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ptrs = [idx_dev[base + k].data_ptr() for k in range(a.steps + 8)]
            op, hp, sp, os_ = out.data_ptr(), hit.data_ptr(), stream.cuda_stream, out.stride(0)
            if pf:
                store.prefetch(idx_dev[base])
            torch.cuda.synchronize()
            e0.record()
            t0 = time.perf_counter()
            if many:
                import ctypes as C
                ips = [(C.c_void_p * many)(*ptrs[k:k + many]) for k in range(0, a.steps, many)]
                ops, hps = (C.c_void_p * many)(*([op] * many)), (C.c_void_p * many)(*([hp] * many))
                for g, k in enumerate(range(0, a.steps, many)):
                    store.lookup_many_ptr(many, ips[g], B, ops, os_, hps, sp)
                    if pf:
                        store.prefetch_ptr(ptrs[k + many], B)
            elif ptr:
                for k in range(a.steps):
                    store.lookup_ptr(ptrs[k], B, op, os_, hp, sp)
                    if pf:
                        store.prefetch_ptr(ptrs[k + 1], B)
            else:
                for k in range(a.steps):
                    store.lookup(idx_dev[base + k], out=out, hit=hit)
                    if pf:
                        store.prefetch(idx_dev[base + k + 1])
            host_us = 1e6 * (time.perf_counter() - t0) / a.steps
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / a.steps
            best = ms if best is None else min(best, ms)
        ph = store.phase_times()
        st = store.stats()
        # per-kernel CUDA-event times (plain launches instead of the graph: the overlap differs slightly)
        store.kernel_times(reset=True)
        store.set_profiling(True)
        base = a.warm + 10
        for k in range(min(100, a.steps)):
            store.lookup(idx_dev[base + k], out=out, hit=hit)
        torch.cuda.synchronize()
        kt = {nm: round(1e3 * ms / max(1, timed), 2) for nm, (ms, timed, _l) in store.kernel_times(reset=True).items() if timed}
        store.set_profiling(False)
        keys = ("avg_serve", "avg_gap1", "avg_update", "avg_gap2", "avg_evict", "evict_plan", "evict_chunks", "evict_wait_last",
                "evict_writeback", "avg_fetch_since_evict_start", "evict_chunks_per_batch", "evict_last_chunk_avg", "evict_last_chunk_max")
        gap = 1e3 * best - sum(ph[k] for k in ("avg_serve", "avg_gap1", "avg_update", "avg_gap2", "avg_evict"))
        print(json.dumps({"variant": var, "us_per_step": 1e3 * best, "batch_to_batch_gap_us": round(gap, 2), "host_us_per_step": host_us, "lookups_per_s": B * T / (best * 1e-3),
                          "evictions_per_step": st["evictions"][0] / (a.steps * a.repeat),
                          "phases_us": {k: round(ph[k], 3) for k in keys if k in ph}, "kernel_event_us": kt}), flush=True)
        store.close()
        del store
        time.sleep(0.2)


if __name__ == "__main__":
    main()
