#!/usr/bin/env python
"""bench.py -- EV lookups/s of the embedding-lookup hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # our CUDA path
    python bench.py --impl reference [--gpus N] [--steps K] ...     # the reference's CPU path
    python bench.py --steps K --dump-outputs DIR                    # + the last timed step's outputs as DIR/*.npy

A *step* is one pass of the hot path over one batch of synthetic Zipf(1.05) indices
(26 tables x B samples): probe -> EvLFU promote -> miss fetch from the host-pinned backing
store -> insert/evict -> dequantise -> fp32 rows [B, 26, dim].

N = 1  : BASELINE configs[1] -- C1 EvLFU cache in HBM, Kaggle-shape tables, batch 2048, fp32 tier.
N > 1  : the same tables table-wise sharded over N GPUs (bench_sharded.py), global batch 2048*N (weak
         scaling), exact groupability (all-reduce of per-sample hit counts) and an NCCL all-to-all of
         the pooled rows; --shape terabyte selects BASELINE configs[4] (dim 64, 40 M-row tables).

One JSON line on stdout (rank 0); everything else goes to stderr.
  value     lookups/s with the index batches already resident in HBM (CUDA events, max over ranks)
  e2e       the same through the host-buffer C-ABI call (pinned host indices in, fp32 rows out)
  roofline  dominant kernel: algorithmic bytes per launch / its CUDA-event time, vs measured HBM peak
  cpu_baseline  the reference's own libcachemanager.so (oracle/_ref) on this box's host cores
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200, help="timed steps of the value line (the e2e and roofline legs time as many)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="samples per step (default 2048)")
    ap.add_argument("--dim", type=int, default=0)
    ap.add_argument("--precision", type=int, default=32)
    ap.add_argument("--scale", type=float, default=1.0, help="shrink table cardinalities (debug only; invalidates the number)")
    ap.add_argument("--cache-warm", type=int, default=-1, help="untimed batches that fill the cache before warm-up")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-baseline-seconds", type=float, default=150.0, help="time budget of the CPU baseline's warm-up")
    ap.add_argument("--cpu-replicas", type=int, default=0,
                    help="leg (iii) of SURVEY 8(d): also time N independent processes of the reference library at once (4 threads "
                         "each; adds about a minute and ~6 GB of host memory per replica)")
    ap.add_argument("--no-clocks", action="store_true")
    ap.add_argument("--no-prefetch", action="store_true", help="A/B: do not announce the next index batch (evs_prefetch)")
    ap.add_argument("--no-b16k", action="store_true", help="skip the batch-16384 roofline leg")
    ap.add_argument("--op", default="", choices=["", "interact", "embedding_bag", "knn"],
                    help="time one of the tensor ops either side of the cache alone (bench_ops.py) instead of the lookup path")
    ap.add_argument("--no-ops", action="store_true", help="skip the interact / embedding_bag legs of the default line")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the short configs[2] / configs[3] legs of the default line")
    ap.add_argument("--no-configs4", action="store_true", help="N = 1: skip the Terabyte-shape (configs[4]) leg (48 GB of pinned host memory)")
    ap.add_argument("--only-main", action="store_true", help="N > 1: only the main leg (no contiguous-placement and configs[4] legs)")
    ap.add_argument("--store-in-hbm", action="store_true", help="debug: backing store copied into HBM (not the BASELINE config)")
    ap.add_argument("--layers", type=int, default=1, help="1 = configs[1] (C1); 2 = configs[2] (C1+C2); 3 = configs[3] (C1+C2+C3, needs 8/4)")
    ap.add_argument("--secondary", type=int, default=0, help="SECONDARY_PRECISION of the C2 tier")
    ap.add_argument("--prop", default="", help='SIZE_PROPORTION "c1-c2-c3" (3 layers)')
    ap.add_argument("--transport", default="p2p", choices=["p2p", "nccl"],
                    help="N > 1 only: exchange fused into the kernels over NVLink peer memory, or NCCL all-reduce + all-to-all")
    ap.add_argument("--policy", default="evlfu", choices=["evlfu", "lru", "lfu"],
                    help="replacement policy: evlfu = the reference's EvLFU (BASELINE configs); lru / lfu = its comparison policies "
                         "cache_algo/LRU.py / LFU.py (1 layer)")
    ap.add_argument("--shape", default="kaggle", choices=["kaggle", "terabyte"],
                    help="table shape: kaggle (configs[1-3]) or terabyte (configs[4]: dim 64, cardinalities capped at 40 M); N = 1 with "
                         "terabyte needs --table-slice (one rank's tables fit one host, all 48 GB of them do not)")
    ap.add_argument("--table-slice", default="", help="N = 1 only: serve tables a:b of the shape, e.g. 0:4 = what rank 0 of an 8-GPU run owns")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="N = 1 only: after the timed steps, write what the last timed step returned (rows [B, T, dim], hit codes "
                         "[B, T]) as DIR/rows.npy and DIR/hit.npy in float32; above 64 MB a seeded sample of the samples, whose "
                         "indices go to DIR/sample.npy.  The same arguments give the same inputs, so two builds compare file by file")
    a = ap.parse_args()
    if a.dump_outputs and (a.impl != "ours" or a.op or a.gpus > 1):
        ap.error("--dump-outputs applies to the N = 1 line of our CUDA path")
    return a


DUMP_BYTES = 64 << 20


def dump_outputs(path: str, rows: np.ndarray, hit: np.ndarray) -> None:
    """rows [B, T, dim] fp32, hit [B, T] uint8 of one step -> path/*.npy (float32), at most DUMP_BYTES in all."""
    os.makedirs(path, exist_ok=True)
    B = rows.shape[0]
    per_sample = rows[0].size * 4 + hit[0].size * 4 + 8
    arrays = {"rows": rows, "hit": hit.astype(np.float32)}
    if B * per_sample > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(B, DUMP_BYTES // per_sample, replace=False))
        arrays = {"rows": rows[keep], "hit": arrays["hit"][keep], "sample": keep.astype(np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a))
    log("outputs of the last timed step written to %s: %s" % (path, {k: list(v.shape) for k, v in arrays.items()}))


class ClockSampler:
    """nvidia-smi sampled every 25 ms while the timed regions run (B200_PROFILING.md)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "25", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception as e:                      # no nvidia-smi: report it, do not fail the bench
            log("clock sampler unavailable:", e)
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def bytes_per_lookup(dim: int, prec: int) -> int:
    """SURVEY.md section 8(d): int64 index + one 16 B index slot + stored row + fp32 output row (P = 1)."""
    return 8 + 16 + dim * prec // 8 + 4 * dim


def build_workload(args, n_batches: int, rows, dim: int, B: int, seed: int = 42):
    pkg = importlib.import_module("ev-store-dlrm_b200")
    t0 = time.time()
    tables = pkg.workload.make_tables(rows, dim)
    t1 = time.time()
    trace = pkg.workload.ZipfTrace(rows, alpha=1.05, seed=seed)
    idx = trace.batches(n_batches, B)
    log(f"workload: tables {sum(t.nbytes for t in tables) / 1e9:.2f} GB in {t1 - t0:.1f}s, "
        f"{n_batches} index batches in {time.time() - t1:.1f}s")
    return pkg, tables, idx


def batches_until_full(idx: np.ndarray, rows, cap: int) -> int:
    """Number of leading batches of the trace after which more than `cap` distinct keys have been requested, i.e. the
    cache (any policy: nothing is evicted before it is full) holds `cap` entries.  idx: int64 [n, T, B].  Both arms
    derive their cache warm-up from this, so they reach the timed region in the same state."""
    n, T, B = idx.shape
    new_per_batch = np.zeros(n, dtype=np.int64)
    batch_of = np.repeat(np.arange(n, dtype=np.int32), B)[::-1]
    for t in range(T):
        # first batch that requests each row: written in reverse trace order, so the earliest batch is the write that stays
        first = np.full(int(rows[t]), n, dtype=np.int32)
        first[idx[:, t].ravel()[::-1]] = batch_of
        new_per_batch += np.bincount(first[first < n], minlength=n)
    cum = np.cumsum(new_per_batch)
    full = int(np.searchsorted(cum, cap, side="left")) + 1
    return min(full, n)


WARM_AFTER_FULL = 300       # batches with evictions running before anything is timed
WARM_SEARCH = 4800          # batches of the trace examined for the fill point


def configs1_config(B: int, dim: int, cache_rows: int, warm: int) -> dict:
    """The `config` object of BASELINE configs[1]; both arms print exactly this."""
    return {"workload": "configs[1]: C1 EvLFU fp32 tier, Kaggle-shape 26 tables (33.76M rows), dim %d, Zipf(1.05), batch %d, "
                        "cache %d rows (13%% of the rows), backing store in host memory" % (dim, B, cache_rows),
            "batch": B, "dim": dim, "precision": 32, "layers": 1, "policy": "evlfu", "cache_rows": cache_rows,
            "cache_warm_batches": warm,
            "cache_warm": "the Zipf trace itself until the cache is full (%d batches, derived from the trace) plus %d batches "
                          "with evictions running" % (warm - WARM_AFTER_FULL, WARM_AFTER_FULL),
            "l2": "no flush: index + slab working set (%.2f GB) exceeds the 126 MB L2 and every step reads a distinct index batch"
                  % (cache_rows * (dim * 4 + 32) / 1e9)}


# ------------------------------------------------------------------------------------ reference arm
def run_cpu_reference(variant, tables_raw, idx, B, warm_batches, timed_batches, budget_s=None):
    """Times the reference's libcachemanager.so (oracle/_ref) through ev_lookup, one sample per
    call, 1 caller thread + the library's 3 reader threads.  idx: int64 [n, 26, B]."""
    from oracle import ref_driver
    v = ref_driver.VARIANTS[variant]
    t0 = time.time()
    ref_driver.write_fixture(variant, {v["main"]: tables_raw})
    log(f"reference fixture written to {ref_driver.fixture_dir(variant)} in {time.time() - t0:.1f}s")
    ref = ref_driver.RefCache(variant)
    perfect = __import__("ctypes").c_int.in_dll(ref.lib, "perfectHit")

    def as_trace(k0, k1):
        # [n, 26, B] -> sample-major int32 [n*B, 26]
        return np.ascontiguousarray(idx[k0:k1].transpose(0, 2, 1).reshape(-1, idx.shape[1]).astype(np.int32))

    warm_s = 0.0
    done = 0
    while done < warm_batches:
        step = min(16, warm_batches - done)
        s, _ = ref.drive(as_trace(done, done + step))
        warm_s += s
        done += step
        if budget_s is not None and warm_s > budget_s:
            break
    warm_done = done
    perfect.value = 0
    per_step = []
    for k in range(timed_batches):
        kk = warm_done + k
        if kk >= idx.shape[0]:
            break
        s, _ = ref.drive(as_trace(kk, kk + 1))
        per_step.append(s)
    total = float(sum(per_step))
    n_samples = len(per_step) * B
    return {
        "seconds": total, "steps": len(per_step), "samples": n_samples, "samples_per_s": n_samples / total,
        "lookups_per_s": n_samples * idx.shape[1] / total, "warm_batches": warm_done, "warm_seconds": warm_s,
        "perfect_hits": int(perfect.value), "ms_per_step": 1e3 * total / max(1, len(per_step)),
    }


def run_cpu_replicas(n: int, args):
    """N concurrent `bench.py --impl reference` processes (the reference's library is process-global and single-caller, so
    more host cores can only be used by more processes, each with its own cache): the sum of their lookups/s."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "40", "--warmup", "3"]
    if args.cache_warm >= 0:
        cmd += ["--cache-warm", str(args.cache_warm)]
    t0 = time.time()
    procs = [subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, cwd=ROOT) for _ in range(n)]
    vals = []
    for p in procs:
        out, _ = p.communicate(timeout=1200)
        lines = [ln for ln in out.splitlines() if ln.startswith("{")]
        if p.returncode == 0 and lines:
            vals.append(float(json.loads(lines[-1])["value"]))
    return {"n": n, "finished": len(vals), "value": float(sum(vals)), "unit": "lookups/s", "cores": 4 * n, "per_replica": vals,
            "wall_s": time.time() - t0, "kind": "reference",
            "sample": "%d processes at once, each: 40 batches of 2048 samples after the full warm-up, 1 caller + 3 reader threads" % n}


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import ref_driver
    pkg = importlib.import_module("ev-store-dlrm_b200")
    B = (args.batch or 2048) * max(1, args.gpus)          # the N-GPU arm's global batch (weak scaling)
    dim = args.dim or 16
    variant = "bench_c1_fp32_d16"
    if not ref_driver.available(variant) or dim != 16 or args.scale != 1.0:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/lib%s.so not built for this config" % variant}))
        return 0
    rows = pkg.workload.KAGGLE_ROWS
    cache_rows = pkg.workload.KAGGLE_CACHE_ROWS
    W = max(args.warmup, 3)
    # the same trace, the same warm-up rule and the same `config` as main_ours (N = 1); at N > 1 the reference still runs
    # unsharded on the host cores, over the N-GPU arm's global batch
    search = max(8, WARM_SEARCH * 2048 // B)
    n_batches = search + 4 * W + 8 * args.steps + 32
    _, tables, idx = build_workload(args, n_batches, rows, dim, B)
    warm = args.cache_warm if args.cache_warm >= 0 else batches_until_full(idx[:search], rows, cache_rows) + WARM_AFTER_FULL * 2048 // B
    log(f"reference arm: {warm} warm batches of {B} (cache full after {warm - WARM_AFTER_FULL * 2048 // B}), then {W} + {args.steps}")
    r = run_cpu_reference(variant, tables, idx, B, warm + W, args.steps)
    cfg = configs1_config(B, dim, cache_rows, warm) if args.gpus <= 1 else sharded_config(args.gpus, B, dim, args.transport)
    line = {
        "impl": "reference", "metric": "ev_lookups_per_s", "value": r["lookups_per_s"], "unit": "lookups/s",
        "n_gpus": args.gpus, "steps": r["steps"], "warmup": W, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "samples_per_s": r["samples_per_s"], "config": cfg,
        "cpu_baseline": {"value": r["lookups_per_s"], "unit": "lookups/s", "cores": 4, "kind": "reference",
                         "sample": "%d full batches of %d samples after %d warm batches (cache full); the reference's own "
                                   "libcachemanager.so compiled from its sources (1 caller + 3 reader threads, "
                                   "N_THD__READ_EVTABLE_32BIT), backing tables as files in /dev/shm" % (r["steps"], B, r["warm_batches"]),
                         "perfect_hits": r["perfect_hits"], "warm_seconds": r["warm_seconds"], "host_cpus": os.cpu_count()},
        "e2e": {"value": r["lookups_per_s"], "unit": "lookups/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def sharded_config(world: int, B: int, dim: int, transport: str = "p2p") -> dict:
    """`config` of the N > 1 line (Kaggle shape, weak scaling); the reference arm prints the same object."""
    return {"workload": "configs[1] tables sharded table-wise over %d GPUs (weak scaling of the N = 1 line): C1 EvLFU fp32 tier, "
                        "Kaggle-shape 26 tables (33.76M rows), dim %d, Zipf(1.05), global batch %d = 2048 per GPU, 13%% of the rows "
                        "cached, backing store in host memory" % (world, dim, B),
            "batch": B, "dim": dim, "precision": 32, "layers": 1, "policy": "evlfu", "n_gpus": world,
            "parallelism": "table-wise x%d, exchange %s" % (world, "fused into the kernels over NVLink peer memory (evs_shard_*)"
                                                            if transport == "p2p" else "NCCL all-reduce + all_to_all_single"),
            "transport": transport,
            "placement": "tables spread over the ranks by row count (sharded.balanced_placement; departs from ext_dist.get_my_slice, "
                         "whose contiguous slices are reported under placement_contiguous)",
            "l2": "no flush: index + slab working set exceeds the 126 MB L2 and every step reads a distinct index batch"}


def extra_config_leg(pkg, dev, device, tables, idx, rows, dim, cache_rows, layers, p0, p1, prop, B, K, W, warm2048):
    """One more BASELINE configuration on the tables and the trace of the main leg: configs[2] (C1 + C2 mixed precision) or
    configs[3] (C1 + C2 + C3, batch 16384; alt keys = workload.make_alt_keys, the documented stand-in for the kNN tables).
    Same memory budget as configs[1] (TOTAL_SIZE = cache_rows fp32-row units), same warm-up rule, 4 batches per call."""
    import ctypes as C
    import torch
    T = len(rows)
    g = B // 2048
    n_need = (warm2048 // g + W + 3 * K + 8) if g > 1 else (warm2048 + W + 3 * K + 8)
    if g > 1:
        n = min(idx.shape[0] // g, n_need)
        ib = np.ascontiguousarray(idx[:n * g].reshape(n, g, T, 2048).transpose(0, 2, 1, 3)).reshape(n, T, B)
    else:
        n = min(idx.shape[0], n_need)
        ib = idx[:n]
    warm = min(warm2048 // g, n - W - 3 * K - 5)
    stores = {p: [pkg.to_host_rows(pkg.codecs.encode_table(t, p), device=device) for t in tables] for p in (p0, p1)}
    alt = pkg.workload.make_alt_keys(rows) if layers == 3 else None
    cfg = pkg.CacheConfig(n_layers=layers, main_precision=p0, secondary_precision=p1, size_proportion=prop, total_size=cache_rows,
                          max_batch=B, device=device)
    store = pkg.EvStore(tables, cfg, stores=stores, alt_keys=alt)
    try:
        idx_dev = torch.from_numpy(ib).to(dev)
        out = torch.empty((B, T, dim), dtype=torch.float32, device=dev)
        hit = torch.empty((B, T), dtype=torch.uint8, device=dev)
        for k in range(warm + W):
            store.lookup(idx_dev[k], out=out, hit=hit)
            store.prefetch(idx_dev[k + 1])
        store.sync()
        store.stats(reset=True)
        base = warm + W
        st_ = torch.cuda.current_stream(dev).cuda_stream
        outp, hitp = (C.c_void_p * 4)(*([out.data_ptr()] * 4)), (C.c_void_p * 4)(*([hit.data_ptr()] * 4))
        regions = []
        for rep in range(3):
            calls = [(k, min(4, K - k), (C.c_void_p * 4)(*[idx_dev[base + k + j].data_ptr() for j in range(4)])) for k in range(0, K, 4)]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for k, nb, ips in calls:
                store.lookup_many_ptr(nb, ips, B, outp, out.stride(0), hitp, st_)
                store.prefetch(idx_dev[base + k + nb])
            e1.record()
            torch.cuda.synchronize()
            regions.append(e0.elapsed_time(e1))
            base += K
        store.check()
        s = store.stats()
        ms = sorted(regions)[1]
        lk = max(1, s["lookups"])
        return {"layers": layers, "main_precision": p0, "secondary_precision": p1, "size_proportion": prop, "batch": B, "steps": K,
                "value": K * B * T / (ms * 1e-3), "unit": "lookups/s", "ms_per_step": ms / K, "value_regions_ms": regions,
                "hit_rate_by_tier": {"c1": s["hits"][0] / lk, "c2": s["hits"][1] / lk, "c3": s["c3_hits"] / lk},
                "capacity": s["capacity"], "c3_capacity": s["c3_capacity"], "cache_warm_batches": warm, "resident": s["size"],
                "note": None if s["size"][0] >= s["capacity"][0] else
                        "C1 is not full after the warm-up (its entries are %d-bit: the same budget holds %dx as many), so every key "
                        "still goes to C1 (evlfu_8.cpp:590-602) and C2 / C3 see no traffic" % (p0, 32 // p0),
                "alt_keys": "workload.make_alt_keys (a more popular row of the same table; the kNN generator is evs_knn)" if layers == 3 else None}
    finally:
        store.close()


# ------------------------------------------------------------------------------------ our arm
def main_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        from bench_sharded import main_sharded          # Terabyte-shape, table-wise sharded
        return main_sharded(args)

    assert torch.cuda.is_available(), "bench.py needs a CUDA device: the product path has no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    B = args.batch or 2048
    dim = args.dim or 16
    prec = args.precision
    K, W = args.steps, max(args.warmup, 3)
    pkg = importlib.import_module("ev-store-dlrm_b200")
    shape_rows = pkg.workload.TERABYTE_ROWS if args.shape == "terabyte" else pkg.workload.KAGGLE_ROWS
    rows = shape_rows if args.scale == 1.0 else pkg.workload.scaled_rows(shape_rows, args.scale)
    sliced = bool(args.table_slice)
    if sliced:
        a_, b_ = (int(x) for x in args.table_slice.split(":"))
        rows = rows[a_:b_]
    if args.shape == "terabyte":
        dim = args.dim or 64
        assert sliced or args.scale < 1.0, "the whole Terabyte shape is 48 GB of host memory: pass --table-slice a:b (one rank's tables)"
    T = len(rows)
    cache_rows = pkg.workload.KAGGLE_CACHE_ROWS if (args.scale == 1.0 and args.shape == "kaggle" and not sliced) else int(sum(rows) * 0.13)
    search = max(8, WARM_SEARCH * 2048 // B)
    n_batches = search + 4 * W + 8 * K + 32                # the reference arm generates the same trace (same n, same B)
    _, tables, idx = build_workload(args, n_batches, rows, dim, B)
    t0 = time.time()
    warm = args.cache_warm if args.cache_warm >= 0 else batches_until_full(idx[:search], rows, cache_rows * 32 // args.precision
                                                                           if args.layers == 1 else cache_rows) + WARM_AFTER_FULL * 2048 // B
    warm = min(warm, search)
    log(f"cache warm-up: {warm} batches (fill point derived from the trace in {time.time() - t0:.1f}s)")

    layers = args.layers
    sec = args.secondary if layers >= 2 else 0
    # TOTAL_SIZE is in fp32-row units (cache_manager.cpp:16): a single tier of `prec` bits holding cache_rows entries
    # takes cache_rows * prec / 32 of them; the multi-layer configs get the same memory budget as configs[1]
    total_size = cache_rows * prec // 32 if layers == 1 else cache_rows
    cfg = pkg.CacheConfig(n_layers=layers, main_precision=prec, secondary_precision=sec, size_proportion=args.prop,
                          total_size=total_size, max_batch=B, device=local_rank, store_in_hbm=args.store_in_hbm, policy=args.policy)
    alt = pkg.workload.make_alt_keys(rows) if layers == 3 else None
    t0 = time.time()
    # backing store in host memory: evs_host_alloc rows (mapped into the device with large pages: about twice the zero-copy row
    # rate of cudaHostAlloc memory over a 2 GB table, profiles/r2_zc_vmm_probe.txt); EVS_BENCH_STORE=pinned selects torch's
    # pinned allocator instead (A/B)
    stores, keep = {}, []
    store_mem = os.environ.get("EVS_BENCH_STORE", "mapped")
    for pr in [prec] + ([sec] if layers >= 2 else []):
        if store_mem == "mapped":
            stores[pr] = [pkg.to_host_rows(pkg.codecs.encode_table(t, pr), device=local_rank) for t in tables]
        else:
            pinned = [torch.from_numpy(pkg.codecs.encode_table(t, pr)).pin_memory() for t in tables]
            keep.append(pinned)
            stores[pr] = [q.numpy() for q in pinned]
    log(f"backing store copied to {store_mem} host allocations in {time.time() - t0:.1f}s")
    store = pkg.EvStore(tables, cfg, stores=stores, alt_keys=alt)
    log(f"EvStore created in {time.time() - t0:.1f}s (cache {cache_rows} rows, backing store host-pinned zero-copy)")

    # everything below is ordered on one explicit stream: the CUDA events that bracket the timed
    # region are recorded on the stream the kernels are launched on
    bench_stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(bench_stream)
    idx_host = torch.from_numpy(idx).pin_memory()                    # [n, T, B] int64
    idx_dev = idx_host.to(dev, non_blocking=True)
    out = torch.empty((B, T, dim), dtype=torch.float32, device=dev)
    hit = torch.empty((B, T), dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()

    # ---- fill the cache (mirrors the reference's --cache-warmup pass) ------------------------
    t0 = time.time()
    use_pf = not args.no_prefetch
    for k in range(warm):
        store.lookup(idx_dev[k], out=out, hit=hit)
        if use_pf:
            store.prefetch(idx_dev[k + 1])
    store.sync()
    st = store.stats(reset=True)
    log(f"cache warm: {warm} batches in {time.time() - t0:.2f}s, resident {st['size'][0]}/{st['capacity'][0]}, "
        f"hit rate so far {st['hits'][0] / max(1, st['lookups']):.3f}")
    fill = st["size"][0] / max(1, st["capacity"][0])

    sampler = ClockSampler(local_rank)
    if not args.no_clocks:
        sampler.start()
        time.sleep(0.3)

    store.phase_times()                           # clears the debug accumulators
    # ---- value: indices resident in HBM ------------------------------------------------------
    # EXACTLY K timed steps, W warm-up steps before them, in up to three back-to-back regions of whole calls (listed in
    # value_regions_ms, so that a region that stands out is visible); the line reports all K steps over the summed region
    # time.  Every step announces the next index batch (evs_prefetch), as a serving loop with its requests queued would.
    base = warm
    for k in range(W):
        store.lookup(idx_dev[base + k], out=out, hit=hit)
        if use_pf:
            store.prefetch(idx_dev[base + k + 1])
    torch.cuda.synchronize()
    base += W
    regions = []
    launches = 0
    # The serving loop has its requests queued, so it hands the library GROUP batches per call (evs_lookup_batches: one
    # captured graph per 4 batches, the batches still strictly ordered on the device) and announces the first batch of
    # the next call; every batch is a full pass of the hot path over its own index batch.
    GROUP = max(1, int(os.environ.get("EVS_BENCH_GROUP", "4")))
    import ctypes as C
    out_ptrs = (C.c_void_p * GROUP)(*([out.data_ptr()] * GROUP))
    hit_ptrs = (C.c_void_p * GROUP)(*([hit.data_ptr()] * GROUP))
    n_calls = -(-K // GROUP)
    region_steps = [GROUP * (n_calls // 3 + (r < n_calls % 3)) for r in range(min(3, n_calls))]
    region_steps[-1] -= sum(region_steps) - K              # the last call may hold fewer than GROUP batches
    for Kr in region_steps:
        l0 = store.launch_count()
        calls = [(k, min(GROUP, Kr - k), (C.c_void_p * GROUP)(*[idx_dev[base + k + j].data_ptr() for j in range(GROUP)]))
                 for k in range(0, Kr, GROUP)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k, n, ips in calls:
            store.lookup_many_ptr(n, ips, B, out_ptrs, out.stride(0), hit_ptrs, bench_stream.cuda_stream)
            if use_pf:
                store.prefetch(idx_dev[base + k + n])
        e1.record()
        torch.cuda.synchronize()
        regions.append(e0.elapsed_time(e1))
        launches += store.launch_count() - l0
        base += Kr
    # every batch of a call writes the same buffers: they hold the last timed step's result until the legs below reuse them
    last_step = (out.cpu().numpy(), hit.cpu().numpy()) if args.dump_outputs else None
    ms_dev = sum(regions)
    base -= W + K                                 # the sections below advance by W + K
    phases = store.phase_times()
    log("device phases of the last timed batch (us):", phases)
    st = store.stats(reset=True)
    KK = K
    log("per step: misses %.0f evictions %.0f flushed %.0f inserts %.0f" % (st["misses"] / KK, st["evictions"][0] / KK,
        st["flushed"][0] / KK, st["inserts"][0] / KK))
    hit_rate = (st["hits"][0] + st["hits"][1] + st["c3_hits"]) / max(1, st["lookups"])
    tier_rates = {"c1": st["hits"][0] / max(1, st["lookups"]), "c2": st["hits"][1] / max(1, st["lookups"]),
                  "c3": st["c3_hits"] / max(1, st["lookups"])}
    perfect_rate = st["perfect_hits"] / max(1, st["samples"])
    lookups = K * B * T
    value = lookups / (ms_dev * 1e-3)

    # ---- e2e: host buffers through the C-ABI -------------------------------------------------
    # (a) evs_lookup_batch_host: one synchronous call per batch, like the reference's ev_lookup;
    # (b) evs_submit_host / evs_wait_host: the same batches, at most 4 in flight, so the copies of
    #     neighbouring batches overlap the kernels.  Both read pinned host indices and deliver the
    #     fp32 rows (and the hit map) into pinned host buffers inside the timed region.
    base += W + K
    out_host = [torch.empty((B, T, dim), dtype=torch.float32).pin_memory() for _ in range(4)]
    hit_host = [torch.empty((B, T), dtype=torch.uint8).pin_memory() for _ in range(4)]
    ih = idx_host
    for k in range(W):
        store.lookup_host_ptr(ih[base + k].data_ptr(), B, out_host[0].data_ptr(), hit_host[0].data_ptr())
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(K):
        store.lookup_host_ptr(ih[base + W + k].data_ptr(), B, out_host[0].data_ptr(), hit_host[0].data_ptr())
    torch.cuda.synchronize()
    e2e_sync_s = time.perf_counter() - t0
    base += W + K
    tickets = []
    for k in range(W):
        tickets.append(store.submit_host_ptr(ih[base + k].data_ptr(), B, out_host[k % 4].data_ptr(), hit_host[k % 4].data_ptr()))
    store.wait_host(tickets[-1])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(K):
        tk = store.submit_host_ptr(ih[base + W + k].data_ptr(), B, out_host[k % 4].data_ptr(), hit_host[k % 4].data_ptr())
    store.wait_host(tk)
    e2e_s = time.perf_counter() - t0
    e2e_value = lookups / e2e_s
    h2d = B * T * 8
    d2h = B * T * dim * 4 + B * T

    clocks = sampler.stop() if not args.no_clocks else {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}

    # ---- roofline: per-kernel CUDA-event times over K more steps ------------------------------
    base += W + K
    store.kernel_times(reset=True)
    store.set_profiling(True)
    for k in range(K):
        store.lookup(idx_dev[base + k], out=out, hit=hit)
    torch.cuda.synchronize()
    kt = store.kernel_times(reset=True)
    store.set_profiling(False)
    per_kernel = {n: {"avg_us": 1e3 * ms / max(1, timed), "launches": timed} for n, (ms, timed, _l) in kt.items() if timed}
    tot_us = sum(v["avg_us"] * v["launches"] for v in per_kernel.values())
    for v in per_kernel.values():
        v["share"] = v["avg_us"] * v["launches"] / max(tot_us, 1e-9)
    dom = max(per_kernel, key=lambda n: per_kernel[n]["share"])
    peak, peak_src = measured_peak_hbm()
    bpl = bytes_per_lookup(dim, prec)
    alg_bytes = B * T * bpl
    # The roofline kernel is k_serve: the fused probe + dequantise + gather kernel is the only HBM-bandwidth-bound
    # kernel of the step and the one SURVEY.md 8(d)'s bytes-per-lookup figure describes (and the north-star's 50 %
    # target names).  The kernels that take more of the step at this batch size are not bandwidth bound: k_update / k_evict
    # are chains of dependent accesses, the miss fetch (a role of k_evict, and the look-ahead k_prefetch) is bound by the
    # PCIe small-read rate (DESIGN.md 5);
    # they are listed under "per_kernel" with their share and named in "dominant_by_time".
    serve_ev_us = per_kernel["k_serve"]["avg_us"]
    # in-kernel %globaltimer span (first CTA start to last CTA end) averaged over the timed batches; the CUDA-event
    # figure additionally holds ~6 us of launch and drain
    serve_us = phases["avg_serve"]
    # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture of this
    # same command (profiles/r2_traffic.json, written by tools/ncu_summary.py); null when no capture is committed
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        if tj.get("batch") == B and tj.get("dim") == dim and tj.get("precision") == prec and layers == 1:
            traffic = tj["dram_bytes_per_launch"].get("k_serve")
    except Exception:
        pass
    n_miss = st["misses"] / max(1, 3 * K)
    roofline = {
        "bound": "hbm", "kernel": "k_serve", "achieved": alg_bytes / (serve_ev_us * 1e-6) / 1e9, "peak": peak, "unit": "GB/s",
        "frac": alg_bytes / (serve_ev_us * 1e-6) / 1e9 / peak, "traffic": traffic, "peak_source": peak_src,
        "algorithmic_bytes_per_launch": alg_bytes, "bytes_per_lookup": bpl, "kernel_avg_us": serve_ev_us,
        "timing": "CUDA events around each launch on its stream (profiling mode: plain launches instead of the graph)",
        "in_kernel": {"avg_us": serve_us, "achieved": alg_bytes / (serve_us * 1e-6) / 1e9, "frac": alg_bytes / (serve_us * 1e-6) / 1e9 / peak,
                      "timing": "%globaltimer, first CTA start to last CTA end, averaged over the timed region of `value` (graph launches)"},
        "k_serve": {"event_avg_us": serve_ev_us, "in_kernel_avg_us": serve_us,
                    "achieved": alg_bytes / (serve_us * 1e-6) / 1e9, "frac": alg_bytes / (serve_us * 1e-6) / 1e9 / peak},
        "dominant_by_time": {"kernel": dom, "share": per_kernel[dom]["share"], "avg_us": per_kernel[dom]["avg_us"],
                             "bound": ("k_evict = eviction roles (latency: dependent HBM / L2 accesses) + miss-fetch role (%.0f missing rows per "
                                       "launch: staged by the look-ahead, else zero-copy PCIe reads at 55-110 rows/us)" % n_miss) if dom == "k_evict"
                             else "latency: chains of dependent HBM / L2 accesses, not bandwidth"},
        "step_frac": lookups * bpl / (ms_dev * 1e-3) / 1e9 / peak, "per_kernel": per_kernel, "phases_us": phases,
    }

    footprint = store.memory_footprint()
    # ---- the same cache at batch 16384: where k_serve reaches its bandwidth regime ---------------------------------
    # (configs[1] is quoted at batch 2048, where 8 MB per launch is latency-bound whatever the kernel does; the
    # north-star's ">= 50 % of HBM peak on the fused probe + dequantise + gather kernel" is a statement about the
    # kernel at a batch that fills the machine, reported here from the same run)
    b16 = None
    if (not args.no_b16k and B == 2048 and layers == 1 and args.scale == 1.0 and not sliced):
        try:
            store.close()
            store = None
            B2, K2 = 16384, min(K, 50)
            n2 = warm // 8 + W + 2 * K2 + 2
            assert n2 * 8 <= idx.shape[0]
            idx2 = np.ascontiguousarray(idx[:n2 * 8].reshape(n2, 8, T, B).transpose(0, 2, 1, 3)).reshape(n2, T, B2)
            idx2_dev = torch.from_numpy(idx2).to(dev)
            cfg2 = pkg.CacheConfig(n_layers=1, main_precision=prec, total_size=total_size, max_batch=B2, device=local_rank, policy=args.policy)
            st2 = pkg.EvStore(tables, cfg2, stores=stores)
            out2 = torch.empty((B2, T, dim), dtype=torch.float32, device=dev)
            hit2 = torch.empty((B2, T), dtype=torch.uint8, device=dev)
            k = 0
            for _ in range(warm // 8 + W):
                st2.lookup(idx2_dev[k], out=out2, hit=hit2)
                st2.prefetch(idx2_dev[k + 1])
                k += 1
            torch.cuda.synchronize()
            st2.phase_times()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(K2):
                st2.lookup(idx2_dev[k], out=out2, hit=hit2)
                st2.prefetch(idx2_dev[k + 1])
                k += 1
            e1.record()
            torch.cuda.synchronize()
            ms2 = e0.elapsed_time(e1)
            ph2 = st2.phase_times()
            st2.kernel_times(reset=True)
            st2.set_profiling(True)
            for _ in range(K2):
                st2.lookup(idx2_dev[k], out=out2, hit=hit2)
                k += 1
            torch.cuda.synchronize()
            kt2 = st2.kernel_times(reset=True)
            st2.set_profiling(False)
            ev_us = 1e3 * kt2["k_serve"][0] / max(1, kt2["k_serve"][1])
            ab2 = B2 * T * bpl
            b16 = {"batch": B2, "steps": K2, "ms_per_step": ms2 / K2, "lookups_per_s": K2 * B2 * T / (ms2 * 1e-3),
                   "algorithmic_bytes_per_launch": ab2, "k_serve_event_us": ev_us, "frac": ab2 / (ev_us * 1e-6) / 1e9 / peak,
                   "achieved": ab2 / (ev_us * 1e-6) / 1e9, "k_serve_in_kernel_us": ph2["avg_serve"],
                   "in_kernel_frac": ab2 / (ph2["avg_serve"] * 1e-6) / 1e9 / peak,
                   "per_kernel_us": {n: 1e3 * ms / max(1, timed) for n, (ms, timed, _l) in kt2.items() if timed}}
            st2.close()
            del idx2_dev, out2, hit2
        except Exception as e:
            log("batch-16384 leg failed:", repr(e))
    roofline["batch16384"] = b16

    # ---- the two tensor ops either side of the cache, alone, against the HBM roofline (bench.py --op ... for more) ----
    ops = None
    if not args.no_ops and args.scale == 1.0:
        try:
            from bench_ops import bench_embedding_bag, bench_interact
            ops = {"interact_d16": bench_interact(pkg, dev, B=16384, d=16, K=30, peak=peak),
                   "interact_d64": bench_interact(pkg, dev, B=16384, d=64, K=30, peak=peak),
                   "embedding_bag_d64": bench_embedding_bag(pkg, dev, B=16384, P=10, d=64, K=30, peak=peak)}
            torch.cuda.empty_cache()
        except Exception as e:
            log("op legs failed:", repr(e))

    # ---- BASELINE configs[2] and configs[3] on the same tables and trace (short legs; bench.py --layers ... for the full lines) ----
    other = None
    if (not args.no_other_configs and layers == 1 and prec == 32 and B == 2048 and args.scale == 1.0 and args.shape == "kaggle"
            and not sliced and args.policy == "evlfu"):
        other = {}
        for name, (ly_, p0, p1, prop_, B3) in {"configs2_32_8": (2, 32, 8, "", 2048), "configs3_8_4_c3": (3, 8, 4, "48-48-4", 16384)}.items():
            try:
                other[name] = extra_config_leg(pkg, dev, local_rank, tables, idx, rows, dim, cache_rows, ly_, p0, p1, prop_, B3,
                                               min(K, 20), W, warm)
            except Exception as e:
                log(name, "leg failed:", repr(e))
            torch.cuda.empty_cache()

    # ---- CPU baseline: the reference's own library on this host -------------------------------
    cpu = None
    if (not args.no_cpu_baseline and args.scale == 1.0 and dim == 16 and prec == 32 and layers == 1 and args.policy == "evlfu"
            and args.shape == "kaggle" and not sliced):
        try:
            from oracle import ref_driver
            variant = "bench_c1_fp32_d16"
            if ref_driver.available(variant):
                # the same warm-up as the GPU arm (until the cache is full, + evictions running), bounded by a time budget
                r = run_cpu_reference(variant, tables, idx, B, warm + W, 40, budget_s=args.cpu_baseline_seconds)
                cpu = {"value": r["lookups_per_s"], "unit": "lookups/s", "cores": 4, "kind": "reference",
                       "sample": "%d batches of %d samples timed after %d warm batches in %.0f s (%s); the reference's own "
                                 "libcachemanager.so, 1 caller + 3 reader threads, backing tables as files in /dev/shm"
                                 % (r["steps"], B, r["warm_batches"], r["warm_seconds"],
                                    "the GPU arm's warm-up: cache full" if r["warm_batches"] >= warm + W else "time budget reached: cache only partly full"),
                       "samples_per_s": r["samples_per_s"], "host_cpus": os.cpu_count()}
                # leg (ii) of SURVEY 8(d): the sequential Python EvLFU (restated EvLFU_C1.py, in-RAM rows), one core
                try:
                    from oracle.evlfu import SeqEvLFU
                    seq = SeqEvLFU(cache_rows, n_tables=T)
                    tr = np.ascontiguousarray(idx[:3].transpose(0, 2, 1).reshape(-1, T))
                    n_py = min(4000, tr.shape[0])
                    t0 = time.perf_counter()
                    for i in range(n_py):
                        seq.request(tr[i])
                    dt = time.perf_counter() - t0
                    cpu["python_evlfu"] = {"value": n_py * T / dt, "unit": "lookups/s", "cores": 1, "kind": "port",
                                           "sample": "%d requests through oracle.evlfu.SeqEvLFU (EvLFU_C1.py restated; policy only, rows not copied), cold cache" % n_py}
                except Exception as e:
                    log("python EvLFU leg failed:", repr(e))
                # leg (iii): N independent processes, each the whole library with its own cache (replicas), all at once
                if args.cpu_replicas > 0:
                    try:
                        cpu["replicas"] = run_cpu_replicas(args.cpu_replicas, args)
                    except Exception as e:
                        log("replica leg failed:", repr(e))
            else:
                log("cpu_baseline: oracle/_ref not built")
        except Exception as e:                          # the baseline must not take the GPU number down
            log("cpu_baseline failed:", repr(e))
    if cpu is None:
        cpu = {"value": None, "unit": "lookups/s", "cores": 0, "kind": "reference", "sample": "not run"}

    std_cfg = (layers == 1 and prec == 32 and args.policy == "evlfu" and args.shape == "kaggle" and not sliced and args.scale == 1.0
               and not args.store_in_hbm)
    # ---- configs[4] on one GPU: the N = 1 point of the Terabyte-shape scaling series (bench_sharded.py runs it at N > 1) ----
    configs4 = None
    if std_cfg and B == 2048 and not args.no_configs4:
        try:
            if store is not None:
                store.close()
                store = None
            del tables, idx, idx_dev, idx_host, stores
            import gc
            gc.collect()
            torch.cuda.empty_cache()
            from bench_sharded import run_one_leg
            ver = {}
            configs4 = run_one_leg(pkg, log, args, 0, 1, local_rank, "terabyte", "balanced", "configs4", min(K, 50), False, ver)
        except Exception as e:
            log("configs[4] leg failed:", repr(e))
    line = {
        "metric": "ev_lookups_per_s", "value": value, "unit": "lookups/s", "n_gpus": 1, "steps": K, "warmup": W,
        "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if prec == 32 else f"u{prec}->f32", "data": "synthetic",
        "samples_per_s": value / T, "hit_rate": hit_rate, "hit_rate_by_tier": tier_rates, "perfect_hit_rate": perfect_rate,
        "config": configs1_config(B, dim, cache_rows, warm) if std_cfg else
                  {"workload": ("%s: C1 %s fp%d tier" % ("configs[1]" if args.shape == "kaggle" else "configs[4], one GPU",
                                                          {"evlfu": "EvLFU", "lru": "LRU (cache_algo/LRU.py, comparison policy)",
                                                           "lfu": "LFU (cache_algo/LFU.py, comparison policy)"}[args.policy], prec) if layers == 1 else
                                "configs[%d]: C1 %d-bit + C2 %d-bit%s, TOTAL_SIZE %d fp32-row units%s" % (
                                    layers, prec, sec, " + C3" if layers == 3 else "", total_size, (" split " + args.prop) if args.prop else ""))
                               + ", %s %d tables (%.2fM rows), dim %d, Zipf(1.05), batch %d, cache %d rows, "
                                 "host-pinned backing store" % (
                                     ("Kaggle-shape" if args.shape == "kaggle" else "Terabyte-shape (configs[4])")
                                     + ((" tables %s only (one rank's shard, local agg_hit)," % args.table_slice) if sliced else ""),
                                     T, sum(rows) / 1e6, dim, B, cache_rows),
                   "layers": layers, "secondary_precision": sec, "policy": args.policy,
                   "batch": B, "dim": dim, "precision": prec, "cache_rows": cache_rows, "cache_warm_batches": warm,
                   "l2": "no flush: index + slab working set exceeds the 126 MB L2 and every step reads a distinct index batch"},
        "cache": {"fill": fill, "hbm_bytes": footprint, "budget_bytes": cache_rows * dim * prec // 8,
                  "note": "hbm_bytes = index (load factor <= 1/3) + slot-indexed slab + bucket rings + look-ahead staging; budget_bytes "
                          "= cache rows x row bytes, the reference's TOTAL_SIZE accounting (cache_manager.cpp:16)"},
        "value_regions_ms": regions, "value_region_steps": region_steps, "look_ahead": use_pf, "batches_per_call": GROUP, "configs4": configs4, "other_configs": other, "ops": ops,
        "e2e": {"value": e2e_value, "unit": "lookups/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": 1e3 * e2e_s / K, "api": "evs_submit_host/evs_wait_host (4 batches in flight)",
                "sync_call_value": lookups / e2e_sync_s, "sync_call_ms_per_step": 1e3 * e2e_sync_s / K},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
    }
    if last_step is not None:
        dump_outputs(args.dump_outputs, *last_step)
    print(json.dumps(line), flush=True)
    if store is not None:
        store.close()
    return 0


def _guard_stdout():
    """Libraries (NCCL's version banner, the reference's printf) write to fd 1; the contract is ONE JSON
    line on stdout.  Everything else is sent to stderr; the JSON line goes to the saved descriptor."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(saved, "w")


if __name__ == "__main__":
    a = parse_args()
    _guard_stdout()
    if a.op:
        from bench_ops import main_ops
        sys.exit(main_ops(a))
    sys.exit(main_reference(a) if a.impl == "reference" else main_ours(a))
