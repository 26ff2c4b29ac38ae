"""Bags on a table-wise sharded cache (evs_shard_lookup_bags) against the plain sharded lookup, on N GPUs of one box.

Kaggle-shape tables (dim 16, fp32 tier), tables placed by row count (sharded.balanced_placement), the 13 % cache budget
split over the ranks (sharded.split_cache_budget), global batch 2048 * N, Zipf(1.05) indices.  For each P the bags of a
batch hold 1..P indices (uniform); P = 1 is the same traffic as the plain line, one index per sample and table.
Each line: a new cache is warmed with `--fill` plain batches and `--warmup` steps of the line's own traffic, then
`--steps` steps are timed (CUDA events between barriers, max over the ranks), one library call per batch for both the bags
and the plain line.  With --gpus 1 the lines are the single-GPU paths (evs_lookup_bags, evs_lookup_batch) through the
same ShardedLookup calls.  Before timing, one bag
step is verified on every rank: each pooled row equals the sum, j ascending in fp32, of the closed-form backing rows of
its bag (workload.synth_rows).

NVLink bytes per step are counted from the shapes: the pooled rows each rank stores into its peers' receive buffers
plus the slice hit counts (one 4-byte word per slice and peer).

    python tools/sharded_bags_bench.py --gpus 2 --steps 50 --warmup 20 --out profiles/sharded_bags_n2.json
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

DIM, BL = 16, 2048


def _card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        power = q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def _bag_batch(trace, T_local, B, P, rng):
    """One bag batch of this rank's tables: lengths uniform in 1..P, indices from the rank's Zipf trace."""
    idx = trace.batch(B * P)
    lS_i, lS_o = [], []
    for t in range(T_local):
        lens = rng.integers(1, P + 1, size=B)
        lS_i.append(np.ascontiguousarray(idx[t, :int(lens.sum())]))
        lS_o.append(np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int64))
    return lS_o, lS_i


def _verify(pkg, rank, world, placement, all_rows, B, P, ly, lS_o, lS_i, dev):
    """Every pooled row this rank received == the fp32 sum, j ascending, of the backing rows of its bag."""
    import torch
    import torch.distributed as dist
    from oracle.evlfu import expand_bags
    tmax = max(len(x) for x in placement)
    mine = torch.full((tmax, B * P), -1, dtype=torch.int64, device=dev)
    mine[:len(lS_i)] = torch.from_numpy(expand_bags(lS_i, lS_o, B, P)).to(dev)
    allv = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(allv, mine)
    Bl = B // world
    ok = True
    for r, ids in enumerate(placement):
        v = allv[r].view(tmax, B, P)[:, rank * Bl:(rank + 1) * Bl]
        for j_t, t in enumerate(ids):
            acc = torch.zeros((Bl, DIM), dtype=torch.float32, device=dev)
            for j in range(P):
                k = v[j_t, :, j]
                rows = pkg.workload.synth_rows(t, k.clamp(min=0), DIM, all_rows[t])
                acc = torch.where((k >= 0)[:, None], acc + rows, acc)
            ok = ok and bool(torch.equal(ly[:, t, :], acc))
    return ok


def _rank(rank, world, port, args, q):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    pkg = importlib.import_module("ev-store-dlrm_b200")
    all_rows = list(pkg.workload.KAGGLE_ROWS)
    T = len(all_rows)
    B = BL * world
    ps = [int(x) for x in args.ps.split(",")]
    placement = pkg.sharded.balanced_placement(all_rows, world)
    ids = placement[rank]
    rows = [all_rows[t] for t in ids]
    cache = pkg.sharded.split_cache_budget([sum(all_rows[t] for t in x) for x in placement], int(sum(all_rows) * 0.13))[rank]
    slices = B * max(ps)
    host = [pkg.workload.synth_table_mapped(t, all_rows[t], DIM, dev) for t in ids]

    def barrier():
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()

    def region(step):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(args.steps):
            step(k)
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1) / args.steps], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    lines = {}
    for P in [0] + ps:                                  # P = 0: the plain sharded line
        cfg = pkg.CacheConfig(n_layers=1, main_precision=32, total_size=cache, max_batch=slices, device=rank, n_tables_total=T,
                              table_ids=tuple(ids))
        store = pkg.EvStore.from_raw_stores(rows, DIM, cfg, {32: host})
        sh = pkg.sharded.ShardedLookup(store, T, DIM, rank, world, transport="p2p", batch_max=slices, placement=placement)
        trace = pkg.workload.ZipfTrace(rows, alpha=1.05, seed=42 + ids[0], perm_seed=7 + ids[0])
        rng = np.random.default_rng(5 + rank)
        n = args.warmup + args.steps
        if P == 0:
            data = [torch.from_numpy(trace.batch(B)).to(dev) for _ in range(n)]
            step = lambda k, base: sh.lookup(data[base + k])
        else:
            data = []
            for _ in range(n):
                o, i = _bag_batch(trace, len(ids), B, P, rng)
                data.append(([torch.from_numpy(x).to(dev) for x in o], [torch.from_numpy(x).to(dev) for x in i], o, i))
            step = lambda k, base: sh.lookup_bags(data[base + k][0], data[base + k][1], P)
        t0 = time.time()
        for _ in range(args.fill):                       # warm the cache with fresh batches of the same distribution
            sh.lookup(torch.from_numpy(trace.batch(B)).to(dev))
        for k in range(args.warmup):
            step(k, 0)
        barrier()
        ok = True
        if P:
            ly, _ = step(0, 0)
            ok = _verify(pkg, rank, world, placement, all_rows, B, P, ly, data[0][2], data[0][3], dev)
        okt = torch.tensor([0.0 if ok else 1.0], dtype=torch.float64, device=dev)
        dist.all_reduce(okt)
        st = store.stats(reset=True)
        ms = region(lambda k: step(k, args.warmup))
        st = store.stats()
        nnz = torch.tensor([float(st["lookups"]) / args.steps], dtype=torch.float64, device=dev)
        hits = torch.tensor([float(st["hits"][0]), float(st["lookups"])], dtype=torch.float64, device=dev)
        dist.all_reduce(nnz)
        dist.all_reduce(hits)
        pooled = B * (world - 1) // world * len(ids) * DIM * 4
        counts = B * max(P, 1) * 4 * (world - 1)
        nv = torch.tensor([float(pooled + counts)], dtype=torch.float64, device=dev)
        dist.all_reduce(nv)
        lines["plain" if P == 0 else f"bags_P{P}"] = dict(
            step_ms=ms, indices_per_step=nnz.item(), indices_per_s=nnz.item() / (ms * 1e-3), hit_rate=hits[0].item() / max(1.0, hits[1].item()),
            nvlink_bytes_per_step_all_ranks=nv.item(), verified=bool(okt.item() == 0.0) if P else None, setup_s=round(time.time() - t0, 1))
        store.close()
    if rank == 0:
        name, power = _card()
        q.put(dict(tool="tools/sharded_bags_bench.py", gpus=world, card=name, power_limit=power, global_batch=B, dim=DIM,
                   shape="kaggle", placement="balanced", cache_budget="13 % of all rows, split_cache_budget", steps=args.steps,
                   warmup=args.warmup, fill=args.fill, lines=lines))
    dist.barrier()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--gpus", type=int, default=2)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--fill", type=int, default=200, help="untimed plain batches that warm the cache before the warm-up")
    ap.add_argument("--ps", default="1,4,10")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < args.gpus:
        sys.exit(f"needs {args.gpus} GPUs, {torch.cuda.device_count()} visible")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 26500 + os.getpid() % 2000
    procs = [ctx.Process(target=_rank, args=(r, args.gpus, port, args, q)) for r in range(args.gpus)]
    for p in procs:
        p.start()
    res = q.get(timeout=3600)
    for p in procs:
        p.join(timeout=120)
    if any(p.exitcode != 0 for p in procs):
        sys.exit("a rank failed")
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    if not all(v["verified"] in (None, True) for v in res["lines"].values()):
        sys.exit("VERIFY FAILED")


if __name__ == "__main__":
    main()
