"""bench.py --op interact | embedding_bag: the two tensor ops either side of the cache in sequential_forward
(dlrm_s_pytorch_C1_C2_C3.py:742-768), each timed alone against the HBM roofline.

  interact       evs_interact (k_interact_mma): T = [x ; ly], Z = T T^t on the tensor cores, strict lower triangle packed
                 behind x  (interact_features, :625-658).  Algorithmic bytes per sample = ((n_f + 1) d + d + pairs) * 4.
  embedding_bag  evs_embedding_bag (k_gather): out[b] = sum of the bag's rows, nn.EmbeddingBag(mode="sum")
                 (apply_emb_ori_dlrm, :191-223).  Algorithmic bytes = nnz * (8 + row bytes) + B * (8 + 4 d).

Inputs rotate through enough buffers that consecutive launches never find their data in the 126 MB L2.
"""
from __future__ import annotations

import ctypes as C
import importlib
import json


def _time_launches(fn, n_sets, K, W=5):
    import torch
    for k in range(W):
        fn(k % n_sets)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(K):
        fn(k % n_sets)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / K


def bench_interact(pkg, dev, B=16384, n_f=26, d=16, K=50, peak=6459.3):
    import torch
    lib = pkg.load_library()
    pairs = (n_f + 1) * n_f // 2
    per_set = B * ((n_f + 1) * d + d + pairs) * 4
    n_sets = max(3, int(400e6 // per_set) + 1)
    xs = [torch.randn((B, d), device=dev) for _ in range(n_sets)]
    lys = [torch.randn((B, n_f, d), device=dev) for _ in range(n_sets)]
    outs = [torch.empty((B, d + pairs), device=dev) for _ in range(n_sets)]
    st = torch.cuda.current_stream(dev).cuda_stream or 1

    def run(i):
        rc = lib.evs_interact(xs[i].data_ptr(), lys[i].data_ptr(), outs[i].data_ptr(), B, n_f, d, st)
        assert rc == 0

    ms = _time_launches(run, n_sets, K)
    # against torch: cat + bmm + tril gather + cat (what the reference runs on the GPU)
    li = torch.tensor([i for i in range(n_f + 1) for j in range(i)], device=dev)
    lj = torch.tensor([j for i in range(n_f + 1) for j in range(i)], device=dev)

    def run_torch(i):
        T = torch.cat([xs[i].unsqueeze(1), lys[i]], dim=1)
        Z = torch.bmm(T, T.transpose(1, 2))
        return torch.cat([xs[i], Z[:, li, lj]], dim=1)

    ms_t = _time_launches(run_torch, n_sets, max(5, K // 5))
    run(0)
    torch.cuda.synchronize()
    err = float((run_torch(0) - outs[0]).abs().max())
    gbs = per_set / (ms * 1e-3) / 1e9
    return {"op": "interact", "kernel": "k_interact_mma (mma.sync m16n8k8 TF32, operands split hi + lo)", "B": B, "n_f": n_f, "dim": d,
            "ms": ms, "algorithmic_bytes": per_set, "achieved_GBps": gbs, "frac_of_hbm_peak": gbs / peak,
            "flop": 2 * (n_f + 1) ** 2 * d * B, "torch_cat_bmm_tril_ms": ms_t, "speedup_vs_torch": ms_t / ms, "max_abs_diff_vs_torch": err,
            "buffers_rotated": n_sets}


def bench_embedding_bag(pkg, dev, B=16384, P=10, d=64, rows=4_000_000, prec=32, K=50, peak=6459.3):
    import torch
    lib = pkg.load_library()
    row_bytes = d * prec // 8
    table = torch.randint(0, 255, (rows, row_bytes), dtype=torch.uint8, device=dev) if prec != 32 else \
        torch.randn((rows, d), device=dev)
    nnz = B * P
    n_sets = 4
    idxs = [torch.randint(0, rows, (nnz,), dtype=torch.int64, device=dev) for _ in range(n_sets)]
    off = torch.arange(0, nnz, P, dtype=torch.int64, device=dev)
    outs = [torch.empty((B, d), device=dev) for _ in range(n_sets)]
    st = torch.cuda.current_stream(dev).cuda_stream or 1

    def run(i):
        rc = lib.evs_embedding_bag(table.data_ptr(), rows, d, prec, idxs[i].data_ptr(), off.data_ptr(), nnz, B, None, outs[i].data_ptr(), d, st)
        assert rc == 0

    ms = _time_launches(run, n_sets, K)
    alg = nnz * (8 + row_bytes) + B * (8 + 4 * d)
    res = {"op": "embedding_bag", "kernel": "k_gather", "B": B, "indices_per_bag": P, "dim": d, "precision": prec, "table_rows": rows,
           "table_bytes": rows * row_bytes, "ms": ms, "algorithmic_bytes": alg, "achieved_GBps": alg / (ms * 1e-3) / 1e9,
           "frac_of_hbm_peak": alg / (ms * 1e-3) / 1e9 / peak,
           "note": "uniform random rows of a table far larger than L2: every row is a separate %d-byte DRAM access" % row_bytes}
    if prec == 32:
        eb = torch.nn.EmbeddingBag(rows, d, mode="sum", _weight=table)
        ms_t = _time_launches(lambda i: eb(idxs[i], off), n_sets, max(5, K // 5))
        res["torch_embedding_bag_ms"] = ms_t
        res["speedup_vs_torch"] = ms_t / ms
        run(0)
        torch.cuda.synchronize()
        res["max_abs_diff_vs_torch"] = float((eb(idxs[0], off) - outs[0]).abs().max())
    return res


def bench_knn(pkg, dev, n=262144, d=16, K=3):
    """evs_knn, every row of an [n, d] matrix against all rows (the alt-key generator's inner loop).  FLOP = 2 d per pair (the
    tensor cores execute 3x that for the hi / lo split: hi rounded to TF32, lo the exact remainder, truncated by the tensor
    core); the kernel is bound by the selection's ALU work, not by the tensor pipe."""
    import torch
    x = torch.randn((n, d), device=dev)
    nbr = pkg.altkeys.knn(x)                              # warm-up (and the result for the spot check)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        pkg.altkeys.knn(x)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / K
    # spot check of 64 rows against torch's fp32 distances
    rows = torch.arange(0, n, n // 64, device=dev)[:64]
    d2 = torch.cdist(x[rows], x).pow(2)
    want = d2.topk(11, dim=1, largest=False).indices[:, 1:]
    agree = float((want == nbr[rows]).float().mean())
    pairs = float(n) * n
    return {"op": "knn", "kernel": "k_knn (mma.sync m16n8k8 TF32, operands split hi + lo; top-11 selection in registers) + k_knn_merge",
            "rows": n, "dim": d, "k": 10, "ms": ms, "pairs_per_s": pairs / (ms * 1e-3), "useful_TFLOPs": pairs * 2 * d / (ms * 1e-3) / 1e12,
            "tensor_TFLOPs_executed": pairs * 2 * ((d + 7) // 8 * 8) * 3 / (ms * 1e-3) / 1e12, "agreement_with_torch_cdist_topk": agree,
            "full_kaggle_estimate_s": (33.76e6 ** 2) / (pairs / (ms * 1e-3))}


def main_ops(args):
    import torch
    from bench import measured_peak_hbm
    assert torch.cuda.is_available(), "bench.py --op needs a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    pkg = importlib.import_module("ev-store-dlrm_b200")
    peak, src = measured_peak_hbm()
    B = args.batch or 16384
    K = max(10, args.steps)
    if args.op == "knn":
        legs = [bench_knn(pkg, dev, n=(args.batch or 262144), d=d) for d in ([args.dim] if args.dim else [16, 64])]
        line = {"metric": "knn_pairs_per_s", "op": "knn", "value": max(l["pairs_per_s"] for l in legs), "unit": "pairs/s", "n_gpus": 1,
                "steps": 3, "legs": legs, "data": "synthetic"}
        print(json.dumps(line), flush=True)
        return 0
    if args.op == "interact":
        legs = [bench_interact(pkg, dev, B=B, d=d, K=K, peak=peak) for d in ([args.dim] if args.dim else [16, 64])]
    else:
        legs = [bench_embedding_bag(pkg, dev, B=B, P=10, d=d, prec=p, K=K, peak=peak)
                for d, p in ([(args.dim, args.precision)] if args.dim else [(16, 32), (64, 32), (64, 8)])]
    line = {"metric": "op_GBps", "op": args.op, "value": max(l["achieved_GBps"] for l in legs), "unit": "GB/s", "n_gpus": 1,
            "steps": K, "peak": peak, "peak_source": src, "legs": legs, "data": "synthetic"}
    print(json.dumps(line), flush=True)
    return 0
