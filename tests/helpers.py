"""Shared helpers for the parity tests."""
import importlib

import numpy as np

from oracle import codecs as ocodecs
from oracle.evlfu import BatchEvLFU, gather_rows
from oracle.lru import BatchLFU, BatchLRU

SMALL_ROWS = [50, 7, 400, 300, 9, 4, 60, 12, 3, 120, 30, 350, 40, 5, 45, 280, 4, 33, 21, 4, 390, 6, 5, 90, 11, 70]
SKEW_ROWS = [3, 5, 4000, 2500, 7, 4, 60, 9, 3, 300, 50, 3500, 40, 4, 80, 3000, 5, 45, 30, 4, 3800, 6, 5, 600, 11, 400]
TINY_ROWS = [4 + (t % 3) for t in range(26)]


def pkg():
    return importlib.import_module("ev-store-dlrm_b200")


def decoded_tables(tables, prec):
    """What a tier of precision `prec` returns for every row (oracle codecs)."""
    if prec == 32:
        return tables
    return [ocodecs.dequantize_rows(ocodecs.quantize_table(t, prec), prec) for t in tables]


def run_single_tier_parity(rows, dim, prec, total_size, B_list, n_batches, seed=42, approx=-1,
                           store_in_hbm=False, host_path=False, check_state_every=1, alpha=1.05, policy="evlfu", prefetch=False):
    """Drive the CUDA path and BatchEvLFU (or BatchLRU) with the same batches; compare everything, every batch.
    prefetch: every batch is announced with evs_prefetch right after the previous batch was enqueued, so the
    look-ahead kernel races the previous batch's update / eviction kernels as it does in production."""
    import torch
    p = pkg()
    tables = p.workload.make_tables(rows, dim)
    dec = decoded_tables(tables, prec)
    trace = p.workload.ZipfTrace(rows, alpha=alpha, seed=seed)
    cap = total_size * (32 // prec)
    cfg = p.CacheConfig(n_layers=1, main_precision=prec, total_size=total_size, max_batch=max(B_list),
                        approx_emb_thres=approx, record_events=True, store_in_hbm=store_in_hbm, policy=policy)
    store = p.EvStore(tables, cfg)
    oracle = {"lru": BatchLRU, "lfu": BatchLFU, "evlfu": BatchEvLFU}[policy](cap, n_tables=len(rows))
    T = len(rows)
    totals = dict(hits=0, lookups=0, evicted=0, flushed=0)
    try:
        all_idx = [trace.batch(B_list[it % len(B_list)]) for it in range(n_batches)]
        dev_idx = [torch.from_numpy(i).cuda() for i in all_idx] if not host_path else None
        if prefetch:
            torch.cuda.synchronize()
            store.prefetch(dev_idx[0])
        for it in range(n_batches):
            B = B_list[it % len(B_list)]
            idx = all_idx[it]
            if host_path:
                out, hit = store.lookup_host(idx)
            else:
                o, h = store.lookup(dev_idx[it])
                if prefetch and it + 1 < n_batches:
                    store.prefetch(dev_idx[it + 1])
                torch.cuda.synchronize()
                out, hit = o.cpu().numpy(), h.cpu().numpy()
            o_hit, st, sr, agg = oracle.lookup_batch(idx, approx_emb_thres=approx)
            want = gather_rows(dec, st, sr)
            assert (hit.astype(bool) == o_hit).all(), f"hit stream, batch {it} (B={B})"
            ok = st >= 0
            assert (out[ok] == want[ok]).all(), f"rows, batch {it} (B={B})"
            ev, fl = store.last_events()
            assert ev.tolist() == oracle.evicted, f"eviction stream, batch {it}: {ev.tolist()[:8]} vs {oracle.evicted[:8]}"
            assert fl.tolist() == oracle.flushed, f"flush stream, batch {it}"
            if it % check_state_every == 0 or it == n_batches - 1:
                state, n_perfect = store.dump_state()
                assert state == oracle.state(), f"resident state / FIFO order, batch {it}"
                assert n_perfect == oracle.n_perfect, f"n_perfect, batch {it}"
            totals["hits"] += int(o_hit.sum())
            totals["lookups"] += B * T
            totals["evicted"] += len(oracle.evicted)
            totals["flushed"] += len(oracle.flushed)
        store.sync()
        s = store.stats()
        assert s["lookups"] == totals["lookups"]
        assert s["evictions"][0] == totals["evicted"] and s["flushed"][0] == totals["flushed"]
        assert s["size"][0] == len(oracle.entries)
    finally:
        store.close()
    return totals


def run_tier_parity(rows, dim, layers, main, sec, total, B_list, n_batches, prop="", seed=42, check_state_every=1,
                    alpha=1.05, store_in_hbm=False, high_thres=0, prefetch=False):
    """Two / three layer CUDA path vs oracle.tiers.BatchTiers: hit codes, fp32 rows (dequantised at the
    answering tier's precision), eviction / flush streams and FIFO state of both tiers, C3 contents."""
    import torch
    from oracle import tiers as otiers
    p = pkg()
    tables = p.workload.make_tables(rows, dim)
    dec = [decoded_tables(tables, main), decoded_tables(tables, sec)]
    alt = p.workload.make_alt_keys(rows) if layers == 3 else None
    trace = p.workload.ZipfTrace(rows, alpha=alpha, seed=seed)
    caps = otiers.capacities(layers, main, sec, total, prop, dim)
    cfg = p.CacheConfig(n_layers=layers, main_precision=main, secondary_precision=sec, total_size=total,
                        size_proportion=prop, max_batch=max(B_list), record_events=True, store_in_hbm=store_in_hbm,
                        high_agghit_threshold=high_thres)
    store = p.EvStore(tables, cfg, alt_keys=alt)
    oracle = otiers.BatchTiers(caps, n_layers=layers, T=len(rows), alt_keys=alt, high_thres=high_thres or 23)
    tot = dict(c1=0, c2=0, c3=0, miss=0, ev1=0, ev2=0, fl1=0, fl2=0)
    try:
        st0 = store.stats()
        assert tuple(st0["capacity"]) == caps[:2] and st0["c3_capacity"] == (caps[2] if layers == 3 else 0), (st0, caps)
        all_idx = [trace.batch(B_list[it % len(B_list)]) for it in range(n_batches)]
        dev_idx = [torch.from_numpy(i).cuda() for i in all_idx]
        if prefetch:
            torch.cuda.synchronize()
            store.prefetch(dev_idx[0])
        for it in range(n_batches):
            B = B_list[it % len(B_list)]
            idx = all_idx[it]
            o, h = store.lookup(dev_idx[it])
            if prefetch and it + 1 < n_batches:
                store.prefetch(dev_idx[it + 1])
            torch.cuda.synchronize()
            out, hit = o.cpu().numpy(), h.cpu().numpy()
            code, val_tier, st, sr, agg = oracle.lookup_batch(idx)
            assert (hit == code).all(), f"hit codes, batch {it} (B={B}): {np.argwhere(hit != code)[:4].tolist()}"
            want = otiers.gather_tier_rows(dec, val_tier, st, sr)
            assert (out == want).all(), f"rows, batch {it} (B={B})"
            for ti, ot in ((0, oracle.c1), (1, oracle.c2)):
                ev, fl = store.last_events(ti)
                assert ev.tolist() == ot.evicted, f"eviction stream of C{ti + 1}, batch {it}: {ev.tolist()[:6]} vs {ot.evicted[:6]}"
                assert fl.tolist() == ot.flushed, f"flush stream of C{ti + 1}, batch {it}"
            if it % check_state_every == 0 or it == n_batches - 1:
                for ti, ot in ((0, oracle.c1), (1, oracle.c2)):
                    state, n_perfect = store.dump_state(ti)
                    assert state == ot.state(), f"FIFO state of C{ti + 1}, batch {it}"
                    assert n_perfect == ot.n_perfect, f"n_perfect of C{ti + 1}, batch {it}"
                if layers == 3:
                    k, a, r = store.dump_c3()
                    ok, oa, orr = oracle.c3.dump() if oracle.c3 is not None else ([], [], [])
                    if not (k.tolist() == ok and a.tolist() == oa and r.tolist() == orr):
                        kk = k.tolist()
                        d = next((i for i in range(min(len(kk), len(ok))) if kk[i] != ok[i] or r[i] != orr[i]), -1)
                        raise AssertionError(f"C3 contents, batch {it}: len {len(kk)} vs {len(ok)}, first diff at {d}: "
                                             f"{kk[max(0, d - 2):d + 3]} / {r.tolist()[max(0, d - 2):d + 3]} vs {ok[max(0, d - 2):d + 3]} / {orr[max(0, d - 2):d + 3]}; "
                                             f"sets equal {sorted(kk) == sorted(ok)}; group sizes ev2 {len(oracle.c2.evicted)} ev1 {len(oracle.c1.evicted)} c3 size {len(oracle.c3.vals)}")
            tot["c1"] += int((code == 1).sum())
            tot["c2"] += int((code == 2).sum())
            tot["c3"] += int((code == 3).sum())
            tot["miss"] += int((code == 0).sum())
            tot["ev1"] += len(oracle.c1.evicted)
            tot["ev2"] += len(oracle.c2.evicted)
            tot["fl1"] += len(oracle.c1.flushed)
            tot["fl2"] += len(oracle.c2.flushed)
        store.sync()
        s = store.stats()
        assert s["hits"] == [tot["c1"], tot["c2"]] and s["c3_hits"] == tot["c3"] and s["misses"] == tot["miss"], (s, tot)
        assert s["evictions"] == [tot["ev1"], tot["ev2"]]
        assert s["size"] == [len(oracle.c1.entries), len(oracle.c2.entries)]
    finally:
        store.close()
    return tot


def load_dlrm_golden(golden_dir):
    """tests/golden/dlrm_forward.npz with the weights and tables of the model it was computed with.  The file holds the
    inputs, the reference's outputs and the SHA-256 of every weight / table array.  The arrays themselves are redrawn
    here in the order DLRM_Net.__init__ draws them from np.random seeded with `seed` (create_emb: uniform(+-sqrt(1/n))
    per table; create_mlp for the bottom, then the top MLP: normal(0, sqrt(2/(m+n))) weights, normal(0, sqrt(1/m))
    biases) and must hash to the stored digests."""
    import hashlib
    import os
    with np.load(os.path.join(golden_dir, "dlrm_forward.npz")) as z:
        g = {k: z[k] for k in z.files}
    rng = np.random.RandomState(int(g["seed"]))
    m_spa = g["R"].shape[1] - 27 * 26 // 2
    for k, n in enumerate(int(x) for x in g["rows"]):
        g[f"emb_{k}"] = rng.uniform(low=-np.sqrt(1 / n), high=np.sqrt(1 / n), size=(n, m_spa)).astype(np.float32)
    for name, ln in (("bot", [g["X"].shape[1], 512, 256, 64, m_spa]), ("top", [g["R"].shape[1], 512, 256, 1])):
        for i in range(len(ln) - 1):
            n, m = ln[i], ln[i + 1]
            g[f"{name}_w{i}"] = rng.normal(0.0, np.sqrt(2 / (m + n)), size=(m, n)).astype(np.float32)
            g[f"{name}_b{i}"] = rng.normal(0.0, np.sqrt(1 / m), size=m).astype(np.float32)
    for k in [k for k in g if k.startswith("sha256_")]:
        assert hashlib.sha256(g[k[7:]].tobytes()).digest() == g[k].tobytes(), f"{k[7:]} differs from the reference's array"
    return g


def dlrm_forward_cpu(g, tables):
    """sequential_forward of the reference's DLRM_Net (dlrm_s_pytorch.py:588-613) restated with plain torch on the
    CPU over the weights of tests/golden/dlrm_forward.npz and the given embedding tables.  Returns (Z [B,1], R [B,367])."""
    import torch

    def mlp(x, name, n, sig):
        for i in range(n):
            x = torch.nn.functional.linear(x, torch.from_numpy(g[f"{name}_w{i}"]), torch.from_numpy(g[f"{name}_b{i}"]))
            x = torch.sigmoid(x) if i == sig else torch.relu(x)
        return x

    x = mlp(torch.from_numpy(g["X"]), "bot", 4, -1)
    ly = [torch.from_numpy(np.ascontiguousarray(tables[k][g["lS_i"][k]])) for k in range(26)]
    T = torch.cat([x.unsqueeze(1), torch.stack(ly, dim=1)], dim=1)
    Zm = torch.bmm(T, T.transpose(1, 2))
    li = torch.tensor([i for i in range(27) for j in range(i)])
    lj = torch.tensor([j for i in range(27) for j in range(i)])
    R = torch.cat([x, Zm[:, li, lj]], dim=1)
    return mlp(R, "top", 3, 2).numpy(), R.numpy()
