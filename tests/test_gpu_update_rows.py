"""evs_update_rows / EvStore.update_rows: new row values, written into the backing store at every precision and into
every cached copy, stream-ordered between batches.

The oracles of the other parity tests (BatchEvLFU, BatchLRU, BatchLFU, BatchTiers) still decide every hit code, eviction,
flush and C3 record -- an update moves no policy state -- and the expected rows are gathered from a MUTABLE copy of the
fp32 tables that each update is applied to, decoded at the serving tier's precision."""
import os

import numpy as np
import pytest

from helpers import SMALL_ROWS, decoded_tables, pkg
from oracle import codecs as ocodecs
from oracle.evlfu import BatchEvLFU, gather_rows
from oracle.lru import BatchLFU, BatchLRU

pytestmark = pytest.mark.gpu

WHERE_C1, WHERE_C2, WHERE_STORE, WHERE_REJECTED = 1, 2, 4, 0x80


def _f32(x):
    return np.asarray(x, dtype=np.float32)


def _edge_values():
    """Every codec edge, both signs of zero, and the float32 neighbours of each, both ways."""
    e = [0.65, -0.65, 1.0, -1.0, 0.00025, 0.015, 0.25, 0.4, 0.6, 0.8, -0.8, -0.6, -0.4, -0.25, -0.015, -0.00025, 0.0, -0.0]
    e = _f32(e)
    return np.concatenate([e, np.nextafter(e, _f32(np.inf)), np.nextafter(e, _f32(-np.inf))])


def _value_pool(golden_dir):
    with np.load(os.path.join(golden_dir, "codecs.npz")) as z:
        x = _f32(z["x"])
    return np.concatenate([_edge_values(), x, _f32([5.9, -5.9, 6.0, -6.0, 3.21, -3.21])])


def _encodable(v, prec):
    """Values `prec` bits can hold: what evs_update_rows accepts."""
    v = _f32(v)
    if prec == 32:
        return np.ones(v.shape, dtype=bool)
    fin = np.isfinite(v)
    if prec == 8:
        return fin & (v >= -1) & (v <= 1)
    if prec == 16:
        w = np.where(fin & (np.abs(v) < 100), v, 0).astype(np.float64)
        below = np.trunc(-100.0 * (0.65 + w)).astype(np.int64)
        below += (below % 2 == 0)
        above = np.trunc(100.0 * (w - 0.65)).astype(np.int64)
        above -= (above % 2 == 1)
        mid = np.trunc((w + 0.65) / 1.3 * 65000).astype(np.int64)
        q = np.where(w < -0.65, 65000 + below, np.where(w > 0.65, 65000 + above, mid))
        return fin & (np.abs(v) < 100) & (q >= 0) & (q <= 65535)
    return fin


def _expect_rows(v, prec):
    """What a lookup served at `prec` bits returns for fp32 rows v [n, d]."""
    return v if prec == 32 else ocodecs.dequantize_rows(ocodecs.quantize_table(v, prec), prec)


def _keys(t, r):
    return (np.asarray(t, dtype=np.int64) << 40) | np.asarray(r, dtype=np.int64)


def _update(store, keys, vals, stream=None):
    """store.update_rows over library-format keys; returns where (numpy)."""
    import torch
    keys = np.asarray(keys, dtype=np.int64)
    t = torch.from_numpy(keys >> 40).cuda()
    r = torch.from_numpy(keys & ((1 << 40) - 1)).cuda()
    w = store.update_rows(t, r, torch.from_numpy(np.ascontiguousarray(vals, dtype=np.float32)).cuda(), stream=stream)
    return w


def _store_bytes(store, table, tier, prec, rows, dim):
    """The backing rows of (tier, table) as the device reads them (host array, or the HBM copy)."""
    import torch
    ptr, p = store.store_ptr(table, tier)
    assert p == prec
    nbytes = rows * dim * prec // 8

    class _U8:
        __cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (int(ptr), False), "version": 2}
    if store.cfg.store_in_hbm:
        return torch.as_tensor(_U8(), device="cuda").cpu().numpy().copy()
    return np.frombuffer(store._stores[prec][table], dtype=np.uint8).copy()


# ---- 1. encoders bit-exact, writes byte-exact ---------------------------------------------------------------------------
@pytest.mark.parametrize("memory", ["host", "hbm", "host_alloc"])
@pytest.mark.parametrize("dim", [16, 18, 36, 64])
@pytest.mark.parametrize("prec", [32, 16, 8, 4])
def test_encoders_and_byte_exact_writes(prec, dim, memory, golden_dir):
    import torch
    p = pkg()
    rng = np.random.default_rng(prec * 1000 + dim)
    pool = _value_pool(golden_dir)
    ok_pool = pool[_encodable(pool, prec)]
    n_rows = 2 * (len(pool) // dim + 8) + 1
    base = rng.uniform(-0.9, 0.9, size=(n_rows, dim)).astype(np.float32)
    stores = {prec: [p.to_host_rows(p.codecs.encode_table(base, prec))]} if memory == "host_alloc" else None
    tables = [p.to_host_rows(base) if (memory == "host_alloc" and prec == 32) else base.copy()]
    store = p.EvStore(tables, p.CacheConfig(total_size=64, max_batch=8, main_precision=prec, store_in_hbm=memory == "hbm"),
                      stores=stores)
    try:
        before = _store_bytes(store, 0, 0, prec, n_rows, dim)
        # odd rows are updated (every pool value once, padded with encodable values); even rows are their untouched neighbours
        upd_rows = np.arange(1, n_rows, 2)
        vals = rng.choice(ok_pool, size=(len(upd_rows), dim))
        flat = vals.reshape(-1)
        flat[:len(ok_pool)] = ok_pool
        bad = {32: None, 16: [np.nan, 7.0, -6.5, np.inf], 8: [np.nan, 1.0000001, -1.5, -np.inf], 4: [np.nan, np.inf, -np.inf]}[prec]
        rejected = []
        if bad is not None:
            for k, b in enumerate(bad):
                i = len(upd_rows) - 1 - k
                vals[i, (3 * k) % dim] = b
                rejected.append(i)
        else:
            vals[-1, :3] = np.array([0x7FC01234, 0xFF800001, 0x80000000], dtype=np.uint32).view(np.float32)  # NaNs, -0.0 as given
        where = _update(store, _keys(0, upd_rows), vals)
        torch.cuda.synchronize()
        w = where.cpu().numpy()
        want_where = np.full(len(upd_rows), WHERE_STORE, dtype=np.uint8)
        want_where[rejected] = WHERE_REJECTED
        assert np.array_equal(w, want_where), np.argwhere(w != want_where)[:4]
        after = _store_bytes(store, 0, 0, prec, n_rows, dim)
        want = before.reshape(n_rows, -1).copy()
        acc = np.setdiff1d(np.arange(len(upd_rows)), rejected)
        want[upd_rows[acc]] = p.codecs.encode_table(vals[acc], prec).view(np.uint8).reshape(len(acc), -1)
        # the device encoders equal both host quantisers
        assert np.array_equal(p.codecs.encode_table(vals[acc], prec).view(np.uint8), ocodecs.quantize_table(vals[acc], prec).view(np.uint8))
        got = after.reshape(n_rows, -1)
        assert np.array_equal(got, want), f"bytes differ in rows {np.unique(np.argwhere(got != want)[:, 0])[:6]}"
        if memory == "hbm":      # the host arrays are left untouched
            assert np.array_equal(np.frombuffer(store._stores[prec][0], dtype=np.uint8), before)
    finally:
        store.close()


# ---- 2. policy invariance and values, every batch ----------------------------------------------------------------------
def _pick_keys(rng, rows, resident_sets, next_idx, c3_targets, k=6):
    """A mix of keys: resident in each tier, not resident, missing in the next batch, C3 alt-key targets."""
    T = len(rows)
    res_all = set().union(*resident_sets)
    out = []
    for s in resident_sets:
        if s:
            out += list(rng.choice(sorted(s), size=min(k, len(s)), replace=False))
    t = rng.integers(0, T, size=4 * k)
    r = (rng.random(4 * k) * np.asarray(rows)[t]).astype(np.int64)
    out += [x for x in _keys(t, r).tolist() if x not in res_all][:k]
    nxt = _keys(np.repeat(np.arange(T)[:, None], next_idx.shape[1], axis=1), next_idx).reshape(-1)
    miss = sorted(set(nxt.tolist()) - res_all)
    if miss:
        out += list(rng.choice(miss, size=min(k, len(miss)), replace=False))
    if c3_targets:
        out += list(rng.choice(sorted(c3_targets), size=min(k, len(c3_targets)), replace=False))
    return np.unique(np.asarray(out, dtype=np.int64))


def _apply(ref, keys, vals):
    for k, v in zip(keys.tolist(), vals):
        ref[k >> 40][k & ((1 << 40) - 1)] = v


def _check_where(where, keys, resident_sets):
    want = np.array([WHERE_STORE | sum((1 << i) for i, s in enumerate(resident_sets) if k in s) for k in keys.tolist()], dtype=np.uint8)
    assert np.array_equal(where, want), (keys[where != want][:4], where[where != want][:4], want[where != want][:4])


@pytest.mark.parametrize("policy,prec,approx", [("evlfu", 16, 10), ("evlfu", 32, 12), ("lru", 32, -1), ("lfu", 8, -1)])
def test_single_tier_policy_invariance_and_values(policy, prec, approx):
    import torch
    p = pkg()
    rows, dim, total, B, n = SMALL_ROWS, 16, 180, 64, 40
    tables = p.workload.make_tables(rows, dim)
    ref = [t.copy() for t in tables]
    trace = p.workload.ZipfTrace(rows, seed=5)
    cap = total * (32 // prec)
    store = p.EvStore(tables, p.CacheConfig(main_precision=prec, total_size=total, max_batch=B, approx_emb_thres=approx,
                                            record_events=True, policy=policy))
    oracle = {"lru": BatchLRU, "lfu": BatchLFU, "evlfu": BatchEvLFU}[policy](cap, n_tables=len(rows))
    rng = np.random.default_rng(3)
    idx = [trace.batch(B) for _ in range(n)]
    n_upd = n_sub = 0
    try:
        for it in range(n):
            o, h = store.lookup(torch.from_numpy(idx[it]).cuda())
            torch.cuda.synchronize()
            o_hit, st, sr, _ = oracle.lookup_batch(idx[it], approx_emb_thres=approx)
            assert (h.cpu().numpy().astype(bool) == o_hit).all(), f"hit stream, batch {it}"
            n_sub += int((h.cpu().numpy() == 4).sum())
            ok = st >= 0
            want = gather_rows(decoded_tables(ref, prec), st, sr)
            assert (o.cpu().numpy()[ok] == want[ok]).all(), f"rows, batch {it}"
            ev, fl = store.last_events()
            assert ev.tolist() == oracle.evicted and fl.tolist() == oracle.flushed, f"eviction / flush stream, batch {it}"
            state, n_perfect = store.dump_state()
            assert state == oracle.state() and n_perfect == oracle.n_perfect, f"state, batch {it}"
            if it + 1 < n:
                resident = [set(k for b in state for k in b)]
                keys = _pick_keys(rng, rows, resident, idx[it + 1], set())
                vals = rng.uniform(-1, 1, size=(len(keys), dim)).astype(np.float32)
                w = _update(store, keys, vals)
                _apply(ref, keys, vals)
                _check_where(w.cpu().numpy(), keys, resident)
                n_upd += len(keys)
        s = store.stats()
        assert s["lookups"] == n * B * len(rows) and s["size"][0] == len(oracle.entries)
        assert n_upd > 0 and (approx < 0 or n_sub > 0)
    finally:
        store.close()


@pytest.mark.parametrize("layers,main,sec,total,prop", [(2, 32, 8, 100, ""), (2, 16, 4, 200, ""), (2, 8, 4, 200, ""),
                                                        (3, 8, 4, 200, "45-45-10")])
def test_tiers_policy_invariance_and_values(layers, main, sec, total, prop):
    import torch
    from oracle import tiers as otiers
    p = pkg()
    rows, dim, B, n = SMALL_ROWS, 16, 64, 40
    tables = p.workload.make_tables(rows, dim)
    ref = [t.copy() for t in tables]
    alt = p.workload.make_alt_keys(rows) if layers == 3 else None
    trace = p.workload.ZipfTrace(rows, seed=9)
    caps = otiers.capacities(layers, main, sec, total, prop, dim)
    store = p.EvStore(tables, p.CacheConfig(n_layers=layers, main_precision=main, secondary_precision=sec, total_size=total,
                                            size_proportion=prop, max_batch=B, record_events=True), alt_keys=alt)
    oracle = otiers.BatchTiers(caps, n_layers=layers, T=len(rows), alt_keys=alt)
    rng = np.random.default_rng(4)
    idx = [trace.batch(B) for _ in range(n)]
    tot = dict(c2=0, c3=0, both=0)
    try:
        for it in range(n):
            o, h = store.lookup(torch.from_numpy(idx[it]).cuda())
            torch.cuda.synchronize()
            code, val_tier, st, sr, _ = oracle.lookup_batch(idx[it])
            assert (h.cpu().numpy() == code).all(), f"hit codes, batch {it}"
            dec = [decoded_tables(ref, main), decoded_tables(ref, sec)]
            assert (o.cpu().numpy() == otiers.gather_tier_rows(dec, val_tier, st, sr)).all(), f"rows, batch {it}"
            states = []
            for ti, ot in ((0, oracle.c1), (1, oracle.c2)):
                ev, fl = store.last_events(ti)
                assert ev.tolist() == ot.evicted and fl.tolist() == ot.flushed, f"streams of C{ti + 1}, batch {it}"
                state, n_perfect = store.dump_state(ti)
                assert state == ot.state() and n_perfect == ot.n_perfect, f"state of C{ti + 1}, batch {it}"
                states.append(set(k for b in state for k in b))
            c3_targets = set()
            if layers == 3:
                k, a, r = store.dump_c3()
                ok, oa, orr = oracle.c3.dump()
                assert k.tolist() == ok and a.tolist() == oa and r.tolist() == orr, f"C3, batch {it}"
                c3_targets = set(_keys(a.astype(np.int64) % 100 - 1, a.astype(np.int64) // 100).tolist())
            tot["c2"] += int((code == 2).sum())
            tot["c3"] += int((code == 3).sum())
            if it + 1 < n:
                keys = _pick_keys(rng, rows, states, idx[it + 1], c3_targets)
                vals = rng.uniform(-1, 1, size=(len(keys), dim)).astype(np.float32)
                w = _update(store, keys, vals).cpu().numpy()
                _apply(ref, keys, vals)
                _check_where(w, keys, states)
                tot["both"] += int(((w & 3) == 3).sum())
        s = store.stats()
        assert s["size"] == [len(oracle.c1.entries), len(oracle.c2.entries)]
        assert tot["c2"] > 0 and (layers < 3 or tot["c3"] > 0), tot
    finally:
        store.close()


# ---- 3. ordering without synchronisation -------------------------------------------------------------------------------
@pytest.mark.parametrize("layers,main,sec", [(1, 32, 0), (1, 4, 0), (2, 32, 8)])
def test_ordered_between_batches_without_synchronisation(layers, main, sec):
    import torch
    p = pkg()
    rows, dim, B = SMALL_ROWS, 16, 32
    tables = p.workload.make_tables(rows, dim)
    old = [t.copy() for t in tables]
    store = p.EvStore(tables, p.CacheConfig(n_layers=layers, main_precision=main, secondary_precision=sec, total_size=2000,
                                            max_batch=B))
    try:
        a = np.zeros((len(rows), B), dtype=np.int64)
        b = np.ones((len(rows), B), dtype=np.int64)                       # row 1 of every table: a miss in batch n + 1
        b[:, ::2] = 0                                                     # row 0: a C1 hit in batch n + 1 (inserted by batch n)
        da, db = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
        keys = np.concatenate([_keys(np.arange(len(rows)), 0), _keys(np.arange(len(rows)), 1)])
        vals = np.random.default_rng(1).uniform(-1, 1, size=(len(keys), dim)).astype(np.float32)
        kt = torch.from_numpy(keys).cuda()
        vt = torch.from_numpy(vals).cuda()
        torch.cuda.synchronize()
        out_a, _ = store.lookup(da)
        store.update_rows(kt >> 40, kt & ((1 << 40) - 1), vt)
        out_b, hit_b = store.lookup(db)
        torch.cuda.synchronize()
        T = len(rows)
        for t in range(T):
            assert np.array_equal(out_a[:, t].cpu().numpy(), np.repeat(_expect_rows(old[t][:1], main), B, axis=0)), t
            new0, new1 = _expect_rows(vals[t:t + 1], main)[0], _expect_rows(vals[T + t:T + t + 1], main)[0]
            got = out_b[:, t].cpu().numpy()
            assert np.array_equal(got[::2], np.repeat(new0[None], B // 2, axis=0)), t
            assert np.array_equal(got[1::2], np.repeat(new1[None], B // 2, axis=0)), t
        assert (hit_b.cpu().numpy()[::2] == 1).all()
    finally:
        store.close()


# ---- 4. look-ahead -----------------------------------------------------------------------------------------------------
def _fresh_batches(rows, B, n, first_row):
    """n batches whose keys are all different from each other and from anything earlier: rows first_row + ..."""
    out = []
    for k in range(n):
        b = np.empty((len(rows), B), dtype=np.int64)
        for t, r in enumerate(rows):
            b[t] = (first_row + k * B + np.arange(B)) % r
        out.append(b)
    return out


@pytest.mark.parametrize("grouped", [False, True])
def test_look_ahead_staged_rows_are_not_served_after_an_update(grouped):
    """The next batch is announced and, after a synchronise, its misses are staged with the OLD bytes; the update in
    between must cancel the announcement.  Without the cancellation the old rows come back every time."""
    import torch
    p = pkg()
    rows, dim, B = [5000] * 8, 16, 256
    tables = p.workload.make_tables(rows, dim)
    ref = [t.copy() for t in tables]
    store = p.EvStore(tables, p.CacheConfig(total_size=50000, max_batch=B, record_events=True))
    oracle = BatchEvLFU(50000, n_tables=len(rows))
    rng = np.random.default_rng(8)
    try:
        batches = [torch.from_numpy(x).cuda() for x in _fresh_batches(rows, B, 12, 0)]
        host = [x.cpu().numpy() for x in batches]

        def check(outs, hits, ks):
            torch.cuda.synchronize()
            for o, h, k in zip(outs, hits, ks):
                o_hit, st, sr, _ = oracle.lookup_batch(host[k])
                assert (h.cpu().numpy().astype(bool) == o_hit).all(), k
                assert np.array_equal(o.cpu().numpy(), gather_rows(ref, st, sr)), f"rows of batch {k}"

        def update_batch(k):
            keys = np.unique(_keys(np.repeat(np.arange(len(rows))[:, None], B, axis=1), host[k]).reshape(-1))
            vals = rng.uniform(-1, 1, size=(len(keys), dim)).astype(np.float32)
            _update(store, keys, vals)
            _apply(ref, keys, vals)

        if grouped:
            outs, hits = store.lookup_many(batches[0:4])
            store.prefetch(batches[4])
            check(outs, hits, range(0, 4))                 # synchronises: batch 4's misses are staged
            update_batch(4)
            update_batch(6)                                # a batch inside the next group, staged by that group itself
            outs, hits = store.lookup_many(batches[4:8])
            check(outs, hits, range(4, 8))
            # update, then announce at once (no synchronise): the look-ahead must read the new bytes
            store.prefetch(batches[8])
            update_batch(8)
            store.prefetch(batches[8])
            outs, hits = store.lookup_many(batches[8:12])
            check(outs, hits, range(8, 12))
        else:
            for k in range(0, 10, 2):
                o, h = store.lookup(batches[k])
                store.prefetch(batches[k + 1])
                check([o], [h], [k])                       # synchronises: batch k + 1's misses are staged
                update_batch(k + 1)
                if k >= 4:
                    store.prefetch(batches[k + 1])         # announced again after the update: stages the new bytes
                o, h = store.lookup(batches[k + 1])
                check([o], [h], [k + 1])
    finally:
        store.close()


# ---- 5. duplicates, n = 0, rejected keys, argument checks -----------------------------------------------------------------
def test_duplicates_last_wins_empty_call_rejected_keys_and_argument_errors():
    import torch
    p = pkg()
    rows, dim = [30, 40, 50, 60], 18
    tables = p.workload.make_tables(rows, dim)
    store = p.EvStore(tables, p.CacheConfig(total_size=64, max_batch=8, n_tables_total=26, table_base=10, main_precision=8))
    try:
        before = [np.frombuffer(a, dtype=np.uint8).copy() for a in store._stores[8]]
        v = np.random.default_rng(2).uniform(-1, 1, size=(7, dim)).astype(np.float32)
        v_bad = v.copy()
        v_bad[6, 5] = 1.5
        keys = _keys([11, 11, 11, 12, 12, 13, 13], [3, 3, 3, 7, 7, 9, 9])
        w = _update(store, keys, v_bad).cpu().numpy()
        torch.cuda.synchronize()
        store.check()                                               # value rejections raise no sticky error
        assert w.tolist() == [0, 0, WHERE_STORE, 0, WHERE_STORE, 0, WHERE_REJECTED]
        got = [np.frombuffer(a, dtype=np.uint8).reshape(r, -1) for a, r in zip(store._stores[8], rows)]
        assert np.array_equal(got[1][3], p.codecs.encode_table(v[2:3], 8)[0])           # the last of three, whole
        assert np.array_equal(got[2][7], p.codecs.encode_table(v[4:5], 8)[0])
        assert np.array_equal(got[3][9], before[3].reshape(rows[3], -1)[9])      # the last one is rejected: nothing written
        for t in (0, 1, 2, 3):
            m = np.ones(rows[t], dtype=bool)
            m[{0: [], 1: [3], 2: [7], 3: []}[t]] = False
            assert np.array_equal(got[t][m], before[t].reshape(rows[t], -1)[m]), t
        # n = 0
        e = store.update_rows(10, torch.empty(0, dtype=torch.int64, device="cuda"), torch.empty((0, dim), device="cuda"))
        assert e.shape == (0,)
        # out of range / foreign / negative: 0x80 and the sticky index error
        w = _update(store, np.array([_keys(10, 30), _keys(13, 60), _keys(9, 0), _keys(14, 0), -1, _keys(10, 29)]),
                    np.zeros((6, dim), dtype=np.float32)).cpu().numpy()
        torch.cuda.synchronize()
        assert w.tolist() == [WHERE_REJECTED] * 5 + [WHERE_STORE]
        with pytest.raises(p.EvsError):
            store.check()
        with pytest.raises(p.EvsError):
            store.check(clear=True)
        store.check()
        r = torch.zeros(2, dtype=torch.int64, device="cuda")
        good = torch.zeros((2, dim), device="cuda")
        for args in ((10, r.float(), good), (10, r, good.double()), (10, r, good[:, :-1]), (10, r, good.cpu()), (10, r.cpu(), good),
                     (torch.zeros(2, device="cuda"), r, good), (torch.zeros(3, dtype=torch.int64, device="cuda"), r, good),
                     (10, r, torch.zeros((3, dim), device="cuda")), (10, r, torch.zeros((dim, 2), device="cuda").t())):
            with pytest.raises(ValueError):
                store.update_rows(*args)
    finally:
        store.close()


def test_update_refused_during_stream_capture():
    import torch
    p = pkg()
    tables = p.workload.make_tables([20] * 3, 16)
    store = p.EvStore(tables, p.CacheConfig(total_size=64, max_batch=8))
    try:
        s = torch.cuda.Stream()
        r = torch.zeros(1, dtype=torch.int64, device="cuda")
        v = torch.zeros((1, 16), device="cuda")
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with pytest.raises(p.EvsError):
            with torch.cuda.graph(g, stream=s):
                store.update_rows(0, r, v)
    finally:
        torch.cuda.synchronize()
        store.close()


# ---- 6. the other read paths --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("prec", [32, 4])
def test_bags_and_storage_paths_see_the_update(prec):
    import torch
    p = pkg()
    rows, dim, B, P = SMALL_ROWS, 16, 16, 4
    tables = p.workload.make_tables(rows, dim)
    ref = [t.copy() for t in tables]
    store = p.EvStore(tables, p.CacheConfig(total_size=400, max_batch=B * P, main_precision=prec))
    rng = np.random.default_rng(6)
    T = len(rows)
    try:
        lens = [rng.integers(0, P + 1, size=B) for _ in range(T)]
        lS_i = [torch.from_numpy((rng.random(int(l.sum())) * rows[t]).astype(np.int64)).cuda() for t, l in enumerate(lens)]
        lS_o = [torch.from_numpy(np.concatenate([[0], np.cumsum(l)[:-1]]).astype(np.int64)).cuda() for l in lens]
        store.lookup_bags(lS_o, lS_i, max_per_bag=P)                   # warm: the bag keys become resident
        keys = np.unique(np.concatenate([_keys(t, x.cpu().numpy()) for t, x in enumerate(lS_i)]))
        keys = np.concatenate([keys, _keys([0, 2, 11], [49, 399, 349])])
        vals = rng.uniform(-1, 1, size=(len(keys), dim)).astype(np.float32)
        w = _update(store, keys, vals).cpu().numpy()
        _apply(ref, keys, vals)
        assert (w[:-3] & WHERE_C1).any()
        out, _ = store.lookup_bags(lS_o, lS_i, max_per_bag=P)
        dec = decoded_tables(ref, prec)
        want = np.zeros((B, T, dim), dtype=np.float32)
        for t in range(T):
            ii, oo = lS_i[t].cpu().numpy(), lS_o[t].cpu().numpy()
            for s in range(B):
                for j in range(oo[s], oo[s] + lens[t][s]):
                    want[s, t] = want[s, t] + dec[t][ii[j]]
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy(), want)
        idx = np.stack([(np.arange(B) * 7 + t) % r for t, r in enumerate(rows)]).astype(np.int64)
        idx[0, 0], idx[2, 1], idx[11, 2] = 49, 399, 349
        got = store.storage_lookup(torch.from_numpy(idx).cuda())
        torch.cuda.synchronize()
        assert np.array_equal(got.cpu().numpy(), np.stack([dec[t][idx[t]] for t in range(T)], axis=1))
    finally:
        store.close()


# ---- 7. sharded -----------------------------------------------------------------------------------------------------------
def test_sharded_update_two_shards_on_one_device():
    import torch
    p = pkg()
    dim, B, cap, world = 16, 64, 260, 2
    tables = p.workload.make_tables(SMALL_ROWS, dim)
    ref = [t.copy() for t in tables]
    trace = p.workload.ZipfTrace(SMALL_ROWS, seed=41)
    rng = np.random.default_rng(12)
    stores, oracles, slices, shs = [], [], [], []
    for r in range(world):
        sl = p.sharded.get_my_slice(26, r, world)
        cfg = p.CacheConfig(total_size=cap, max_batch=B, n_tables_total=26, table_base=sl.start, record_events=True)
        stores.append(p.EvStore(tables[sl], cfg))
        oracles.append(BatchEvLFU(cap, n_tables=26))
        slices.append(sl)
        shs.append(p.sharded.ShardedLookup(stores[-1], 26, dim, r, world, transport="nccl"))
    try:
        for it in range(20):
            idx = trace.batch(B)
            aggs = [st.probe(torch.from_numpy(np.ascontiguousarray(idx[sl])).cuda()) for st, sl in zip(stores, slices)]
            agg = torch.stack([x.to(torch.int32) for x in aggs]).sum(dim=0).to(torch.uint8)
            o_agg = agg.cpu().numpy()
            for st, o, sl in zip(stores, oracles, slices):
                out, hit = st.lookup(torch.from_numpy(np.ascontiguousarray(idx[sl])).cuda(), agg_in=agg)
                torch.cuda.synchronize()
                o_hit, s_t, s_r, _ = o.lookup_batch(idx[sl], agg=o_agg, table_base=sl.start)
                assert np.array_equal(hit.cpu().numpy().astype(bool), o_hit), (it, sl)
                assert np.array_equal(out.cpu().numpy(), gather_rows(ref[sl], s_t - sl.start, s_r)), (it, sl)
                ev, fl = st.last_events()
                assert ev.tolist() == o.evicted and fl.tolist() == o.flushed, (it, sl)
                state, n_perfect = st.dump_state()
                assert state == o.state() and n_perfect == o.n_perfect
            resident = [set(k for b in st.dump_state()[0] for k in b) for st in stores]
            keys = _pick_keys(rng, SMALL_ROWS, [resident[0] | resident[1]], np.zeros((26, 1), dtype=np.int64), set())
            vals = rng.uniform(-1, 1, size=(len(keys), dim)).astype(np.float32)
            kt = torch.from_numpy(keys).cuda()
            vt = torch.from_numpy(vals).cuda()
            wheres = [sh.update_rows(kt >> 40, kt & ((1 << 40) - 1), vt).cpu().numpy() for sh in shs]
            _apply(ref, keys, vals)
            for r, (w, sl) in enumerate(zip(wheres, slices)):
                mine = np.isin(keys >> 40, np.arange(sl.start, sl.stop))
                assert (w[~mine] == 0).all()
                want = np.array([WHERE_STORE | (k in resident[r]) for k in keys[mine].tolist()], dtype=np.uint8)
                assert np.array_equal(w[mine], want)
    finally:
        for st in stores:
            st.close()


CASE = (SMALL_ROWS, 16, 64, 260, 10)


def _update_plan(k):
    """Keys and values the ranks apply after global batch k (the same on every rank)."""
    rows, dim = CASE[0], CASE[1]
    rng = np.random.default_rng(100 + k)
    t = rng.integers(0, 26, size=40)
    r = (rng.random(40) * np.asarray(rows)[t]).astype(np.int64)
    keys = np.unique(_keys(t, r))
    return keys, rng.uniform(-1, 1, size=(len(keys), dim)).astype(np.float32)


def _worker(rank, world, port, q, same_device, many):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    devno = 0 if same_device else rank
    torch.cuda.set_device(devno)
    if same_device:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    else:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", devno))
    p = pkg()
    rows, dim, B, cap, n = CASE
    tables = p.workload.make_tables(rows, dim)
    batches = p.workload.ZipfTrace(rows, seed=43).batches(n, B)
    ids = p.sharded.contiguous_placement(26, world)[rank]
    store = p.EvStore([tables[t] for t in ids], p.CacheConfig(total_size=cap, max_batch=B, n_tables_total=26,
                                                              table_ids=tuple(ids), device=devno))
    sh = p.sharded.ShardedLookup(store, 26, dim, rank, world, transport="p2p", batch_max=B)
    res, err = [], None
    try:
        dev = [torch.from_numpy(np.ascontiguousarray(idx[ids])).cuda() for idx in batches]
        torch.cuda.synchronize()
        k = 0
        while k < n:
            step = 4 if (many and k + 4 <= n) else 1
            got = sh.lookup_many(dev[k:k + step]) if step > 1 else [sh.lookup(dev[k])]
            for ly, hit in got:
                torch.cuda.synchronize()
                res.append((ly.cpu().numpy().copy(), hit.cpu().numpy().copy()))
            k += step
            keys, vals = _update_plan(k)
            kt = torch.from_numpy(keys).cuda()
            sh.update_rows(kt >> 40, kt & ((1 << 40) - 1), torch.from_numpy(vals).cuda())
        store.sync()
    except Exception as e:                               # report instead of hanging the peer
        err = repr(e)
    q.put((rank, res, err))
    dist.barrier()
    store.close()
    dist.destroy_process_group()


def _run_sharded_updates(same_device, many):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    world = 2
    port = 31700 + (os.getpid() + 7 * int(many) + 3 * int(same_device)) % 2000
    procs = [ctx.Process(target=_worker, args=(r, world, port, q, same_device, many)) for r in range(world)]
    for pr in procs:
        pr.start()
    got = {}
    for _ in range(world):
        r, res, err = q.get(timeout=300)
        assert err is None, f"rank {r}: {err}"
        got[r] = res
    for pr in procs:
        pr.join(timeout=60)
        assert pr.exitcode == 0
    p = pkg()
    rows, dim, B, cap, n = CASE
    ref = [t.copy() for t in p.workload.make_tables(rows, dim)]
    batches = p.workload.ZipfTrace(rows, seed=43).batches(n, B)
    placement = p.sharded.contiguous_placement(26, world)
    oracles = [BatchEvLFU(cap, n_tables=26) for _ in range(world)]
    Bl = B // world
    k = 0
    while k < n:
        step = 4 if (many and k + 4 <= n) else 1
        for kk in range(k, k + step):
            idx = batches[kk]
            agg = sum(np.array([[(ids[t] << 40 | int(idx[ids[t], s])) in o.entries for t in range(len(ids))]
                                for s in range(B)]).sum(axis=1) for o, ids in zip(oracles, placement))
            full = np.empty((B, 26, dim), dtype=np.float32)
            for r, (o, ids) in enumerate(zip(oracles, placement)):
                o_hit, s_t, s_r, _ = o.lookup_batch(idx[ids], agg=agg, table_ids=ids)
                full[:, ids] = gather_rows(ref, s_t, s_r)
                assert np.array_equal(got[r][kk][1].astype(bool), o_hit), (kk, r)
            for r in range(world):
                assert np.array_equal(got[r][kk][0], full[r * Bl:(r + 1) * Bl]), (kk, r)
        k += step
        keys, vals = _update_plan(k)
        _apply(ref, keys, vals)


@pytest.mark.parametrize("many", [False, True])
def test_sharded_update_p2p_two_processes_on_one_gpu(many):
    _run_sharded_updates(True, many)


def test_sharded_update_p2p_two_gpus():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    _run_sharded_updates(False, True)


# ---- 8. size -------------------------------------------------------------------------------------------------------------
def test_one_million_keys_with_duplicates():
    import torch
    p = pkg()
    n, dim, R = 1 << 20, 64, 600000
    tables = p.workload.make_tables([R, 1000], dim)
    store = p.EvStore(tables, p.CacheConfig(total_size=20000, max_batch=1024))
    rng = np.random.default_rng(5)
    try:
        warm = np.stack([rng.integers(0, 1000, size=1024), rng.integers(0, 1000, size=1024)]).astype(np.int64)
        store.lookup(torch.from_numpy(warm).cuda())
        t = (rng.random(n) < 0.01).astype(np.int64)
        r = np.where(t == 1, rng.integers(0, 1000, size=n), rng.integers(0, R, size=n))
        vals = torch.randn((n, dim), device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
        old = [x.copy() for x in tables]
        w = store.update_rows(torch.from_numpy(t).cuda(), torch.from_numpy(r).cuda(), vals)
        torch.cuda.synchronize()
        keys = _keys(t, r)
        order = np.lexsort((np.arange(n), keys))                 # by key, then position
        last = np.ones(n, dtype=bool)
        last[order[:-1]] = keys[order[:-1]] != keys[order[1:]]
        w = w.cpu().numpy()
        assert ((w != 0) == last).all() and ((w[last] & WHERE_STORE) != 0).all() and ((w[last] & WHERE_C1) != 0).any()
        v = vals.cpu().numpy()
        for tt in (0, 1):
            want = old[tt].copy()
            m = last & (t == tt)
            want[r[m]] = v[m]
            assert np.array_equal(tables[tt], want), tt          # the caller's fp32 arrays are the backing store
        out, _ = store.lookup(torch.from_numpy(warm).cuda())
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy(), np.stack([tables[0][warm[0]], tables[1][warm[1]]], axis=1))
    finally:
        store.close()
