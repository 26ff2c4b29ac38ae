"""evs_save_state / evs_load_state: a snapshot of a warm cache's policy state, restored into another handle.

The guarantee under test: handle A serves some batches and saves; handle B (fresh, or one that has served other traffic)
loads the snapshot; from then on A and B, given the same batches, return bit-identical rows, identical hit codes and
agg_hit, the same eviction / flush streams, the same evs_dump_state / evs_dump_c3 after every batch and the same deltas
of the statistics counters.  B is also followed by the batch oracle (BatchEvLFU, BatchLRU, BatchLFU or BatchTiers at B's
capacities) seeded from the snapshot, which pins B's decisions where its capacities differ from A's.  Small caches make evictions, flushes and C3 second chances happen within a few dozen
batches, as in test_gpu_update_rows.py."""
import numpy as np
import pytest

from helpers import SMALL_ROWS, pkg
from state_seed import Follower, parse_snapshot, rewrite, sections_equal

pytestmark = pytest.mark.gpu

DIM, B = 16, 64
DELTA_KEYS = ("lookups", "samples", "hits", "c3_hits", "approx_subst", "misses", "perfect_hits", "inserts", "evictions",
              "flushed", "batches")


def _store(p, tables, alt=None, **kw):
    kw.setdefault("max_batch", B)
    kw.setdefault("record_events", True)
    return p.EvStore(tables, p.CacheConfig(**kw), alt_keys=alt)


def _tiers(store):
    return 2 if store.cfg.n_layers >= 2 else 1


def _snapshot(store):
    """Everything observable about the policy state."""
    s = {"tiers": [store.dump_state(t) for t in range(_tiers(store))]}
    if store.cfg.n_layers == 3:
        s["c3"] = [x.tolist() for x in store.dump_c3()]
    st = store.stats()
    s["size"], s["c3_size"] = st["size"], st["c3_size"]
    return s


def _run(store, idx_list, path, dev):
    """Serve the batches; returns per batch (rows, hit codes, agg_hit, events per tier) -- agg_hit by a probe before it."""
    import torch
    res = []
    if path == "many":
        d = [torch.from_numpy(i).to(dev) for i in idx_list]
        outs, hits = store.lookup_many(d)
        torch.cuda.synchronize()
        for o, h in zip(outs, hits):
            res.append((o.cpu().numpy(), h.cpu().numpy(), None, None))
        return res
    for idx in idx_list:
        if path == "bags":
            T = idx.shape[0]
            lS_i = [torch.from_numpy(idx[t]).to(dev) for t in range(T)]
            lS_o = [torch.arange(0, idx.shape[1], 2, dtype=torch.int64, device=dev) for _ in range(T)]   # bags of 2
            o, h = store.lookup_bags(lS_o, lS_i, max_per_bag=2)
            h = torch.stack(h)
        else:
            d = torch.from_numpy(idx).to(dev)
            agg = store.probe(d).clone()
            o, h = store.lookup(d)
        torch.cuda.synchronize()
        ev = [store.last_events(t) for t in range(_tiers(store))]
        res.append((o.cpu().numpy(), h.cpu().numpy(), None if path == "bags" else agg.cpu().numpy(),
                    [(e.tolist(), f.tolist()) for e, f in ev]))
    return res


def _deltas(s1, s0):
    return {k: (np.asarray(s1[k]) - np.asarray(s0[k])).tolist() for k in DELTA_KEYS}


def _continue_both(a, b, idx_list, path, dev, same_rows=True, per_batch_state=True, follower=None):
    sa0, sb0 = a.stats(), b.stats()
    step = 4 if path == "many" else 1
    for k in range(0, len(idx_list), step):
        chunk = idx_list[k:k + step]
        ra, rb = _run(a, chunk, path, dev), _run(b, chunk, path, dev)
        for j, (x, y) in enumerate(zip(ra, rb)):
            if same_rows:
                assert np.array_equal(x[0].view(np.uint32), y[0].view(np.uint32)), f"rows, batch {k + j}"
            assert np.array_equal(x[1], y[1]), f"hit codes, batch {k + j}"
            if x[2] is not None:
                assert np.array_equal(x[2], y[2]), f"agg_hit, batch {k + j}"
            if x[3] is not None:
                assert x[3] == y[3], f"eviction / flush streams, batch {k + j}"
            if follower is not None:
                follower.check(chunk[j], y[0], y[1], y[3], f", batch {k + j}")
        if per_batch_state or k + step >= len(idx_list):
            assert _snapshot(a) == _snapshot(b), f"state after batch {k + step - 1}"
    assert _deltas(a.stats(), sa0) == _deltas(b.stats(), sb0)


# ---- 1. continuation ------------------------------------------------------------------------------------------------------
CASES = {
    # name: (config, batches before the save)
    "c1_32": (dict(main_precision=32, total_size=300), 30),
    "c1_16": (dict(main_precision=16, total_size=150), 30),
    "c1_8": (dict(main_precision=8, total_size=80), 30),
    "c1_4": (dict(main_precision=4, total_size=40), 30),
    "c1_32_approx": (dict(main_precision=32, total_size=300, approx_emb_thres=12), 30),
    "c1_8_approx": (dict(main_precision=8, total_size=80, approx_emb_thres=10), 30),
    "c2_32_8": (dict(n_layers=2, main_precision=32, secondary_precision=8, total_size=240), 30),
    "c2_32_8_c1_not_full": (dict(n_layers=2, main_precision=32, secondary_precision=8, total_size=2000), 2),
    "c2_8_4": (dict(n_layers=2, main_precision=8, secondary_precision=4, total_size=100), 30),
    "c3_8_4": (dict(n_layers=3, main_precision=8, secondary_precision=4, total_size=60, size_proportion="25-25-50"), 40),
    "lru": (dict(main_precision=32, total_size=300, policy="lru"), 30),
    "lfu": (dict(main_precision=32, total_size=300, policy="lfu"), 30),
}


def _setup(name, seed=3):
    p = pkg()
    cfg, n0 = CASES[name]
    tables = p.workload.make_tables(SMALL_ROWS, DIM)
    alt = p.workload.make_alt_keys(SMALL_ROWS) if cfg.get("n_layers") == 3 else None
    trace = p.workload.ZipfTrace(SMALL_ROWS, seed=seed)
    return p, cfg, n0, tables, alt, trace


@pytest.mark.parametrize("b_warm", [False, True])
@pytest.mark.parametrize("name", list(CASES))
def test_continuation(name, b_warm):
    import torch
    p, cfg, n0, tables, alt, trace = _setup(name)
    dev = torch.device("cuda")
    a = _store(p, tables, alt, **cfg)
    b = _store(p, tables, alt, **cfg)
    try:
        _run(a, [trace.batch(B) for _ in range(n0)], "single", dev)
        if b_warm:        # B has served other traffic: the load replaces all of it
            other = p.workload.ZipfTrace(SMALL_ROWS, seed=99)
            _run(b, [other.batch(B) for _ in range(7)], "single", dev)
        before = _snapshot(a)
        blob = a.save_state()
        info = p.state_info(blob)
        assert info["n_layers"] == cfg.get("n_layers", 1) and info["rows"] == SMALL_ROWS
        assert _snapshot(a) == before                    # saving changes nothing
        b.load_state(blob)
        assert _snapshot(b) == before
        # what B holds is the whole snapshot: C3's window with its stale and duplicate records included
        assert sections_equal(parse_snapshot(b.save_state()), parse_snapshot(blob))
        follower = Follower(b, cfg, blob, tables, alt)
        if name == "c2_32_8_c1_not_full":
            assert before["size"][0] < a.stats()["capacity"][0]
        if name == "c2_32_8":
            r1 = {k for bk in before["tiers"][0][0] for k in bk}
            r2 = {k for bk in before["tiers"][1][0] for k in bk}
            assert r1 & r2, "a state with keys resident in both tiers"
        if name == "c3_8_4":
            assert info["c3"]["window"] > info["c3"]["size"] > 0, info["c3"]    # stale / duplicate records in the window
        _continue_both(a, b, [trace.batch(B) for _ in range(40)], "single", dev, follower=follower)
    finally:
        a.close()
        b.close()


# ---- 2. stream order and the other lookup paths ----------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["c1_32", "c2_32_8", "c3_8_4"])
def test_save_follows_unsynchronised_batches_and_load_on_a_caller_stream(name):
    import torch
    p, cfg, n0, tables, alt, trace = _setup(name, seed=5)
    dev = torch.device("cuda")
    a, ref, b = (_store(p, tables, alt, **cfg) for _ in range(3))
    try:
        idx = [torch.from_numpy(trace.batch(B)).to(dev) for _ in range(n0)]
        s = torch.cuda.Stream()
        torch.cuda.synchronize()
        with torch.cuda.stream(s):
            for x in idx:                                # enqueued, not waited for
                a.lookup(x)
            blob = a.save_state()
        for x in idx:
            ref.lookup(x)
        torch.cuda.synchronize()
        assert _snapshot(a) == _snapshot(ref)
        other = p.workload.ZipfTrace(SMALL_ROWS, seed=77)
        for _ in range(5):
            b.lookup(torch.from_numpy(other.batch(B)).to(dev))
        nxt = [trace.batch(B) for _ in range(12)]
        s.wait_stream(torch.cuda.current_stream())      # b's batches ran on the default stream
        with torch.cuda.stream(s):
            b.load_state(blob)
        torch.cuda.current_stream().wait_stream(s)
        _continue_both(a, b, nxt, "single", dev)
    finally:
        for x in (a, ref, b):
            x.close()


@pytest.mark.parametrize("name", ["c1_32", "c2_8_4", "c3_8_4"])
def test_batch_announced_before_the_load(name):
    import torch
    p, cfg, n0, tables, alt, trace = _setup(name, seed=8)
    dev = torch.device("cuda")
    a, b = _store(p, tables, alt, **cfg), _store(p, tables, alt, **cfg)
    try:
        other = p.workload.ZipfTrace(SMALL_ROWS, seed=21)
        _run(a, [trace.batch(B) for _ in range(n0)], "single", dev)
        _run(b, [other.batch(B) for _ in range(n0)], "single", dev)
        blob = a.save_state()
        nxt = torch.from_numpy(trace.batch(B)).to(dev)
        b.prefetch(nxt)                                  # staged against b's old state
        a.prefetch(nxt)
        b.load_state(blob)
        oa, ha = a.lookup(nxt)
        ob, hb = b.lookup(nxt)
        torch.cuda.synchronize()
        assert np.array_equal(oa.cpu().numpy().view(np.uint32), ob.cpu().numpy().view(np.uint32))
        assert np.array_equal(ha.cpu().numpy(), hb.cpu().numpy())
        assert _snapshot(a) == _snapshot(b)
        _continue_both(a, b, [trace.batch(B) for _ in range(8)], "single", dev)
    finally:
        a.close()
        b.close()


@pytest.mark.parametrize("path", ["many", "bags"])
@pytest.mark.parametrize("name", ["c1_32_approx", "c2_32_8", "c3_8_4", "lfu"])
def test_continuation_through_grouped_and_bag_lookups(name, path):
    import torch
    p, cfg, n0, tables, alt, trace = _setup(name, seed=11)
    dev = torch.device("cuda")
    cfg = dict(cfg, max_batch=2 * B)
    a, b = _store(p, tables, alt, **cfg), _store(p, tables, alt, **cfg)
    try:
        _run(a, [trace.batch(B) for _ in range(n0)], path, dev)
        b.load_state(a.save_state())
        _continue_both(a, b, [trace.batch(B) for _ in range(16)], path, dev, per_batch_state=path == "bags")
    finally:
        a.close()
        b.close()


# ---- 3. across configurations --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("src,dst", [
    (dict(main_precision=32, total_size=300), dict(main_precision=8, total_size=75)),
    (dict(main_precision=32, total_size=300), dict(main_precision=32, total_size=600)),          # larger capacity
    (dict(main_precision=32, total_size=300), dict(main_precision=16, total_size=150, store_in_hbm=True, max_batch=256)),
    (dict(main_precision=32, total_size=300, policy="lfu"), dict(main_precision=32, total_size=450, policy="lfu")),
    (dict(n_layers=2, main_precision=32, secondary_precision=8, total_size=240),
     dict(n_layers=2, main_precision=16, secondary_precision=4, total_size=480)),
    (dict(n_layers=3, main_precision=8, secondary_precision=4, total_size=60, size_proportion="25-25-50"),
     dict(n_layers=3, main_precision=8, secondary_precision=4, total_size=90, size_proportion="25-25-50")),
])
def test_load_into_other_precisions_and_capacities(src, dst):
    """The dumped state equals A's; from then on B follows the oracle seeded from the snapshot at B's own capacities
    (hit codes, rows decoded at B's precisions, eviction / flush streams, FIFO state, n_perfect, C3), and with equal
    capacities B also takes A's decisions."""
    import torch
    p = pkg()
    dev = torch.device("cuda")
    tables = p.workload.make_tables(SMALL_ROWS, DIM)
    alt = p.workload.make_alt_keys(SMALL_ROWS) if src.get("n_layers") == 3 else None
    trace = p.workload.ZipfTrace(SMALL_ROWS, seed=13)
    a, b = _store(p, tables, alt, **src), _store(p, tables, alt, **dst)
    try:
        _run(a, [trace.batch(B) for _ in range(40)], "single", dev)
        before = _snapshot(a)
        blob = a.save_state()
        b.load_state(blob)
        got = _snapshot(b)
        assert got["tiers"] == before["tiers"] and got.get("c3") == before.get("c3")
        follower = Follower(b, dst, blob, tables, alt)
        nxt = [trace.batch(B) for _ in range(40)]
        if b.stats()["capacity"] == a.stats()["capacity"] and b.stats()["c3_capacity"] == a.stats()["c3_capacity"]:
            _continue_both(a, b, nxt, "single", dev, same_rows=src == dst, follower=follower)
        else:
            for k, x in enumerate(nxt):
                r = _run(b, [x], "single", dev)[0]
                follower.check(x, r[0], r[1], r[3], f", batch {k}")
    finally:
        a.close()
        b.close()


def test_load_after_update_rows_reads_the_new_values():
    import torch
    p = pkg()
    dev = torch.device("cuda")
    tables = p.workload.make_tables(SMALL_ROWS, DIM)
    trace = p.workload.ZipfTrace(SMALL_ROWS, seed=17)
    a = _store(p, tables, main_precision=32, total_size=300)
    try:
        _run(a, [trace.batch(B) for _ in range(20)], "single", dev)
        state, _ = a.dump_state()
        keys = np.array([k for bk in state for k in bk][:50], dtype=np.int64)
        vals = np.random.default_rng(1).uniform(-1, 1, size=(len(keys), DIM)).astype(np.float32)
        kt = torch.from_numpy(keys).cuda()
        a.update_rows(kt >> 40, kt & ((1 << 40) - 1), torch.from_numpy(vals).cuda())     # writes `tables` in place
        blob = a.save_state()
        b = _store(p, tables, main_precision=32, total_size=300)
        try:
            b.load_state(blob)
            idx = np.zeros((26, len(keys)), dtype=np.int64)
            tab = keys >> 40
            for j, k in enumerate(keys):
                idx[:, j] = 0
                idx[tab[j], j] = k & ((1 << 40) - 1)
            out, hit = b.lookup(torch.from_numpy(idx).cuda())
            torch.cuda.synchronize()
            o, h = out.cpu().numpy(), hit.cpu().numpy()
            for j in range(len(keys)):
                assert h[j, tab[j]] == 1
                assert np.array_equal(o[j, tab[j]], vals[j])
        finally:
            b.close()
    finally:
        a.close()


# ---- 4. rejections -----------------------------------------------------------------------------------------------------
HDR = 464


def _patch(blob, off, dtype, value):
    b = blob.copy()
    b[off:off + np.dtype(dtype).itemsize] = np.frombuffer(np.array([value], dtype=dtype).tobytes(), dtype=np.uint8)
    return b


def _host_rejections(blob, info):
    """(name, blob, config overrides of the loading handle) that the host checks refuse."""
    yield "magic", _patch(blob, 0, "<u1", ord("X")), {}
    yield "version", _patch(blob, 8, "<u4", 2), {}
    yield "length", _patch(blob, 16, "<u8", len(blob) + 8), {}
    yield "truncated", blob[:-8], {}
    yield "truncated_consistent", _patch(blob[:-8], 16, "<u8", len(blob) - 8), {}
    yield "header_only", _patch(blob[:HDR], 16, "<u8", HDR), {}
    yield "short", blob[:100], {}
    yield "policy", blob, {"policy": "lru"}
    yield "n_layers", blob, {"n_layers": 2, "secondary_precision": 8}
    yield "n_tables_total", blob, {"n_tables_total": 27}
    yield "table_ids", _patch(blob, 80 + 4 * 25, "<i4", 26), {}          # header: table_ids[32] at 80, rows[32] at 208
    yield "rows", _patch(blob, 208 + 8 * 3, "<i8", SMALL_ROWS[3] + 1), {}
    yield "capacity", blob, {"total_size": sum(info["tiers"][0]["counts"]) - 1}


def test_host_checks_refuse_and_leave_the_handle_untouched():
    import torch
    p = pkg()
    dev = torch.device("cuda")
    tables = p.workload.make_tables(SMALL_ROWS, DIM)
    trace = p.workload.ZipfTrace(SMALL_ROWS, seed=19)
    a = _store(p, tables, main_precision=32, total_size=300)
    try:
        _run(a, [trace.batch(B) for _ in range(20)], "single", dev)
        blob = a.save_state()
        info = p.state_info(blob)
        for name, bad, over in _host_rejections(blob, info):
            cfg = dict(main_precision=32, total_size=300)
            cfg.update(over)
            b = _store(p, tables, **cfg)
            try:
                other = p.workload.ZipfTrace(SMALL_ROWS, seed=23)
                _run(b, [other.batch(B) for _ in range(3)], "single", dev)
                before = _snapshot(b)
                with pytest.raises(p.EvsError) as e:
                    b.load_state(bad)
                assert "evs_load_state" in str(e.value) and "empty" not in str(e.value), name
                assert _snapshot(b) == before, name
            finally:
                b.close()
    finally:
        a.close()


def test_c3_window_that_leaves_no_room_for_a_batch_is_refused():
    """The window must fit the loading handle's ring with room for one batch's appends (the victims of both tiers)."""
    import torch
    p, cfg, n0, tables, alt, trace = _setup("c3_8_4", seed=31)
    dev = torch.device("cuda")
    a = _store(p, tables, alt, **cfg)
    b = _store(p, tables, alt, **dict(cfg, max_batch=1))
    ring = 1 << (4 * b.stats()["c3_capacity"] + 8 * 26 - 1).bit_length()      # next_pow2(4 c3_cap + 8 n_max)
    try:
        _run(a, [trace.batch(B) for _ in range(n0)], "single", dev)
        snap = parse_snapshot(a.save_state())
        window, entries = snap["c3"]
        pad = [entries[0][0]] * (ring - 2 * 26 - len(window))     # duplicate records of a mapped key
        fits = rewrite(a.save_state(), dict(snap, c3=(pad + window, entries)))
        over = rewrite(a.save_state(), dict(snap, c3=([entries[0][0]] + pad + window, entries)))
        before = _snapshot(b)
        with pytest.raises(p.EvsError, match="no room"):
            b.load_state(over)
        assert _snapshot(b) == before
        b.load_state(fits)
        assert p.state_info(b.save_state())["c3"]["window"] == len(pad) + len(window)
    finally:
        a.close()
        b.close()


def test_load_and_save_refused_during_stream_capture():
    import torch
    p = pkg()
    tables = p.workload.make_tables([20] * 3, 16)
    store = p.EvStore(tables, p.CacheConfig(total_size=64, max_batch=8))
    try:
        blob = store.save_state()
        s = torch.cuda.Stream()
        torch.cuda.synchronize()
        for op in (lambda: store.load_state(blob), lambda: store.save_state()):
            g = torch.cuda.CUDAGraph()
            with pytest.raises(p.EvsError):
                with torch.cuda.graph(g, stream=s):
                    op()
    finally:
        torch.cuda.synchronize()
        store.close()


def _body_tier0(blob, nb):
    """Offsets of tier 0's counts and keys in the blob."""
    counts = np.frombuffer(blob[HDR + 8:HDR + 8 + 8 * nb].tobytes(), dtype="<u8")
    return HDR + 8 + 8 * nb, counts


@pytest.mark.parametrize("what", ["row_out_of_range", "unserved_table", "duplicate_in_tier", "duplicate_c3"])
def test_device_checks_leave_the_handle_empty(what):
    import torch
    name = "c3_8_4" if what == "duplicate_c3" else "c1_32"
    p, cfg, n0, tables, alt, trace = _setup(name, seed=29)
    dev = torch.device("cuda")
    a = _store(p, tables, alt, **cfg)
    try:
        _run(a, [trace.batch(B) for _ in range(n0)], "single", dev)
        blob = a.save_state()
        info = p.state_info(blob)
        nb = info["n_tables_total"] + 1
        kofs, counts = _body_tier0(blob, nb)
        n0k = int(counts.sum())
        assert n0k >= 2
        keys = np.frombuffer(blob[kofs:kofs + 8 * n0k].tobytes(), dtype="<u8").copy()
        if what == "row_out_of_range":
            t = int(keys[0] >> 40)
            keys[0] = (t << 40) | SMALL_ROWS[t]
        elif what == "unserved_table":
            keys[0] = (30 << 40) | 1
        elif what == "duplicate_in_tier":
            keys[1] = keys[0]
        bad = blob.copy()
        bad[kofs:kofs + 8 * n0k] = np.frombuffer(keys.astype("<u8").tobytes(), dtype=np.uint8)
        if what == "duplicate_c3":
            w = np.frombuffer(bad[HDR:].tobytes(), dtype="<u8").copy()
            o = 0
            for t in range(2):
                o += 1 + nb + int(w[o + 1:o + 1 + nb].sum())
            size, W = int(w[o]), int(w[o + 1])
            assert size >= 2
            m = o + 2 + W
            w[m + 2] = w[m]                              # entry 1's key := entry 0's key
            bad = np.concatenate([bad[:HDR], np.frombuffer(w.astype("<u8").tobytes(), dtype=np.uint8)])
        b = _store(p, tables, alt, **cfg)
        cold = _store(p, tables, alt, **cfg)
        try:
            _run(b, [trace.batch(B) for _ in range(3)], "single", dev)
            with pytest.raises(p.EvsError) as e:
                b.load_state(bad)
            assert "empty" in str(e.value)
            s = _snapshot(b)
            assert all(len(k) == 0 for t in s["tiers"] for k in t[0]) and s["size"] == [0, 0]
            assert s.get("c3", [[]])[0] == []
            # the next batches run as on a cold handle (statistics excepted: they are cumulative)
            nxt = [trace.batch(B) for _ in range(6)]
            for x in nxt:
                rb, rc = _run(b, [x], "single", dev)[0], _run(cold, [x], "single", dev)[0]
                assert np.array_equal(rb[0], rc[0]) and np.array_equal(rb[1], rc[1]) and rb[3] == rc[3]
                assert _snapshot(b) == _snapshot(cold)
        finally:
            b.close()
            cold.close()
    finally:
        a.close()


# ---- 5. full size ------------------------------------------------------------------------------------------------------
def test_kaggle_shape_full_size_save_load_continue():
    """configs[1]: Kaggle-shape tables (33.76 M rows, fp32, evs_host_alloc store), cache 4 389 135 entries, B = 2048."""
    import torch
    import bench
    p = pkg()
    rows, dim, Bf = p.workload.KAGGLE_ROWS, 16, 2048
    cap = p.workload.KAGGLE_CACHE_ROWS
    tables = [p.to_host_rows(t) for t in p.workload.make_tables(rows, dim)]
    n_search, n_after = 4200, 200
    idx = p.workload.ZipfTrace(rows, seed=42).batches(n_search + n_after, Bf)
    warm = min(n_search, bench.batches_until_full(idx[:n_search], rows, cap) + 50)
    cfg = dict(total_size=cap, max_batch=Bf)
    a = p.EvStore(tables, p.CacheConfig(**cfg))
    b = p.EvStore(tables, p.CacheConfig(**cfg))
    try:
        d = torch.from_numpy(idx[:warm]).cuda()
        for k in range(warm):
            a.lookup(d[k])
        torch.cuda.synchronize()
        assert a.stats()["size"][0] == cap
        blob = a.save_state()
        assert p.state_info(blob)["tiers"][0]["counts"] and sum(p.state_info(blob)["tiers"][0]["counts"]) == cap
        b.load_state(blob)
        del d
        d = torch.from_numpy(idx[warm:warm + n_after]).cuda()
        oa = torch.empty((Bf, 26, dim), device="cuda")
        ob = torch.empty_like(oa)
        ha = torch.empty((Bf, 26), dtype=torch.uint8, device="cuda")
        hb = torch.empty_like(ha)
        for k in range(n_after):
            a.lookup(d[k], out=oa, hit=ha)
            b.lookup(d[k], out=ob, hit=hb)
            assert torch.equal(oa.view(torch.int32), ob.view(torch.int32)), f"rows, batch {k}"
            assert torch.equal(ha, hb), f"hit codes, batch {k}"
        torch.cuda.synchronize()
        assert a.dump_state() == b.dump_state()
    finally:
        a.close()
        b.close()


# ---- 6. sharded ---------------------------------------------------------------------------------------------------------
def test_sharded_two_shards_on_one_device_save_load_continue():
    import torch
    p = pkg()
    dim, cap, world = 16, 260, 2
    tables = p.workload.make_tables(SMALL_ROWS, dim)
    trace = p.workload.ZipfTrace(SMALL_ROWS, seed=41)

    def pair():
        stores, shs = [], []
        for r in range(world):
            sl = p.sharded.get_my_slice(26, r, world)
            cfg = p.CacheConfig(total_size=cap, max_batch=B, n_tables_total=26, table_base=sl.start, record_events=True)
            stores.append(p.EvStore(tables[sl], cfg))
            shs.append(p.sharded.ShardedLookup(stores[-1], 26, dim, r, world, transport="nccl"))
        return stores, shs

    def step(stores, idx):
        slices = [p.sharded.get_my_slice(26, r, world) for r in range(world)]
        aggs = [st.probe(torch.from_numpy(np.ascontiguousarray(idx[sl])).cuda()) for st, sl in zip(stores, slices)]
        agg = torch.stack([x.to(torch.int32) for x in aggs]).sum(dim=0).to(torch.uint8)
        res = []
        for st, sl in zip(stores, slices):
            out, hit = st.lookup(torch.from_numpy(np.ascontiguousarray(idx[sl])).cuda(), agg_in=agg)
            torch.cuda.synchronize()
            res.append((out.cpu().numpy(), hit.cpu().numpy(), st.last_events(), st.dump_state()))
        return res

    sa, ha = pair()
    sb, hb = pair()
    try:
        for _ in range(20):
            step(sa, trace.batch(B))
        blobs = [h.save_state() for h in ha]
        for h, bl in zip(hb, blobs):
            h.load_state(bl)
        for it in range(15):
            idx = trace.batch(B)
            ra, rb = step(sa, idx), step(sb, idx)
            for x, y in zip(ra, rb):
                assert np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1]), it
                assert [e.tolist() for e in x[2]] == [e.tolist() for e in y[2]] and x[3] == y[3], it
    finally:
        for st in sa + sb:
            st.close()
