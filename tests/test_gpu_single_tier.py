"""CUDA path vs the batch-granular oracle, through the C-ABI: hit stream, fp32 rows,
eviction / flush streams and the resident FIFO state must be bit-exact, every batch."""
import numpy as np
import pytest

from helpers import SKEW_ROWS, SMALL_ROWS, TINY_ROWS, pkg, run_single_tier_parity

pytestmark = pytest.mark.gpu


def test_fp32_small_batches():
    t = run_single_tier_parity(SMALL_ROWS, 16, 32, 600, [64], 30)
    assert t["evicted"] > 0


def test_fp32_batch_of_one_and_ragged_sizes():
    run_single_tier_parity(SMALL_ROWS, 16, 32, 500, [1, 3, 8, 9, 31, 64, 2, 100], 64)


def test_fp32_dim36_reference_dimension():
    run_single_tier_parity(SMALL_ROWS, 36, 32, 700, [48], 25)


def test_fp32_dim64_skewed_tables_large_batch():
    t = run_single_tier_parity(SKEW_ROWS, 64, 32, 6000, [512], 24, check_state_every=4)
    assert t["evicted"] > 0


def test_fp32_flush_rule():
    """Tiny tables: most samples are perfect hits, bucket 26 fills and gets flushed."""
    t = run_single_tier_parity(TINY_ROWS, 16, 32, 110, [4, 16], 220, check_state_every=5)
    assert t["flushed"] > 0


@pytest.mark.parametrize("prec", [16, 8, 4])
def test_quantised_single_tier(prec):
    run_single_tier_parity(SMALL_ROWS, 16, prec, 150, [64, 17], 30, check_state_every=3)


@pytest.mark.parametrize("prec", [16, 8, 4])
def test_quantised_dim36(prec):
    run_single_tier_parity(SMALL_ROWS, 36, prec, 150, [33], 16, check_state_every=3)


def test_approximate_embedding_threshold():
    run_single_tier_parity(SMALL_ROWS, 16, 32, 900, [64], 40, approx=20, check_state_every=4)


def test_host_buffer_path_and_hbm_store():
    run_single_tier_parity(SMALL_ROWS, 16, 32, 600, [64, 5], 20, host_path=True)
    run_single_tier_parity(SMALL_ROWS, 16, 8, 200, [64], 10, store_in_hbm=True)


def test_empty_batch_and_bad_index():
    import torch
    p = pkg()
    tables = p.workload.make_tables(SMALL_ROWS, 16)
    store = p.EvStore(tables, p.CacheConfig(total_size=300, max_batch=32))
    out, hit = store.lookup(torch.zeros((26, 0), dtype=torch.int64, device="cuda"))
    assert out.shape == (0, 26, 16)
    bad = torch.zeros((26, 4), dtype=torch.int64, device="cuda")
    bad[3, 2] = 10 ** 9
    store.lookup(bad)
    with pytest.raises(p.EvsError):
        store.sync()
    with pytest.raises(p.EvsError):
        store.lookup(torch.zeros((26, 33), dtype=torch.int64, device="cuda"))
    store.close()


def test_ring_compaction_keeps_order(monkeypatch):
    """Many small batches on a tiny cache with the smallest rings the library makes: the bucket rings wrap and get compacted
    (k_compact, host-triggered from the ring-occupancy mirror)."""
    monkeypatch.setenv("EVSTORE_B200_RING_SLACK", "5")
    run_single_tier_parity(SMALL_ROWS, 16, 32, 64, [8], 700, check_state_every=50)
    # every hit of an LRU cache appends a record: the one ring fills within a few batches
    run_single_tier_parity(SMALL_ROWS, 16, 32, 400, [64], 60, check_state_every=10, policy="lru")


def test_back_to_back_batches_without_host_sync():
    """Batches queued back to back (no host synchronisation in between, as bench.py does): every
    batch must still see the state its predecessor left (stream order of the whole kernel graph)."""
    import torch
    from oracle.evlfu import BatchEvLFU, gather_rows
    p = pkg()
    rows, dim, B, cap, n = SKEW_ROWS, 16, 256, 3000, 60
    tables = p.workload.make_tables(rows, dim)
    trace = p.workload.ZipfTrace(rows, seed=5)
    idx = trace.batches(n, B)
    store = p.EvStore(tables, p.CacheConfig(total_size=cap, max_batch=B))
    oracle = BatchEvLFU(cap, n_tables=len(rows))
    d_idx = torch.from_numpy(idx).cuda()
    outs = torch.empty((n, B, len(rows), dim), dtype=torch.float32, device="cuda")
    hits = torch.empty((n, B, len(rows)), dtype=torch.uint8, device="cuda")
    for k in range(n):
        store.lookup(d_idx[k], out=outs[k], hit=hits[k])
    torch.cuda.synchronize()
    store.sync()
    outs, hits = outs.cpu().numpy(), hits.cpu().numpy()
    for k in range(n):
        o_hit, st, sr, _ = oracle.lookup_batch(idx[k])
        assert (hits[k].astype(bool) == o_hit).all(), f"hit stream, batch {k}"
        assert (outs[k] == gather_rows(tables, st, sr)).all(), f"rows, batch {k}"
    state, n_perfect = store.dump_state()
    assert state == oracle.state() and n_perfect == oracle.n_perfect
    store.close()


def test_pipelined_host_buffer_path():
    """evs_submit_host / evs_wait_host: 4 batches in flight, results identical to the oracle."""
    import torch
    from oracle.evlfu import BatchEvLFU, gather_rows
    p = pkg()
    rows, dim, B, cap, n = SMALL_ROWS, 16, 128, 700, 24
    tables = p.workload.make_tables(rows, dim)
    idx = p.workload.ZipfTrace(rows, seed=9).batches(n, B)
    store = p.EvStore(tables, p.CacheConfig(total_size=cap, max_batch=B))
    oracle = BatchEvLFU(cap, n_tables=len(rows))
    ih = torch.from_numpy(idx).pin_memory()
    outs = torch.empty((n, B, len(rows), dim), dtype=torch.float32).pin_memory()
    hits = torch.empty((n, B, len(rows)), dtype=torch.uint8).pin_memory()
    tickets = [store.submit_host_ptr(ih[k].data_ptr(), B, outs[k].data_ptr(), hits[k].data_ptr()) for k in range(n)]
    for t in tickets:
        store.wait_host(t)
    store.sync()
    for k in range(n):
        o_hit, st, sr, _ = oracle.lookup_batch(idx[k])
        assert (hits[k].numpy().astype(bool) == o_hit).all(), f"hit stream, batch {k}"
        assert (outs[k].numpy() == gather_rows(tables, st, sr)).all(), f"rows, batch {k}"
    store.close()


def test_fp32_very_large_batch_scan_path():
    """More than 512 serve-CTAs (B > 4096): ring positions come from the k_scan prefix pass."""
    t = run_single_tier_parity(SKEW_ROWS, 16, 32, 5000, [17000, 16500, 3], 5)
    assert t["evicted"] > 0


def test_fp32_direct_prefix_beyond_the_preloaded_rounds_and_medium_scan_path():
    """257..512 serve-CTAs: k_update sums its predecessors' counts itself, the first 256 from registers
    loaded before the claim and the rest in a loop after it; 513+ CTAs: k_scan."""
    t = run_single_tier_parity(SKEW_ROWS, 16, 32, 5000, [4096, 2049, 3000, 1], 6)
    assert t["evicted"] > 0
    t = run_single_tier_parity(SKEW_ROWS, 16, 32, 5000, [4097, 6000, 2], 5)
    assert t["evicted"] > 0


def test_without_programmatic_dependent_launch(monkeypatch):
    """EVSTORE_B200_PDL=0: plain stream order between the batch's kernels (the A/B baseline of the PDL chain)."""
    monkeypatch.setenv("EVSTORE_B200_PDL", "0")
    run_single_tier_parity(SMALL_ROWS, 16, 32, 600, [64, 5], 12)
    run_single_tier_parity(SMALL_ROWS, 36, 8, 150, [33], 8)


@pytest.mark.parametrize("dim,prec", [(16, 32), (64, 32), (16, 16), (64, 8), (36, 32)])
def test_look_ahead_prefetch_changes_nothing(dim, prec):
    """evs_prefetch announces every next batch: its probable misses are staged in HBM by a kernel that races the
    batch in flight.  Hit stream, rows, eviction / flush streams and FIFO state must stay bit-exact (dim 36 fp32 rows
    are 144 B: aligned; dim 36 at 8 bits would not be, and then the announcement is a no-op)."""
    t = run_single_tier_parity(SKEW_ROWS, dim, prec, 2500 * prec // 32, [700, 64, 257, 2048, 1], 30, prefetch=True, check_state_every=3)
    assert t["evicted"] > 0
    run_single_tier_parity(SMALL_ROWS, dim, prec, 600 * prec // 32, [64, 5], 14, prefetch=True)


def test_look_ahead_prefetch_unaligned_rows_and_lru():
    run_single_tier_parity(SMALL_ROWS, 36, 8, 150, [33, 64], 10, prefetch=True)          # 36-byte rows: no staging, same results
    run_single_tier_parity(SKEW_ROWS, 16, 32, 2500, [300, 64], 16, prefetch=True, policy="lru", check_state_every=4)


def test_look_ahead_announcement_that_does_not_match_is_ignored():
    """Announce batch A, then look B up; announce twice before one lookup; announce and never look up."""
    import torch
    from helpers import pkg
    from oracle.evlfu import BatchEvLFU, gather_rows
    p = pkg()
    dim, B, cap = 16, 128, 700
    tables = p.workload.make_tables(SMALL_ROWS, dim)
    trace = p.workload.ZipfTrace(SMALL_ROWS, seed=5)
    store = p.EvStore(tables, p.CacheConfig(total_size=cap, max_batch=B, record_events=True))
    oracle = BatchEvLFU(cap)
    batches = [trace.batch(B) for _ in range(24)]
    dev = [torch.from_numpy(b).cuda() for b in batches]
    torch.cuda.synchronize()
    for it in range(0, 24, 3):
        store.prefetch(dev[it + 1])                 # wrong announcement for batch `it`
        store.prefetch(dev[it + 2])                 # a second one for the same slot
        for k in (it, it + 1):
            out, hit = store.lookup(dev[k])
            if k == it:
                store.prefetch(dev[it + 1])         # the right one for the next call
            torch.cuda.synchronize()
            o_hit, st, sr, _ = oracle.lookup_batch(batches[k])
            assert (hit.cpu().numpy().astype(bool) == o_hit).all(), k
            assert (out.cpu().numpy() == gather_rows(tables, st, sr)).all(), k
            ev, fl = store.last_events()
            assert ev.tolist() == oracle.evicted and fl.tolist() == oracle.flushed, k
    store.sync()
    store.close()


@pytest.mark.parametrize("n_tables", [1, 2, 3, 5, 13, 16, 17])
def test_fewer_tables_pack_several_samples_per_warp(n_tables):
    """A handle with T <= 16 tables packs 32 / next_pow2(T) samples into each warp (what a rank of a
    table-wise sharded run does); every stream must still equal the oracle's."""
    rows = SKEW_ROWS[2:2 + n_tables]
    cap = max(40, int(sum(rows) * 0.2))
    t = run_single_tier_parity(rows, 16, 32, cap, [257, 64, 1, 33, 700], 25, check_state_every=2)
    assert t["evicted"] > 0


def test_fewer_tables_approx_threshold_and_quantised():
    rows = SMALL_ROWS[:6]
    run_single_tier_parity(rows, 16, 32, 300, [96, 7], 30, approx=4, check_state_every=3)
    run_single_tier_parity(SMALL_ROWS[3:7], 36, 8, 60, [130], 12, check_state_every=3)


@pytest.mark.parametrize("prec,mapped", [(32, False), (32, True), (8, True)])
def test_grouped_submission_equals_single_batches(prec, mapped):
    """evs_lookup_batches: groups of 4 batches as one graph (+ look-ahead of the batches inside a call) deliver what the same
    batches deliver one call each -- hit maps and rows of EVERY batch, the last batch's eviction stream, the final FIFO
    state -- against the oracle; `mapped`: backing rows in evs_host_alloc memory (managed, resident on the host)."""
    import torch
    from helpers import decoded_tables
    from oracle.evlfu import BatchEvLFU, gather_rows
    p = pkg()
    rows, dim, B = SKEW_ROWS, 16, 96
    tables = p.workload.make_tables(rows, dim)
    dec = decoded_tables(tables, prec)
    total = 3000 * prec // 32
    cfg = p.CacheConfig(n_layers=1, main_precision=prec, total_size=total, max_batch=B, record_events=True)
    stores = {prec: [p.to_host_rows(p.codecs.encode_table(t, prec)) for t in tables]} if mapped else None
    store = p.EvStore(tables, cfg, stores=stores)
    oracle = BatchEvLFU(total * (32 // prec), n_tables=len(rows))
    trace = p.workload.ZipfTrace(rows, seed=5)
    try:
        for call, n in enumerate([4, 9, 1, 8, 3, 12]):
            idx = [trace.batch(B) for _ in range(n)]
            dev = [torch.from_numpy(i).cuda() for i in idx]
            torch.cuda.synchronize()
            if call % 2 == 0:
                store.prefetch(dev[0])                      # the first batch of a call announced by the caller, or not
            outs, hits = store.lookup_many(dev)
            torch.cuda.synchronize()
            store.check()
            for k in range(n):
                o_hit, st, sr, _ = oracle.lookup_batch(idx[k])
                assert (hits[k].cpu().numpy().astype(bool) == o_hit).all(), f"hit map, call {call} batch {k}"
                assert (outs[k].cpu().numpy() == gather_rows(dec, st, sr)).all(), f"rows, call {call} batch {k}"
            ev, fl = store.last_events()
            assert ev.tolist() == oracle.evicted and fl.tolist() == oracle.flushed, f"eviction stream after call {call}"
            state, n_perfect = store.dump_state()
            assert state == oracle.state() and n_perfect == oracle.n_perfect, f"FIFO state after call {call}"
        assert store.stats()["evictions"][0] > 0
    finally:
        store.close()
