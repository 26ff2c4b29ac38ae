"""k_evict's per-batch scratch (chunk tickets, look-back entries, kept / scan_end, batch totals, the arrival counter) is reset
by the CTA that closes each batch.  Whatever way batches reach the device -- one call each, groups of a captured graph,
a flush batch, a replay of a graph the caller captured -- the next batch must start from clean scratch: the hit maps,
rows, eviction / flush streams and FIFO state stay equal to the batch-granular oracle."""
import numpy as np
import pytest

from helpers import SMALL_ROWS, TINY_ROWS, pkg

pytestmark = pytest.mark.gpu


def _open(rows, total, B, seed):
    from oracle.evlfu import BatchEvLFU
    p = pkg()
    tables = p.workload.make_tables(rows, 16)
    store = p.EvStore(tables, p.CacheConfig(n_layers=1, total_size=total, max_batch=B, record_events=True))
    return p, tables, store, BatchEvLFU(total, n_tables=len(rows)), p.workload.ZipfTrace(rows, seed=seed)


def _agree(store, oracle, tables, idx, out, hit, what):
    import torch
    from oracle.evlfu import gather_rows
    torch.cuda.synchronize()
    store.check()
    o_hit, st, sr, _ = oracle.lookup_batch(idx)
    assert (hit.cpu().numpy().astype(bool) == o_hit).all(), f"hit map, {what}"
    assert (out.cpu().numpy() == gather_rows(tables, st, sr)).all(), f"rows, {what}"


def _state(store, oracle, what):
    ev, fl = store.last_events()
    assert ev.tolist() == oracle.evicted and fl.tolist() == oracle.flushed, f"eviction / flush stream, {what}"
    state, n_perfect = store.dump_state()
    assert state == oracle.state() and n_perfect == oracle.n_perfect, f"FIFO state, {what}"


@pytest.mark.parametrize("plan", [[1, 4, 1, 1, 3], [2, 4, 1, 5, 1, 1]])
def test_single_and_grouped_calls_odd_and_even_batch_counts(plan):
    """An odd and an even number of batches in all, single calls and grouped calls mixed."""
    import torch
    p, tables, store, oracle, trace = _open(SMALL_ROWS, 600, 64, seed=11)
    try:
        for call, n in enumerate(plan):
            idx = [trace.batch(64) for _ in range(n)]
            dev = [torch.from_numpy(i).cuda() for i in idx]
            if n == 1 or call % 2 == 0:
                res = [store.lookup(d) for d in dev]
            else:
                outs, hits = store.lookup_many(dev)
                res = list(zip(outs, hits))
            for k in range(n):
                _agree(store, oracle, tables, idx[k], res[k][0], res[k][1], f"call {call} batch {k}")
            _state(store, oracle, f"after call {call}")
        assert store.stats()["evictions"][0] > 0
    finally:
        store.close()


def test_flush_batch_then_normal_batches():
    """Tiny tables: bucket 26 fills and is flushed; the batches after a flush run the parallel eviction again."""
    import torch
    p, tables, store, oracle, trace = _open(TINY_ROWS, 110, 16, seed=3)
    flushes = after_flush = 0
    try:
        for it in range(160):
            idx = trace.batch(16 if it % 3 else 4)
            out, hit = store.lookup(torch.from_numpy(idx).cuda())
            _agree(store, oracle, tables, idx, out, hit, f"batch {it}")
            _state(store, oracle, f"batch {it}")
            if oracle.flushed:
                flushes += 1
            elif flushes and oracle.evicted:
                after_flush += 1
        assert flushes > 0 and after_flush > 0
    finally:
        store.close()


def test_replays_of_a_caller_captured_graph():
    """A graph the caller captured around lookup: the device numbers every replay itself; replays, single calls and a
    grouped call follow each other."""
    import torch
    p, tables, store, oracle, trace = _open(SMALL_ROWS, 600, 64, seed=7)
    B = 64
    try:
        first = trace.batch(B)                                     # warm-up outside the graph (also a batch)
        out, hit = store.lookup(torch.from_numpy(first).cuda())
        _agree(store, oracle, tables, first, out, hit, "warm-up")
        s_idx = torch.from_numpy(trace.batch(B)).cuda()
        s_out = torch.empty((B, len(SMALL_ROWS), 16), dtype=torch.float32, device="cuda")
        s_hit = torch.empty((B, len(SMALL_ROWS)), dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            store.lookup(s_idx, out=s_out, hit=s_hit)
        for it in range(7):
            idx = trace.batch(B)
            s_idx.copy_(torch.from_numpy(idx))
            g.replay()
            store.note_replays(1)
            _agree(store, oracle, tables, idx, s_out, s_hit, f"replay {it}")
            _state(store, oracle, f"replay {it}")
            if it % 3 == 1:
                idx = trace.batch(B)
                out, hit = store.lookup(torch.from_numpy(idx).cuda())
                _agree(store, oracle, tables, idx, out, hit, f"single call after replay {it}")
            if it == 4:
                idx = [trace.batch(B) for _ in range(5)]                 # one group of 4 and one single batch
                outs, hits = store.lookup_many([torch.from_numpy(i).cuda() for i in idx])
                for k in range(5):
                    _agree(store, oracle, tables, idx[k], outs[k], hits[k], f"grouped call after replay {it}, batch {k}")
            _state(store, oracle, f"after replay {it}")
    finally:
        store.close()


def test_replays_of_a_caller_captured_grouped_call():
    """A graph the caller captured around lookup_many of 5 batches (outside a capture: one group and one single): every
    batch goes in as plain kernels the device numbers itself, replay after replay; single and grouped calls follow."""
    import torch
    p, tables, store, oracle, trace = _open(SMALL_ROWS, 600, 64, seed=13)
    B, n, T = 64, 5, len(SMALL_ROWS)
    try:
        first = trace.batch(B)                                     # warm-up outside the graph (also a batch)
        out, hit = store.lookup(torch.from_numpy(first).cuda())
        _agree(store, oracle, tables, first, out, hit, "warm-up")
        s_idx = [torch.from_numpy(trace.batch(B)).cuda() for _ in range(n)]
        s_out = [torch.empty((B, T, 16), dtype=torch.float32, device="cuda") for _ in range(n)]
        s_hit = [torch.empty((B, T), dtype=torch.uint8, device="cuda") for _ in range(n)]
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            store.lookup_many(s_idx, outs=s_out, hits=s_hit)
        for it in range(3):
            idx = [trace.batch(B) for _ in range(n)]
            for d, i in zip(s_idx, idx):
                d.copy_(torch.from_numpy(i))
            g.replay()
            store.note_replays(n)
            for k in range(n):
                _agree(store, oracle, tables, idx[k], s_out[k], s_hit[k], f"replay {it}, batch {k}")
            _state(store, oracle, f"replay {it}")
            idx = trace.batch(B)
            out, hit = store.lookup(torch.from_numpy(idx).cuda())
            _agree(store, oracle, tables, idx, out, hit, f"single call after replay {it}")
            idx = [trace.batch(B) for _ in range(n)]
            outs, hits = store.lookup_many([torch.from_numpy(i).cuda() for i in idx])
            for k in range(n):
                _agree(store, oracle, tables, idx[k], outs[k], hits[k], f"grouped call after replay {it}, batch {k}")
            _state(store, oracle, f"after replay {it}")
    finally:
        store.close()
