"""Host logic of ShardedLookup.lookup_bags with the "nccl" transport on CPU: two processes, gloo.  Each rank drives a CPU
stand-in for its EvStore (the oracle's batch policy over the slices of its own tables); the test checks what the product
adds around the store: the all-reduce of the per-slice hit counts, the all-to-all of the POOLED rows and the reassembly
into [B/size, 26, d], against all ranks simulated in one process (tests/sharded_bags_case.py)."""
import os

import numpy as np
import pytest

from helpers import SMALL_ROWS, pkg
from sharded_bags_case import make_bags, oracle_bags

WORLD = 2
DIM, B, CAP = 16, 16, 300
PS = [3, 10, 1, 32, 3, 10]


class OracleBagStore:
    """CPU test double with EvStore's probe_bags / lookup_bags signatures."""

    def __init__(self, tables_all, cap, ids):
        from oracle.evlfu import BatchEvLFU
        self.o = BatchEvLFU(cap, n_tables=26)
        self.tables, self.ids = tables_all, list(ids)

    @staticmethod
    def _lists(lS_o, lS_i):
        return [x.numpy() for x in lS_i], [x.numpy() for x in lS_o]

    def probe_bags(self, lS_o, lS_i, max_per_bag):
        import torch
        from oracle.evlfu import expand_bags
        from sharded_bags_case import slice_counts
        idx_lists, off_lists = self._lists(lS_o, lS_i)
        iv = expand_bags(idx_lists, off_lists, len(off_lists[0]), max_per_bag)
        return torch.from_numpy(slice_counts(self.o, self.ids, iv).astype(np.uint8))

    def lookup_bags(self, lS_o, lS_i, max_per_bag, out=None, agg_in=None):
        import torch
        from oracle.evlfu import expand_bags, gather_rows, pool_bags
        idx_lists, off_lists = self._lists(lS_o, lS_i)
        Bq, P = len(off_lists[0]), max_per_bag
        iv = expand_bags(idx_lists, off_lists, Bq, P)
        h, st, sr, _ = self.o.lookup_batch(iv, agg=None if agg_in is None else agg_in.numpy(), table_ids=self.ids)
        out.copy_(torch.from_numpy(pool_bags(gather_rows(self.tables, st, sr), iv, Bq, P)))
        hits = []
        for t in range(len(self.ids)):
            off = list(off_lists[t]) + [len(idx_lists[t])]
            hits.append(torch.from_numpy(np.concatenate([h[s * P:s * P + off[s + 1] - off[s], t] for s in range(Bq)]).astype(np.uint8)))
        return out, hits


def _placement(kind):
    p = pkg()
    return p.sharded.balanced_placement(SMALL_ROWS, WORLD) if kind == "balanced" else p.sharded.contiguous_placement(26, WORLD)


def _worker(rank, port, q, kind):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=WORLD)
    p = pkg()
    tables = p.workload.make_tables(SMALL_ROWS, DIM)
    placement = _placement(kind)
    ids = placement[rank]
    sh = p.sharded.ShardedLookup(OracleBagStore(tables, CAP, ids), 26, DIM, rank, WORLD, placement=placement)
    res = []
    for k, P in enumerate(PS):
        idx_lists, off_lists = make_bags(k, SMALL_ROWS, B, P)
        ly, hit = sh.lookup_bags([torch.from_numpy(off_lists[t]) for t in ids], [torch.from_numpy(idx_lists[t]) for t in ids], P)
        res.append((ly.numpy().copy(), [h.numpy().copy() for h in hit]))
    q.put((rank, res))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("kind", ["contiguous", "balanced"])
def test_sharded_lookup_bags_two_ranks_gloo(kind):
    import torch.multiprocessing as mp
    from oracle.evlfu import BatchEvLFU
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 25500 + (os.getpid() + (7 if kind == "balanced" else 0)) % 2000
    procs = [ctx.Process(target=_worker, args=(r, port, q, kind)) for r in range(WORLD)]
    for pr in procs:
        pr.start()
    got = dict(q.get(timeout=180) for _ in range(WORLD))
    for pr in procs:
        pr.join(timeout=60)
        assert pr.exitcode == 0
    p = pkg()
    tables = p.workload.make_tables(SMALL_ROWS, DIM)
    placement = _placement(kind)
    oracles = [BatchEvLFU(CAP, n_tables=26) for _ in range(WORLD)]
    Bl = B // WORLD
    n_hits = 0
    for k, P in enumerate(PS):
        idx_lists, off_lists = make_bags(k, SMALL_ROWS, B, P)
        want = oracle_bags(oracles, placement, tables, idx_lists, off_lists, B, P)
        full = np.empty((B, 26, DIM), dtype=np.float32)
        for ids, (pooled, _, _, _) in zip(placement, want):
            full[:, ids] = pooled
        for r in range(WORLD):
            ly, hit = got[r][k]
            assert ly.shape == (Bl, 26, DIM)
            assert np.array_equal(ly, full[r * Bl:(r + 1) * Bl]), f"batch {k} rank {r}: pooled rows after the all-to-all"
            for t, c in enumerate(want[r][1]):
                assert np.array_equal(hit[t], c), f"batch {k} rank {r} table {placement[r][t]}: hit codes"
                n_hits += int(c.sum())
    assert n_hits > 0
