"""Table-wise sharding of the lookup path over the GPUs of one box (BASELINE configs[4]).

Semantics of the reference's distributed forward (dlrm_s_pytorch.py:529-586 with
extend_distributed.py): rank r owns a contiguous slice of the tables (``get_split_lengths`` /
``get_my_slice``, extend_distributed.py:47-62), looks the FULL batch up in its tables, and one
all-to-all turns the table-sharded pooled rows ``[B, T_local*d]`` into batch-sharded ones
``[B/size, 26*d]`` (``ext_dist.alltoall``, extend_distributed.py:541-576; ``all_to_all_single``
at :414).  One process per GPU, ``torch.distributed`` (NCCL over NVLink on GPUs; gloo in the CPU
tests of this host logic).

EvLFU's only cross-table coupling is agg_hit, the number of a sample's keys that hit.  The
reference never ran its cache sharded; here the ranks probe (``evs_probe_batch``), all-reduce the
per-sample hit counts (uint8[B], 2-16 KB) and pass the sum to ``evs_lookup_batch`` as ``agg_in``,
so the union of the ranks' hit / eviction streams equals the single-GPU policy's.
"""
from __future__ import annotations


def get_split_lengths(n: int, size: int):
    """extend_distributed.py:54-62: the first n % size ranks get one extra table."""
    k, m = divmod(n, size)
    return [k + 1] * m + [k] * (size - m) if m else [k] * size


def get_my_slice(n: int, rank: int, size: int) -> slice:
    """extend_distributed.py:47-51."""
    k, m = divmod(n, size)
    return slice(rank * k + min(rank, m), (rank + 1) * k + min(rank + 1, m), 1)


def contiguous_placement(n: int, size: int):
    """The reference's placement: rank r serves the tables of get_my_slice(n, r, size)."""
    return [list(range(n))[get_my_slice(n, r, size)] for r in range(size)]


def balanced_placement(rows, size: int):
    """Tables spread over the ranks by ROW COUNT, keeping get_split_lengths' tables-per-rank (so every rank still
    handles the same number of lookups per sample).  This DEPARTS from the reference's contiguous split
    (extend_distributed.py:47-62): Criteo's few huge tables sit next to each other, so the contiguous slices leave
    most ranks with a handful of rows -- and almost no misses, evictions or backing-store traffic -- while one or
    two ranks carry everything.  Largest table first, each to the rank with the fewest rows that still has a free
    slot; ids ascending within a rank."""
    n = len(rows)
    cap = get_split_lengths(n, size)
    load = [0] * size
    out = [[] for _ in range(size)]
    for t in sorted(range(n), key=lambda t: (-int(rows[t]), t)):
        r = min((r for r in range(size) if len(out[r]) < cap[r]), key=lambda r: (load[r], r))
        out[r].append(t)
        load[r] += int(rows[t])
    return [sorted(x) for x in out]


def split_cache_budget(rows_per_rank, total_rows_cached: int, floor: int = 1024):
    """The one cache's budget (TOTAL_SIZE, cache_manager.cpp:16: entries of the whole model) split over the ranks of a
    table-wise sharded cache.  Every GPU contributes the same memory; a rank whose tables are smaller than its share caches
    them whole and the rest of its share goes to the others (water filling): cap_r = min(rows_r, level), sum = budget.
    Sizing every rank at the same FRACTION of its own rows instead leaves a rank that owns only small tables with a cache
    far smaller than one batch's keys -- it thrashes, and the whole step waits for its miss fetches."""
    rows = [int(r) for r in rows_per_rank]
    budget = min(int(total_rows_cached), sum(rows))
    caps = [0] * len(rows)
    open_ranks = sorted(range(len(rows)), key=lambda r: rows[r])
    left = budget
    while open_ranks:
        level = left // len(open_ranks)
        r = open_ranks[0]
        if rows[r] <= level:
            caps[r] = rows[r]
            left -= rows[r]
            open_ranks.pop(0)
        else:
            for q in open_ranks:
                caps[q] = level
            break
    return [max(floor, c) for c in caps]


class ShardedLookup:
    """One rank's part of the sharded lookup.  ``store`` serves this rank's tables
    (``EvStore`` built with table_base / n_tables_total; any object with ``probe`` and ``lookup`` -- and ``probe_bags`` /
    ``lookup_bags`` for bags -- of the same signatures works, which is how the CPU tests drive the host logic)."""

    def __init__(self, store, n_tables_total: int, dim: int, rank: int, world: int, group=None, exact_agg: bool = True,
                 transport: str = "nccl", batch_max: int = 0, placement=None):
        """transport "nccl": torch.distributed all-reduce + all_to_all_single (any backend; what the reference does).
        transport "p2p": the exchange is fused into the kernels over NVLink peer memory (evs_shard_*); needs
        ``batch_max`` (the global batch) and a store with shard_create / shard_connect / shard_lookup.
        placement: per rank the global ids of its tables (default: the reference's contiguous slices); the store of
        a rank with a non-contiguous set must have been built with ``CacheConfig.table_ids``."""
        self.store, self.T, self.dim = store, n_tables_total, dim
        self.rank, self.world, self.group = rank, world, group
        self.exact_agg = exact_agg
        self.transport = transport if world > 1 else "nccl"
        if self.transport == "p2p":
            import torch.distributed as dist
            mine = store.shard_create(rank, world, batch_max)
            handles = [None] * world
            dist.all_gather_object(handles, mine, group=group)
            store.shard_connect(handles)
            dist.barrier(group=group)
        self.placement = [list(x) for x in placement] if placement is not None else contiguous_placement(n_tables_total, world)
        assert sorted(t for x in self.placement for t in x) == list(range(n_tables_total)), "every table on exactly one rank"
        self.splits = [len(x) for x in self.placement]
        self.my = self.placement[rank]
        self.T_local = self.splits[rank]
        self._bufs = {}

    def _buffers(self, B, device):
        import torch
        key = (B, str(device))
        if key not in self._bufs:
            Bl = B // self.world
            send = torch.empty((B, self.T_local, self.dim), dtype=torch.float32, device=device)
            recv = torch.empty((Bl * self.T * self.dim,), dtype=torch.float32, device=device)
            out = torch.empty((Bl, self.T, self.dim), dtype=torch.float32, device=device)
            hit = torch.empty((B, self.T_local), dtype=torch.uint8, device=device)
            agg = torch.empty((B,), dtype=torch.uint8, device=device)
            self._bufs[key] = (send, recv, out, hit, agg)
        return self._bufs[key]

    def lookup(self, lS_i_local, next_idx=None):
        """lS_i_local: int64 [T_local, B], this rank's tables for the whole batch (B % world == 0).
        next_idx: the tensor the NEXT call will pass (look-ahead, EvStore.prefetch), or None.
        Returns (ly [B/world, 26, dim] for this rank's slice of the batch, hit [B, T_local])."""
        import torch.distributed as dist
        T_local, B = lS_i_local.shape
        assert T_local == self.T_local and B % self.world == 0
        if self.transport == "p2p":
            r = self.store.shard_lookup(lS_i_local)
            if next_idx is not None:
                self.store.prefetch(next_idx)
            return r
        send, recv, out, hit, agg = self._buffers(B, lS_i_local.device)
        agg_in = None
        if self.exact_agg and self.world > 1:
            self.store.probe(lS_i_local, agg_out=agg)
            dist.all_reduce(agg, op=dist.ReduceOp.SUM, group=self.group)
            agg_in = agg
        self.store.lookup(lS_i_local, out=send, hit=hit, agg_in=agg_in)
        if next_idx is not None and hasattr(self.store, "prefetch"):
            self.store.prefetch(next_idx)
        if self.world == 1:
            return send, hit
        return self._exchange(send, recv, out, B), hit

    def lookup_bags(self, lS_o_local, lS_i_local, max_per_bag: int = 10):
        """Bags (pooling factor > 1) of this rank's tables for the whole batch: lS_o_local / lS_i_local are apply_emb's
        per-table offset and index tensors of this rank's T_local tables (B bags each, B % world == 0, bags of at most
        max_per_bag indices).  A batch of bags is looked up as B * max_per_bag slices whose agg_hit is summed over the
        ranks; each rank pools its own tables and only pooled rows cross between the ranks.
        Returns (ly [B/world, 26, dim] for this rank's slice of the batch, hit: per local table uint8 [nnz_t])."""
        import torch.distributed as dist
        assert len(lS_o_local) == self.T_local and len(lS_i_local) == self.T_local
        B = int(lS_o_local[0].numel())
        assert B % self.world == 0
        if self.transport == "p2p":
            return self.store.shard_lookup_bags(lS_o_local, lS_i_local, max_per_bag)
        send, recv, out, _, _ = self._buffers(B, lS_i_local[0].device)
        agg_in = None
        if self.exact_agg and self.world > 1:
            agg_in = self.store.probe_bags(lS_o_local, lS_i_local, max_per_bag)
            dist.all_reduce(agg_in, op=dist.ReduceOp.SUM, group=self.group)
        _, hit = self.store.lookup_bags(lS_o_local, lS_i_local, max_per_bag, out=send, agg_in=agg_in)
        if self.world == 1:
            return send, hit
        return self._exchange(send, recv, out, B), hit

    def _exchange(self, send, recv, out, B):
        """Table-sharded pooled rows [B, T_local, d] -> this rank's batch-sharded [B/world, 26, d] (all_to_all_single)."""
        import torch
        import torch.distributed as dist
        Bl = B // self.world
        # send: [B, T_local*d] split along the batch; recv: world blocks [Bl, T_src, d], source-rank major
        in_splits = [Bl * self.T_local * self.dim] * self.world
        out_splits = [Bl * t * self.dim for t in self.splits]
        dist.all_to_all_single(recv, send.view(-1), out_splits, in_splits, group=self.group)
        o = 0
        for ids in self.placement:
            t = len(ids)
            n = Bl * t * self.dim
            blk = recv[o:o + n].view(Bl, t, self.dim)
            if ids == list(range(ids[0], ids[0] + t)):
                out[:, ids[0]:ids[0] + t, :] = blk
            else:
                out[:, torch.as_tensor(ids, device=out.device), :] = blk
            o += n
        return out

    def lookup_many(self, idx_list, next_idx=None, hits=None):
        """Consecutive batches in one call: [(ly, hit)] as ``lookup`` on each in turn.  With the fused transport groups of 4
        batches reach every rank's device as one captured graph (evs_shard_lookup_many) and a returned ``ly`` is valid until
        four batches later; the other transports run the batches one by one."""
        if self.transport == "p2p":
            outs, hits = self.store.shard_lookup_many(idx_list, hits=hits)
            if next_idx is not None:
                self.store.prefetch(next_idx)
            return list(zip(outs, hits))
        res = []
        for k, idx in enumerate(idx_list):
            ly, hit = self.lookup(idx, next_idx=idx_list[k + 1] if k + 1 < len(idx_list) else next_idx)
            res.append((ly.clone(), hit.clone()))         # lookup() reuses its buffers from call to call
        return res

    def update_rows(self, tables, rows, values, stream=None):
        """New values for rows of the model (``EvStore.update_rows``), called with the same arguments on every rank.
        Each rank applies the entries of the tables it owns; no collective is needed, because a rank serves rows of its
        own tables only.  Returns this rank's ``where`` [n]: the entries of other ranks' tables read 0."""
        import torch
        n = int(rows.shape[0])
        where = torch.zeros((n,), dtype=torch.uint8, device=rows.device)
        if torch.is_tensor(tables):
            mine = torch.isin(tables, torch.as_tensor(self.my, dtype=tables.dtype, device=tables.device))
        else:
            mine = torch.full((n,), int(tables) in self.my, dtype=torch.bool, device=rows.device)
        sel = mine.nonzero().flatten()
        if sel.numel():
            t = tables[sel] if torch.is_tensor(tables) else int(tables)
            where[sel] = self.store.update_rows(t, rows[sel], values[sel], stream=stream)
        return where

    def save_state(self):
        """Snapshot of this rank's cache (``EvStore.save_state``)."""
        return self.store.save_state()

    def load_state(self, blob):
        """Restore a snapshot of a rank that served the same tables (``EvStore.load_state``); re-sharding is not supported."""
        self.store.load_state(blob)

    def alltoall_bytes(self, B: int) -> int:
        """Bytes this rank sends to its peers per batch (SURVEY.md section 8(d))."""
        return B * self.T_local * self.dim * 4 * (self.world - 1) // self.world
