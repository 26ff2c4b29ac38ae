"""Inputs and oracle shared by the sharded-bags tests (tests/test_gpu_sharded_bags.py, tests/test_sharded_bags_gloo.py).

A sharded bag batch must give exactly what single-GPU bags give with every table: every rank expands its own tables'
bags into B*P slices (oracle.evlfu.expand_bags), a slice's agg_hit is the sum over the ranks of the hits among its present
keys, every rank runs the batch policy on its slices (BatchEvLFU.lookup_batch(agg=...)), and the pooled rows are the
slice rows summed in ascending j (pool_bags)."""
import numpy as np

from oracle.evlfu import expand_bags, gather_rows, make_key, pool_bags


def make_bags(k, rows, B, P):
    """Step k's bags of every table: ragged lengths uniform in 0..P, with an empty bag and a bag of exactly P in every
    table.  Returns (idx_lists, off_lists) in apply_emb's layout (offsets [B] per table)."""
    rng = np.random.default_rng(1000 + k)
    idx_lists, off_lists = [], []
    for n in rows:
        lens = rng.integers(0, P + 1, size=B)
        lens[rng.integers(0, B)] = 0
        lens[rng.integers(0, B)] = P
        tot = int(lens.sum())
        r = np.minimum((n * rng.random(tot) ** 1.3 * rng.random(tot)).astype(np.int64), n - 1)
        idx_lists.append(r)
        off_lists.append(np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int64))
    return idx_lists, off_lists


def make_plain(k, rows, B):
    """Step k's plain batch: int64 [26, B]."""
    rng = np.random.default_rng(2000 + k)
    return np.stack([np.minimum((n * rng.random(B) ** 1.3 * rng.random(B)).astype(np.int64), n - 1) for n in rows])


def slice_counts(o, ids, idx_v):
    """Per slice: how many of this rank's present keys are resident in its oracle."""
    T, V = idx_v.shape
    return np.array([sum(idx_v[t, v] >= 0 and make_key(ids[t], int(idx_v[t, v])) in o.entries for t in range(T))
                     for v in range(V)], dtype=np.int64)


def oracle_bags(oracles, placement, tables, idx_lists, off_lists, B, P):
    """One sharded bag batch on the oracles (one per rank).  Returns per rank (pooled [B, T_r, d], hit codes per local
    table [nnz_t] (1 = hit), present keys, misses)."""
    idx_vs = [expand_bags([idx_lists[t] for t in ids], [off_lists[t] for t in ids], B, P) for ids in placement]
    agg = sum(slice_counts(o, ids, iv) for o, ids, iv in zip(oracles, placement, idx_vs))
    out = []
    for o, ids, iv in zip(oracles, placement, idx_vs):
        o_hit, s_t, s_r, _ = o.lookup_batch(iv, agg=agg, table_ids=ids)
        pooled = pool_bags(gather_rows(tables, s_t, s_r), iv, B, P)
        codes = []
        for t, g in enumerate(ids):
            off = list(off_lists[g]) + [len(idx_lists[g])]
            codes.append(np.concatenate([o_hit[s * P:s * P + off[s + 1] - off[s], t] for s in range(B)]).astype(np.uint8))
        present = int((iv >= 0).sum())
        out.append((pooled, codes, present, present - int(o_hit.sum())))
    return out
