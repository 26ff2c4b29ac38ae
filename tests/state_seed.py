"""Snapshots (evs_save_state) on the oracle side: parse a blob's sections, seed a batch oracle from them, and follow a
seeded oracle next to a handle.  Used by test_gpu_state.py and, without a GPU, by test_state_format.py."""
from collections import OrderedDict, deque

import numpy as np

from oracle import tiers as otiers
from oracle.evlfu import BatchEvLFU, gather_rows
from oracle.lru import BatchLFU, BatchLRU

HDR = 464


def parse_snapshot(blob):
    """Sections of a snapshot: {"n_layers", "tiers": [(n_perfect, [keys of bucket b] ...)], "c3": None or
    (window records, [(key, alt, flag)])}.  The header is checked by state_info."""
    import importlib
    info = importlib.import_module("ev-store-dlrm_b200").state_info(blob)
    w = np.frombuffer(np.asarray(blob, dtype=np.uint8)[HDR:].tobytes(), dtype="<u8")
    nb = info["n_tables_total"] + 1
    o, tiers = 0, []
    for _ in info["tiers"]:
        counts = [int(x) for x in w[o + 1:o + 1 + nb]]
        keys = [int(x) for x in w[o + 1 + nb:o + 1 + nb + sum(counts)]]
        off = np.concatenate([[0], np.cumsum(counts)]).astype(int)
        tiers.append((int(w[o]), [keys[off[b]:off[b + 1]] for b in range(nb)]))
        o += 1 + nb + sum(counts)
    c3 = None
    if info["c3"] is not None:
        size, W = int(w[o]), int(w[o + 1])
        window = [int(x) for x in w[o + 2:o + 2 + W]]
        m = w[o + 2 + W:o + 2 + W + 2 * size]
        c3 = (window, [(int(m[2 * i]), int(m[2 * i + 1]) & 0xFFFFFFFF, int(m[2 * i + 1]) >> 32) for i in range(size)])
    return {"n_layers": info["n_layers"], "tiers": tiers, "c3": c3}


def _seed_tier(t, n_perfect, buckets, lru=False):
    if lru:
        t.entries = OrderedDict((k, None) for k in buckets[0])
    else:
        t.entries = {k: b for b, ks in enumerate(buckets) for k in ks}
        t.lists = [OrderedDict((k, None) for k in ks) for ks in buckets]
    t.n_perfect = n_perfect


def seed_oracle(oracle, snap):
    """Put a fresh BatchEvLFU / BatchLRU / BatchLFU / oracle.tiers.BatchTiers into the state a snapshot holds."""
    if isinstance(oracle, otiers.BatchTiers):
        for t, (n_perfect, buckets) in zip((oracle.c1, oracle.c2), snap["tiers"]):
            _seed_tier(t, n_perfect, buckets)
        if oracle.c3 is not None:
            window, entries = snap["c3"]
            oracle.c3.fifo = deque(window)
            oracle.c3.vals = {k: [alt, bool(flag & 1)] for k, alt, flag in entries}
    else:
        _seed_tier(oracle, *snap["tiers"][0], lru=isinstance(oracle, BatchLRU))
    return oracle


def snapshot_of(oracle):
    """The inverse of seed_oracle: the sections a snapshot of the oracle's state holds."""
    if isinstance(oracle, otiers.BatchTiers):
        tiers = [(t.n_perfect, t.state()) for t in (oracle.c1, oracle.c2)]
        c3 = None
        if oracle.c3 is not None:
            c3 = (list(oracle.c3.fifo), [(k, int(v[0]), int(v[1])) for k, v in oracle.c3.vals.items()])
        return {"n_layers": oracle.n_layers, "tiers": tiers, "c3": c3}
    return {"n_layers": 1, "tiers": [(oracle.n_perfect, oracle.state())], "c3": None}


def make_oracle(cfg, caps, c3_cap, alt=None, T=26):
    """The batch oracle of a handle's configuration (CacheConfig fields as a dict) and capacities."""
    layers = cfg.get("n_layers", 1)
    if layers >= 2:
        return otiers.BatchTiers((caps[0], caps[1], c3_cap), n_layers=layers, T=T, alt_keys=alt)
    return {"evlfu": BatchEvLFU, "lru": BatchLRU, "lfu": BatchLFU}[cfg.get("policy", "evlfu")](caps[0], n_tables=T)


class Follower:
    """A batch oracle seeded from a snapshot, checked against a handle after each batch it serves."""

    def __init__(self, store, cfg, blob, tables, alt=None):
        from helpers import decoded_tables
        st = store.stats()
        self.cfg, self.store = cfg, store
        self.oracle = seed_oracle(make_oracle(cfg, st["capacity"], st["c3_capacity"], alt), parse_snapshot(blob))
        self.layers = cfg.get("n_layers", 1)
        precs = [cfg.get("main_precision", 32)] + ([cfg["secondary_precision"]] if self.layers >= 2 else [])
        self.dec = [decoded_tables(tables, q) for q in precs]

    def check(self, idx, out, hit, events, where=""):
        o, store = self.oracle, self.store
        if self.layers >= 2:
            code, val_tier, st, sr, _agg = o.lookup_batch(idx)
            assert np.array_equal(hit, code), f"hit codes vs the seeded oracle{where}"
            assert np.array_equal(out, otiers.gather_tier_rows(self.dec, val_tier, st, sr)), f"rows vs the seeded oracle{where}"
            tiers = [o.c1, o.c2]
        else:
            o_hit, st, sr, _agg = o.lookup_batch(idx, approx_emb_thres=self.cfg.get("approx_emb_thres", -1))
            assert np.array_equal(hit.astype(bool), o_hit), f"hit map vs the seeded oracle{where}"
            ok = st >= 0
            assert np.array_equal(out[ok], gather_rows(self.dec[0], st, sr)[ok]), f"rows vs the seeded oracle{where}"
            tiers = [o]
        for ti, ot in enumerate(tiers):
            assert events[ti] == (ot.evicted, ot.flushed), f"eviction / flush streams of tier {ti} vs the seeded oracle{where}"
            state, n_perfect = store.dump_state(ti)
            assert state == ot.state() and n_perfect == ot.n_perfect, f"state of tier {ti} vs the seeded oracle{where}"
        if self.layers == 3:
            k, a, r = store.dump_c3()
            assert (k.tolist(), a.tolist(), r.tolist()) == tuple(list(x) for x in o.c3.dump()), f"C3 vs the seeded oracle{where}"


def rewrite(blob, snap):
    """blob's header (with its length field updated) followed by the body of the sections `snap`."""
    words = []
    for n_perfect, buckets in snap["tiers"]:
        words += [n_perfect] + [len(b) for b in buckets] + [k for b in buckets for k in b]
    if snap["c3"] is not None:
        window, entries = snap["c3"]
        words += [len(entries), len(window)] + list(window)
        for key, alt, flag in entries:
            words += [key, alt | (flag << 32)]
    body = np.array(words, dtype="<u8").view(np.uint8)
    out = np.concatenate([np.asarray(blob, dtype=np.uint8)[:HDR], body])
    out[16:24] = np.array([len(out)], dtype="<u8").view(np.uint8)
    return out


def sections_equal(x, y):
    """Snapshot sections equal up to the order of C3's map entries (slot order: slot assignments may differ)."""
    cx = None if x["c3"] is None else (x["c3"][0], sorted(x["c3"][1]))
    cy = None if y["c3"] is None else (y["c3"][0], sorted(y["c3"][1]))
    return x["tiers"] == y["tiers"] and cx == cy
