"""The snapshot format of evs_save_state (include/evstore_b200.h), read by state_info without a GPU: a blob written by a
pure-Python writer of the documented layout round-trips, and truncated or foreign blobs are refused."""
import struct

import numpy as np
import pytest

from helpers import SMALL_ROWS, pkg


def write_blob(policy, n_layers, table_ids, rows, tiers, c3=None, n_tables_total=26, dim=16, precisions=(32, 0),
               caps=(300, 0), c3_cap=0):
    """tiers: [(n_perfect, [keys of bucket 0], [keys of bucket 1], ...)] with n_tables_total + 1 buckets each;
    c3: (size, window records, [(key, alt, flag)]) or None."""
    nb = n_tables_total + 1
    words = []
    for n_perfect, buckets in tiers:
        assert len(buckets) == nb
        words += [n_perfect] + [len(b) for b in buckets] + [k for b in buckets for k in b]
    if c3 is not None:
        size, window, entries = c3
        words += [size, len(window)] + list(window)
        for key, alt, flag in entries:
            words += [key, alt | (flag << 32)]
    body = np.array(words, dtype="<u8").tobytes()
    n = len(table_ids)
    hdr = struct.pack("<8sIIQ8i3Q32i32q", b"EVSSTATE", 1, 464, 464 + len(body), policy, n_layers, n_tables_total, n,
                      dim, precisions[0], precisions[1], nb, caps[0], caps[1], c3_cap,
                      *(list(table_ids) + [-1] * (32 - n)), *(list(rows) + [0] * (32 - n)))
    assert len(hdr) == 464
    return np.frombuffer(hdr + body, dtype=np.uint8).copy()


def _key(t, r):
    return (t << 40) | r


def _buckets(rng, nb, n):
    out = [[] for _ in range(nb)]
    for i in range(n):
        out[int(rng.integers(0, nb))].append(_key(int(rng.integers(0, 26)), i))
    return out


def test_single_tier_round_trip():
    rng = np.random.default_rng(0)
    bk = _buckets(rng, 27, 200)
    blob = write_blob(0, 1, range(26), SMALL_ROWS, [(17, bk)])
    info = pkg().state_info(blob)
    assert info["policy"] == "evlfu" and info["n_layers"] == 1 and info["n_tables_total"] == 26
    assert info["table_ids"] == list(range(26)) and info["rows"] == SMALL_ROWS
    assert info["tiers"] == [{"n_perfect": 17, "counts": [len(b) for b in bk]}] and info["c3"] is None
    assert info["bytes"] == len(blob) == 464 + 8 * (1 + 27 + 200)
    assert pkg().state_info(blob.tobytes()) == info


def test_three_layers_round_trip_with_stale_window_records():
    rng = np.random.default_rng(1)
    t0, t1 = _buckets(rng, 27, 50), _buckets(rng, 27, 80)
    window = [_key(3, 1), _key(3, 1), _key(4, 2), _key(5, 9)]          # a duplicate and a stale record
    entries = [(_key(3, 1), 201, 1), (_key(4, 2), 1503, 0)]
    blob = write_blob(0, 3, range(26), SMALL_ROWS, [(0, t0), (2, t1)], c3=(2, window, entries), precisions=(8, 4),
                      caps=(80, 160), c3_cap=320)
    info = pkg().state_info(blob)
    assert info["c3"] == {"size": 2, "window": 4}
    assert [t["n_perfect"] for t in info["tiers"]] == [0, 2]
    assert info["capacity"] == [80, 160] and info["c3_capacity"] == 320
    assert (info["main_precision"], info["secondary_precision"]) == (8, 4)


def test_sharded_rank_and_other_policies():
    blob = write_blob(2, 1, [13, 14, 15], [5, 6, 7], [(0, [[] for _ in range(27)])])
    info = pkg().state_info(blob)
    assert info["policy"] == "lfu" and info["table_ids"] == [13, 14, 15] and info["rows"] == [5, 6, 7]
    assert info["tiers"][0]["counts"] == [0] * 27


@pytest.mark.parametrize("cut", [0, 8, 100, 463, 464, -8, -1])
def test_truncated_blobs_are_refused(cut):
    rng = np.random.default_rng(2)
    blob = write_blob(0, 2, range(26), SMALL_ROWS, [(0, _buckets(rng, 27, 30)), (0, _buckets(rng, 27, 40))])
    with pytest.raises(ValueError):
        pkg().state_info(blob[:cut] if cut else blob[:0])


def test_truncated_body_with_a_consistent_length_is_refused():
    rng = np.random.default_rng(3)
    blob = write_blob(0, 1, range(26), SMALL_ROWS, [(0, _buckets(rng, 27, 30))])
    short = blob[:-8].copy()
    short[16:24] = np.frombuffer(struct.pack("<Q", len(short)), dtype=np.uint8)
    with pytest.raises(ValueError, match="sections"):
        pkg().state_info(short)


def test_foreign_blobs_are_refused():
    rng = np.random.default_rng(4)
    blob = write_blob(0, 1, range(26), SMALL_ROWS, [(0, _buckets(rng, 27, 10))])
    bad = blob.copy()
    bad[0] = ord("X")
    with pytest.raises(ValueError, match="magic"):
        pkg().state_info(bad)
    bad = blob.copy()
    bad[8:12] = np.frombuffer(struct.pack("<I", 2), dtype=np.uint8)
    with pytest.raises(ValueError, match="version"):
        pkg().state_info(bad)
    with pytest.raises(ValueError):
        pkg().state_info(np.random.default_rng(5).integers(0, 256, size=2000).astype(np.uint8))


# ---- the oracle seeding helper (tests/state_seed.py) -------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["evlfu", "evlfu_approx", "lru", "lfu", "tiers2", "tiers3"])
def test_an_oracle_seeded_from_a_snapshot_continues_identically(kind):
    """An oracle runs n batches; a fresh oracle seeded from a snapshot of its state (written in the blob format and parsed
    back) then continues exactly as it does: hit maps, sources, agg_hit, eviction / flush streams, state, C3."""
    from oracle import tiers as otiers
    from state_seed import make_oracle, parse_snapshot, rewrite, seed_oracle, snapshot_of
    p = pkg()
    rows = SMALL_ROWS
    alt = p.workload.make_alt_keys(rows) if kind == "tiers3" else None
    cfg = {"evlfu": dict(), "evlfu_approx": dict(approx_emb_thres=12), "lru": dict(policy="lru"), "lfu": dict(policy="lfu"),
           "tiers2": dict(n_layers=2), "tiers3": dict(n_layers=3)}[kind]
    caps = {"tiers2": (120, 1920, 0), "tiers3": (60, 120, 480)}.get(kind, (300, 0, 0))
    approx = cfg.get("approx_emb_thres", -1)
    trace = p.workload.ZipfTrace(rows, seed=7)
    a = make_oracle(cfg, caps[:2], caps[2], alt)

    def step(o, idx):
        r = o.lookup_batch(idx) if isinstance(o, otiers.BatchTiers) else o.lookup_batch(idx, approx_emb_thres=approx)
        tiers = [o.c1, o.c2] if isinstance(o, otiers.BatchTiers) else [o]
        ev = [(t.evicted, t.flushed, t.state(), t.n_perfect) for t in tiers]
        c3 = o.c3.dump() if getattr(o, "c3", None) is not None else None
        return [x.tolist() for x in r], ev, c3

    for _ in range(40):
        step(a, trace.batch(64))
    snap = snapshot_of(a)
    if kind == "tiers3":
        assert len(snap["c3"][0]) > len(snap["c3"][1]) > 0          # stale / duplicate records in the window
    header = write_blob(0, snap["n_layers"], range(26), rows, [(0, [[] for _ in range(27)])] * (2 if snap["n_layers"] > 1 else 1),
                        c3=(0, [], []) if snap["c3"] is not None else None, c3_cap=caps[2])
    blob = rewrite(header, snap)
    back = parse_snapshot(blob)
    assert back["tiers"] == snap["tiers"] and back["c3"] == snap["c3"]
    b = seed_oracle(make_oracle(cfg, caps[:2], caps[2], alt), back)
    for it in range(40):
        idx = trace.batch(64)
        assert step(a, idx) == step(b, idx), f"batch {it}"
