"""The multi-layer oracles (oracle/tiers.py) against the reference itself.

The reference's two-layer path exists only in C++; oracle/build_ref.py (run by build()) compiles it
from the checkout of the original project named by EVSTORE_REFERENCE into oracle/_ref/lib<variant>.so;
without one these pins skip.  ``SeqTiers(order="stdset", flush="cpp")``
must reproduce it request by request: every returned row has to be the dequantised row of the
tier the restatement says answered (fp32 / 16 / 8 / 4-bit rows of one key differ, so the floats
identify the tier), over thousands of requests with evictions, promotions and the C1-full
routing switch.  Positions where the C++ reads a dangling pointer (evlfu_32.cpp:352 "TODO: This
is buggy") are excluded -- and counted, they must stay rare.

The batch-granular ``BatchTiers`` is then tied to the sequential restatement at batch size 1.
"""
import ctypes as C

import numpy as np
import pytest

from helpers import SMALL_ROWS, pkg
from oracle import codecs as ocodecs
from oracle import ref_driver, tiers
from oracle.evlfu import BatchEvLFU, split_key
from oracle.ref_variants import VARIANTS

T = 26
DIM = 36
PRECS = (32, 16, 8, 4)


@pytest.fixture(scope="module")
def fixture_tables():
    p = pkg()
    tables = p.workload.make_tables(SMALL_ROWS, DIM)
    raw = {prec: [ocodecs.quantize_table(t, prec) for t in tables] for prec in PRECS}
    dec = {prec: [ocodecs.dequantize_rows(r, prec) for r in raw[prec]] for prec in PRECS}
    return tables, raw, dec


def _trace(n, seed, alpha=1.05):
    p = pkg()
    tr = p.workload.ZipfTrace(SMALL_ROWS, alpha=alpha, seed=seed)
    return np.ascontiguousarray(tr.batches(1, n)[0].T.astype(np.int32))        # [n, 26]


def _run_pin(variant, fixture_tables, n, seed, alpha=1.05, fresh=False):
    if not (ref_driver.available(variant) and tiers.shim_available()):
        pytest.skip("needs the original project's compiled cache (set EVSTORE_REFERENCE to its checkout, run build())")
    _tables, raw, dec = fixture_tables
    v = VARIANTS[variant]
    ref_driver.write_fixture(variant, {prec: raw[prec] for prec in PRECS})
    ref = ref_driver.RefCache(variant, fresh_copy=fresh)       # fresh: a private, empty instance of the library
    trace = _trace(n, seed, alpha)
    _sec, out = ref.drive(trace, want_out=True)                                 # [n, 26, 36]
    perfect_ref = int(C.c_int.in_dll(ref.lib, "perfectHit").value)
    caps = tiers.capacities(v["layers"], v["main"], v["sec"], v["total"], v["prop"], v["dim"])
    o = tiers.SeqTiers(caps, n_layers=v["layers"], order="stdset", flush="cpp")
    precs = (v["main"], v["sec"])
    n_stale = n_evict = n_flush = n_c2 = perfect = 0
    for i in range(n):
        code, val_tier, src, stale, pf = o.request(trace[i])
        perfect += pf
        n_evict += len(o.c1.evicted) + len(o.c2.evicted)
        n_flush += len(o.c1.flushed) + len(o.c2.flushed)
        for t in range(T):
            if stale[t]:
                n_stale += 1
                continue
            n_c2 += val_tier[t]
            tt, rr = split_key(src[t])
            want = dec[precs[val_tier[t]]][tt][rr]
            assert (out[i, t] == want).all(), f"{variant}: request {i} table {t}: code {code[t]} tier {val_tier[t]}"
    assert perfect == perfect_ref, "perfect-hit counter (cache_manager.cpp:59)"
    return dict(stale=n_stale, evict=n_evict, flush=n_flush, c2=n_c2, perfect=perfect)


def test_seq_single_tier_fp32_equals_compiled_reference(fixture_tables):
    r = _run_pin("test_c1_fp32_d36", fixture_tables, 6000, seed=3)
    assert r["evict"] > 1000 and r["stale"] < 60


def test_seq_single_tier_8bit_equals_compiled_reference(fixture_tables):
    r = _run_pin("test_c1_8_d36", fixture_tables, 6000, seed=4)
    assert r["evict"] > 1000


@pytest.mark.parametrize("variant", ["test_c2_8_4_small_d36", "test_c2_32_8_small_d36", "test_c2_16_4_small_d36"])
def test_seq_two_tier_equals_compiled_reference(fixture_tables, variant):
    r = _run_pin(variant, fixture_tables, 8000, seed=5)
    assert r["evict"] > 500, r          # C1 filled up, the odd/even routing and evictions ran
    assert r["c2"] > 1000, r            # rows were answered at C2's precision
    assert r["stale"] < 100, r


def test_seq_two_tier_never_full_equals_compiled_reference(fixture_tables):
    """TOTAL_SIZE 100000: C1 never fills, everything goes to C1 (evlfu_8.cpp:590-602)."""
    r = _run_pin("test_c2_8_4_d36", fixture_tables, 3000, seed=6)
    assert r["evict"] == 0 and r["c2"] == 0


def test_seq_flush_rule_equals_compiled_reference(fixture_tables):
    """A hot trace (alpha 2.5) makes most requests perfect hits, so bucket 26 reaches 95 % of the
    capacity and the C++ flush (int(0.3*cap) keys, n_perfect -= that) runs."""
    # a separate process-global library instance would be needed to restart from an empty cache,
    # so this uses the one variant no other test loads
    if "test_c1_flush_d36" not in VARIANTS:
        pytest.skip("variant not configured")
    r = _run_pin("test_c1_flush_d36", fixture_tables, 6000, seed=8, alpha=2.5)
    assert r["flush"] > 0, r


@pytest.mark.parametrize("variant,seed,alpha", [
    ("test_c2_8_4_small_d36", 21, 0.7), ("test_c2_8_4_small_d36", 22, 1.4), ("test_c2_32_8_small_d36", 23, 0.7),
    ("test_c2_16_4_small_d36", 24, 1.4), ("test_c1_fp32_d36", 25, 0.7), ("test_c1_8_d36", 26, 1.4)])
def test_more_traces_on_fresh_library_instances(fixture_tables, variant, seed, alpha):
    """Other seeds and skews (flatter: more evictions; steeper: more promotions) through private copies of the
    compiled reference, each starting from an empty cache."""
    r = _run_pin(variant, fixture_tables, 4000, seed=seed, alpha=alpha, fresh=True)
    assert r["evict"] > 100 and r["stale"] < 200, r


# ---- batch-granular policy vs the sequential restatement ------------------------------------------
def _clone(seq_tier, batch_tier):
    from collections import OrderedDict
    batch_tier.entries = dict(seq_tier.vals)
    batch_tier.lists = [OrderedDict((k, None) for k in b.keys()) for b in seq_tier.lists]
    batch_tier.n_perfect = seq_tier.n_perfect


@pytest.mark.parametrize("layers,caps", [(2, (120, 500, 0)), (2, (300, 300, 0)), (3, (120, 400, 90))])
def test_batch_tiers_at_b1_equal_sequential(layers, caps):
    """From the same pre-state, one sample through BatchTiers == SeqTiers(fifo, py): codes, value
    sources, both tiers' FIFO states, C3 contents -- except requests that take the same-request
    eviction corner (a hit key evicted by an earlier insert of the same request)."""
    p = pkg()
    alt = p.workload.make_alt_keys(SMALL_ROWS) if layers == 3 else None
    seq = tiers.SeqTiers(caps, n_layers=layers, order="fifo", flush="py", alt_keys=alt)
    trace = _trace(2500, seed=11)
    corners = c3_hits = 0
    for i in range(len(trace)):
        bt = tiers.BatchTiers(caps, n_layers=layers, alt_keys=alt)
        _clone(seq.c1, bt.c1)
        _clone(seq.c2, bt.c2)
        if layers == 3:
            bt.c3.vals = {k: list(v) for k, v in seq.c3.vals.items()}
            bt.c3.fifo = type(seq.c3.fifo)(seq.c3.fifo)
        code, val_tier, src, stale, pf = seq.request(trace[i])
        bcode, bval, bst, bsr, bagg = bt.lookup_batch(trace[i].reshape(T, 1))
        if any(stale):
            corners += 1
            continue
        c3_hits += sum(1 for c in code if c == tiers.HIT_C3)
        assert list(bcode[0]) == code, i
        assert list(bval[0]) == val_tier, i
        for t in range(T):
            assert (bst[0, t], bsr[0, t]) == split_key(src[t]), (i, t)
        assert bt.c1.state() == seq.c1.state() and bt.c2.state() == seq.c2.state(), i
        assert bt.c1.n_perfect == seq.c1.n_perfect and bt.c2.n_perfect == seq.c2.n_perfect, i
        assert sorted(bt.c1.evicted) == sorted(seq.c1.evicted) and sorted(bt.c2.evicted) == sorted(seq.c2.evicted), i
        if layers == 3:
            # same mapping and flags; the queue order inside one request's group may differ, because
            # the sequential policy evicts one victim per insert and the batch policy all at the end
            assert bt.c3.vals == seq.c3.vals, i
            assert sorted(bt.c3.fifo) == sorted(seq.c3.fifo), i
    assert corners < len(trace) // 5
    if layers == 3:
        assert c3_hits > 0


def test_batch_tiers_single_layer_equals_batch_evlfu():
    p = pkg()
    tr = p.workload.ZipfTrace(SMALL_ROWS, seed=13)
    a = tiers.BatchTiers((400, 0, 0), n_layers=1)
    b = BatchEvLFU(400)
    for it in range(40):
        idx = tr.batch([64, 5, 1, 33][it % 4])
        code, _vt, st, sr, agg = a.lookup_batch(idx)
        hit, bst, bsr, bagg = b.lookup_batch(idx)
        assert ((code > 0) == hit).all() and (st == bst).all() and (sr == bsr).all() and (agg == bagg).all()
        assert a.c1.evicted == b.evicted and a.c1.flushed == b.flushed and a.c1.state() == b.state()


def test_capacities_follow_reference_constructors():
    assert tiers.capacities(1, 32, 0, 600) == (600, 0, 0)
    assert tiers.capacities(1, 8, 0, 150) == (600, 0, 0)
    assert tiers.capacities(2, 8, 4, 400) == (800, 1600, 0)
    assert tiers.capacities(2, 32, 8, 300) == (150, 2400, 0)        # 8-bit C2 built through EVLFU_8BIT(cap*4): x4 twice
    assert tiers.capacities(2, 32, 16, 300) == (150, 300, 0)
    assert tiers.capacities(2, 16, 8, 200) == (200, 1600, 0)
    assert tiers.capacities(3, 8, 4, 75425, "48-48-4", 36) == (36204 * 4, 36204 * 8, 3017 * 36)
