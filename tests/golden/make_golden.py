#!/usr/bin/env python
"""Generate golden vectors by running the UNMODIFIED reference code.

Needs a checkout of the original project, named by EVSTORE_REFERENCE; the outputs
(``tests/golden/*.npz``) are committed, this script is how they were made.

  EVSTORE_REFERENCE=<checkout> python tests/golden/make_golden.py

1. ``evlfu_c1_*.npz``   -- /root/reference/cache_algo/EvLFU_C1.py driven one request
   at a time on synthetic Zipf traces with a stub ``storage_manager`` whose rows
   encode (table,row), so the returned tensors reveal which backing row answered.
   Per request: hit vector, evicted keys, flushed keys, answering (table,row);
   plus the final per-bucket FIFO lists.
2. ``codecs.npz``       -- the reference's offline quantisers / dequantisers
   (script/reduce_precision.py) evaluated on a fixed vector of floats.
3. ``lru_*.npz``        -- /root/reference/cache_algo/LRU.py (the comparison policy) the same way:
   per request hit vector and evicted keys, plus the final recency order.
6. ``lfu_*.npz``        -- /root/reference/cache_algo/LFU.py: per request hit vector and the set of evicted keys,
   plus the final frequency lists and least_freq.
5. ``dlrm_forward.npz`` -- the reference's DLRM_Net (BASELINE configs[0] architecture, small tables) run on the CPU:
   one input batch, interaction output, click probabilities and the SHA-256 of every weight / table array
   (tests/helpers.py load_dlrm_golden redraws them from the seed).
4. ``formats/``         -- files written by the reference's own writers: the big-endian alt-key binary
   (script/convert_altkeys_to_binary.py) from ``altkeys.txt``, and ``training_config.txt`` (evstore_utils.py).
"""
import os
import sys
import types

import numpy as np

REF = os.environ.get("EVSTORE_REFERENCE", "")
HERE = os.path.dirname(os.path.abspath(__file__))
T = 26
DIM = 36                     # the reference's hard-coded EV_DIMENSION
KEY_SHIFT = 40


def zipf_trace(rng, rows, n_req, alpha=1.05):
    """[n_req, T] int64: per table, rank ~ r^-alpha mapped through a fixed permutation."""
    out = np.empty((n_req, T), dtype=np.int64)
    for t in range(T):
        n = rows[t]
        w = np.arange(1, n + 1, dtype=np.float64) ** (-alpha)
        cdf = np.cumsum(w) / w.sum()
        ranks = np.searchsorted(cdf, rng.random(n_req), side="left")
        perm = np.random.default_rng(7 + t).permutation(n)
        out[:, t] = perm[np.minimum(ranks, n - 1)]
    return out


class LogList(list):
    """list that records pop(0) -- the only way EvLFU_C1 removes victims (:40,:55)."""

    def __init__(self, events, bucket):
        super().__init__()
        self.events = events
        self.bucket = bucket

    def pop(self, i=-1):
        k = super().pop(i)
        self.events.append(("pop", self.bucket, k))
        return k


def str_key_to_int(k):
    t, r = k.split("-")
    return ((int(t) - 1) << KEY_SHIFT) | int(r)


def run_reference_evlfu(trace, cap, approx_thres):
    # stub storage_manager: row value = [table0, row, 0.5, ...] (exact in fp32)
    sm = types.ModuleType("storage_manager")

    def get_val(table_id, row_id):
        v = [0.5] * DIM
        v[0] = float(table_id - 1)
        v[1] = float(row_id)
        return v

    sm.get_val_from_storage = get_val
    sm.get_arr_val_from_storage = lambda keys: [get_val(t, r) for t, r in keys]
    sys.modules["storage_manager"] = sm
    sys.path.insert(0, os.path.join(REF, "cache_algo"))
    sys.modules.pop("EvLFU_C1", None)
    import EvLFU_C1 as ref  # noqa: the reference module itself

    ref.init(cap)
    events = []
    for b in range(T + 1):
        ref.lists_C1[b] = LogList(events, b)

    def ref_print(*a, **k):           # the reference announces a flush with print (:37)
        if a and a[0] == "flushing!":
            events.append(("flush",))

    ref.print = ref_print             # module-global lookup wins over the builtin
    nf = int(0.3 * cap) + 1           # :39 -- pops that follow the announcement are the flush
    n = len(trace)
    hits = np.zeros((n, T), dtype=bool)
    src_t = np.zeros((n, T), dtype=np.int32)
    src_r = np.zeros((n, T), dtype=np.int64)
    ev_keys, ev_off = [], [0]
    fl_keys, fl_off = [], [0]
    for i in range(n):
        events.clear()
        hit, embs = ref.request_to_ev_lfu([int(x) for x in trace[i]], False, approx_thres, DIM)
        hits[i] = hit
        for t in range(T):
            v = embs[t][0]
            tt, rr = float(v[0]), float(v[1])
            if v[2] == 0.5 and tt == int(tt) and 0 <= tt < T:
                src_t[i, t], src_r[i, t] = int(tt), int(rr)
            else:                       # the reference's random fill (:104-107)
                src_t[i, t], src_r[i, t] = -1, 0
        flush_left = 0
        for e in events:
            if e[0] == "flush":
                flush_left = nf
            elif flush_left > 0:
                assert e[1] == T
                fl_keys.append(str_key_to_int(e[2]))
                flush_left -= 1
            else:
                ev_keys.append(str_key_to_int(e[2]))
        ev_off.append(len(ev_keys))
        fl_off.append(len(fl_keys))
    state_keys, state_off = [], [0]
    for b in range(T + 1):
        state_keys.extend(str_key_to_int(k) for k in ref.lists_C1[b])
        state_off.append(len(state_keys))
    return dict(hits=np.packbits(hits, axis=1), src_t=src_t.astype(np.int8), src_r=src_r.astype(np.int32),
                ev_keys=np.array(ev_keys, dtype=np.int64), ev_off=np.array(ev_off, dtype=np.int32),
                fl_keys=np.array(fl_keys, dtype=np.int64), fl_off=np.array(fl_off, dtype=np.int32),
                state_keys=np.array(state_keys, dtype=np.int64), state_off=np.array(state_off, dtype=np.int32),
                n_perfect=np.int64(ref.n_perfect_item_C1), min_bucket=np.int64(ref.min_C1))


def golden_evlfu():
    cases = [
        # name, rows per table, n_req, cap, approx_thres, seed
        ("evlfu_c1_small", [40 + 13 * t for t in range(T)], 2500, 300, -1, 42),
        ("evlfu_c1_skew", [3, 5, 4000, 2500, 7, 4, 60, 9, 3, 300, 50, 3500, 40, 4, 80, 3000,
                           5, 45, 30, 4, 3800, 6, 5, 600, 11, 400], 4000, 1500, -1, 43),
        ("evlfu_c1_flush", [4 + (t % 3) for t in range(T)], 3000, 110, -1, 44),   # tiny tables -> perfect hits -> flushes
        ("evlfu_c1_approx", [40 + 13 * t for t in range(T)], 2000, 400, 20, 45),
    ]
    for name, rows, n_req, cap, thres, seed in cases:
        rng = np.random.default_rng(seed)
        trace = zipf_trace(rng, rows, n_req)
        g = run_reference_evlfu(trace, cap, thres)
        np.savez_compressed(os.path.join(HERE, name + ".npz"), trace=trace.astype(np.int32),
                            rows=np.array(rows, dtype=np.int64), cap=np.int64(cap),
                            approx_thres=np.int64(thres), **g)
        print(name, "requests", n_req, "evictions", len(g["ev_keys"]), "flushed", len(g["fl_keys"]),
              "hit rate %.3f" % np.unpackbits(g["hits"], axis=1)[:, :T].mean())


def golden_codecs():
    sys.path.insert(0, os.path.join(REF, "script"))
    sys.modules.pop("reduce_precision", None)
    import reduce_precision as rp  # the reference's quantisers

    rng = np.random.default_rng(99)
    x = np.concatenate([
        rng.uniform(-0.65, 0.65, 3000), rng.uniform(-1.0, 1.0, 1000), rng.normal(0, 0.01, 1000),
        np.array([0.0, -0.0, 0.65, -0.65, 0.6501, -0.6501, 1.0, -1.0, 0.25, -0.25, 0.8, -0.8, 0.6, 0.4,
                  0.015, 0.00025, -0.015, -0.00025, 1e-7, -1e-7, 0.999, -0.999]),
    ]).astype(np.float32)
    # the reference applies the lambdas to a float32 pandas column under NumPy 1.x, where
    # np.float32 (op) python-float promotes to float64; feed python floats to get that.
    xs = [float(v) for v in x]
    q16 = np.array([rp.convert_ev_float_to_ushort(v) for v in xs], dtype=np.int64)
    d16 = np.array([rp.convert_ushort_to_evfloat(int(v)) for v in q16], dtype=np.float64)
    q8 = np.array([round(((v + 1) / 2) * 254) for v in xs], dtype=np.int64)          # :270
    d8 = np.array([round(((int(v) / 254) * 2) - 1, 3) for v in q8], dtype=np.float64)  # :283
    q4 = np.array([rp.convert_to_4bit_int_posit(v) for v in xs], dtype=np.int64)
    d4 = np.array([rp.convert_from_4bit_int_posit(int(min(v, 14))) for v in q4], dtype=np.float64)
    np.savez_compressed(os.path.join(HERE, "codecs.npz"), x=x, q16=q16, d16=d16, q8=q8, d8=d8, q4=q4, d4=d4)
    print("codecs", len(x), "values; q16 max", q16.max(), "q4 range", q4.min(), q4.max())


def run_reference_lru(trace, cap):
    """/root/reference/cache_algo/LRU.py driven one request at a time; the module's OrderedDict is
    replaced by a subclass that logs popitem (the only way LRU.py evicts, :19)."""
    import collections
    sm = types.ModuleType("storage_manager")
    sm.get_val_from_storage = lambda table_id, row_id: [float(table_id - 1), float(row_id)] + [0.5] * (DIM - 2)
    sys.modules["storage_manager"] = sm
    sys.path.insert(0, os.path.join(REF, "cache_algo"))
    sys.modules.pop("LRU", None)
    import LRU as ref  # noqa: the reference module itself

    events = []

    class LogOD(collections.OrderedDict):
        def popitem(self, last=True):
            k, v = super().popitem(last)
            events.append(k)
            return k, v

    ref.LRUCache = LogOD()
    ref.init(cap)
    n = len(trace)
    hits = np.zeros((n, T), dtype=bool)
    ev_keys, ev_off = [], [0]
    for i in range(n):
        events.clear()
        hit, embs = ref.request_to_lru([int(x) for x in trace[i]], False)
        hits[i] = hit
        for t in range(T):                       # the value returned is the row of the requested key
            v = embs[t][0]
            assert int(v[0]) == t and int(v[1]) == int(trace[i, t])
        ev_keys.extend(str_key_to_int(k) for k in events)
        ev_off.append(len(ev_keys))
    state = [str_key_to_int(k) for k in ref.LRUCache.keys()]
    return dict(hits=np.packbits(hits, axis=1), ev_keys=np.array(ev_keys, dtype=np.int64),
                ev_off=np.array(ev_off, dtype=np.int32), state_keys=np.array(state, dtype=np.int64))


def golden_lru():
    cases = [
        ("lru_small", [40 + 13 * t for t in range(T)], 2500, 300, 52),
        ("lru_skew", [3, 5, 4000, 2500, 7, 4, 60, 9, 3, 300, 50, 3500, 40, 4, 80, 3000,
                      5, 45, 30, 4, 3800, 6, 5, 600, 11, 400], 4000, 1500, 53),
    ]
    for name, rows, n_req, cap, seed in cases:
        rng = np.random.default_rng(seed)
        trace = zipf_trace(rng, rows, n_req)
        g = run_reference_lru(trace, cap)
        np.savez_compressed(os.path.join(HERE, name + ".npz"), trace=trace.astype(np.int32),
                            rows=np.array(rows, dtype=np.int64), cap=np.int64(cap), **g)
        print(name, "requests", n_req, "evictions", len(g["ev_keys"]),
              "hit rate %.3f" % np.unpackbits(g["hits"], axis=1)[:, :T].mean())


def run_reference_lfu(trace, cap):
    """/root/reference/cache_algo/LFU.py driven one request at a time; evictions are read off node_for_key
    (the keys that disappeared during the request, in the order of the frequency lists they left)."""
    sm = types.ModuleType("storage_manager")
    sm.get_val_from_storage = lambda table_id, row_id: [float(table_id - 1), float(row_id)] + [0.5] * (DIM - 2)
    sys.modules["storage_manager"] = sm
    sys.path.insert(0, os.path.join(REF, "cache_algo"))
    sys.modules.pop("LFU", None)
    import LFU as ref  # noqa: the reference module itself

    ref.init(cap)
    n = len(trace)
    hits = np.zeros((n, T), dtype=bool)
    ev_keys, ev_off = [], [0]
    for i in range(n):
        before = list(ref.node_for_key.keys())
        hit, _embs = ref.request_to_lfu([int(x) for x in trace[i]], False)
        hits[i] = hit
        after = ref.node_for_key
        gone = [k for k in before if k not in after]        # (a key evicted and re-inserted by the same request stays)
        ev_keys.extend(sorted(str_key_to_int(k) for k in gone))
        ev_off.append(len(ev_keys))
    state_keys, state_off = [], [0]
    for f in range(1, len(ref.node_for_freq)):
        state_keys.extend(str_key_to_int(k) for k in ref.node_for_freq[f])
        state_off.append(len(state_keys))
    return dict(hits=np.packbits(hits, axis=1), ev_keys=np.array(ev_keys, dtype=np.int64), ev_off=np.array(ev_off, dtype=np.int32),
                state_keys=np.array(state_keys, dtype=np.int64), state_off=np.array(state_off, dtype=np.int32),
                least_freq=np.int64(ref.least_freq))


def golden_lfu():
    cases = [
        ("lfu_small", [40 + 13 * t for t in range(T)], 2500, 300, 62),
        ("lfu_skew", [3, 5, 4000, 2500, 7, 4, 60, 9, 3, 300, 50, 3500, 40, 4, 80, 3000,
                      5, 45, 30, 4, 3800, 6, 5, 600, 11, 400], 3000, 1500, 63),
    ]
    for name, rows, n_req, cap, seed in cases:
        rng = np.random.default_rng(seed)
        trace = zipf_trace(rng, rows, n_req)
        g = run_reference_lfu(trace, cap)
        np.savez_compressed(os.path.join(HERE, name + ".npz"), trace=trace.astype(np.int32),
                            rows=np.array(rows, dtype=np.int64), cap=np.int64(cap), **g)
        print(name, "requests", n_req, "evictions", len(g["ev_keys"]),
              "hit rate %.3f" % np.unpackbits(g["hits"], axis=1)[:, :T].mean(), "max freq", len(g["state_off"]) - 1)


def golden_cdf():
    """calculate_and_write_cdf (dlrm_s_pytorch_C1_C2_C3.py:291-319) executed from the reference file itself (the
    module cannot be imported: it needs the Cython EvLFU build) on seeded request start times."""
    import ast
    import subprocess
    from pathlib import Path
    import pandas as pd
    path = os.path.join(REF, "dlrm_s_pytorch_C1_C2_C3.py")
    tree = ast.parse(open(path).read())
    fn = next(n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "calculate_and_write_cdf")
    ns = dict(Path=Path, pd=pd, os=os, subprocess=subprocess)
    exec(compile(ast.Module(body=[fn], type_ignores=[]), path, "exec"), ns)
    rng = np.random.default_rng(321)
    t = np.concatenate([[100.0], 100.0 + np.cumsum(rng.gamma(2.0, 0.0004, size=5003))])
    out = os.path.join(HERE, "formats")
    cwd = os.getcwd()
    os.chdir("/tmp")                       # the function shells out to ./script/plot_cdf.py; let that fail quietly
    try:
        ns["calculate_and_write_cdf"](out, "evlfu_golden", [float(x) for x in t])
    finally:
        os.chdir(cwd)
    np.save(os.path.join(out, "cdf_time_start.npy"), t)
    print("cdf:", sum(1 for _ in open(os.path.join(out, "evlfu_golden-cdf.csv"))), "lines")


def golden_formats():
    """On-disk formats written by the reference's own code: the alt-key binary
    (script/convert_altkeys_to_binary.py:27-57) and training_config.txt (evstore_utils.py:31-41)."""
    out = os.path.join(HERE, "formats")
    os.makedirs(out, exist_ok=True)
    rng = np.random.default_rng(123)
    lines = [f"{int(rng.integers(1, 27))}-{int(rng.integers(0, 10131227))}" for _ in range(200)]
    lines += ["1-0", "26-10131226", "3-42949671"]            # smallest key, a big row, near the uint32 limit
    txt = os.path.join(out, "altkeys.txt")
    with open(txt, "w") as f:
        f.write("\n".join(lines) + "\n")
    sys.path.insert(0, os.path.join(REF, "script"))
    sys.modules.pop("convert_altkeys_to_binary", None)
    import convert_altkeys_to_binary as cab  # the reference's converter
    cab.convert_altkeys_to_binary(txt, os.path.join(out, "altkeys.bin"))
    sys.path.insert(0, REF)
    import evstore_utils as eu  # the reference's training-config writer
    ln_emb = np.array([1460, 583, 10131227, 2202608, 305, 24, 12517, 633, 3, 93145, 5683, 8351593, 3194, 27, 14992,
                       5461306, 10, 5652, 2173, 4, 7046547, 18, 15, 286181, 105, 142572])
    eu.store_training_config(os.path.join(out, "training_config.txt"), {i: i for i in range(26)}, 306969, 3274, ln_emb, 13)
    print("formats:", os.listdir(out))


def golden_dlrm():
    """BASELINE configs[0]: the reference's DLRM_Net (dlrm_s_pytorch.py:206-613) itself, Kaggle architecture
    (13 dense, 26 tables, dim 16, bot 13-512-256-64-16, top 367-512-256-1, dot interaction), small random
    tables, one batch of 128 through sequential_forward on the CPU.  Saved: every weight, the inputs, the
    click probabilities -- the end-to-end known answer for bottom MLP -> lookup -> interaction -> top MLP."""
    import hashlib

    import torch
    sys.path.insert(0, REF)
    sys.path.insert(0, os.path.join(REF, "script"))
    import dlrm_s_pytorch as ref  # the reference model
    np.random.seed(777)
    torch.manual_seed(777)
    rows = [50, 7, 400, 300, 9, 4, 60, 12, 3, 120, 30, 350, 40, 5, 45, 280, 4, 33, 21, 4, 390, 6, 5, 90, 11, 70]
    m_spa, B = 16, 128
    ln_bot = np.array([13, 512, 256, 64, m_spa])
    ln_top = np.array([m_spa + 27 * 26 // 2, 512, 256, 1])
    net = ref.DLRM_Net(m_spa, np.array(rows), ln_bot, ln_top, arch_interaction_op="dot", arch_interaction_itself=False,
                       sigmoid_bot=-1, sigmoid_top=ln_top.size - 2, sync_dense_params=True, loss_threshold=0.0, ndevices=-1)
    net.eval()
    rng = np.random.default_rng(778)
    X = torch.from_numpy(rng.random((B, 13), dtype=np.float32))
    lS_i = torch.from_numpy(np.stack([rng.integers(0, r, size=B) for r in rows]).astype(np.int64))
    lS_o = torch.arange(B, dtype=torch.int64).repeat(len(rows), 1)
    with torch.no_grad():
        Z = net.sequential_forward(X, lS_o, lS_i)
        x = net.apply_mlp(X, net.bot_l)
        ly = net.apply_emb(lS_o, lS_i, net.emb_l, net.v_W_l)
        R = net.interact_features(x, ly)
    out = dict(rows=np.array(rows), X=X.numpy(), lS_i=lS_i.numpy(), Z=Z.numpy(), R=R.numpy(), seed=np.array(777))
    # the weights and tables are ~2 MB of random floats: store their digests; tests/helpers.load_dlrm_golden redraws them
    arrays = {f"emb_{k}": e.weight for k, e in enumerate(net.emb_l)}
    for name, mlp in (("bot", net.bot_l), ("top", net.top_l)):
        lin = [l for l in mlp if isinstance(l, torch.nn.Linear)]
        for i, l in enumerate(lin):
            arrays[f"{name}_w{i}"], arrays[f"{name}_b{i}"] = l.weight, l.bias
    for k, a in arrays.items():
        digest = hashlib.sha256(np.ascontiguousarray(a.detach().numpy()).tobytes()).digest()
        out["sha256_" + k] = np.frombuffer(digest, dtype=np.uint8)
    np.savez_compressed(os.path.join(HERE, "dlrm_forward.npz"), **out)
    print("dlrm_forward: Z", Z.shape, float(Z.min()), float(Z.max()), "R", R.shape)


if __name__ == "__main__":
    which = sys.argv[1:] or ["evlfu", "codecs", "lru", "formats", "dlrm", "lfu", "cdf"]
    if "dlrm" in which:
        golden_dlrm()
    if "lfu" in which:
        golden_lfu()
    if "cdf" in which:
        golden_cdf()
    if "formats" in which:
        golden_formats()
    if "evlfu" in which:
        golden_evlfu()
    if "codecs" in which:
        golden_codecs()
    if "lru" in which:
        golden_lru()
