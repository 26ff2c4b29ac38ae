"""BASELINE configs[0] end to end: the reference's own DLRM_Net (Kaggle architecture, small random tables) was
run on the CPU by tests/golden/make_golden.py; one input batch, the interaction output, the click probabilities
and digests of its weights are in tests/golden/dlrm_forward.npz (helpers.load_dlrm_golden redraws the weights).  ``dlrm_ops.DLRMInference.sequential_forward``
(bottom MLP on cuBLAS next to the cached lookup, our interaction kernel, top MLP) must reproduce them:
fp32 rows from the cache are exact copies, so only GEMM summation order differs -- tolerance 2e-6 absolute on
the probabilities (they lie in 0.29..0.37), 1e-4 / 1e-5 (atol / rtol) on the 367 interaction features."""
import numpy as np
import pytest

from helpers import load_dlrm_golden, pkg

pytestmark = pytest.mark.gpu


def _golden(golden_dir):
    return load_dlrm_golden(golden_dir)


@pytest.mark.parametrize("use_cache,policy", [(True, "evlfu"), (True, "lru"), (False, "evlfu")])
def test_sequential_forward_equals_reference_model(golden_dir, use_cache, policy):
    import torch
    p = pkg()
    g = _golden(golden_dir)
    tables = [np.ascontiguousarray(g[f"emb_{k}"]) for k in range(26)]
    bot = [(g[f"bot_w{i}"], g[f"bot_b{i}"]) for i in range(4)]
    top = [(g[f"top_w{i}"], g[f"top_b{i}"]) for i in range(3)]
    store = p.EvStore(tables, p.CacheConfig(total_size=700, max_batch=128, policy=policy))
    saved = p.dlrm_ops.cache_algo
    p.dlrm_ops.cache_algo = "lru" if policy == "lru" else "cpp_algo"
    try:
        net = p.dlrm_ops.DLRMInference(bot, top, store, use_emb_cache=use_cache)
        X = torch.from_numpy(g["X"]).cuda()
        lS_i = torch.from_numpy(g["lS_i"]).cuda()
        lS_o = torch.arange(128, device="cuda").repeat(26, 1)
        for attempt in range(3):                       # cold cache, then warm: same answer
            Z = net.sequential_forward(X, lS_o, lS_i)
            torch.cuda.synchronize()
            assert tuple(Z.shape) == (128, 1)
            assert np.allclose(Z.cpu().numpy(), g["Z"], rtol=0, atol=2e-6), float(np.abs(Z.cpu().numpy() - g["Z"]).max())
        # the interaction features on their own
        x = net.apply_mlp(X, net.bot, -1)
        ly = p.dlrm_ops.apply_emb_evstore(lS_o, lS_i, use_emb_cache=use_cache, store=store)
        R = p.dlrm_ops.interact_features(x, ly)
        assert np.allclose(R.cpu().numpy(), g["R"], rtol=1e-5, atol=1e-4)
        if use_cache:
            store.sync()
            s = store.stats()
            assert s["hits"][0] > 0 and s["misses"] > 0
        with pytest.raises(ValueError):                  # a cache of the other policy is refused, not silently used
            p.dlrm_ops.cache_algo = "cpp_algo" if policy == "lru" else "lru"
            p.dlrm_ops.apply_emb_evstore(lS_o, lS_i, use_emb_cache=True, store=store)
    finally:
        p.dlrm_ops.cache_algo = saved
        store.close()


@pytest.mark.parametrize("prec,tol_row,tol_z", [(16, 1e-3, 2e-5), (8, 4e-3, 2e-3), (4, 0.25, 6e-2)])
def test_quantised_tier_predictions_within_the_stated_tolerance(golden_dir, prec, tol_row, tol_z):
    """North-star part two: rows served from a quantised tier and the final CTR predictions stay within a stated
    tolerance of the fp32 reference model.  The tolerances are the reference codecs' own resolution -- 16-bit:
    step 2e-5, rows within 1e-3 (the north-star's figure) and probabilities within 2e-5; 8-bit: half a step of
    2/254 = 3.94e-3 on rows, 2e-3 on probabilities; 4-bit (a 15-entry table, evlfu_4.hpp:46): 0.25 / 6e-2 --
    and the CUDA path adds nothing to them: it equals the reference's dequantisers bit for bit, so its
    probabilities equal a CPU forward over the dequantised tables within the GEMM tolerance (2e-6)."""
    import torch
    from helpers import dlrm_forward_cpu
    from oracle import codecs as ocodecs
    p = pkg()
    g = _golden(golden_dir)
    tables = [np.ascontiguousarray(g[f"emb_{k}"]) for k in range(26)]
    dec = [ocodecs.dequantize_rows(ocodecs.quantize_table(t, prec), prec) for t in tables]
    Zq, _ = dlrm_forward_cpu(g, dec)
    bot = [(g[f"bot_w{i}"], g[f"bot_b{i}"]) for i in range(4)]
    top = [(g[f"top_w{i}"], g[f"top_b{i}"]) for i in range(3)]
    store = p.EvStore(tables, p.CacheConfig(main_precision=prec, total_size=700 * prec // 32 + 40, max_batch=128))
    try:
        net = p.dlrm_ops.DLRMInference(bot, top, store)
        X = torch.from_numpy(g["X"]).cuda()
        lS_i = torch.from_numpy(g["lS_i"]).cuda()
        lS_o = torch.arange(128, device="cuda").repeat(26, 1)
        for attempt in range(2):
            Z = net.sequential_forward(X, lS_o, lS_i).cpu().numpy()
            assert float(np.abs(Z - Zq).max()) <= 2e-6
            assert float(np.abs(Z - g["Z"]).max()) <= tol_z
        ly = p.dlrm_ops.apply_emb_evstore(lS_o, lS_i, store=store)
        for k in range(26):
            rows = ly[k].cpu().numpy()
            assert np.array_equal(rows, dec[k][g["lS_i"][k]])                      # the reference's dequantiser, bit for bit
            assert float(np.abs(rows - tables[k][g["lS_i"][k]]).max()) <= tol_row
    finally:
        store.close()


def test_captured_forward_equals_eager_forward(golden_dir):
    """DLRMInference.capture: the whole sequential_forward (bottom MLP branch, the cache's three kernels, interaction, top MLP)
    as ONE CUDA graph.  Replaying it over a stream of batches gives the eager path's probabilities, and the cache goes
    through the same states (hit statistics, eviction counts, final FIFO lists) -- the device numbers the replays itself."""
    import torch
    p = pkg()
    g = _golden(golden_dir)
    tables = [np.ascontiguousarray(g[f"emb_{k}"]) for k in range(26)]
    rows = [t.shape[0] for t in tables]
    bot = [(g[f"bot_w{i}"], g[f"bot_b{i}"]) for i in range(4)]
    top = [(g[f"top_w{i}"], g[f"top_b{i}"]) for i in range(3)]
    B = 128
    trace = p.workload.ZipfTrace(rows, seed=17)
    batches = [trace.batch(B) for _ in range(12)]
    dense = [torch.rand((B, 13), device="cuda", generator=torch.Generator(device="cuda").manual_seed(k)) for k in range(12)]
    out = {}
    for mode in ("eager", "graph"):
        store = p.EvStore(tables, p.CacheConfig(total_size=500, max_batch=B, record_events=True))
        net = p.dlrm_ops.DLRMInference(bot, top, store)
        if mode == "graph":
            net.capture(B)                                   # its warm-up pass looks batch-of-zeros up once, eagerly
        else:
            net.sequential_forward(torch.zeros((B, 13), device="cuda"), None, torch.zeros((26, B), dtype=torch.int64, device="cuda"))
        probs = []
        for k in range(12):
            idx = torch.from_numpy(batches[k]).cuda()
            z = net.replay(dense[k], idx) if mode == "graph" else net.sequential_forward(dense[k], None, idx)
            torch.cuda.synchronize()
            probs.append(z.cpu().numpy().copy())
        store.sync()
        st = store.stats()
        state, n_perfect = store.dump_state()
        out[mode] = (probs, st, state, n_perfect)
        store.close()
    for k in range(12):
        assert np.allclose(out["eager"][0][k], out["graph"][0][k], rtol=0, atol=1e-6), k
    se, sg = out["eager"][1], out["graph"][1]
    assert sg["lookups"] == se["lookups"] and sg["hits"] == se["hits"] and sg["evictions"] == se["evictions"] and sg["batches"] == se["batches"]
    assert se["evictions"][0] > 0
    assert out["eager"][2] == out["graph"][2] and out["eager"][3] == out["graph"][3]
