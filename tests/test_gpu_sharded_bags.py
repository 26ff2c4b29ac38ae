"""Bags on a table-wise sharded cache (evs_shard_lookup_bags, evs_probe_bags / evs_lookup_bags_agg) against the oracle of
tests/sharded_bags_case.py after every batch: pooled rows bit for bit, per-index hit codes, eviction streams, statistics,
and the FIFO state at the end.  Two processes on one GPU for the fused exchange (as tests/test_gpu_sharded.py), and the
"nccl" / "p2p" transports on two GPUs when the box has them."""
import os

import numpy as np
import pytest

from helpers import SMALL_ROWS, pkg
from oracle.evlfu import BatchEvLFU, expand_bags, gather_rows
from sharded_bags_case import make_bags, make_plain, oracle_bags, slice_counts

pytestmark = pytest.mark.gpu

DIM, B, CAP, SLICES = 16, 16, 300, 512          # global batch B, B * 32 slices at most
# bag batches with P = 1, 3, 10, 32 interleaved with plain batches on the same shard; more than four batches, so the
# receive buffers rotate
SCHEDULE = [3, 0, 10, 1, 0, 32, 3, 0, 10, 32, 1, 3]
HIT_ABSENT = 255


def _placement(kind, world):
    p = pkg()
    return p.sharded.balanced_placement(SMALL_ROWS, world) if kind == "balanced" else p.sharded.contiguous_placement(26, world)


def _to_dev(lists):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in lists]


def test_bags_shards_on_one_device_probe_and_agg_in():
    """Without the exchange: several stores on one GPU, evs_probe_bags, the slice counts summed (what the all-reduce does),
    then evs_lookup_bags_agg."""
    import torch
    p = pkg()
    tables = p.workload.make_tables(SMALL_ROWS, DIM)
    for world in (2, 8):
        placement = p.sharded.contiguous_placement(26, world)
        stores = [p.EvStore([tables[t] for t in ids], p.CacheConfig(total_size=CAP * 2 // world, max_batch=SLICES, n_tables_total=26,
                                                                     table_ids=tuple(ids), record_events=True)) for ids in placement]
        oracles = [BatchEvLFU(CAP * 2 // world, n_tables=26) for _ in placement]
        n_ev = 0
        try:
            for k, P in enumerate(x for x in SCHEDULE if x):
                idx_lists, off_lists = make_bags(k, SMALL_ROWS, B, P)
                args = [(_to_dev([off_lists[t] for t in ids]), _to_dev([idx_lists[t] for t in ids])) for ids in placement]
                aggs = [st.probe_bags(o, i, P) for st, (o, i) in zip(stores, args)]
                for a, o, ids in zip(aggs, oracles, placement):       # the probe equals the oracle's local slice counts
                    iv = expand_bags([idx_lists[t] for t in ids], [off_lists[t] for t in ids], B, P)
                    assert np.array_equal(a.cpu().numpy().astype(np.int64), slice_counts(o, ids, iv)), (world, k)
                agg = torch.stack([x.to(torch.int32) for x in aggs]).sum(dim=0).to(torch.uint8)
                want = oracle_bags(oracles, placement, tables, idx_lists, off_lists, B, P)
                for st, (o_dev, i_dev), o, (pooled, codes, _, _) in zip(stores, args, oracles, want):
                    out, hit = st.lookup_bags(o_dev, i_dev, P, agg_in=agg)
                    torch.cuda.synchronize()
                    st.check()
                    assert np.array_equal(out.cpu().numpy(), pooled), (world, k)
                    for h, c in zip(hit, codes):
                        h = h.cpu().numpy()
                        assert not (h == HIT_ABSENT).any() and np.array_equal((h != 0).astype(np.uint8), c), (world, k)
                    ev, fl = st.last_events()
                    assert ev.tolist() == o.evicted and fl.tolist() == o.flushed, (world, k)
                    n_ev += len(o.evicted)
            for st, o in zip(stores, oracles):
                state, n_perfect = st.dump_state()
                assert state == o.state() and n_perfect == o.n_perfect
            assert n_ev > 0
        finally:
            for st in stores:
                st.close()


def _refusals(p, store, sh, ids):
    """Host-side refusals of evs_shard_lookup_bags: nothing reaches the device, so the peers are not waited for."""
    import torch
    bad = []

    def bags(Bq, P):
        lS_o = [torch.arange(Bq, dtype=torch.int64, device="cuda") for _ in ids]
        lS_i = [torch.zeros(Bq, dtype=torch.int64, device="cuda") for _ in ids]
        return lS_o, lS_i, P

    for what, (lS_o, lS_i, P) in (("B*P > batch_max", bags(32, 32)), ("P = 0", bags(B, 0)), ("P = 33", bags(B, 33)),
                                   ("B not a multiple of world", bags(B - 1, 2))):
        try:
            store.shard_lookup_bags(lS_o, lS_i, P)
            bad.append(what)
        except p.EvsError:
            pass
    return bad


def _worker(rank, world, port, q, backend, transport, same_device, kind, env, cross_check):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ.update(env)
    devno = 0 if same_device else rank
    torch.cuda.set_device(devno)
    if backend == "nccl":
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", devno))
    else:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    p = pkg()
    tables = p.workload.make_tables(SMALL_ROWS, DIM)
    placement = _placement(kind, world)
    ids = placement[rank]

    def make():
        cfg = p.CacheConfig(total_size=CAP, max_batch=SLICES, n_tables_total=26, table_ids=tuple(ids), device=devno, record_events=True)
        store = p.EvStore([tables[t] for t in ids], cfg)
        return store, p.sharded.ShardedLookup(store, 26, DIM, rank, world, transport=transport, batch_max=SLICES, placement=placement)

    res, err = {}, None
    stores = []
    try:
        store, sh = make()
        stores.append(store)
        if cross_check:
            # P = 1 with one index per bag against the plain sharded lookup on a second cache: rows, hit codes, state
            store2, sh2 = make()
            stores.append(store2)
            steps = []
            for k in range(10):
                idx = make_plain(k, SMALL_ROWS, B)[ids]
                ly, hit = sh.lookup(torch.from_numpy(np.ascontiguousarray(idx)).cuda())
                ly2, hit2 = sh2.lookup_bags([torch.arange(B, dtype=torch.int64, device="cuda") for _ in ids], _to_dev(list(idx)), 1)
                torch.cuda.synchronize()
                steps.append((ly.cpu().numpy().copy(), hit.cpu().numpy().copy(), ly2.cpu().numpy().copy(),
                              np.stack([h.cpu().numpy() for h in hit2], axis=1), store.last_events(), store2.last_events()))
            res["cross"] = steps
            res["state"] = [store.dump_state(), store2.dump_state()]
        else:
            steps = []
            for k, P in enumerate(SCHEDULE):
                if P:
                    idx_lists, off_lists = make_bags(k, SMALL_ROWS, B, P)
                    ly, hit = sh.lookup_bags(_to_dev([off_lists[t] for t in ids]), _to_dev([idx_lists[t] for t in ids]), P)
                    torch.cuda.synchronize()
                    hit = [h.cpu().numpy().copy() for h in hit]
                else:
                    ly, hit = sh.lookup(torch.from_numpy(np.ascontiguousarray(make_plain(k, SMALL_ROWS, B)[ids])).cuda())
                    torch.cuda.synchronize()
                    hit = hit.cpu().numpy().copy()
                store.check()
                steps.append((ly.cpu().numpy().copy(), hit, store.last_events()))
            res["steps"] = steps
            res["state"] = store.dump_state()
            res["stats"] = store.stats()
            if transport == "p2p":
                res["refusals_missed"] = _refusals(p, store, sh, ids)
        for st in stores:
            st.sync()
    except Exception as e:                               # report instead of hanging the peer
        err = repr(e)
    q.put((rank, res, err))
    dist.barrier()
    for st in stores:
        st.close()
    dist.destroy_process_group()


def _spawn(world, backend, transport, same_device, kind="contiguous", env=None, cross_check=False):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 27600 + (os.getpid() + hash((backend, transport, kind, str(env), cross_check))) % 2000
    procs = [ctx.Process(target=_worker, args=(r, world, port, q, backend, transport, same_device, kind, env or {}, cross_check))
             for r in range(world)]
    for pr in procs:
        pr.start()
    got = {}
    for _ in range(world):
        r, res, err = q.get(timeout=600)
        assert err is None, f"rank {r}: {err}"
        got[r] = res
    for pr in procs:
        pr.join(timeout=60)
        assert pr.exitcode == 0
    return got


def _check(got, world, kind):
    """Replay the schedule on the oracles and compare every rank after every batch."""
    p = pkg()
    tables = p.workload.make_tables(SMALL_ROWS, DIM)
    placement = _placement(kind, world)
    oracles = [BatchEvLFU(CAP, n_tables=26) for _ in range(world)]
    Bl = B // world
    lookups, misses = [0] * world, [0] * world
    n_ev = 0
    for k, P in enumerate(SCHEDULE):
        if P:
            idx_lists, off_lists = make_bags(k, SMALL_ROWS, B, P)
            want = oracle_bags(oracles, placement, tables, idx_lists, off_lists, B, P)
            full = np.empty((B, 26, DIM), dtype=np.float32)
            for r, (ids, (pooled, codes, present, miss)) in enumerate(zip(placement, want)):
                full[:, ids] = pooled
                lookups[r] += present
                misses[r] += miss
                for t, c in enumerate(codes):
                    h = got[r]["steps"][k][1][t]
                    assert not (h == 255).any(), f"batch {k} rank {r}: an index reported as absent"
                    assert np.array_equal((h != 0).astype(np.uint8), c), f"batch {k} rank {r} table {ids[t]}: hit codes"
        else:
            idx = make_plain(k, SMALL_ROWS, B)
            agg = sum(np.array([[(ids[t] << 40 | int(idx[ids[t], s])) in o.entries for t in range(len(ids))]
                                for s in range(B)]).sum(axis=1) for o, ids in zip(oracles, placement))
            full = np.empty((B, 26, DIM), dtype=np.float32)
            for r, (o, ids) in enumerate(zip(oracles, placement)):
                o_hit, s_t, s_r, _ = o.lookup_batch(idx[ids], agg=agg, table_ids=ids)
                full[:, ids] = gather_rows(tables, s_t, s_r)
                lookups[r] += o_hit.size
                misses[r] += int(o_hit.size - o_hit.sum())
                assert np.array_equal(got[r]["steps"][k][1].astype(bool), o_hit), f"batch {k} rank {r}: hit map"
        for r, o in enumerate(oracles):
            assert np.array_equal(got[r]["steps"][k][0], full[r * Bl:(r + 1) * Bl]), f"batch {k} rank {r}: pooled rows"
            ev, fl = got[r]["steps"][k][2]
            assert ev.tolist() == o.evicted and fl.tolist() == o.flushed, f"batch {k} rank {r}: eviction stream"
            n_ev += len(o.evicted)
    for r, o in enumerate(oracles):
        state, n_perfect = got[r]["state"]
        assert state == o.state() and n_perfect == o.n_perfect, f"rank {r}: FIFO state"
        s = got[r]["stats"]
        assert s["lookups"] == lookups[r] and s["misses"] == misses[r], f"rank {r}: statistics"
        assert not got[r].get("refusals_missed"), f"rank {r}: not refused: {got[r]['refusals_missed']}"
    assert n_ev > 0


def test_sharded_bags_p2p_two_processes_on_one_gpu():
    """The fused exchange with contiguous placement: counts by slice, pooled rows into the owners' receive buffers."""
    _check(_spawn(2, "gloo", "p2p", True), 2, "contiguous")


def test_sharded_bags_p2p_one_gpu_two_pass_balanced():
    """The separate probe pass (forced) and a non-contiguous placement: pooled rows land at the global ids' columns."""
    _check(_spawn(2, "gloo", "p2p", True, kind="balanced", env={"EVSTORE_B200_SHARD_TWO_PASS": "1"}), 2, "balanced")


def test_sharded_bags_p_1_equals_plain_sharded_lookup():
    """One index per bag: evs_shard_lookup_bags with P = 1 gives what evs_shard_lookup gives on a second cache."""
    got = _spawn(2, "gloo", "p2p", True, kind="balanced", cross_check=True)
    for r in range(2):
        for k, (ly, hit, ly2, hit2, ev, ev2) in enumerate(got[r]["cross"]):
            assert np.array_equal(ly, ly2), f"batch {k} rank {r}: rows"
            assert np.array_equal(hit, hit2), f"batch {k} rank {r}: hit codes"
            assert ev[0].tolist() == ev2[0].tolist() and ev[1].tolist() == ev2[1].tolist(), f"batch {k} rank {r}: eviction stream"
        assert got[r]["state"][0] == got[r]["state"][1], f"rank {r}: FIFO state"


@pytest.mark.parametrize("transport", ["nccl", "p2p"])
@pytest.mark.parametrize("kind", ["contiguous", "balanced"])
def test_sharded_bags_two_gpus(transport, kind):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    _check(_spawn(2, "nccl", transport, False, kind=kind), 2, kind)
