"""evs_knn (csrc/evs_knn.cuh) against oracle/altkeys.py: the neighbour lists of get_neighbors_GPU.ipynb (11 nearest, entry [0]
dropped) and the alt keys of most_popular_neighbor.ipynb.  Neighbour lists and distances are held to the float64 bound of
tests/test_gpu_knn.py (check_knn, whose module docstring derives it); that file covers every launch configuration."""
import numpy as np
import pytest

from helpers import pkg
from oracle import altkeys
from test_gpu_knn import check_knn

pytestmark = pytest.mark.gpu


def check_lists(x, q, got, got_d, k):
    check_knn(x, x if q is None else q, got, got_d, k)


@pytest.mark.parametrize("n,d,seed", [(1000, 16, 0), (777, 36, 1), (300, 64, 2), (2500, 8, 3), (130, 20, 4)])
def test_knn_every_row(n, d, seed):
    import torch
    p = pkg()
    x = np.random.default_rng(seed).standard_normal((n, d)).astype(np.float32)
    nbr, dist = p.altkeys.knn(torch.from_numpy(x).cuda(), return_dist=True)
    torch.cuda.synchronize()
    check_lists(x, None, nbr.cpu().numpy(), dist.cpu().numpy(), 10)


def test_knn_few_queries_split_database_and_small_k():
    import torch
    p = pkg()
    rng = np.random.default_rng(7)
    x = rng.standard_normal((20000, 16)).astype(np.float32)
    q = x[rng.integers(0, 20000, size=70)] + rng.standard_normal((70, 16)).astype(np.float32) * 0.01
    nbr, dist = p.altkeys.knn(torch.from_numpy(x).cuda(), torch.from_numpy(q).cuda(), k=4, return_dist=True)
    torch.cuda.synchronize()
    check_lists(x, q, nbr.cpu().numpy(), dist.cpu().numpy(), 4)


def test_knn_fewer_rows_than_neighbours_and_duplicates():
    import torch
    p = pkg()
    x = np.random.default_rng(9).standard_normal((6, 16)).astype(np.float32)
    x[4] = x[1]                                          # two identical rows: entry [0] is the lower index of the pair
    nbr = p.altkeys.knn(torch.from_numpy(x).cuda()).cpu().numpy()
    want, _ = altkeys.knn_bruteforce(x, k=10)
    assert (nbr == want).all() and (nbr[:, 5:] == -1).all()
    assert nbr[1, 0] == 4 and nbr[4, 0] == 4            # row 4's own list starts with itself once row 1 was dropped


def test_alt_keys_most_popular_neighbour():
    p = pkg()
    rng = np.random.default_rng(11)
    tables = [rng.standard_normal((r, 16)).astype(np.float32) * 0.1 for r in (400, 30, 7, 900, 3)]
    freq = [rng.integers(0, 50, size=t.shape[0]).astype(np.uint32) for t in tables]
    for f in (None, freq):
        got = p.altkeys.generate_alt_keys(tables, f)
        want = altkeys.alt_keys(tables, f)
        for t in range(len(tables)):
            assert got[t].dtype == np.uint32 and np.array_equal(got[t], want[t]), t


def test_generated_alt_keys_serve_a_three_layer_cache():
    """The generated tables are in the format the C3 tier reads: a 3-layer EvStore built over them runs, and the double misses
    it answers from an alternative row (hit code 3) are the ones its counter reports."""
    import torch
    p = pkg()
    rows = [300, 40, 900, 25, 600, 12]
    tables = p.workload.make_tables(rows, 16)
    alt = p.altkeys.generate_alt_keys(tables)
    cfg = p.CacheConfig(n_layers=3, main_precision=8, secondary_precision=4, total_size=60, size_proportion="40-40-20", max_batch=64)
    store = p.EvStore(tables, cfg, alt_keys=alt)
    trace = p.workload.ZipfTrace(rows, seed=2)
    c3 = 0
    for _ in range(40):
        idx = trace.batch(64)
        out, hit = store.lookup(torch.from_numpy(idx).cuda())
        torch.cuda.synchronize()
        c3 += int((hit == 3).sum())
    store.sync()
    assert store.stats()["c3_hits"] == c3
    store.close()
