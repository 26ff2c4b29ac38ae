"""Alternative keys for C3 (aprx_embedding): the reference's offline generator
(script/approximate_embedding/phase2_similarity_analysis/get_neighbors_GPU.ipynb + most_popular_neighbor.ipynb) on the GPU.

``get_neighbors_GPU.ipynb`` stacks the rows of all 26 tables into one matrix, asks cuML for the 11 nearest rows (Euclidean,
brute force) of every row and drops entry [0] (the row itself); ``most_popular_neighbor.ipynb`` keeps, of those 10, the one
that occurs most often in the workload (first maximum; absent rows count 0).  The result per table is the alt-key array the
C3 tier reads: ``alt_row * 100 + alt_table`` with tables numbered from 1 (convert_altkeys_to_binary.py:50).

Here both steps are ``evs_knn`` (csrc/evs_knn.cuh): one fused tensor-core kernel (3xTF32 ``mma.sync`` distances: every
operand split into hi, rounded to TF32, and the exact remainder lo, which the tensor core truncates; fp32 accurate, with
the top-11 selection in registers) and a merge kernel that also makes the popularity pick.  A row with a NaN or ±Inf
element (or one whose squared norm overflows fp32) is never a neighbour or an alt key; such a row's own neighbours are
all -1 and its alt key is 0.
"""
from __future__ import annotations

import numpy as np

from . import _native

MAX_K = 10
N_NEIGHBORS = 10                      # n_neighbors = 11 minus the row itself


def knn(x, q=None, k: int = N_NEIGHBORS, return_dist: bool = False, stream=None):
    """x: fp32 CUDA tensor [n, d] (the database); q: fp32 CUDA tensor [nq, d] (default: x itself, i.e. every row's
    neighbours).  Returns int64 [nq, k] row ids of x, nearest first with the nearest of all (q itself when q is x) dropped;
    with ``return_dist`` also the fp32 squared distances."""
    import torch
    lib = _native.load_library()
    assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous() and x.dim() == 2
    q = x if q is None else q
    assert q.is_cuda and q.dtype == torch.float32 and q.is_contiguous() and q.shape[1] == x.shape[1]
    nq = q.shape[0]
    nbr = torch.empty((nq, k), dtype=torch.int64, device=x.device)
    dist = torch.empty((nq, k), dtype=torch.float32, device=x.device) if return_dist else None
    st = stream if stream is not None else (torch.cuda.current_stream(x.device).cuda_stream or 1)
    with torch.cuda.device(x.device):
        rc = lib.evs_knn(x.data_ptr(), x.shape[0], q.data_ptr(), nq, x.shape[1], k, nbr.data_ptr(),
                         dist.data_ptr() if dist is not None else None, None, None, 0, None, st)
    _native.check(rc, "evs_knn")
    return (nbr, dist) if return_dist else nbr


def generate_alt_keys(tables, freq=None, k: int = N_NEIGHBORS, device: int = 0, query_chunk: int = 1 << 22):
    """tables: list of fp32 [rows_t, d] arrays (numpy or torch; the trained embedding tables).  freq: optional list of
    per-table request counts (uint32 [rows_t]; ``rankedWorkload.csv`` of the reference).  Returns one uint32 numpy array per
    table: alt_key[row] = alt_row * 100 + alt_table (1-based), the format ``EvStore(..., alt_keys=...)`` takes."""
    import torch
    lib = _native.load_library()
    dev = torch.device("cuda", device)
    rows = [int(t.shape[0]) for t in tables]
    off = np.concatenate([[0], np.cumsum(rows)]).astype(np.int64)
    n = int(off[-1])
    with torch.cuda.device(dev):
        x = torch.cat([torch.as_tensor(np.ascontiguousarray(t) if isinstance(t, np.ndarray) else t, dtype=torch.float32).to(dev) for t in tables]).contiguous()
        off_dev = torch.from_numpy(off).to(dev)
        f_dev = None
        if freq is not None:
            f_dev = torch.cat([torch.as_tensor(np.asarray(f).astype(np.int64)).to(dev) for f in freq]).to(torch.int32).contiguous()
            assert f_dev.numel() == n
        alt = torch.empty((n,), dtype=torch.int32, device=dev)
        st = torch.cuda.current_stream(dev).cuda_stream or 1
        for q0 in range(0, n, query_chunk):
            q1 = min(n, q0 + query_chunk)
            rc = lib.evs_knn(x.data_ptr(), n, x[q0:q1].data_ptr(), q1 - q0, x.shape[1], k, None, None,
                             f_dev.data_ptr() if f_dev is not None else None, off_dev.data_ptr(), len(rows), alt[q0:q1].data_ptr(), st)
            _native.check(rc, "evs_knn")
        out = alt.cpu().numpy().view(np.uint32)
    return [np.ascontiguousarray(out[off[t]:off[t + 1]]) for t in range(len(rows))]
