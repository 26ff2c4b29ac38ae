"""Host-side handle of the GPU cache: the runtime-configured counterpart of the reference's
mixed_precs_caching/cache_manager.cpp (whose configuration is compile-time #defines).

``EvStore`` owns one evs_handle (include/evstore_b200.h).  Device tensors go straight to
``evs_lookup_batch``; host arrays go through ``evs_lookup_batch_host``.  There is no CPU
fallback: construction raises when the CUDA library or a CUDA device is missing.
"""
from __future__ import annotations

import ctypes as C
import struct
from dataclasses import dataclass, field

import numpy as np

from . import _native
from .codecs import encode_table, row_bytes


@dataclass
class CacheConfig:
    """Mirrors cache_manager.cpp:13-20 (+ EV_DIMENSION / N_EV_TABLE)."""
    n_layers: int = 1                 # N_CACHING_LAYER
    main_precision: int = 32          # MAIN_PRECISION
    secondary_precision: int = 0      # SECONDARY_PRECISION
    total_size: int = 75425           # TOTAL_SIZE (fp32-row units)
    size_proportion: str = ""         # SIZE_PROPORTION "c1-c2-c3"
    max_batch: int = 2048
    approx_emb_thres: int = -1        # EvLFU_C1.request_to_ev_lfu(approx_emb_thres)
    device: int = 0
    n_tables_total: int = 0           # agg_hit range; 0 = n_tables
    table_base: int = 0
    table_ids: tuple = ()             # global ids of the local tables (non-contiguous placement); () = table_base + t
    store_in_hbm: bool = False
    record_events: bool = False
    flush_rate: float = 0.0
    perfect_item_cap: float = 0.0
    high_agghit_threshold: int = 0
    policy: str = "evlfu"             # "evlfu" (EvLFU_C1.py / mixed_precs_caching), "lru" (cache_algo/LRU.py) or "lfu" (cache_algo/LFU.py); the last two: one layer
    extra: dict = field(default_factory=dict)

    def proportions(self):
        if not self.size_proportion:
            return 0, 0, 0
        a, b, c = (int(x) for x in self.size_proportion.split("-"))
        return a, b, c


def _ptr_array(arrays):
    arr = (C.c_void_p * len(arrays))()
    for i, a in enumerate(arrays):
        arr[i] = a.ctypes.data
    return arr


CUDA_STREAM_LEGACY = 1     # cudaStreamLegacy: the C-ABI treats a NULL stream as "the handle's own stream"


def _stream_handle(stream, device):
    """The cudaStream_t the work is ordered on: an explicit handle, else torch's current stream."""
    if stream is not None:
        return stream
    import torch
    return torch.cuda.current_stream(device).cuda_stream or CUDA_STREAM_LEGACY


STATE_MAGIC = b"EVSSTATE"
STATE_VERSION = 1
STATE_HEADER = struct.Struct("<8sIIQ8i3Q32i32q")         # include/evstore_b200.h: the snapshot header, 464 bytes


def state_info(blob) -> dict:
    """Header and section sizes of a snapshot from ``EvStore.save_state`` (no GPU): policy, n_layers, n_tables_total,
    table_ids, rows, dim, precisions, capacities, and per tier n_perfect and the keys per bucket, C3's size and window
    length.  Raises ValueError for a truncated or foreign blob."""
    b = memoryview(np.ascontiguousarray(np.frombuffer(blob, dtype=np.uint8) if isinstance(blob, (bytes, bytearray)) else blob,
                                        dtype=np.uint8)).cast("B")
    if len(b) < STATE_HEADER.size:
        raise ValueError(f"not a snapshot: {len(b)} bytes, shorter than the {STATE_HEADER.size}-byte header")
    f = STATE_HEADER.unpack_from(b, 0)
    magic, version, hdr, total = f[0], f[1], f[2], f[3]
    if magic != STATE_MAGIC:
        raise ValueError("not a snapshot (bad magic)")
    if version != STATE_VERSION or hdr != STATE_HEADER.size:
        raise ValueError(f"unsupported snapshot version {version}")
    if total != len(b):
        raise ValueError(f"snapshot of {len(b)} bytes, its header says {total}")
    policy, n_layers, t_total, n_tables, dim, mp, sp, nb = f[4:12]
    caps, c3_cap = list(f[12:14]), f[14]
    ids, rows = list(f[15:15 + 32])[:n_tables], list(f[47:47 + 32])[:n_tables]
    if not 1 <= n_layers <= 3 or not 1 <= n_tables <= 32 or not 2 <= nb <= 32:
        raise ValueError("snapshot header out of range")
    w = np.frombuffer(b, dtype="<u8", offset=STATE_HEADER.size) if (len(b) - STATE_HEADER.size) % 8 == 0 else None
    if w is None:
        raise ValueError("the snapshot body is not a whole number of 8-byte words")
    o, tiers = 0, []
    for _ in range(2 if n_layers >= 2 else 1):
        if o + 1 + nb > len(w):
            raise ValueError("truncated snapshot")
        counts = [int(x) for x in w[o + 1:o + 1 + nb]]
        tiers.append({"n_perfect": int(w[o]), "counts": counts})
        o += 1 + nb + sum(counts)
    c3 = None
    if n_layers == 3 and c3_cap > 0:
        if o + 2 > len(w):
            raise ValueError("truncated snapshot")
        c3 = {"size": int(w[o]), "window": int(w[o + 1])}
        o += 2 + c3["window"] + 2 * c3["size"]
    if o != len(w):
        raise ValueError(f"snapshot body of {len(w)} words, its sections need {o}")
    return {"version": version, "bytes": total, "policy": ("evlfu", "lru", "lfu")[policy] if 0 <= policy <= 2 else policy,
            "n_layers": n_layers, "n_tables_total": t_total, "table_ids": ids, "rows": rows, "dim": dim,
            "main_precision": mp, "secondary_precision": sp, "capacity": caps[:len(tiers)], "c3_capacity": c3_cap,
            "tiers": tiers, "c3": c3}


class _DevArray:
    """A device buffer owned by the library, exposed through __cuda_array_interface__ (zero copy)."""

    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<f4", "data": (int(ptr), False), "version": 2}


def _tensor_from_ptr(ptr, shape, device):
    import torch
    return torch.as_tensor(_DevArray(ptr, shape), device=device)


def host_rows(shape, dtype=np.float32, device: int = 0) -> np.ndarray:
    """An uninitialised host array for backing rows from ``evs_host_alloc``: host memory the device maps with large
    pages, so that the zero-copy miss fetch over a multi-GB table runs at about twice the row rate of page-locked
    numpy / cudaHostAlloc memory.  Fill it like any array (``np.copyto``, ``np.fromfile`` into it, ...); it is freed
    when the array and every view of it are gone (destroy the EvStore built over it first)."""
    import weakref
    lib = _native.load_library()
    shape = tuple(int(x) for x in (shape if hasattr(shape, "__len__") else (shape,)))
    dt = np.dtype(dtype)
    nbytes = int(np.prod(shape, dtype=np.int64)) * dt.itemsize
    ptr = C.c_void_p()
    _native.check(lib.evs_host_alloc(C.byref(ptr), max(nbytes, 1), int(device)), "evs_host_alloc")
    buf = (C.c_uint8 * max(nbytes, 1)).from_address(ptr.value)
    weakref.finalize(buf, lib.evs_host_free, ptr.value)        # the numpy array below keeps `buf` alive
    return np.frombuffer(buf, dtype=dt, count=int(np.prod(shape, dtype=np.int64))).reshape(shape)


def to_host_rows(array: np.ndarray, device: int = 0) -> np.ndarray:
    """Copy of ``array`` in ``host_rows`` memory."""
    out = host_rows(array.shape, array.dtype, device)
    np.copyto(out, array)
    return out


class _ShapeOnly:
    """Stands in for an fp32 table whose rows are only available quantised / on disk."""

    def __init__(self, rows: int, dim: int):
        self.shape = (rows, dim)


class EvStore:
    def __init__(self, tables_fp32, cfg: CacheConfig, stores: dict | None = None, alt_keys=None):
        """tables_fp32: list of [rows, dim] float32 arrays (the trained embedding tables).
        stores: optional {precision: [raw rows per table]} if the quantised files already exist;
        otherwise they are derived from the fp32 tables with the reference's quantisers."""
        self._init_config(tables_fp32, cfg, stores, alt_keys)
        self.handle = C.c_void_p()
        self._owns_handle = True
        _native.check(self.lib.evs_create(C.byref(self._c), C.byref(self.handle)), "evs_create")

    @classmethod
    def from_raw_stores(cls, rows, dim: int, cfg: CacheConfig, stores: dict, alt_keys=None):
        """Build the cache over backing rows that already exist in the reference's on-disk layout
        (``storage_manager.open_model_dir`` / ``load_ev_table_into_emb_stor``): ``stores`` maps every precision
        the configuration uses to its per-table raw arrays; no fp32 copy of the tables is needed."""
        need = [cfg.main_precision] + ([cfg.secondary_precision] if cfg.n_layers >= 2 else [])
        missing = [p for p in need if p not in stores]
        if missing:
            raise ValueError(f"stores lacks the rows at {missing} bits")
        return cls([_ShapeOnly(int(r), int(dim)) for r in rows], cfg, stores=stores, alt_keys=alt_keys)

    def _init_config(self, tables_fp32, cfg: CacheConfig, stores=None, alt_keys=None):
        """Marshal the tables and the configuration into an evs_config (kept alive in self._c)."""
        self.lib = _native.load_library()
        self.cfg = cfg
        self.n_tables = len(tables_fp32)
        self.dim = int(tables_fp32[0].shape[1])
        self.rows = np.array([t.shape[0] for t in tables_fp32], dtype=np.int64)
        stores = dict(stores or {})
        need = [cfg.main_precision] + ([cfg.secondary_precision] if cfg.n_layers >= 2 else [])
        self._stores = {}
        for p in need:
            rb = row_bytes(self.dim, p)
            tabs = stores.get(p) or [encode_table(t, p) for t in tables_fp32]
            for t, a in zip(tables_fp32, tabs):
                if not a.flags["C_CONTIGUOUS"] or a.nbytes != t.shape[0] * rb:
                    raise ValueError(f"backing rows at {p} bits must be C-contiguous [rows, {rb} B]")
            self._stores[p] = tabs                                   # keep alive: the GPU reads them in place
        self._alt = None
        c = _native.EvsConfig()
        c.device = cfg.device
        c.n_tables = self.n_tables
        c.n_tables_total = cfg.n_tables_total or self.n_tables
        c.table_base = cfg.table_base
        c.dim = self.dim
        c.n_layers = cfg.n_layers
        c.main_precision = cfg.main_precision
        c.secondary_precision = cfg.secondary_precision
        c.total_size = cfg.total_size
        c.prop_c1, c.prop_c2, c.prop_c3 = cfg.proportions()
        c.max_batch = cfg.max_batch
        c.approx_emb_thres = cfg.approx_emb_thres
        c.high_agghit_threshold = cfg.high_agghit_threshold
        c.flush_rate = cfg.flush_rate
        c.perfect_item_cap = cfg.perfect_item_cap
        c.rows = self.rows.ctypes.data_as(C.POINTER(C.c_int64))
        self._main_ptrs = _ptr_array(self._stores[cfg.main_precision])
        c.store_main = C.cast(self._main_ptrs, C.POINTER(C.c_void_p))
        if cfg.n_layers >= 2:
            self._sec_ptrs = _ptr_array(self._stores[cfg.secondary_precision])
            c.store_secondary = C.cast(self._sec_ptrs, C.POINTER(C.c_void_p))
        if cfg.n_layers == 3:
            if alt_keys is None:
                raise ValueError("n_layers == 3 needs alt_keys (one uint32 array per table)")
            self._alt = [np.ascontiguousarray(a, dtype=np.uint32) for a in alt_keys]
            self._alt_ptrs = _ptr_array(self._alt)
            c.alt_keys = C.cast(self._alt_ptrs, C.POINTER(C.c_void_p))
        c.store_in_hbm = int(cfg.store_in_hbm)
        c.record_events = int(cfg.record_events)
        if cfg.policy not in ("evlfu", "lru", "lfu"):
            raise ValueError(f"unknown policy {cfg.policy!r} (evlfu | lru | lfu)")
        c.policy = {"evlfu": 0, "lru": 1, "lfu": 2}[cfg.policy]
        if cfg.table_ids:
            if len(cfg.table_ids) != self.n_tables:
                raise ValueError("table_ids needs one global id per local table")
            self._table_ids = (C.c_int32 * self.n_tables)(*[int(g) for g in cfg.table_ids])
            c.table_ids = C.cast(self._table_ids, C.POINTER(C.c_int32))
        self._c = c

    # ---- hot path ------------------------------------------------------------------------
    def prefetch(self, lS_i_next, ready_event=None):
        """Look-ahead (evs_prefetch): announce the index batch the NEXT lookup / shard_lookup call will pass (the same
        tensor).  Its probable misses are staged from the pinned backing store into HBM while the batch in flight
        runs.  ``ready_event``: a torch.cuda.Event recorded after the tensor was filled; None = already complete."""
        T, B = lS_i_next.shape
        assert lS_i_next.is_cuda and lS_i_next.is_contiguous() and T == self.n_tables
        ev = ready_event.cuda_event if ready_event is not None else None
        _native.check(self.lib.evs_prefetch(self.handle, lS_i_next.data_ptr(), B, ev), "evs_prefetch")

    def update_rows(self, tables, rows, values, stream=None):
        """Refresh a model in service (evs_update_rows): new fp32 values for rows of the tables this store serves.

        tables: a global table id (int) or an integer CUDA tensor [n] of them; rows: integer CUDA tensor [n];
        values: float32 CUDA tensor [n, dim] (rows may be strided, elements contiguous).  Returns ``where``, a uint8 CUDA
        tensor [n]: bit 0 = the C1 copy was refreshed, bit 1 = the C2 copy, bit 2 = the backing store was written,
        0x80 = rejected (row out of range or table not served here -- which also makes ``check`` raise -- or a value the
        stored precision cannot hold).  A key given twice takes its last row; the earlier occurrences report 0.

        The backing store is written IN PLACE: with host backing rows that is the caller's own arrays -- for a 32-bit
        store the fp32 tables passed to the constructor -- and, with ``store_in_hbm``, the HBM copy only.  Ordered on
        ``stream`` (default: torch's current stream): lookups enqueued before see the old rows, lookups after the new
        ones; cache contents, eviction order and statistics do not change.  Raises ValueError before any launch on a bad
        dtype, device or shape."""
        import torch
        dev = torch.device("cuda", self.cfg.device)

        def on_dev(x):
            return torch.is_tensor(x) and x.is_cuda and x.device == dev

        int_types = (torch.int64, torch.int32)
        if not on_dev(rows) or rows.dtype not in int_types or rows.dim() != 1:
            raise ValueError(f"rows must be a 1-D int64 / int32 tensor on {dev}")
        n = int(rows.shape[0])
        if not on_dev(values) or values.dtype != torch.float32 or values.dim() != 2 or tuple(values.shape) != (n, self.dim) \
                or (n > 0 and self.dim > 1 and values.stride(1) != 1) or (n > 1 and values.stride(0) < self.dim):
            raise ValueError(f"values must be a float32 tensor [{n}, {self.dim}] on {dev} with contiguous rows")
        if torch.is_tensor(tables):
            if not on_dev(tables) or tables.dtype not in int_types or tuple(tables.shape) != (n,):
                raise ValueError(f"tables must be an int or a 1-D int64 / int32 tensor [{n}] on {dev}")
            tab = tables.to(torch.int64)
        elif isinstance(tables, (int, np.integer)):
            tab = torch.full((n,), int(tables), dtype=torch.int64, device=dev)
        else:
            raise ValueError("tables must be an int or an integer CUDA tensor")
        where = torch.empty((n,), dtype=torch.uint8, device=dev)
        if n == 0:
            return where
        r = rows.to(torch.int64)
        # (table << 40) | row; a negative table or row gives a negative key, which the library rejects
        keys = torch.where((tab < 0) | (r < 0), torch.full_like(r, -1), (tab << 40) | r)
        st = _stream_handle(stream, dev)
        vstride = values.stride(0) if n > 1 else self.dim
        rc = self.lib.evs_update_rows(self.handle, keys.data_ptr(), n, values.data_ptr(), vstride, where.data_ptr(), st)
        _native.check(rc, "evs_update_rows")
        return where

    def save_state(self, stream=None) -> np.ndarray:
        """Snapshot of the cache's policy state (evs_save_state): resident keys per tier in eviction order, n_perfect,
        C3's raw FIFO window and map -- keys only, no row bytes.  Reflects every lookup enqueued on ``stream`` (default:
        torch's current stream) before the call; synchronises.  Returns the blob as a uint8 array (``state_info``
        parses its header); ``load_state`` restores it into a handle serving the same tables."""
        import torch
        st = _stream_handle(stream, torch.device("cuda", self.cfg.device))
        bound = C.c_uint64(0)
        _native.check(self.lib.evs_state_bytes(self.handle, C.byref(bound)), "evs_state_bytes")
        buf = np.empty(int(bound.value), dtype=np.uint8)
        n = C.c_uint64(0)
        _native.check(self.lib.evs_save_state(self.handle, buf.ctypes.data, buf.nbytes, C.byref(n), st), "evs_save_state")
        return buf[:n.value].copy()

    def load_state(self, blob, stream=None):
        """Replace the cache's policy state with a snapshot from ``save_state`` (evs_load_state); rows are read from this
        store's backing rows at its own precisions.  Lookups enqueued on ``stream`` after the call see the loaded state;
        synchronises.  Raises EvsError for a snapshot of another configuration (the cache is then unchanged) or one whose
        keys fail the device checks (the cache is then empty)."""
        import torch
        st = _stream_handle(stream, torch.device("cuda", self.cfg.device))
        b = np.ascontiguousarray(np.frombuffer(blob, dtype=np.uint8) if isinstance(blob, (bytes, bytearray)) else blob,
                                 dtype=np.uint8)
        _native.check(self.lib.evs_load_state(self.handle, b.ctypes.data, b.nbytes, st), "evs_load_state")

    def check(self, clear: bool = False):
        """Raise if a batch that has already run saw an out-of-range index or a silent peer (no synchronisation)."""
        _native.check(self.lib.evs_check(self.handle, int(clear)), "evs_check")

    def memory_footprint(self) -> int:
        """Bytes of HBM the handle holds (index + slot-indexed slabs + rings + staging)."""
        n = C.c_uint64(0)
        _native.check(self.lib.evs_memory_footprint(self.handle, C.byref(n)), "evs_memory_footprint")
        return int(n.value)

    def lookup(self, lS_i, out=None, hit=None, agg_in=None, stream=None):
        """lS_i: int64 CUDA tensor [n_tables, B].  Returns (out [B, n_tables, dim] fp32, hit [B, n_tables] uint8)."""
        import torch
        assert lS_i.is_cuda and lS_i.dtype == torch.int64 and lS_i.is_contiguous()
        T, B = lS_i.shape
        assert T == self.n_tables
        if out is None:
            out = torch.empty((B, T, self.dim), dtype=torch.float32, device=lS_i.device)
        if hit is None:
            hit = torch.empty((B, T), dtype=torch.uint8, device=lS_i.device)
        st = _stream_handle(stream, lS_i.device)
        stride = out.stride(0)
        rc = self.lib.evs_lookup_batch(self.handle, lS_i.data_ptr(), B, out.data_ptr(), stride, hit.data_ptr(),
                                       agg_in.data_ptr() if agg_in is not None else None, st)
        _native.check(rc, "evs_lookup_batch")
        return out, hit

    def note_replays(self, n: int = 1, stream=None):
        """A CUDA graph the caller captured around ``lookup`` was launched ``n`` times (evs_note_replays)."""
        import torch
        st = _stream_handle(stream, torch.device("cuda", self.cfg.device))
        _native.check(self.lib.evs_note_replays(self.handle, int(n), st), "evs_note_replays")

    def _pack_bags(self, lS_o, lS_i):
        """apply_emb's per-table lists -> (B, nnz per table, idx int64 [nnz] table 0 first, off int64 [n_tables*B + 1])."""
        import torch
        T = self.n_tables
        assert len(lS_i) == T and len(lS_o) == T
        B = int(lS_o[0].numel())
        dev = lS_i[0].device
        nnz_t = [int(x.numel()) for x in lS_i]
        base = np.concatenate([[0], np.cumsum(nnz_t)]).astype(np.int64)
        idx = torch.cat([x.reshape(-1).to(torch.int64) for x in lS_i]) if base[-1] > 0 else torch.zeros(1, dtype=torch.int64, device=dev)
        off = torch.cat([lS_o[t].reshape(-1).to(torch.int64) + int(base[t]) for t in range(T)] +
                        [torch.tensor([int(base[-1])], dtype=torch.int64, device=dev)])
        return B, base, idx, off

    def lookup_bags(self, lS_o, lS_i, max_per_bag: int = 10, out=None, stream=None, agg_in=None):
        """Pooled lookup (evs_lookup_bags): lS_i / lS_o are the per-table index and offset tensors of apply_emb
        (lS_i[t] int64 CUDA [nnz_t], lS_o[t] int64 CUDA [B], nn.EmbeddingBag's offsets).  Returns (pooled fp32
        [B, n_tables, dim], hit: list of n_tables uint8 tensors [nnz_t]).  agg_in: uint8 CUDA [B * max_per_bag], each
        slice's agg_hit summed over the ranks of a sharded cache (evs_lookup_bags_agg, after ``probe_bags``), or None."""
        import torch
        T = self.n_tables
        B, base, idx, off = self._pack_bags(lS_o, lS_i)
        dev = idx.device
        if out is None:
            out = torch.empty((B, T, self.dim), dtype=torch.float32, device=dev)
        hit = torch.empty((max(int(base[-1]), 1),), dtype=torch.uint8, device=dev)
        st = _stream_handle(stream, dev)
        if agg_in is None:
            rc = self.lib.evs_lookup_bags(self.handle, idx.data_ptr(), off.data_ptr(), B, int(base[-1]), int(max_per_bag),
                                          out.data_ptr(), out.stride(0), hit.data_ptr(), st)
            _native.check(rc, "evs_lookup_bags")
        else:
            assert agg_in.is_cuda and agg_in.dtype == torch.uint8 and agg_in.numel() >= B * int(max_per_bag)
            rc = self.lib.evs_lookup_bags_agg(self.handle, idx.data_ptr(), off.data_ptr(), B, int(base[-1]), int(max_per_bag),
                                              out.data_ptr(), out.stride(0), hit.data_ptr(), agg_in.data_ptr(), st)
            _native.check(rc, "evs_lookup_bags_agg")
        return out, [hit[int(base[t]):int(base[t + 1])] for t in range(T)]

    def probe_bags(self, lS_o, lS_i, max_per_bag: int = 10, agg_out=None, stream=None):
        """Local hit count of every slice of a bag batch (evs_probe_bags): uint8 [B * max_per_bag].  State is unchanged."""
        import torch
        B, base, idx, off = self._pack_bags(lS_o, lS_i)
        if agg_out is None:
            agg_out = torch.empty((max(B * int(max_per_bag), 1),), dtype=torch.uint8, device=idx.device)
        st = _stream_handle(stream, idx.device)
        _native.check(self.lib.evs_probe_bags(self.handle, idx.data_ptr(), off.data_ptr(), B, int(base[-1]), int(max_per_bag),
                                              agg_out.data_ptr(), st), "evs_probe_bags")
        return agg_out

    def lookup_many(self, lS_i_list, outs=None, hits=None, stream=None):
        """Consecutive batches in one call (evs_lookup_batches): the same results as ``lookup`` on each in turn, but groups
        of 4 batches reach the device as one captured graph and their misses are staged by the look-ahead.
        lS_i_list: int64 CUDA tensors [n_tables, B] (same B).  outs / hits: one tensor per batch, or a single tensor every
        batch overwrites (a caller that consumes only the last), or None.  Returns (outs, hits) as lists."""
        import torch
        n = len(lS_i_list)
        T, B = lS_i_list[0].shape
        dev = lS_i_list[0].device
        assert all(x.is_cuda and x.dtype == torch.int64 and x.is_contiguous() and x.shape == (T, B) for x in lS_i_list) and T == self.n_tables
        if outs is None:
            outs = [torch.empty((B, T, self.dim), dtype=torch.float32, device=dev) for _ in range(n)]
        elif torch.is_tensor(outs):
            outs = [outs] * n
        if hits is None:
            hits = [torch.empty((B, T), dtype=torch.uint8, device=dev) for _ in range(n)]
        elif torch.is_tensor(hits):
            hits = [hits] * n
        ip = (C.c_void_p * n)(*[x.data_ptr() for x in lS_i_list])
        op = (C.c_void_p * n)(*[x.data_ptr() for x in outs])
        hp = (C.c_void_p * n)(*[x.data_ptr() for x in hits])
        st = _stream_handle(stream, dev)
        _native.check(self.lib.evs_lookup_batches(self.handle, n, ip, B, op, outs[0].stride(0), hp, st), "evs_lookup_batches")
        return outs, hits

    def lookup_many_ptr(self, n: int, idx_ptrs, B: int, out_ptrs, out_stride: int, hit_ptrs, stream: int = 0):
        """Raw form: idx_ptrs / out_ptrs / hit_ptrs are ctypes arrays of n device pointers (built once by a serving loop)."""
        rc = self.lib.evs_lookup_batches(self.handle, n, idx_ptrs, B, out_ptrs, out_stride, hit_ptrs, stream or None)
        if rc:
            _native.check(rc, "evs_lookup_batches")

    def probe(self, lS_i, agg_out=None, stream=None):
        import torch
        T, B = lS_i.shape
        if agg_out is None:
            agg_out = torch.empty((B,), dtype=torch.uint8, device=lS_i.device)
        st = _stream_handle(stream, lS_i.device)
        _native.check(self.lib.evs_probe_batch(self.handle, lS_i.data_ptr(), B, agg_out.data_ptr(), st), "evs_probe_batch")
        return agg_out

    # raw-pointer forms of the two hot calls: what a C / cgo caller does, and what a Python serving loop that has
    # its buffers set up uses to keep the per-batch host cost at the two library calls
    def lookup_ptr(self, idx_ptr: int, B: int, out_ptr: int, out_stride: int = 0, hit_ptr: int = 0, stream: int = 0):
        rc = self.lib.evs_lookup_batch(self.handle, idx_ptr, B, out_ptr, out_stride, hit_ptr or None, None, stream or None)
        if rc:
            _native.check(rc, "evs_lookup_batch")

    def prefetch_ptr(self, idx_ptr: int, B: int):
        rc = self.lib.evs_prefetch(self.handle, idx_ptr, B, None)
        if rc:
            _native.check(rc, "evs_prefetch")

    def lookup_host(self, idx: np.ndarray, out: np.ndarray | None = None, hit: np.ndarray | None = None):
        """idx: int64 host array [n_tables, B] (numpy or a pinned torch tensor's numpy view)."""
        idx = np.ascontiguousarray(idx, dtype=np.int64)
        T, B = idx.shape
        assert T == self.n_tables
        if out is None:
            out = np.empty((B, T, self.dim), dtype=np.float32)
        if hit is None:
            hit = np.empty((B, T), dtype=np.uint8)
        rc = self.lib.evs_lookup_batch_host(self.handle, idx.ctypes.data, B, out.ctypes.data, hit.ctypes.data)
        _native.check(rc, "evs_lookup_batch_host")
        return out, hit

    def lookup_host_ptr(self, idx_ptr: int, B: int, out_ptr: int, hit_ptr: int = 0):
        _native.check(self.lib.evs_lookup_batch_host(self.handle, idx_ptr, B, out_ptr, hit_ptr or None),
                      "evs_lookup_batch_host")

    def submit_host_ptr(self, idx_ptr: int, B: int, out_ptr: int, hit_ptr: int = 0) -> int:
        """Pipelined host-buffer lookup (evs_submit_host); returns the ticket for wait_host."""
        t = C.c_int64(0)
        _native.check(self.lib.evs_submit_host(self.handle, idx_ptr, B, out_ptr, hit_ptr or None, C.byref(t)), "evs_submit_host")
        return t.value

    def wait_host(self, ticket: int):
        _native.check(self.lib.evs_wait_host(self.handle, ticket), "evs_wait_host")

    def interact(self, x, ly, out=None, stream=None):
        """dlrm interact_features (dot): x [B, d], ly [B, n_f, d] -> [B, d + (n_f+1) n_f / 2] (dlrm_ops.interact_features)."""
        from . import dlrm_ops
        return dlrm_ops.interact_features(x, ly, out=out, stream=stream)

    def store_ptr(self, table: int, tier: int = 0):
        """(device-visible pointer, precision) of the backing rows of a table (evs_store_ptr)."""
        p = C.c_void_p()
        prec = C.c_int32(0)
        _native.check(self.lib.evs_store_ptr(self.handle, tier, table, C.byref(p), C.byref(prec)), "evs_store_ptr")
        return p.value, prec.value

    def storage_lookup(self, lS_i, out=None, stream=None):
        """The no-cache path (apply_emb_evstore with use_emb_cache=False -> request_to_emb_storage,
        emb_storage/storage_manager.py:125): every row straight from the pinned backing store,
        pooling factor 1.  lS_i int64 CUDA [n_tables, B] -> fp32 [B, n_tables, dim]."""
        import torch
        T, B = lS_i.shape
        if out is None:
            out = torch.empty((B, T, self.dim), dtype=torch.float32, device=lS_i.device)
        off = torch.arange(B, dtype=torch.int64, device=lS_i.device)
        st = _stream_handle(stream, lS_i.device)
        for t in range(T):
            ptr, prec = self.store_ptr(t)
            rc = self.lib.evs_embedding_bag(ptr, int(self.rows[t]), self.dim, prec, lS_i[t].data_ptr(), off.data_ptr(), B, B,
                                            None, out[:, t, :].data_ptr(), out.stride(0), st)
            _native.check(rc, "evs_embedding_bag")
        return out

    # ---- table-wise sharding over peer memory (evs_shard_*) -------------------------------------
    def shard_create(self, rank: int, world: int, batch_max: int):
        self._shard = C.c_void_p()
        self._shard_world, self._shard_batch_max = world, batch_max
        _native.check(self.lib.evs_shard_create(self.handle, rank, world, batch_max, C.byref(self._shard)), "evs_shard_create")
        buf = C.create_string_buffer(64)
        _native.check(self.lib.evs_shard_export(self._shard, buf), "evs_shard_export")
        return buf.raw

    def shard_connect(self, handles):
        """handles: the 64-byte exports of all ranks, in rank order."""
        blob = b"".join(handles)
        assert len(blob) == 64 * self._shard_world
        _native.check(self.lib.evs_shard_connect(self._shard, blob), "evs_shard_connect")

    def shard_lookup(self, lS_i, hit=None, stream=None):
        """lS_i int64 CUDA [n_tables_local, B_global] -> (this rank's [B/world, n_tables_total, dim] rows, hit)."""
        import torch
        T, B = lS_i.shape
        assert lS_i.is_cuda and lS_i.dtype == torch.int64 and lS_i.is_contiguous() and T == self.n_tables
        if hit is None:
            hit = torch.empty((B, T), dtype=torch.uint8, device=lS_i.device)
        st = _stream_handle(stream, lS_i.device)
        ptr = C.c_void_p()
        _native.check(self.lib.evs_shard_lookup(self._shard, lS_i.data_ptr(), B, hit.data_ptr(), C.byref(ptr), st), "evs_shard_lookup")
        shape = (B // self._shard_world, self.cfg.n_tables_total or self.n_tables, self.dim)
        return _tensor_from_ptr(ptr.value, shape, lS_i.device), hit

    def shard_lookup_many(self, lS_i_list, hits=None, stream=None):
        """Consecutive global batches in one call (evs_shard_lookup_many; groups of 4 batches = one captured graph).  Returns
        ([this rank's [B/world, n_tables_total, dim] rows per batch], hits); a buffer is valid until four batches later."""
        import torch
        n = len(lS_i_list)
        T, B = lS_i_list[0].shape
        dev = lS_i_list[0].device
        assert all(x.is_cuda and x.dtype == torch.int64 and x.is_contiguous() and x.shape == (T, B) for x in lS_i_list) and T == self.n_tables
        if hits is None:
            hits = [torch.empty((B, T), dtype=torch.uint8, device=dev) for _ in range(n)]
        elif torch.is_tensor(hits):
            hits = [hits] * n
        ip = (C.c_void_p * n)(*[x.data_ptr() for x in lS_i_list])
        hp = (C.c_void_p * n)(*[x.data_ptr() for x in hits])
        op = (C.c_void_p * n)()
        st = _stream_handle(stream, dev)
        _native.check(self.lib.evs_shard_lookup_many(self._shard, n, ip, B, hp, op, st), "evs_shard_lookup_many")
        shape = (B // self._shard_world, self.cfg.n_tables_total or self.n_tables, self.dim)
        return [_tensor_from_ptr(op[i], shape, dev) for i in range(n)], hits

    def shard_lookup_bags(self, lS_o, lS_i, max_per_bag: int = 10, stream=None):
        """Bags on a rank of a sharded cache (evs_shard_lookup_bags): lS_o / lS_i as ``lookup_bags`` for this rank's tables
        over the whole global batch.  Returns (this rank's pooled [B/world, n_tables_total, dim] rows, valid until four
        batches later; hit: list of n_tables uint8 tensors [nnz_t])."""
        import torch
        B, base, idx, off = self._pack_bags(lS_o, lS_i)
        dev = idx.device
        hit = torch.empty((max(int(base[-1]), 1),), dtype=torch.uint8, device=dev)
        st = _stream_handle(stream, dev)
        ptr = C.c_void_p()
        _native.check(self.lib.evs_shard_lookup_bags(self._shard, idx.data_ptr(), off.data_ptr(), B, int(base[-1]), int(max_per_bag),
                                                     hit.data_ptr(), C.byref(ptr), st), "evs_shard_lookup_bags")
        shape = (B // self._shard_world, self.cfg.n_tables_total or self.n_tables, self.dim)
        return _tensor_from_ptr(ptr.value, shape, dev), [hit[int(base[t]):int(base[t + 1])] for t in range(self.n_tables)]

    def shard_destroy(self):
        if getattr(self, "_shard", None):
            self.lib.evs_shard_destroy(self._shard)
            self._shard = None

    # ---- bookkeeping ---------------------------------------------------------------------
    def sync(self):
        _native.check(self.lib.evs_sync(self.handle), "evs_sync")

    def stats(self, reset: bool = False) -> dict:
        s = _native.EvsStats()
        _native.check(self.lib.evs_stats(self.handle, C.byref(s), int(reset)), "evs_stats")
        return s.as_dict()

    def set_profiling(self, on: bool):
        _native.check(self.lib.evs_set_profiling(self.handle, int(on)), "evs_set_profiling")

    def kernel_times(self, reset: bool = False) -> dict:
        """{kernel name: (summed device ms over timed launches, timed launches, launches)}."""
        cap = 32
        n = C.c_int32(cap)
        names = (C.c_char_p * cap)()
        ms = (C.c_double * cap)()
        timed = (C.c_uint64 * cap)()
        launches = (C.c_uint64 * cap)()
        _native.check(self.lib.evs_kernel_times(self.handle, C.byref(n), names, ms, timed, launches, int(reset)),
                      "evs_kernel_times")
        return {names[i].decode(): (ms[i], int(timed[i]), int(launches[i])) for i in range(n.value)}

    def phase_times(self) -> dict:
        """Device-side phase durations (us) of the last batch, from %globaltimer stamps."""
        t = (C.c_uint64 * 32)()
        _native.check(self.lib.evs_phase_times(self.handle, t), "evs_phase_times")
        v = [int(x) for x in t]
        us = lambda a, b: (v[b] - v[a]) / 1e3
        n = max(1, v[13])
        return {"avg_over_batches": n, "avg_serve": v[8] / n / 1e3, "avg_gap1": v[9] / n / 1e3, "avg_update": v[10] / n / 1e3,
                "avg_gap2": v[11] / n / 1e3, "avg_evict": v[12] / n / 1e3,
                "overlapped_batches": v[14], "evict_plan": v[22] / n / 1e3, "evict_chunks": v[23] / n / 1e3,
                "evict_wait_last": v[24] / n / 1e3, "evict_writeback": v[25] / n / 1e3, "evict_chunks_per_batch": v[20] / n,
                "evict_records_per_batch": v[21] / n, "avg_fetch_since_evict_start": v[28] / n / 1e3, "avg_peer_wait": v[29] / n / 1e3, "avg_count_wait_cta0": v[30] / n / 1e3, "evict_last_chunk_avg": v[26] / n, "evict_last_chunk_max": v[27], "evict_scanned_total": v[15], "appends_total": v[1],
                "serve": us(0, 7), "serve_to_update_gap": us(7, 2), "update": us(2, 3), "update_to_evict_gap": us(3, 4),
                "evict": us(4, 5), "c3": us(5, 6), "total": us(0, 6)}

    def launch_count(self) -> int:
        return int(self.lib.evs_launch_count(self.handle))

    def last_events(self, tier: int = 0):
        cap_e = self.cfg.max_batch * self.n_tables
        cap_f = int(self.stats()["capacity"][tier] * 0.35) + 8
        ev = np.empty(cap_e, dtype=np.int64)
        fl = np.empty(cap_f, dtype=np.int64)
        ne, nf = C.c_int64(cap_e), C.c_int64(cap_f)
        _native.check(self.lib.evs_last_events(self.handle, tier, ev.ctypes.data, C.byref(ne), fl.ctypes.data, C.byref(nf)),
                      "evs_last_events")
        return ev[:ne.value].copy(), fl[:nf.value].copy()

    def dump_state(self, tier: int = 0):
        """Per agg_hit bucket, the resident keys in eviction (FIFO) order, and n_perfect."""
        st = self.stats()
        cap = int(st["size"][tier]) + 8
        keys = np.empty(cap, dtype=np.int64)
        nb = (self.cfg.n_tables_total or self.n_tables) + 2
        off = np.zeros(nb, dtype=np.int64)
        n = C.c_int64(cap)
        npf = C.c_int64(0)
        _native.check(self.lib.evs_dump_state(self.handle, tier, keys.ctypes.data, C.byref(n), off.ctypes.data, C.byref(npf)),
                      "evs_dump_state")
        return [keys[off[b]:off[b + 1]].tolist() for b in range(nb - 1)], int(npf.value)

    def dump_c3(self):
        st = self.stats()
        # the queue may hold several records of one key (aprx_embedding.cpp:322), so size for the ring
        cap = 8 * int(st["c3_capacity"]) + 16 * self.cfg.max_batch * self.n_tables + 8
        keys = np.empty(cap, dtype=np.int64)
        alt = np.empty(cap, dtype=np.uint32)
        rec = np.empty(cap, dtype=np.uint8)
        n = C.c_int64(cap)
        _native.check(self.lib.evs_dump_c3(self.handle, keys.ctypes.data, alt.ctypes.data, rec.ctypes.data, C.byref(n)),
                      "evs_dump_c3")
        return keys[:n.value].copy(), alt[:n.value].copy(), rec[:n.value].copy()

    def close(self):
        if getattr(self, "handle", None) is not None and self.handle:
            self.shard_destroy()
            if getattr(self, "_owns_handle", True):
                self.lib.evs_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
