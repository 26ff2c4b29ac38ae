"""ctypes binding of libevstore_b200.so (include/evstore_b200.h).

The product path has no CPU fallback: if the CUDA library is missing or a call fails this
module raises.  Build the library with ``python -c "import __graft_entry__ as g; g.build()"``.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libevstore_b200.so")

EVS_MAX_TIERS = 2
EVS_OK = 0


class EvsConfig(C.Structure):
    _fields_ = [
        ("device", C.c_int32), ("n_tables", C.c_int32), ("n_tables_total", C.c_int32), ("table_base", C.c_int32),
        ("dim", C.c_int32), ("n_layers", C.c_int32), ("main_precision", C.c_int32), ("secondary_precision", C.c_int32),
        ("total_size", C.c_int64),
        ("prop_c1", C.c_int32), ("prop_c2", C.c_int32), ("prop_c3", C.c_int32),
        ("max_batch", C.c_int32), ("approx_emb_thres", C.c_int32), ("high_agghit_threshold", C.c_int32),
        ("flush_rate", C.c_float), ("perfect_item_cap", C.c_float),
        ("rows", C.POINTER(C.c_int64)),
        ("store_main", C.POINTER(C.c_void_p)), ("store_secondary", C.POINTER(C.c_void_p)),
        ("alt_keys", C.POINTER(C.c_void_p)),
        ("store_in_hbm", C.c_int32), ("record_events", C.c_int32), ("policy", C.c_int32),
        ("table_ids", C.POINTER(C.c_int32)),
    ]


class EvsStats(C.Structure):
    _fields_ = [
        ("lookups", C.c_uint64), ("samples", C.c_uint64), ("hits", C.c_uint64 * EVS_MAX_TIERS),
        ("c3_hits", C.c_uint64), ("approx_subst", C.c_uint64), ("misses", C.c_uint64), ("perfect_hits", C.c_uint64),
        ("inserts", C.c_uint64 * EVS_MAX_TIERS), ("evictions", C.c_uint64 * EVS_MAX_TIERS),
        ("flushed", C.c_uint64 * EVS_MAX_TIERS), ("size", C.c_uint64 * EVS_MAX_TIERS),
        ("capacity", C.c_uint64 * EVS_MAX_TIERS), ("c3_size", C.c_uint64), ("c3_capacity", C.c_uint64),
        ("batches", C.c_uint64),
    ]

    def as_dict(self):
        out = {}
        for name, _ in self._fields_:
            v = getattr(self, name)
            out[name] = list(v) if hasattr(v, "__len__") else int(v)
        return out


# every symbol include/evstore_b200.h declares
SYMBOLS = [
    "evs_create", "evs_destroy", "evs_last_error", "evs_version", "evs_lookup_batch", "evs_lookup_batches", "evs_lookup_bags", "evs_lookup_bags_agg", "evs_probe_bags", "evs_note_replays", "evs_prefetch", "evs_update_rows", "evs_state_bytes", "evs_save_state", "evs_load_state", "evs_probe_batch", "evs_check",
    "evs_memory_footprint", "evs_host_alloc", "evs_host_free",
    "evs_lookup_batch_host", "evs_submit_host", "evs_wait_host", "evs_sync", "evs_stats", "evs_last_events", "evs_dump_state", "evs_dump_c3",
    "evs_interact", "evs_knn", "evs_embedding_bag", "evs_embedding_bag_status", "evs_store_ptr", "evs_shard_create", "evs_shard_export",
    "evs_shard_connect", "evs_shard_lookup", "evs_shard_lookup_many", "evs_shard_lookup_bags", "evs_shard_destroy", "evs_set_profiling", "evs_kernel_times", "evs_launch_count", "evs_phase_times", "evs_legacy_configure", "evs_legacy_handle", "ev_lookup", "get_ev_values", "print_perfect_hit",
    "test_arr", "ev_lookup_based_on_list_keys",
]

_lib = None


def load_library(path: str | None = None):
    """dlopen the CUDA library and declare its prototypes.  Raises if it is not built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise RuntimeError(f"{p} is not built: run __graft_entry__.build() (needs nvcc); there is no CPU fallback")
    lib = C.CDLL(p)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    lib.evs_create.argtypes = [C.POINTER(EvsConfig), C.POINTER(vp)]
    lib.evs_create.restype = C.c_int
    lib.evs_destroy.argtypes = [vp]
    lib.evs_destroy.restype = C.c_int
    lib.evs_last_error.argtypes = []
    lib.evs_last_error.restype = C.c_char_p
    lib.evs_version.argtypes = []
    lib.evs_version.restype = C.c_int
    lib.evs_lookup_batch.argtypes = [vp, vp, i32, vp, i64, vp, vp, vp]
    lib.evs_lookup_batch.restype = C.c_int
    lib.evs_lookup_batches.argtypes = [vp, i32, vp, i32, vp, i64, vp, vp]
    lib.evs_lookup_batches.restype = C.c_int
    lib.evs_lookup_bags.argtypes = [vp, vp, vp, i32, i64, i32, vp, i64, vp, vp]
    lib.evs_lookup_bags.restype = C.c_int
    lib.evs_lookup_bags_agg.argtypes = [vp, vp, vp, i32, i64, i32, vp, i64, vp, vp, vp]
    lib.evs_lookup_bags_agg.restype = C.c_int
    lib.evs_probe_bags.argtypes = [vp, vp, vp, i32, i64, i32, vp, vp]
    lib.evs_probe_bags.restype = C.c_int
    lib.evs_note_replays.argtypes = [vp, i64, vp]
    lib.evs_note_replays.restype = C.c_int
    lib.evs_prefetch.argtypes = [vp, vp, i32, vp]
    lib.evs_prefetch.restype = C.c_int
    lib.evs_update_rows.argtypes = [vp, vp, i64, vp, i64, vp, vp]
    lib.evs_update_rows.restype = C.c_int
    lib.evs_state_bytes.argtypes = [vp, C.POINTER(C.c_uint64)]
    lib.evs_state_bytes.restype = C.c_int
    lib.evs_save_state.argtypes = [vp, vp, C.c_uint64, C.POINTER(C.c_uint64), vp]
    lib.evs_save_state.restype = C.c_int
    lib.evs_load_state.argtypes = [vp, vp, C.c_uint64, vp]
    lib.evs_load_state.restype = C.c_int
    lib.evs_check.argtypes = [vp, C.c_int]
    lib.evs_check.restype = C.c_int
    lib.evs_memory_footprint.argtypes = [vp, C.POINTER(C.c_uint64)]
    lib.evs_memory_footprint.restype = C.c_int
    lib.evs_host_alloc.argtypes = [C.POINTER(vp), C.c_uint64, i32]
    lib.evs_host_alloc.restype = C.c_int
    lib.evs_host_free.argtypes = [vp]
    lib.evs_host_free.restype = C.c_int
    lib.evs_probe_batch.argtypes = [vp, vp, i32, vp, vp]
    lib.evs_probe_batch.restype = C.c_int
    lib.evs_lookup_batch_host.argtypes = [vp, vp, i32, vp, vp]
    lib.evs_lookup_batch_host.restype = C.c_int
    lib.evs_submit_host.argtypes = [vp, vp, i32, vp, vp, C.POINTER(i64)]
    lib.evs_submit_host.restype = C.c_int
    lib.evs_wait_host.argtypes = [vp, i64]
    lib.evs_wait_host.restype = C.c_int
    lib.evs_sync.argtypes = [vp]
    lib.evs_sync.restype = C.c_int
    lib.evs_stats.argtypes = [vp, C.POINTER(EvsStats), C.c_int]
    lib.evs_stats.restype = C.c_int
    lib.evs_last_events.argtypes = [vp, C.c_int, vp, C.POINTER(i64), vp, C.POINTER(i64)]
    lib.evs_last_events.restype = C.c_int
    lib.evs_dump_state.argtypes = [vp, C.c_int, vp, C.POINTER(i64), vp, C.POINTER(i64)]
    lib.evs_dump_state.restype = C.c_int
    lib.evs_dump_c3.argtypes = [vp, vp, vp, vp, C.POINTER(i64)]
    lib.evs_dump_c3.restype = C.c_int
    lib.evs_interact.argtypes = [vp, vp, vp, i32, i32, i32, vp]
    lib.evs_interact.restype = C.c_int
    lib.evs_knn.argtypes = [vp, i64, vp, i64, i32, i32, vp, vp, vp, vp, i32, vp, vp]
    lib.evs_knn.restype = C.c_int
    lib.evs_embedding_bag.argtypes = [vp, i64, i32, i32, vp, vp, i64, i32, vp, vp, i64, vp]
    lib.evs_embedding_bag.restype = C.c_int
    lib.evs_embedding_bag_status.argtypes = []
    lib.evs_embedding_bag_status.restype = C.c_int
    lib.evs_store_ptr.argtypes = [vp, C.c_int, C.c_int, C.POINTER(vp), C.POINTER(i32)]
    lib.evs_store_ptr.restype = C.c_int
    lib.evs_shard_create.argtypes = [vp, i32, i32, i32, C.POINTER(vp)]
    lib.evs_shard_create.restype = C.c_int
    lib.evs_shard_export.argtypes = [vp, vp]
    lib.evs_shard_export.restype = C.c_int
    lib.evs_shard_connect.argtypes = [vp, vp]
    lib.evs_shard_connect.restype = C.c_int
    lib.evs_shard_lookup.argtypes = [vp, vp, i32, vp, C.POINTER(vp), vp]
    lib.evs_shard_lookup.restype = C.c_int
    lib.evs_shard_lookup_many.argtypes = [vp, i32, vp, i32, vp, vp, vp]
    lib.evs_shard_lookup_many.restype = C.c_int
    lib.evs_shard_lookup_bags.argtypes = [vp, vp, vp, i32, i64, i32, vp, C.POINTER(vp), vp]
    lib.evs_shard_lookup_bags.restype = C.c_int
    lib.evs_shard_destroy.argtypes = [vp]
    lib.evs_shard_destroy.restype = C.c_int
    lib.evs_set_profiling.argtypes = [vp, C.c_int]
    lib.evs_set_profiling.restype = C.c_int
    lib.evs_kernel_times.argtypes = [vp, C.POINTER(i32), C.POINTER(C.c_char_p), C.POINTER(C.c_double),
                                     C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_int]
    lib.evs_kernel_times.restype = C.c_int
    lib.evs_phase_times.argtypes = [vp, C.POINTER(C.c_uint64)]
    lib.evs_phase_times.restype = C.c_int
    lib.evs_launch_count.argtypes = [vp]
    lib.evs_launch_count.restype = C.c_uint64
    lib.evs_legacy_configure.argtypes = [C.POINTER(EvsConfig)]
    lib.evs_legacy_configure.restype = C.c_int
    lib.evs_legacy_handle.argtypes = []
    lib.evs_legacy_handle.restype = vp
    # the reference's own prototypes, as cpp_socket_client.init_ctypes_lib declares them (:63-83)
    lib.ev_lookup.argtypes = [C.POINTER(C.c_int)]
    lib.ev_lookup.restype = C.POINTER(C.c_float)
    lib.get_ev_values.argtypes = [C.POINTER(C.c_int)]
    lib.get_ev_values.restype = C.POINTER(C.c_float)
    lib.print_perfect_hit.argtypes = None
    lib.print_perfect_hit.restype = None
    lib.test_arr.argtypes = [C.POINTER(C.c_int)]
    lib.test_arr.restype = None
    lib.ev_lookup_based_on_list_keys.argtypes = [C.POINTER(C.c_int)]
    lib.ev_lookup_based_on_list_keys.restype = C.c_int
    if path is None:
        _lib = lib
    return lib


class EvsError(RuntimeError):
    pass


def check(rc: int, what: str):
    if rc != EVS_OK:
        msg = load_library().evs_last_error()
        raise EvsError(f"{what} failed with status {rc}: {msg.decode() if msg else ''}")
