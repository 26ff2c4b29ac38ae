"""Run the compiled reference cache (oracle/_ref/lib<variant>.so) on a trace.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py): used by tests/ as a checker and by
bench.py's ``cpu_baseline`` / ``--impl reference`` legs as the timed CPU baseline.

The reference builds its cache in static initialisers at dlopen time and opens its table files
there (cache_manager.cpp:45-55, evlfu_32.cpp:38-50), so the fixture files must exist before
``RefCache`` is constructed.  One process can hold one instance per variant (the state is
process-global in the library and is never reset).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from .ref_variants import FIXTURE_ROOT, PRECISION_DIRS, VARIANTS, lib_name

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(HERE, "_ref")


def available(variant: str) -> bool:
    return os.path.exists(os.path.join(REF_DIR, lib_name(variant))) and os.path.exists(os.path.join(REF_DIR, "libref_drive.so"))


def fixture_dir(variant: str) -> str:
    return FIXTURE_ROOT + VARIANTS[variant]["fixture"] + "/"


def write_fixture(variant: str, raw_tables: dict, alt_keys=None, overwrite: bool = False):
    """raw_tables: {precision: [raw row array per table]} in the binary/ev-table-N.bin layout
    (script/convert_ev_to_binary.py): row-major, dim*bits/8 bytes per row.  alt_keys: per table
    uint32 array, written big-endian (script/convert_altkeys_to_binary.py:35)."""
    root = fixture_dir(variant)
    for prec, tabs in raw_tables.items():
        d = os.path.join(root, PRECISION_DIRS[prec], "binary")
        os.makedirs(d, exist_ok=True)
        for t, a in enumerate(tabs):
            path = os.path.join(d, f"ev-table-{t + 1}.bin")
            a = np.ascontiguousarray(a)
            if overwrite or not os.path.exists(path) or os.path.getsize(path) != a.nbytes:
                a.tofile(path)
    if alt_keys is not None:
        d = os.path.join(root, "alt-keys", "binary")
        os.makedirs(d, exist_ok=True)
        for t, a in enumerate(alt_keys):
            np.asarray(a, dtype=">u4").tofile(os.path.join(d, f"ev-table-{t + 1}.bin"))
    return root


def needed_precisions(variant: str):
    v = VARIANTS[variant]
    out = [v["main"]]
    if v["layers"] >= 2:
        out.append(v["sec"])
    return out


class RefCache:
    def __init__(self, variant: str, fresh_copy: bool = False):
        """fresh_copy: dlopen a private copy of the library, i.e. a second, empty cache instance in
        this process (the library's state is process-global per loaded file)."""
        v = VARIANTS[variant]
        self.variant, self.dim, self.n_tables = variant, v["dim"], 26
        path = os.path.join(REF_DIR, lib_name(variant))
        if not os.path.exists(path):
            raise RuntimeError(f"{path} missing: run oracle/build_ref.py with EVSTORE_REFERENCE set")
        if fresh_copy:
            import shutil
            import tempfile
            fd, tmp = tempfile.mkstemp(prefix="evs_ref_", suffix=".so")
            os.close(fd)
            shutil.copyfile(path, tmp)
            path = tmp
        self.lib = C.CDLL(path)                       # static ctors run here
        if fresh_copy:
            os.unlink(path)                           # the mapping stays valid
        self.lib.ev_lookup.argtypes = [C.POINTER(C.c_int)]
        self.lib.ev_lookup.restype = C.POINTER(C.c_float)
        self.lib.print_perfect_hit.restype = None
        self.drv = C.CDLL(os.path.join(REF_DIR, "libref_drive.so"))
        self.drv.ref_drive.argtypes = [C.c_void_p, C.c_void_p, C.c_long, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_double)]
        self.drv.ref_drive.restype = C.c_double

    def drive(self, trace: np.ndarray, want_out: bool = False):
        """trace: int32 [n, 26] (sample-major).  Returns (seconds, out [n, 26, dim] or None)."""
        trace = np.ascontiguousarray(trace, dtype=np.int32)
        n = trace.shape[0]
        out = np.empty((n, self.n_tables, self.dim), dtype=np.float32) if want_out else None
        chk = C.c_double(0.0)
        fn = C.cast(self.lib.ev_lookup, C.c_void_p)
        sec = self.drv.ref_drive(fn, trace.ctypes.data, n, self.n_tables, self.dim,
                                 out.ctypes.data if want_out else None, C.byref(chk))
        if sec < 0:
            raise RuntimeError("reference ev_lookup returned NULL")
        return sec, out

    def drive_slow(self, trace: np.ndarray, gap_s: float):
        """One ev_lookup per sample with a pause after each, so that the library's C3 worker threads
        (aprx_embedding.cpp:36-101) finish their queued group before the next request probes C3."""
        import time
        trace = np.ascontiguousarray(trace, dtype=np.int32)
        out = np.empty((trace.shape[0], self.n_tables, self.dim), dtype=np.float32)
        for i in range(trace.shape[0]):
            p = self.lib.ev_lookup(trace[i].ctypes.data_as(C.POINTER(C.c_int)))
            out[i] = np.ctypeslib.as_array(p, shape=(self.n_tables, self.dim))
            time.sleep(gap_s)
        return out

    def lookup(self, row_ids):
        arr = (C.c_int * self.n_tables)(*[int(x) for x in row_ids])
        p = self.lib.ev_lookup(arr)
        return np.ctypeslib.as_array(p, shape=(self.n_tables, self.dim)).copy()
