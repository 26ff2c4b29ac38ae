"""CPU-side checks: the C-ABI library loads and exports every symbol the header declares (no compute
calls without a GPU), storage_manager keeps the reference's API and file layout, table split."""
import os
import re

import numpy as np
import pytest

from helpers import SMALL_ROWS, pkg
from oracle import codecs as ocodecs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    p = pkg()
    lib = p.load_library()
    text = open(os.path.join(ROOT, "include", "evstore_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    names = re.findall(r"\b([a-z_][a-z0-9_]*)\s*\([^;{]*\)\s*;", text)
    names = [n for n in names if n not in ("defined",)]
    assert len(names) >= 25, names
    for n in names:
        assert hasattr(lib, n), f"{n} is declared in include/evstore_b200.h but not exported"
    assert sorted(set(names)) == sorted(set(p.SYMBOLS)), set(names) ^ set(p.SYMBOLS)
    assert lib.evs_version() >= 100


def test_product_path_refuses_to_run_without_its_library(tmp_path):
    p = pkg()
    with pytest.raises(RuntimeError):
        p.load_library(str(tmp_path / "missing.so"))


def test_no_product_module_imports_the_oracle():
    pk = os.path.join(ROOT, "ev-store-dlrm_b200")
    for dirpath, _d, files in os.walk(pk):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f


@pytest.mark.parametrize("prec", [32, 16, 8, 4])
def test_storage_manager_api_and_file_layout(tmp_path, prec):
    p = pkg()
    sm = p.storage_manager
    tables = p.workload.make_tables(SMALL_ROWS, 36)
    sm.ev_precs, sm.ev_dimension, sm.n_tables = prec, 36, 26
    sm.storage_type = sm.EmbStorage.FILEPY
    sm.load_tables(tables, precisions=(prec,))
    sm.save_ev_tables(str(tmp_path), prec)
    # the file is the reference's binary/ev-table-N.bin: row-major, dim*bits/8 bytes per row
    raw = ocodecs.quantize_table(tables[2], prec)
    assert open(tmp_path / "binary" / "ev-table-3.bin", "rb").read() == np.ascontiguousarray(raw).tobytes()
    sm.close_any_db_conn()
    sm.load_ev_table_into_emb_stor(str(tmp_path), rows=SMALL_ROWS)
    want = ocodecs.dequantize_rows(raw, prec)
    v = sm.get_val_from_storage(3, 17)                   # tableId is 1-based
    assert len(v) == 36 and np.array_equal(np.float32(v), want[17])
    vals = sm.get_arr_val_from_storage([(3, 0), (1, 5)])
    assert np.array_equal(np.float32(vals[0]), want[0])
    _, ly = sm.request_to_emb_storage([0] * 26)
    assert len(ly) == 26 and tuple(ly[0].shape) == (1, 36)
    with pytest.raises(sm.StorageError):
        sm.get_val_from_storage(27, 0)
    sm.close_any_db_conn()


def test_table_split_matches_extend_distributed():
    s = pkg().sharded
    assert s.get_split_lengths(26, 2) == [13, 13]
    assert s.get_split_lengths(26, 4) == [7, 7, 6, 6]
    assert s.get_split_lengths(26, 8) == [4, 4, 3, 3, 3, 3, 3, 3]
    for size in (1, 2, 4, 8):
        got = []
        for r in range(size):
            sl = s.get_my_slice(26, r, size)
            got += list(range(26))[sl]
            assert sl.stop - sl.start == s.get_split_lengths(26, size)[r]
        assert got == list(range(26))


# ---- on-disk formats of the reference (SURVEY.md section 8(f) rank 2) --------------------------------
def test_alt_key_file_format_equals_reference_writer(tmp_path, golden_dir):
    """tests/golden/formats/altkeys.bin was written by the reference's convert_altkeys_to_binary from altkeys.txt
    (tests/golden/make_golden.py formats): our text -> key conversion, writer and reader agree with it byte for byte."""
    sm = pkg().storage_manager
    fdir = os.path.join(golden_dir, "formats")
    lines = open(os.path.join(fdir, "altkeys.txt")).read().split()
    keys = sm.alt_keys_from_text(lines)
    want = open(os.path.join(fdir, "altkeys.bin"), "rb").read()
    assert np.asarray(keys, dtype=">u4").tobytes() == want
    sm.n_tables = 1
    try:
        sm.save_alt_keys(str(tmp_path), [keys])
        assert open(tmp_path / "binary" / "ev-table-1.bin", "rb").read() == want
        sm.n_tables = 26                                        # the file only holds table 1 of 26
        with pytest.raises(sm.StorageError):
            sm.load_alt_keys(str(tmp_path))
        sm.n_tables = 1
        with pytest.raises(sm.StorageError):                    # table ids reach 26 > n_tables = 1
            sm.load_alt_keys(str(tmp_path))
        (back,) = [np.fromfile(tmp_path / "binary" / "ev-table-1.bin", dtype=">u4").astype(np.uint32)]
        assert np.array_equal(back, keys) and back.dtype == np.uint32
        assert int(back[-1]) // 100 == 42949671 and int(back[-1]) % 100 == 3       # alt_row*100 + alt_table
    finally:
        sm.n_tables = 26


def test_training_config_reader_reads_the_reference_file(tmp_path, golden_dir):
    sm = pkg().storage_manager
    path = os.path.join(golden_dir, "formats", "training_config.txt")
    tfm, nb, nbt, ln_emb, m_den = sm.read_training_config(path)
    assert (nb, nbt, m_den) == (306969, 3274, 13) and tfm[25] == 25
    assert ln_emb.tolist() == pkg().workload.KAGGLE_ROWS
    sm.store_training_config(str(tmp_path / "training_config.txt"), tfm, nb, nbt, ln_emb, m_den)
    assert open(tmp_path / "training_config.txt").read() == open(path).read()


def test_open_model_dir_reads_every_precision_and_the_alt_keys(tmp_path):
    """A stored model laid out like the reference's (ev-table-8/binary, ev-table-4/binary, training_config.txt,
    alt-key binaries) comes back as the raw stores evs_config takes."""
    p = pkg()
    sm = p.storage_manager
    tables = p.workload.make_tables(SMALL_ROWS, 36)
    alt = p.workload.make_alt_keys(SMALL_ROWS)
    sm.ev_dimension, sm.n_tables = 36, 26
    try:
        for prec in (8, 4):
            sm.load_tables(tables, precisions=(prec,))
            sm.save_ev_tables(str(tmp_path / sm.PRECISION_DIRS[prec]), prec)
        sm.store_training_config(str(tmp_path / "training_config.txt"), {i: i for i in range(26)}, 10, 2, np.array(SMALL_ROWS), 13)
        sm.save_alt_keys(str(tmp_path / "alt"), alt)
        rows, stores, alt_back = sm.open_model_dir(str(tmp_path), (8, 4), dim=36, alt_path=str(tmp_path / "alt"))
        assert rows == SMALL_ROWS and sorted(stores) == [4, 8]
        assert np.array_equal(stores[8][3], ocodecs.quantize_table(tables[3], 8))
        assert np.array_equal(stores[4][11], ocodecs.quantize_table(tables[11], 4))
        assert all(np.array_equal(a, b) for a, b in zip(alt, alt_back))
        # a cardinality that disagrees with the file sizes is an error, not a silent truncation
        bad = list(SMALL_ROWS)
        bad[0] += 1
        sm.store_training_config(str(tmp_path / "training_config.txt"), {}, 10, 2, np.array(bad), 13)
        with pytest.raises(sm.StorageError):
            sm.open_model_dir(str(tmp_path), (8,), dim=36)
    finally:
        sm.ev_precs, sm.ev_dimension, sm.n_tables = 32, 36, 26
        sm.close_any_db_conn()


def test_dlrm_forward_golden_describes_the_reference_model(golden_dir):
    """The fixture is self-consistent: recomputing sequential_forward (dlrm_s_pytorch.py:588-613) from the saved
    weights with plain torch on the CPU gives the saved interaction features and probabilities; and the stated
    tolerances of the quantised tiers (tests/test_gpu_dlrm_forward.py) hold for the reference's own codecs."""
    from helpers import dlrm_forward_cpu, load_dlrm_golden
    g = load_dlrm_golden(golden_dir)
    tables = [g[f"emb_{k}"] for k in range(26)]
    Z, R = dlrm_forward_cpu(g, tables)
    assert np.allclose(R, g["R"], rtol=1e-5, atol=1e-6)
    assert np.allclose(Z, g["Z"], rtol=0, atol=1e-6)
    for prec, tol_row, tol_z in ((16, 1e-3, 2e-5), (8, 4e-3, 2e-3), (4, 0.25, 6e-2)):
        dec = [ocodecs.dequantize_rows(ocodecs.quantize_table(t, prec), prec) for t in tables]
        assert max(float(np.abs(d - t).max()) for d, t in zip(dec, tables)) <= tol_row, prec
        Zq, _ = dlrm_forward_cpu(g, dec)
        assert float(np.abs(Zq - g["Z"]).max()) <= tol_z, prec


def test_latency_cdf_file_equals_the_reference_function(tmp_path, golden_dir):
    """tests/golden/formats/evlfu_golden-cdf.csv was written by the reference's calculate_and_write_cdf
    (dlrm_s_pytorch_C1_C2_C3.py:291-319, executed from the reference file by make_golden.py cdf) from
    cdf_time_start.npy; ours writes the same bytes."""
    p = pkg()
    t = np.load(os.path.join(golden_dir, "formats", "cdf_time_start.npy"))
    out = p.evstore_utils.calculate_and_write_cdf(str(tmp_path), "evlfu_golden", [float(x) for x in t])
    want = open(os.path.join(golden_dir, "formats", "evlfu_golden-cdf.csv")).read()
    assert open(out).read() == want
    # fewer requests than CDF points: every latency is kept
    out = p.evstore_utils.calculate_and_write_cdf(str(tmp_path), "few", [0.0, 0.5, 0.75, 2.0, 9.0])
    assert open(out).read().splitlines() == ["y,latency_ms", "0.3333333333333333,250.0", "0.6666666666666666,500.0", "1.0,1250.0"]


def test_split_cache_budget_water_filling():
    """sharded.split_cache_budget: one budget over the ranks, equal shares, a rank smaller than its share is cached whole
    and passes the rest on; the sum is the budget (up to the integer division) and never exceeds a rank's rows."""
    from helpers import pkg
    sh = pkg().sharded
    assert sh.split_cache_budget([100, 100], 50, floor=0) == [25, 25]
    assert sh.split_cache_budget([10, 1000, 1000], 410, floor=0) == [10, 200, 200]
    assert sh.split_cache_budget([5, 8, 1000], 113, floor=0) == [5, 8, 100]
    assert sh.split_cache_budget([5, 8], 1000, floor=0) == [5, 8]
    rows = pkg().workload.KAGGLE_ROWS
    per = [sum(rows[t] for t in x) for x in sh.balanced_placement(rows, 8)]
    caps = sh.split_cache_budget(per, int(sum(rows) * 0.13))
    assert all(c <= r for c, r in zip(caps, per)) and abs(sum(caps) - int(sum(rows) * 0.13)) < 8


def test_placements_cover_every_table_once_and_keep_the_split_lengths():
    from helpers import pkg
    sh = pkg().sharded
    rng = np.random.default_rng(5)
    for _ in range(50):
        n = int(rng.integers(1, 32))
        size = int(rng.integers(1, 9))
        if size > n:
            continue
        rows = rng.integers(1, 10 ** 7, size=n).tolist()
        for pl in (sh.balanced_placement(rows, size), sh.contiguous_placement(n, size)):
            assert sorted(t for x in pl for t in x) == list(range(n))
            assert [len(x) for x in pl] == sh.get_split_lengths(n, size)
            assert all(x == sorted(x) for x in pl)
        caps = sh.split_cache_budget([sum(rows[t] for t in x) for x in sh.balanced_placement(rows, size)], int(sum(rows) * 0.13), floor=0)
        assert sum(caps) <= int(sum(rows) * 0.13) and all(c >= 0 for c in caps)
