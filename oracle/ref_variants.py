"""Build variants of the reference's libcachemanager.so (TEST INFRASTRUCTURE ONLY).

The reference fixes its cache configuration, its embedding dimension and its data root at
compile time (mixed_precs_caching/cache_manager.cpp:13-20, cache_manager.hpp:30-31,
evlfu_32.hpp:61 ...), so every configuration we time or compare against is a separate .so.
``oracle/build_ref.py`` compiles each entry below from the sources of a checkout of the
original project (the directory named by the EVSTORE_REFERENCE environment variable) into
``oracle/_ref/lib<name>.so``; the fixture files the library opens at dlopen time are written by
the caller (bench.py / tests) under FIXTURE_ROOT/<fixture>/.
"""
import os

# checkout of the original project (its cache_algo/ and mixed_precs_caching/), or "" when there is none
REFERENCE = os.environ.get("EVSTORE_REFERENCE", "")

# the compiled-in data root; /dev/shm keeps the CPU baseline off the disk (BASELINE.md section 3)
FIXTURE_ROOT = "/dev/shm/evstore_b200_ref/"

KAGGLE_TOTAL_ROWS = 33762577
# the reference's operating point "30000 is 13%" (cache_manager.cpp:16) scaled to all Kaggle rows
KAGGLE_CACHE_13PCT = int(KAGGLE_TOTAL_ROWS * 0.13)

VARIANTS = {
    # bench.py configs[1]: C1, fp32, Kaggle shape, dim 16
    "bench_c1_fp32_d16": dict(layers=1, main=32, sec=4, total=KAGGLE_CACHE_13PCT, prop="", dim=16, fixture="kaggle_d16"),
    # small fixtures for the CPU tests (dim 36 = the reference's own EV_DIMENSION)
    "test_c1_fp32_d36": dict(layers=1, main=32, sec=4, total=600, prop="", dim=36, fixture="test_d36"),
    "test_c1_8_d36": dict(layers=1, main=8, sec=4, total=150, prop="", dim=36, fixture="test_d36"),
    "test_c2_32_8_small_d36": dict(layers=2, main=32, sec=8, total=100, prop="", dim=36, fixture="test_d36"),
    "test_c1_flush_d36": dict(layers=1, main=32, sec=4, total=100, prop="", dim=36, fixture="test_d36"),
    "test_c2_16_4_small_d36": dict(layers=2, main=16, sec=4, total=200, prop="", dim=36, fixture="test_d36"),
    "test_c2_8_4_d36": dict(layers=2, main=8, sec=4, total=100000, prop="", dim=36, fixture="test_d36"),
    "test_c2_8_4_small_d36": dict(layers=2, main=8, sec=4, total=200, prop="", dim=36, fixture="test_d36"),
    # three layers (C1 8-bit 192 entries, C2 4-bit 384, C3 144 alt keys); needs alt-keys/binary/ in the fixture.
    # Only usable when driven slowly: C3 is populated by the library's worker threads (tests/test_oracle_c3_pin.py)
    "test_c3_8_4_d36": dict(layers=3, main=8, sec=4, total=100, prop="48-48-4", dim=36, fixture="test_d36"),
}

PRECISION_DIRS = {32: "ev-table", 16: "ev-table-16", 8: "ev-table-8", 4: "ev-table-4"}


def lib_name(variant: str) -> str:
    return f"lib{variant}.so"
