#!/usr/bin/env python
"""Compile the reference's own C++ cache (mixed_precs_caching/) into oracle/_ref/*.so.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  The sources are read where they lie
in the checkout named by EVSTORE_REFERENCE; nothing of them is copied into this repository.  Because the
reference's configuration is compile-time text (cache_manager.cpp:13-20 #defines,
EV_DIMENSION in every header, hard-coded /mnt/extra/... data roots in evlfu_*.hpp:58-64 and
aprx_embedding.hpp:39), each variant is built from a *patched stream* of those files placed
in a scratch directory under /tmp (the `sed` step of BASELINE.md section 3), with the
reference's own compile line (cache_manager.cpp:10):

    g++ -shared -o libcachemanager.so -fPIC -O3 evlfu_4.cpp evlfu_8.cpp evlfu_16.cpp
        evlfu_32.cpp [aprx_embedding.cpp] cache_manager.cpp -pthread

Outputs go to oracle/_ref/ only (git-ignored).  Without a reference checkout only our own
helpers are built (libref_drive.so, libstdset_shim.so).
"""
import os
import re
import shutil
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle.ref_variants import FIXTURE_ROOT, REFERENCE, VARIANTS, lib_name  # noqa: E402

REF_SRC = os.path.join(REFERENCE, "mixed_precs_caching") if REFERENCE else ""
OUT = os.path.join(HERE, "_ref")
SOURCES = ["evlfu_4.cpp", "evlfu_8.cpp", "evlfu_16.cpp", "evlfu_32.cpp", "aprx_embedding.cpp", "cache_manager.cpp"]
HEADERS = ["evlfu_4.hpp", "evlfu_8.hpp", "evlfu_16.hpp", "evlfu_32.hpp", "aprx_embedding.hpp", "cache_manager.hpp"]

EV_ROOT = "/mnt/extra/ev-store-dlrm/stored_model/criteo_kaggle_all_mmap/epoch-00/"
ALT_ROOT_RE = re.compile(r'(\n\s*string APRX_EV_FILE_PATH = ")[^"]*(";)')


def patch(text: str, name: str, v: dict) -> str:
    root = FIXTURE_ROOT + v["fixture"] + "/"
    text = text.replace(EV_ROOT, root)
    text = ALT_ROOT_RE.sub(lambda m: m.group(1) + root + "alt-keys/binary/" + m.group(2), text)
    text = re.sub(r"#define EV_DIMENSION\s+36", f"#define EV_DIMENSION {v['dim']}", text)
    if name == "cache_manager.cpp":
        text = re.sub(r"#define N_CACHING_LAYER\s+\d+", f"#define N_CACHING_LAYER {v['layers']}", text)
        text = re.sub(r"#define MAIN_PRECISION\s+\d+", f"#define MAIN_PRECISION {v['main']}", text)
        text = re.sub(r"#define SECONDARY_PRECISION\s+\d+", f"#define SECONDARY_PRECISION {v['sec']}", text)
        text = re.sub(r"#define TOTAL_SIZE\s+\d+", f"#define TOTAL_SIZE {v['total']}", text)
        text = re.sub(r'#define SIZE_PROPORTION\s+"[^"]*"', f'#define SIZE_PROPORTION "{v["prop"]}"', text)
    return text


def build_variant(name: str, v: dict, force: bool = False) -> str:
    os.makedirs(OUT, exist_ok=True)
    target = os.path.join(OUT, lib_name(name))
    stamp = target + ".cfg"
    cfg_text = repr(sorted(v.items())) + FIXTURE_ROOT
    if not force and os.path.exists(target) and os.path.exists(stamp) and open(stamp).read() == cfg_text:
        return target
    scratch = tempfile.mkdtemp(prefix="evs_ref_build_")
    try:
        for f in SOURCES + HEADERS:
            with open(os.path.join(REF_SRC, f)) as fh:
                text = fh.read()
            with open(os.path.join(scratch, f), "w") as fh:
                fh.write(patch(text, f, v))
        cmd = ["g++", "-shared", "-o", target, "-fPIC", "-O3", "-w"] + SOURCES + ["-pthread"]
        subprocess.run(cmd, cwd=scratch, check=True)
        with open(stamp, "w") as fh:
            fh.write(cfg_text)
    finally:
        shutil.rmtree(scratch, ignore_errors=True)
    return target


def build_driver(force: bool = False) -> str:
    """oracle/ref_drive.c (our own trace replayer) -> oracle/_ref/libref_drive.so."""
    os.makedirs(OUT, exist_ok=True)
    src = os.path.join(HERE, "ref_drive.c")
    target = os.path.join(OUT, "libref_drive.so")
    if force or not os.path.exists(target) or os.path.getmtime(src) > os.path.getmtime(target):
        subprocess.run(["gcc", "-O2", "-shared", "-fPIC", "-o", target, src], check=True)
    return target


def build_shim(force: bool = False) -> str:
    """oracle/stdset_shim.cpp (libstdc++ unordered_set<string> behind a C ABI) -> oracle/_ref/libstdset_shim.so."""
    os.makedirs(OUT, exist_ok=True)
    src = os.path.join(HERE, "stdset_shim.cpp")
    target = os.path.join(OUT, "libstdset_shim.so")
    if force or not os.path.exists(target) or os.path.getmtime(src) > os.path.getmtime(target):
        subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-o", target, src], check=True)
    return target


def main(argv):
    build_driver(force="--force" in argv)
    build_shim(force="--force" in argv)
    if not REF_SRC or not os.path.isdir(REF_SRC):
        print("oracle/build_ref.py: no reference checkout (EVSTORE_REFERENCE); built the oracle's own helpers only")
        return 0
    names = [a for a in argv if not a.startswith("-")] or list(VARIANTS)
    for n in names:
        t = build_variant(n, VARIANTS[n], force="--force" in argv)
        print("built", os.path.relpath(t, os.path.dirname(HERE)))
    return 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
