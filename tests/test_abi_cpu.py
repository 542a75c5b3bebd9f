"""CPU-only checks of the boundary: the C-ABI library loads and exports every symbol that
include/lsbsort.h declares, ctypes mirrors match the C structs, and the product path refuses to
run without a GPU instead of falling back."""
import ctypes
import os
import subprocess
import sys

import pytest

import distributed_lsb_b200 as lsb
from distributed_lsb_b200 import lsbsort as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    if not os.path.exists(lsb.library_path()):
        pytest.skip("liblsbsort.so not built (run __graft_entry__.build())")
    declared = lsb.header_symbols()
    assert len(declared) >= 20 and "lsb_sort" in declared and "lsb_pass" in declared
    assert lsb.abi_symbols() == declared
    assert lsb.load_library().lsb_abi_version() == 1


def test_struct_layouts_match_header(tmp_path):
    """compile a tiny C program against the header and compare sizeof/offsetof"""
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "lsbsort.h"\n'
                   'int main(){printf("%zu %zu %zu %zu %zu %zu %zu\\n", sizeof(lsb_config), sizeof(lsb_stats),'
                   'sizeof(lsb_verify), sizeof(lsb_elt), offsetof(lsb_config, seed_base),'
                   'offsetof(lsb_stats, sent), offsetof(lsb_stats, subpass_ms));return 0;}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    want = [ctypes.sizeof(L._Config), ctypes.sizeof(L.Stats), ctypes.sizeof(L.Verify), L.ELT.itemsize,
            L._Config.seed_base.offset, L.Stats.sent.offset, L.Stats.subpass_ms.offset]
    assert got == want


def test_no_cpu_fallback():
    """with no CUDA device visible the library raises instead of sorting on the host; the check runs in a child
    process with CUDA_VISIBLE_DEVICES empty, so it holds on a machine with a GPU as well"""
    if not os.path.exists(lsb.library_path()):
        pytest.skip("liblsbsort.so not built")
    code = ("import sys; sys.path.insert(0, sys.argv[1]); import distributed_lsb_b200 as lsb\n"
            "try:\n    lsb.DistributedSorter(100)\nexcept lsb.LsbError as e:\n    print(e)\n")
    out = subprocess.run([sys.executable, "-c", code, ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         capture_output=True, text=True, check=True).stdout
    assert "no CPU fallback" in out


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "distributed-lsb_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", ".hpp")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.lower().replace("# oracle", ""), f


def test_tune_keys_match_the_header_and_conftest():
    """every lsb_tune key the header documents is accepted, out-of-range values and unknown keys are LSB_ERR_ARG, and
    the partition_kernel defaults tests/conftest.py restores are values the library accepts"""
    import re
    if not os.path.exists(lsb.library_path()):
        pytest.skip("liblsbsort.so not built")
    from conftest import LIB_DEFAULT_TUNE, apply_session_tune
    from patterns import TUNE_DEFAULTS
    header = open(os.path.join(ROOT, "include", "lsbsort.h")).read()
    doc = header[header.index("process-wide tunable"):header.index("int lsb_tune(")]
    keys = set(re.findall(r'"([a-z0-9_]+)"', doc))
    assert {"op_t1", "vparts", "ex_u", "pt_direct", "pt_chunks", "pt_variant", "pt_pf_tiles"} <= keys
    sane = dict(TUNE_DEFAULTS)
    sane.update(LIB_DEFAULT_TUNE)
    assert keys == set(sane), keys ^ set(sane)
    try:
        for k, v in sane.items():
            lsb.tune(k, v)  # the library's own defaults: accepted, and nothing changes for later tests
        for k, bad in [("pt_variant", 2), ("pt_variant", -1), ("pt_chunks", 5), ("pt_direct", 2), ("pt_pf_tiles", -1),
                       ("pt_pf_tiles", 1 << 20), ("vparts", 0), ("ex_u", 5), ("no_such_key", 1)]:
            with pytest.raises(lsb.LsbError):
                lsb.tune(k, bad)
    finally:
        apply_session_tune()
