"""Key orders without a GPU: order_key as compiled from csrc/lsb_keyorder.cuh (host code, nvcc) sorts special values
exactly as numpy sorts the typed view, the tests' numpy restatement (tests/key_orders.py) computes the same bits, and
the flag constants of the Python layer are the header's."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import distributed_lsb_b200 as lsb
import key_orders as KO
from distributed_lsb_b200 import lsbsort as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROG = r'''
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "lsb_keyorder.cuh"
int main(int argc, char** argv) {  // flags as argv[1]; uint64 keys on stdin -> order_key(key, flags) on stdout
  const uint32_t flags = (uint32_t)strtoul(argv[1], nullptr, 0);
  std::vector<uint64_t> k;
  uint64_t x;
  while (fread(&x, 8, 1, stdin) == 1) k.push_back(x);
  for (uint64_t& v : k) v = lsb::order_key(v, flags);
  fwrite(k.data(), 8, k.size(), stdout);
  return 0;
}
'''


@pytest.fixture(scope="module")
def device_order_key(tmp_path_factory):
    nvcc = shutil.which("nvcc") or ("/usr/local/cuda/bin/nvcc" if os.path.exists("/usr/local/cuda/bin/nvcc") else None)
    if nvcc is None:
        pytest.skip("nvcc not found")
    d = tmp_path_factory.mktemp("keyorder")
    (d / "prog.cu").write_text(PROG)
    exe = d / "prog"
    subprocess.check_call([nvcc, "-std=c++17", "-I", os.path.join(ROOT, "distributed-lsb_b200", "csrc"),
                           str(d / "prog.cu"), "-o", str(exe)])

    def run(keys, flags):
        out = subprocess.run([str(exe), str(flags)], input=np.ascontiguousarray(keys, dtype=np.uint64).tobytes(),
                             capture_output=True, check=True).stdout
        return np.frombuffer(out, dtype=np.uint64)
    return run


def _keys():
    rng = np.random.default_rng(7)
    return np.concatenate([KO.SPECIAL_BITS, KO.SPECIAL_BITS[rng.integers(0, len(KO.SPECIAL_BITS), 4000)],
                           rng.integers(0, 1 << 64, 3000, dtype=np.uint64),
                           rng.standard_normal(3000).view(np.uint64)])[rng.permutation(len(KO.SPECIAL_BITS) + 10000)]


@pytest.mark.parametrize("order", sorted(KO.ORDERS))
def test_order_key_sorts_like_numpy(order, device_order_key):
    flags = KO.ORDERS[order]
    keys = _keys()
    enc = device_order_key(keys, flags)
    assert np.array_equal(np.argsort(enc, kind="stable"), KO.argsort(keys, flags)), order


@pytest.mark.parametrize("order", sorted(KO.ORDERS))
def test_numpy_restatement_matches_the_header(order, device_order_key):
    flags = KO.ORDERS[order]
    keys = _keys()
    assert np.array_equal(KO.order_key(keys, flags), device_order_key(keys, flags)), order


def test_float_specials_in_order(device_order_key):
    """-0.0 == +0.0, every NaN equal and last ascending (first descending), -inf < -max < -subnormal < 0"""
    b = KO.f64_bits([-np.inf, -1.7976931348623157e308, -5e-324, -0.0, 0.0, 5e-324, 1.0, np.inf])
    enc = device_order_key(b, KO.F64)
    assert (np.diff(enc.astype(object)) >= 0).all() and enc[3] == enc[4] and len(set(enc.tolist())) == 7
    nans = np.array([0x7FF8000000000000, 0xFFF8000000000000, 0x7FF0000000000001, 0xFFF4000000000042], dtype=np.uint64)
    assert set(device_order_key(nans, KO.F64).tolist()) == {(1 << 64) - 1}
    assert set(device_order_key(nans, KO.F64 | KO.DESC).tolist()) == {0}


def test_flag_constants_match_the_header():
    header = open(os.path.join(ROOT, "include", "lsbsort.h")).read()
    defs = {k: int(v) for k, v in re.findall(r"#define LSB_FLAG_([A-Z0-9_]+) (\d+)u", header)}
    assert defs["KEY_I64"] == L.FLAG_KEY_I64 == 16
    assert defs["KEY_F64"] == L.FLAG_KEY_F64 == 32
    assert defs["DESCENDING"] == L.FLAG_DESCENDING == 64
    for name in ("PHASE_EVENTS", "TWO_LEVEL", "ONE_PASS", "NO_SKIP"):
        assert defs[name] == getattr(L, "FLAG_" + name)


def test_sort_pairs_rejects_other_dtypes():
    for dt in (np.float32, np.int32, np.uint32):
        with pytest.raises(TypeError):
            lsb.sort_pairs(np.zeros(4, dtype=dt))
    with pytest.raises(TypeError):
        lsb.sort_pairs(np.zeros(4, dtype=np.float64), np.zeros(4, dtype=np.int32))
