"""Narrow key types without a GPU: order_key_narrow as compiled from csrc/lsb_keyorder.cuh (host code, nvcc) sorts every
type exactly as numpy sorts the typed values, hostlogic.plan_pass covers exactly the key's bits at every radix, sort /
argsort / key_dtype refuse bad arguments before the library is reached, and the typed entry points are declared in the
header and bound in load_library."""
import inspect
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import distributed_lsb_b200 as lsb
import narrow_keys as NK
from distributed_lsb_b200 import hostlogic as H
from distributed_lsb_b200 import lsbsort as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROG = r'''
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "lsb_keyorder.cuh"
int main(int argc, char** argv) {  // key_type, flags as argv; uint32 keys on stdin -> order_key_narrow on stdout
  const uint32_t key_type = (uint32_t)strtoul(argv[1], nullptr, 0), flags = (uint32_t)strtoul(argv[2], nullptr, 0);
  std::vector<uint32_t> k;
  uint32_t x;
  while (fread(&x, 4, 1, stdin) == 1) k.push_back(x);
  for (uint32_t& v : k) {
    const uint64_t w = lsb::narrow_key_word(v, key_type, flags);
    if ((uint32_t)(w >> 32) != v) return 1;  // the raw bits travel unchanged above the order key
    v = (uint32_t)w;
  }
  fwrite(k.data(), 4, k.size(), stdout);
  return 0;
}
'''


@pytest.fixture(scope="module")
def order_narrow(tmp_path_factory):
    nvcc = shutil.which("nvcc") or ("/usr/local/cuda/bin/nvcc" if os.path.exists("/usr/local/cuda/bin/nvcc") else None)
    if nvcc is None:
        pytest.skip("nvcc not found")
    d = tmp_path_factory.mktemp("narrow")
    (d / "prog.cu").write_text(PROG)
    exe = d / "prog"
    subprocess.check_call([nvcc, "-std=c++17", "-I", os.path.join(ROOT, "distributed-lsb_b200", "csrc"),
                           str(d / "prog.cu"), "-o", str(exe)])

    def run(bits, name, descending=False):
        flags = L.FLAG_DESCENDING if descending else 0
        out = subprocess.run([str(exe), str(NK.KEY_TYPE[name]), str(flags)],
                             input=np.asarray(bits).astype(np.uint32).tobytes(), capture_output=True, check=True).stdout
        return np.frombuffer(out, dtype=np.uint32)
    return run


def _keys(name):
    rng = np.random.default_rng(NK.KEY_TYPE[name])
    sp = NK.special_bits(name)
    w = NK.BITS[name]
    k = np.concatenate([sp, sp[rng.integers(0, len(sp), 3000)], NK.special_mix(6000, name, seed=1),
                        rng.integers(0, 1 << w, 3000, dtype=np.uint64).astype(NK.UINT[w])])
    return k[rng.permutation(len(k))]


@pytest.mark.parametrize("descending", [False, True])
@pytest.mark.parametrize("name", NK.NAMES)
def test_order_key_narrow_sorts_like_numpy(name, descending, order_narrow):
    bits = _keys(name)
    enc = order_narrow(bits, name, descending)
    assert int(enc.max()) < 1 << NK.BITS[name]  # the order key stays in the low W bits
    assert np.array_equal(np.argsort(enc, kind="stable"), NK.argsort(bits, name, descending)), (name, descending)


@pytest.mark.parametrize("name", ["float32", "float16", "bfloat16"])
def test_float_specials(name, order_narrow):
    """-0 == +0, every NaN all ones ascending (zero descending), -inf < -max < -subnormal < 0 < subnormal < max < inf"""
    w = NK.BITS[name]
    sp = NK.special_bits(name)
    x = NK.typed(sp, name)
    nans, ordered = sp[np.isnan(x)], sp[~np.isnan(x)]
    assert len(nans) == 9  # quiet, signalling, payloads, both signs, all ones
    assert set(order_narrow(nans, name).tolist()) == {(1 << w) - 1}
    assert set(order_narrow(nans, name, True).tolist()) == {0}
    ordered = ordered[np.argsort(NK.typed(ordered, name), kind="stable")]
    enc = order_narrow(ordered, name).astype(np.int64)
    assert (np.diff(enc) >= 0).all()
    zeros = order_narrow(sp[:2], name)
    assert zeros[0] == zeros[1] == 1 << (w - 1)


@pytest.mark.parametrize("name", ["uint32", "int32", "uint16", "int16"])
def test_integer_extremes(name, order_narrow):
    w = NK.BITS[name]
    bits = np.array([0, 1, (1 << (w - 1)) - 1, 1 << (w - 1), (1 << w) - 1], dtype=np.uint64)
    enc = order_narrow(bits, name).tolist()
    if name.startswith("u"):
        assert enc == bits.tolist()
    else:
        assert enc == [x ^ (1 << (w - 1)) for x in bits.tolist()]
    assert order_narrow(bits, name, True).tolist() == [((1 << w) - 1) ^ e for e in enc]


@pytest.mark.parametrize("key_bits", [16, 32])
@pytest.mark.parametrize("radix", range(1, 17))
def test_plan_pass_clamps_to_the_key(radix, key_bits):
    n = H.num_passes(radix, key_bits=key_bits)
    assert n == -(-key_bits // radix)
    covered = 0
    for d in range(n):
        shift, bits, lo, hi = H.plan_pass(radix, d, key_bits=key_bits)
        assert shift == covered and 1 <= bits <= radix and lo + hi == bits
        covered += bits
    assert covered == key_bits  # no digit reads a bit above the order key (radix 13 at 32 bits: 13, 13, 6)
    assert [H.plan_pass(radix, d) for d in range(H.num_passes(radix))] == \
        [H.plan_pass(radix, d, key_bits=64) for d in range(H.num_passes(radix, key_bits=64))]


def test_header_constants_and_symbols():
    header = open(os.path.join(ROOT, "include", "lsbsort.h")).read()
    defs = {k.lower(): int(v) for k, v in re.findall(r"#define LSB_KEY_([A-Z0-9_]+) (\d+)", header)}
    assert defs.pop("context") == L.KEY_CONTEXT == 0
    short = {"u32": "uint32", "i32": "int32", "f32": "float32", "u16": "uint16", "i16": "int16", "f16": "float16",
             "bf16": "bfloat16"}
    assert {short[k]: v for k, v in defs.items()} == NK.KEY_TYPE
    for name in ("lsb_sort_device_typed", "lsb_sort_segments_device_typed"):
        assert name in lsb.header_symbols()
        assert f"L.{name}.argtypes" in inspect.getsource(L.load_library)


# ---- Python argument checks (the library must not be reached) -------------------------------------------------------
torch = pytest.importorskip("torch")


class _NoLibrary:
    def __getattr__(self, name):
        raise AssertionError(f"library called ({name}) before the arguments were checked")


@pytest.fixture
def no_library(monkeypatch):
    def refuse(*a, **k):
        raise AssertionError("library loaded before the arguments were checked")
    monkeypatch.setattr(L, "load_library", refuse)
    monkeypatch.setattr(L.DistributedSorter, "__init__", refuse)


def test_sort_and_argsort_refuse(no_library):
    cases = [([1.0, 2.0], TypeError), (np.zeros(4, dtype=np.float32), TypeError),
             (torch.zeros(4, dtype=torch.int8), TypeError), (torch.zeros(4, dtype=torch.bool), TypeError),
             (torch.zeros(4, dtype=torch.complex64), TypeError), (torch.zeros(4, dtype=torch.uint8), TypeError),
             (torch.zeros(4, dtype=torch.float32), ValueError), (torch.zeros(2, 3, dtype=torch.bfloat16), ValueError),
             (torch.zeros(4, dtype=torch.int64), ValueError), (torch.zeros((), dtype=torch.float16), ValueError),
             (torch.zeros(0, dtype=torch.uint16), ValueError)]
    for x, err in cases:
        for fn in (lsb.sort, lsb.argsort):
            with pytest.raises(err):
                fn(x)


def test_sorter_key_dtype_refusals(no_library):
    for dt in (torch.float64, torch.int64, torch.uint64, torch.int8, torch.bool, np.float32, "float32"):
        with pytest.raises(TypeError):
            _real_init(key_dtype=dt)
    for flags in (L.FLAG_KEY_I64, L.FLAG_KEY_F64, L.FLAG_KEY_F64 | L.FLAG_DESCENDING):
        with pytest.raises(ValueError):
            _real_init(key_dtype=torch.float32, flags=flags)


_INIT = L.DistributedSorter.__init__  # the constructor as written, kept before no_library replaces it


def _real_init(**kw):
    """DistributedSorter.__init__ on a shell object, with load_library refusing to run"""
    _INIT(object.__new__(L.DistributedSorter), 16, **kw)


def _sorter(key_dtype, here=16, flags=0):
    s = object.__new__(L.DistributedSorter)
    s._L, s._ctx = _NoLibrary(), None
    s.here, s.device, s.flags, s.key_dtype = here, 0, flags, key_dtype
    return s


def test_sorter_with_key_dtype_checks_tensors():
    s = _sorter(torch.float32)
    for keys, err in [(torch.zeros(16, dtype=torch.float64), TypeError), (torch.zeros(16, dtype=torch.int32), TypeError),
                      (torch.zeros(16, dtype=torch.bfloat16), TypeError), (torch.zeros(4, 4, dtype=torch.float32), ValueError),
                      (torch.zeros(32, dtype=torch.float32)[::2], ValueError), (torch.zeros(15, dtype=torch.float32), ValueError),
                      (torch.zeros(16, dtype=torch.float32), ValueError)]:  # the last: on the CPU
        with pytest.raises(err):
            s.sort_device(keys)
    with pytest.raises(ValueError, match="both"):
        s.sort_device(torch.zeros(16, dtype=torch.float32), keys_out=False, vals_out=False)


def test_default_sorter_still_refuses_narrow_keys():
    """without key_dtype a sorter takes the 8-byte key its flags name, as before"""
    for dt in (torch.float32, torch.int32, torch.bfloat16):
        with pytest.raises(TypeError):
            _sorter(None).sort_device(torch.zeros(16, dtype=dt))
