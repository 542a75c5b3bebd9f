"""CPU-only checks of the device-tensor entry points (sort_tensor, DistributedSorter.sort_device): malformed tensors are
refused in Python with TypeError / ValueError before the library is called, and lsb_sort_device is declared in the
header and bound in load_library."""
import inspect

import pytest

torch = pytest.importorskip("torch")

import distributed_lsb_b200 as lsb  # noqa: E402
from distributed_lsb_b200 import lsbsort as L  # noqa: E402


class _NoLibrary:
    def __getattr__(self, name):
        raise AssertionError(f"library called ({name}) before the arguments were checked")


def _sorter(here=16, flags=0, device=0):
    """a DistributedSorter shell whose library must not be reached"""
    s = object.__new__(L.DistributedSorter)
    s._L, s._ctx = _NoLibrary(), None
    s.here, s.device, s.flags = here, device, flags
    return s


def test_lsb_sort_device_declared_and_bound():
    assert "lsb_sort_device" in lsb.header_symbols()
    assert "L.lsb_sort_device.argtypes" in inspect.getsource(L.load_library)


def test_module_imports_without_torch_at_import_time():
    src = inspect.getsource(L)
    assert "\nimport torch" not in src and "\nfrom torch" not in src


BAD_KEYS = [
    (lambda: [1, 2, 3], TypeError),                                          # not a tensor
    (lambda: torch.zeros(16, dtype=torch.int32), TypeError),                 # 4-byte keys
    (lambda: torch.zeros(16, dtype=torch.float32), TypeError),
    (lambda: torch.zeros(4, 4, dtype=torch.int64), ValueError),              # 2-D
    (lambda: torch.zeros(16, dtype=torch.int64), ValueError),                # on the CPU
]


@pytest.mark.parametrize("case", range(len(BAD_KEYS)))
def test_sort_tensor_rejects(case):
    make, err = BAD_KEYS[case]
    with pytest.raises(err):
        lsb.sort_tensor(make())


def test_vals_checks():
    """the checks sort_tensor and sort_device apply to vals and outputs (CPU tensors, so each case must fail a check
    that comes before the device check)"""
    for vals, err in [(torch.zeros(16, dtype=torch.int32), TypeError), (torch.zeros(16, dtype=torch.float32), TypeError),
                      (torch.zeros(15, dtype=torch.int64), ValueError), (torch.zeros(16, 1, dtype=torch.int64), ValueError),
                      (torch.zeros(32, dtype=torch.int64)[::2], ValueError), ([0] * 16, TypeError)]:
        with pytest.raises(err):
            L._check_vector(torch, vals, "vals", 16)
    with pytest.raises(ValueError, match="CUDA"):
        L._check_vector(torch, torch.zeros(16, dtype=torch.float64), "vals", 16)


@pytest.mark.parametrize("flags,dtype", [(0, torch.int64), (L.FLAG_KEY_I64, torch.uint64), (L.FLAG_KEY_F64, torch.int64),
                                         (L.FLAG_KEY_I64 | L.FLAG_DESCENDING, torch.float64), (0, torch.int32)])
def test_sort_device_rejects_key_dtype_not_matching_flags(flags, dtype):
    with pytest.raises(TypeError):
        _sorter(flags=flags).sort_device(torch.zeros(16, dtype=dtype))


def test_sort_device_rejects_shapes_layouts_and_devices():
    s = _sorter(here=16, flags=L.FLAG_KEY_I64)
    i64 = lambda *shape: torch.zeros(*shape, dtype=torch.int64)  # noqa: E731
    for keys, err, what in [(i64(4, 4), ValueError, "1-D"), (i64(32)[::2], ValueError, "contiguous"),
                            (i64(15), ValueError, "elements"), (i64(16), ValueError, "CUDA"),
                            (i64(16).numpy(), TypeError, "torch.Tensor")]:
        with pytest.raises(err, match=what):
            s.sort_device(keys)


def test_sort_device_rejects_no_outputs():
    with pytest.raises(ValueError, match="both"):
        _sorter(here=16, flags=L.FLAG_KEY_F64).sort_device(torch.zeros(16, dtype=torch.float64), keys_out=False,
                                                           vals_out=False)
