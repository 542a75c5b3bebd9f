"""Narrow keys past 2^31 elements through lsb.sort -- needs a B200 with the memory named in each skip.

float32 at 2^31 + 2^20 + 7 elements (1-D: sort_device with 32-bit indices) and bfloat16 rows of 2^30 + 2^19 + 3 (two
rows: the segmented sort packs global input indices past 2^31 and returns row-local ones).  Each result is checked by
tests/sort_check.py on the keys widened exactly to float64, and by a chunked bit-for-bit check that out == in[idx] at
the key's own width.
"""
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import distributed_lsb_b200 as lsb  # noqa: E402
import sort_check as C  # noqa: E402
from test_gpu_large import GiB, _room  # noqa: E402

BIG = (1 << 31) + (1 << 20) + 7
ROW = (1 << 30) + (1 << 19) + 3


def _keys(n, dtype, seed):
    """special doubles narrowed to the key type (NaNs, infinities, -0.0 and subnormals survive the cast)"""
    out = torch.empty(n, dtype=dtype, device="cuda")
    for lo in range(0, n, C.CHUNK):
        hi = min(n, lo + C.CHUNK)
        out[lo:hi] = C.special_doubles(hi - lo, "cuda", seed=seed * 4096 + lo // C.CHUNK).view(torch.float64).to(dtype)
    return out


def _widened(t):
    out = torch.empty(t.numel(), dtype=torch.float64, device=t.device)
    for lo in range(0, t.numel(), C.CHUNK):
        out[lo:lo + C.CHUNK] = t[lo:lo + C.CHUNK].to(torch.float64)
    return out


def _same_bits(keys_in, keys_out, idx):
    w = torch.int32 if keys_in.element_size() == 4 else torch.int16
    a, b = keys_in.view(w), keys_out.view(w)
    for lo in range(0, a.numel(), C.CHUNK):
        assert torch.equal(b[lo:lo + C.CHUNK], a[idx[lo:lo + C.CHUNK]]), lo


def test_float32_past_2p31():
    n = BIG
    _room("float32 sort of 2^31 + 2^20 + 7", 32 * n + 4 * 2 * n + 8 * n + n + 12 * 8 * C.CHUNK + 2 * 8 * n)
    x = _keys(n, torch.float32, seed=1)
    for descending in (False, True):
        values, indices = lsb.sort(x, descending=descending)
        torch.cuda.empty_cache()
        _same_bits(x, values, indices)
        wi, wo = _widened(x), _widened(values)
        msg = C.check_sort(wi, wo, indices, C.F64 | (C.DESC if descending else 0))
        assert msg is None, "\n" + msg
        del values, indices, wi, wo


def test_bfloat16_rows_past_2p31():
    rows, n = 2, 2 * ROW
    _room("bfloat16 rows of 2 x (2^30 + 2^19 + 3)", 32 * n + 2 * 2 * n + 8 * n + n + 12 * 8 * C.CHUNK + 2 * 8 * n + GiB)
    x = _keys(n, torch.bfloat16, seed=2).view(rows, ROW)
    values, indices = lsb.sort(x, dim=1)
    torch.cuda.empty_cache()
    offsets = torch.arange(rows + 1, dtype=torch.int64, device="cuda") * ROW
    glob = (indices + offsets[:-1, None]).reshape(-1)
    _same_bits(x.reshape(-1), values.reshape(-1), glob)
    del glob
    local = C.LocalIndex(indices.reshape(-1), offsets)
    msg = C.check_sort(_widened(x.reshape(-1)), _widened(values.reshape(-1)), local, C.F64, offsets)
    assert msg is None, "\n" + msg
