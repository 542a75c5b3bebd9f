"""unique without a GPU: the reference of tests/unique_ref.py against numpy and torch, the mapping of dim to key columns,
the Python layer's refusals, and the header's declaration of lsb_unique_device.
"""
import numpy as np
import pytest

import lexsort_ref as LR
import unique_ref as U

torch = pytest.importorskip("torch")

import distributed_lsb_b200 as lsb  # noqa: E402
from distributed_lsb_b200 import lsbsort as L  # noqa: E402

NUMPY_TYPED = [x for x in LR.NAMES if x != "bfloat16"]  # numpy has no bfloat16: its reference widens it to float32


@pytest.mark.parametrize("name", NUMPY_TYPED)
def test_reference_is_numpy_unique(name):
    """1-D keys with NaN payloads of both signs, +-0, infinities and subnormals: np.unique(equal_nan=True)"""
    for n, seed in ((1, 0), (2, 1), (1000, 2), (50000, 3)):
        for bits in (LR.special_mix(n, name, seed=seed), LR.few_values(n, name, 7, seed=seed)):
            x = LR.typed(bits, name)
            values, index, inverse, counts = np.unique(x, return_index=True, return_inverse=True, return_counts=True,
                                                       equal_nan=True)
            got = U.reference([bits], [name])
            assert np.array_equal(got[0], index) and np.array_equal(got[1], inverse.reshape(-1))
            assert np.array_equal(got[2], counts)
            assert np.array_equal(x[got[0]].view(bits.dtype), values.view(bits.dtype))  # the first occurrence's bits


def test_reference_descending_and_consecutive():
    bits = LR.few_values(5000, "float32", 9, seed=4)
    x = LR.typed(bits, "float32")
    index, inverse, counts = U.reference([bits], ["float32"], [True])
    asc = U.reference([bits], ["float32"])
    assert np.array_equal(index, asc[0][::-1]) and np.array_equal(counts, asc[2][::-1])
    assert np.array_equal(inverse, len(index) - 1 - asc[1])
    index, inverse, counts = U.reference([bits], ["float32"], consecutive=True)
    same = (x[1:] == x[:-1]) | (np.isnan(x[1:]) & np.isnan(x[:-1]))
    assert np.array_equal(index, np.concatenate([[0], np.flatnonzero(~same) + 1]))
    assert counts.sum() == len(x) and np.array_equal(inverse, np.cumsum(np.concatenate([[0], ~same])))


@pytest.mark.parametrize("dtype", [np.int64, np.int32, np.uint16, np.int16])
def test_reference_rows_are_numpy_axis0(dtype):
    """NaN-free integer rows: np.unique(axis=0), with the first entry of a row the primary key"""
    rng = np.random.default_rng(5)
    names = {np.int64: "int64", np.int32: "int32", np.uint16: "uint16", np.int16: "int16"}
    for m in (1, 2, 3, 5):
        x = rng.integers(-3 if dtype != np.uint16 else 0, 3, (4000, m)).astype(dtype)
        _, index, inverse, counts = np.unique(x, axis=0, return_index=True, return_inverse=True, return_counts=True)
        bits = [np.ascontiguousarray(x[:, j]).view(LR.UINT[np.dtype(dtype).itemsize * 8]) for j in reversed(range(m))]
        got = U.reference(bits, [names[dtype]] * m)
        assert np.array_equal(got[0], index) and np.array_equal(got[1], inverse.reshape(-1))
        assert np.array_equal(got[2], counts)


def _bits(t):
    """a CPU tensor's bit patterns as numpy unsigned integers"""
    w = t.element_size() * 8
    return t.view({64: torch.int64, 32: torch.int32, 16: torch.int16}[w]).numpy().view(LR.UINT[w])


@pytest.mark.parametrize("dtype", [torch.int64, torch.float32, torch.int16])
def test_dim_columns_against_torch(dtype):
    """_unique_columns for every dim of a 3-D tensor: the reference over its columns, values = x.index_select(dim,
    index), gives torch.unique(dim=d)'s values, inverse and counts"""
    name = str(dtype).replace("torch.", "")
    rng = np.random.default_rng(6)
    x = torch.from_numpy(rng.integers(-2, 2, (7, 5, 6)).astype(np.int64)).to(dtype)
    x[3] = x[1]  # equal slices along every dim somewhere
    x[:, 4] = x[:, 0]
    x[:, :, 5] = x[:, :, 2]
    for dim in (0, 1, 2, -1, -3):
        size, shape, cols = L._unique_columns(torch, x, dim)
        assert size == x.shape[dim] and shape == (size,) and all(c.is_contiguous() for c in cols)
        index, inverse, counts = U.reference([_bits(c) for c in cols], [name] * len(cols))
        values = x.index_select(dim % 3, torch.from_numpy(index))
        want = torch.unique(x, dim=dim, return_inverse=True, return_counts=True)
        assert torch.equal(values, want[0]) and np.array_equal(inverse, want[1].numpy())
        assert np.array_equal(counts, want[2].numpy()), dim
    size, shape, cols = L._unique_columns(torch, x, None)
    assert size == x.numel() and shape == x.shape and len(cols) == 1
    index, inverse, counts = U.reference([_bits(cols[0])], [name])
    want = torch.unique(x, return_inverse=True, return_counts=True)
    assert torch.equal(x.reshape(-1)[torch.from_numpy(index)], want[0])
    assert np.array_equal(inverse.reshape(x.shape), want[1].numpy()) and np.array_equal(counts, want[2].numpy())


def test_refusals_before_the_device():
    x = torch.zeros(4, dtype=torch.int64)
    for fn in (lsb.unique, lsb.unique_consecutive):
        with pytest.raises(TypeError):
            fn([1, 2, 3])
        for dtype in (torch.int8, torch.uint8, torch.bool, torch.complex64):
            with pytest.raises(TypeError):
                fn(torch.zeros(4, dtype=dtype))
        with pytest.raises(ValueError, match="CUDA"):
            fn(x)
        with pytest.raises(TypeError):
            fn(x, dim=True)
        with pytest.raises(TypeError):
            fn(x, dim=0.0)
        for dim in (1, -2):
            with pytest.raises(IndexError):
                fn(x, dim=dim)
        with pytest.raises(IndexError):
            fn(torch.tensor(3), dim=0)
        with pytest.raises(ValueError, match="empty"):
            fn(torch.zeros(3, 0), dim=0)


def test_header_declares_unique():
    assert "lsb_unique_device" in lsb.header_symbols()
    with open(L._HEADER) as f:
        assert "#define LSB_UNIQUE_CONSECUTIVE 1u" in f.read()
    assert L.UNIQUE_CONSECUTIVE == 1
