"""lsb_unique_device at every radix from 1 to 16, in every pass shape, sorted and consecutive, on the inputs
tests/test_unique_decisive_cpu.py proves -- needs a B200.

There every fault of the unique kernels' model (a bit of a round's word left out of the compare, an earlier round's
flag dropped or overwritten, lane 0 reading the wrong neighbour, tile and grid-stride starts forced, a tile numbered
from the next tile's base, raw bits compared instead of order keys, inverse, index or counts written wrong) changes the
output, so a comparison of the whole output here sees it.  Results are compared bit for bit with tests/unique_ref.py,
which builds groups from numpy's own comparison of the typed values and shares no code with order_key.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import distributed_lsb_b200 as lsb  # noqa: E402
import lexsort_ref as R  # noqa: E402
import unique_decisive as U  # noqa: E402
import unique_ref as UR  # noqa: E402
from distributed_lsb_b200 import hostlogic as H  # noqa: E402
from test_gpu_every_radix import RADICES, SHAPES, SHAPE_IDS, _close_sorters, _sorter  # noqa: E402,F401

CASES = sorted(U.cases())


def _inputs():
    """(mix, flipped, consecutive) -> (columns, reference): built once for the module"""
    if not _inputs.cache:
        for (mix, flipped), (names, desc) in U.cases().items():
            for consecutive in (False, True):
                _, cols = U.block_input(mix, flipped, consecutive)
                _inputs.cache[mix, flipped, consecutive] = cols, UR.reference(cols, names, list(desc), consecutive)
    return _inputs.cache


_inputs.cache = {}


def _check(s, cols, names, desc, consecutive, want):
    n = len(cols[0])
    ts = [R.to_device(torch, b, x) for b, x in zip(cols, names)]
    before = [t.clone() for t in ts]
    outs = [torch.full((n,), U.SENTINEL, dtype=torch.int64, device="cuda") for _ in range(3)]
    index, inverse, counts, u, st = s.unique_device(ts, descending=list(desc), consecutive=consecutive,
                                                    index_out=outs[0], inverse_out=outs[1], counts_out=outs[2])
    what = (names, desc, consecutive, s.radix_bits, n)
    assert u == len(want[0]), what
    for got, w, full in ((index, want[0], True), (inverse, want[1], False), (counts, want[2], True)):
        g = got.cpu().numpy()
        assert np.array_equal(g[:len(w)], w), what
        assert not full or (g[len(w):] == U.SENTINEL).all(), what
    rounds = H.lexsort_rounds([R.WIDTH[x] for x in names], s.radix_bits)
    assert st.passes == (0 if consecutive else sum(r[3] for r in rounds)), what
    for t, b in zip(ts, before):
        assert torch.equal(t.view(torch.uint8), b.view(torch.uint8)), what


def _params():
    return [pytest.param(r, f, id=f"r{r}-{SHAPE_IDS[f]}") for r in RADICES for f in SHAPES]


# ---- 1. every mix in both directions, sorted and consecutive, at every radix and pass shape -----------------------------------
@pytest.mark.parametrize("radix,shape", _params())
def test_unique(radix, shape):
    s = _sorter(U.BLOCK_N, radix, shape)
    for (mix, flipped, consecutive), (cols, want) in sorted(_inputs().items()):
        names, desc = U.cases()[mix, flipped]
        _check(s, cols, names, desc, consecutive, want)


# ---- 2. the flag kernel over at least three IO_U steps of its grid stride --------------------------------------------------
@pytest.mark.parametrize("mix", [2, 6])
@pytest.mark.parametrize("consecutive", [False, True], ids=["sorted", "consecutive"])
def test_grid_stride_boundaries(mix, consecutive):
    """group starts decided by each earlier round alone, and non-starts, on the grid-stride and IO_U-step boundaries of
    unique_flag_kernel, at the stride of this card's SM count"""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    names, desc = U.cases()[mix, False]
    b, cols, stride = U.large_input(mix, False, consecutive, sms)
    assert set(U.grid_targets(b, stride, U.LARGE_N).values()) - {None} == set(range(len(U.rounds(names)) - 1))
    want = UR.reference(cols, names, list(desc), consecutive)
    for radix, shape in ((16, 0), (8, SHAPES[-1])):
        s = lsb.DistributedSorter(U.LARGE_N, ranks=1, radix_bits=radix, flags=shape)
        try:
            _check(s, cols, names, desc, consecutive, want)
        finally:
            s.close()


# ---- 3. rows through lsb.unique / lsb.unique_consecutive -------------------------------------------------------------------
ROW_MIXES = [("float32",) * 3, ("bfloat16",) * 5, ("int64", "int64"), ("float64",) * 2]


@pytest.mark.parametrize("names", ROW_MIXES, ids=lambda x: f"{x[0]}x{len(x)}")
def test_rows(names):
    """rows (slices along dim) built from a decisive block of columns of one type: entry 0 of a row is the primary
    column"""
    desc = (False,) * len(names)
    for consecutive in (False, True):
        b = U.Block(names, desc, consecutive)
        cols = U.elements(b, U.block_lengths(b))
        want = UR.reference(cols, names, list(desc), consecutive)
        ts = [R.to_device(torch, c, names[0]) for c in cols]
        x = torch.stack(ts[::-1], dim=1)  # x[i] = element i, most significant column first
        for t, dim in ((x, 0), (x.t().contiguous(), 1), (x.t().contiguous().unsqueeze(0), -1)):
            before = t.clone()
            if consecutive:
                v, inverse, counts = lsb.unique_consecutive(t, return_inverse=True, return_counts=True, dim=dim)
            else:
                v, index, inverse, counts = lsb.unique(t, return_index=True, return_inverse=True, return_counts=True, dim=dim)
                assert np.array_equal(index.cpu().numpy(), want[0]), (names, dim)
            assert np.array_equal(inverse.cpu().numpy(), want[1]) and np.array_equal(counts.cpu().numpy(), want[2]), (names, dim)
            rows = torch.index_select(t.view({8: torch.int64, 4: torch.int32, 2: torch.int16}[t.element_size()]), dim % t.dim(),
                                      torch.from_numpy(want[0]).cuda())
            assert torch.equal(v.view(rows.dtype), rows), (names, dim, consecutive)
            assert torch.equal(t.view(torch.uint8), before.view(torch.uint8))
