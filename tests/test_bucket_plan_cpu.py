"""The bucket plan of a one-GPU sort of 64-bit keys (hostlogic.bucket_plan, the rule of plan_bucket / bucket_accepts in
csrc/lsbsort.cu): how many top bytes are scattered before the bucket pass, and which inputs stay on the byte steps."""
import numpy as np
import pytest

from distributed_lsb_b200 import hostlogic as H


@pytest.mark.parametrize("here,k", [(1, 2), (1 << 20, 2), (1 << 23, 2), ((1 << 23) + 1, 3), (1 << 30, 3), (1 << 31, 3),
                                    ((1 << 31) + 1, 4), (1 << 39, 4), ((1 << 39) + 1, 5)])
def test_bytes_keep_the_mean_bucket_at_most_128(here, k):
    assert H.bucket_bytes(here) == k
    assert here <= 128 * 256 ** k and (k == 2 or here > 128 * 256 ** (k - 1))
    assert H.bucket_bytes(here, forced=4) == 4


def uniform_counts(here):
    return np.full((8, 256), here // 256)


def test_uniform_keys_take_the_plan_above_2_pow_20():
    for here in (1 << 20, 1 << 26, 1 << 30):
        assert H.bucket_plan(uniform_counts(here), here) == H.bucket_bytes(here)
        assert H.bucket_plan(uniform_counts(here), here, radix_bits=8) == H.bucket_bytes(here)
    here = (1 << 20) - 256
    assert H.bucket_plan(uniform_counts(here), here) == 0
    assert H.bucket_plan(uniform_counts(here), here, mode=2) == 2


@pytest.mark.parametrize("radix", [1, 4, 7, 11, 12, 13, 15])
def test_other_radixes_never_take_it(radix):
    assert H.bucket_plan(uniform_counts(1 << 24), 1 << 24, radix_bits=radix, mode=2) == 0


def test_a_crowded_top_byte_declines():
    here = 1 << 23
    c = uniform_counts(here)
    c[7, 3] = 2 * here // 256  # exactly twice its share: accepted
    assert H.bucket_plan(c, here) == 2
    c[7, 3] += 1
    assert H.bucket_plan(c, here) == 0
    assert H.bucket_plan(c, here, mode=2) == 2  # mode 2 skips the histogram test
    assert H.bucket_plan(c, here, mode=1) == 0
    c = uniform_counts(here)
    c[0, 0] = here // 2  # a low byte may be skewed: the bucket pass sorts it on chip
    assert H.bucket_plan(c, here) == 2


def test_a_constant_byte_declines_unless_skipping_is_off():
    here = 1 << 23
    c = uniform_counts(here)
    c[1] = 0
    c[1, 9] = here
    assert H.bucket_plan(c, here) == 0
    assert H.bucket_plan(c, here, mode=2) == 0
    assert H.bucket_plan(c, here, no_skip=True) == 2


def test_masked_and_and_of_draws_keys_decline():
    rng = np.random.default_rng(5)
    here = 1 << 21
    k = rng.integers(0, 1 << 64, size=here, dtype=np.uint64, endpoint=False)
    assert H.bucket_plan(H.byte_counts(k), here) == 2
    assert H.bucket_plan(H.byte_counts(k & np.uint64(0xFFFFFF)), here) == 0
    assert H.bucket_plan(H.byte_counts(k & np.uint64(0xFFFFFF)), here, no_skip=True) == 0
    k3 = k & rng.integers(0, 1 << 64, size=here, dtype=np.uint64) & rng.integers(0, 1 << 64, size=here, dtype=np.uint64)
    assert H.bucket_plan(H.byte_counts(k3), here) == 0


def test_stats_count_scatter_launches():
    assert H.sort_stats(0) == (8, 8, 10)
    assert H.sort_stats(0, skipped=5) == (3, 3, 5)
    assert H.sort_stats(3) == (8, 4, 6)
    assert H.sort_stats(3, overflow=True) == (11, 12, 14)
    assert H.sort_stats(2) == (8, 3, 5)
