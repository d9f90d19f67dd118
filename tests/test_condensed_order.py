"""CPU: locohd_condensed_unit, the unit order of the condensed mode of score_tile_kernel (the same inline function the
kernel calls).  A chunk of row blocks [rb0, rb1) of a range of n environments (nb = ceil(n / 4) blocks of 4) owns the
4 x 4 blocks (rb, cb) with rb0 <= rb < rb1 and rb <= cb < nb; its units must visit each of them once, column block
major, row blocks ascending within a column block - at small sizes, where every unit is compared, and at 64-bit unit
counts, where the closed form's square root has to be corrected to the exact integer."""
import pytest

from loco_hd_b200 import _capi
from loco_hd_b200._capi import LocoHDError


def _blocks(n):
    return (n + 3) // 4


def _expected(n, rb0, row_blocks):
    rb1 = rb0 + row_blocks
    return [(rb, cb) for cb in range(rb0, _blocks(n)) for rb in range(rb0, min(cb + 1, rb1))]


def _chunks(n):
    nb = _blocks(n)
    out = {(0, nb), (0, 1), (nb - 1, 1)}                       # whole range, first and last single row block
    if nb >= 3:
        out |= {(nb // 3, max(1, nb // 4)), (nb // 2, 1), (1, nb - 1)}   # chunks that start inside the range
    return sorted(out)


@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 37, 4096])
def test_units_are_the_chunks_upper_blocks_in_column_block_major_order(n):
    for rb0, row_blocks in _chunks(n):
        want = _expected(n, rb0, row_blocks)
        got = [_capi.condensed_unit(n, rb0, row_blocks, u) for u in range(len(want))]
        assert got == want, (n, rb0, row_blocks)
        with pytest.raises(LocoHDError) as e:   # one past the last unit
            _capi.condensed_unit(n, rb0, row_blocks, len(want))
        assert e.value.status == 10


def _triangle(k):
    return k * (k + 1) // 2


@pytest.mark.parametrize("k", [2 ** 31 - 1, 2 ** 31, 2 ** 31 + 1, 2 ** 32 - 1, 2 ** 32, 2 ** 32 + 1])
def test_exact_at_64_bit_unit_counts(k):
    """Column block k of the triangle starts at unit T(k): T(k) - 1 is the diagonal block of column block k - 1,
    T(k) and T(k) + 1 the first two row blocks of column block k.  The chunk has 2^32 + 8 row blocks (T ~ 2^63) and
    three column blocks after them."""
    rb0, row_blocks, rect = 5, 2 ** 32 + 8, 3
    n = 4 * (rb0 + row_blocks + rect) - 1
    assert _triangle(row_blocks) + row_blocks * rect < 2 ** 64
    T = _triangle(k)
    assert _capi.condensed_unit(n, rb0, row_blocks, T - 1) == (rb0 + k - 1, rb0 + k - 1)
    assert _capi.condensed_unit(n, rb0, row_blocks, T) == (rb0, rb0 + k)
    assert _capi.condensed_unit(n, rb0, row_blocks, T + 1) == (rb0 + 1, rb0 + k)


def test_rectangle_and_limits_at_64_bit_unit_counts():
    rb0, row_blocks, rect = 5, 2 ** 32 + 8, 3
    n = 4 * (rb0 + row_blocks + rect)
    tri = _triangle(row_blocks)
    rb1 = rb0 + row_blocks
    assert _capi.condensed_unit(n, rb0, row_blocks, tri - 1) == (rb1 - 1, rb1 - 1)   # last diagonal block
    assert _capi.condensed_unit(n, rb0, row_blocks, tri) == (rb0, rb1)
    assert _capi.condensed_unit(n, rb0, row_blocks, tri + row_blocks + 7) == (rb0 + 7, rb1 + 1)
    last = tri + row_blocks * rect - 1
    assert _capi.condensed_unit(n, rb0, row_blocks, last) == (rb1 - 1, rb1 + rect - 1)
    with pytest.raises(LocoHDError):
        _capi.condensed_unit(n, rb0, row_blocks, last + 1)
    # a chunk of 2^33 row blocks has more than 2^64 units
    with pytest.raises(LocoHDError):
        _capi.condensed_unit(4 * 2 ** 33, 0, 2 ** 33, 0)


@pytest.mark.parametrize("n,rb0,row_blocks", [(37, 0, 0), (37, 10, 1), (37, 9, 2), (0, 0, 1), (2 ** 64 - 1, 2 ** 62, 1)])
def test_chunks_outside_the_blocks_are_refused(n, rb0, row_blocks):
    with pytest.raises(LocoHDError) as e:
        _capi.condensed_unit(n, rb0, row_blocks, 0)
    assert e.value.status == 10
