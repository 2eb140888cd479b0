"""CPU: box_ranges turns a C-order sub-box into the element ranges numpy's slicing lists, merged where they touch."""
import numpy as np
import pytest

from dctz_b200.regions import box_ranges


def _expand(r):
    return np.concatenate([np.arange(a, a + c, dtype=np.int64) for a, c in r.astype(np.int64)])


def _check(shape, lo, hi):
    r = box_ranges(shape, lo, hi)
    assert r.dtype == np.uint64 and r.ndim == 2 and r.shape[1] == 2
    want = np.arange(int(np.prod(shape))).reshape(shape)[tuple(slice(a, b) for a, b in zip(lo, hi))].reshape(-1)
    assert np.array_equal(_expand(r), want)
    # merged: no range ends where the next one starts
    assert not np.any(r[1:, 0] == r[:-1, 0] + r[:-1, 1])
    return r


def test_random_boxes():
    rng = np.random.default_rng(11)
    for _ in range(300):
        nd = int(rng.integers(1, 5))
        shape = tuple(int(v) for v in rng.integers(1, 9, size=nd))
        lo, hi = [], []
        for s in shape:
            a = int(rng.integers(0, s))
            lo.append(a)
            hi.append(int(rng.integers(a + 1, s + 1)))
        _check(shape, lo, hi)


def test_full_rows_become_one_range_per_plane():
    r = _check((5, 6, 7), (1, 2, 0), (4, 5, 7))
    assert r.tolist() == [[1 * 42 + 2 * 7, 21], [2 * 42 + 14, 21], [3 * 42 + 14, 21]]


def test_full_planes_become_one_range():
    assert _check((5, 6, 7), (1, 0, 0), (4, 6, 7)).tolist() == [[42, 126]]
    assert _check((5, 6, 7), (0, 0, 0), (5, 6, 7)).tolist() == [[0, 210]]


def test_planes_of_a_large_field():
    shape = (256, 2048, 2048)
    assert box_ranges(shape, (7, 0, 0), (8, 2048, 2048)).tolist() == [[7 << 22, 1 << 22]]  # z-plane
    y = box_ranges(shape, (0, 9, 0), (256, 10, 2048))                                     # y-plane: one row per z
    assert y.shape == (256, 2) and np.all(y[:, 1] == 2048) and y[1, 0] - y[0, 0] == 1 << 22
    x = box_ranges(shape, (0, 0, 5), (256, 2048, 6))                                      # x-plane: single elements
    assert x.shape == (1 << 19, 2) and np.all(x[:, 1] == 1) and x[-1, 0] == (1 << 30) - 2048 + 5


@pytest.mark.parametrize("shape,lo,hi", [((100,), (3,), (97,)), ((100,), (0,), (100,)), ((10, 12), (2, 3), (9, 4)),
                                         ((10, 12), (2, 0), (9, 12)), ((10, 12), (0, 5), (10, 12))])
def test_one_and_two_dimensional_fields(shape, lo, hi):
    _check(shape, lo, hi)


@pytest.mark.parametrize("lo,hi", [((0, 3, 0), (2, 3, 4)), ((0, 0, 0), (2, 5, 4)), ((-1, 0, 0), (2, 2, 2)), ((1, 1, 1), (1, 2, 2))])
def test_empty_or_outside_extents_are_rejected(lo, hi):
    with pytest.raises(ValueError):
        box_ranges((3, 4, 4), lo, hi)


def test_axis_count_must_match():
    with pytest.raises(ValueError):
        box_ranges((3, 4), (0,), (1,))
