"""Element ranges of sub-boxes of a field, for Context.decompress_ranges_dev.

The codec sees a field as one flat run of N elements in C order, the way dctz-test.c flattens r1 x r2 x ... fields, so
a sub-box is a set of contiguous runs along the fastest axis.  box_ranges merges runs that touch: full rows of a plane
become one range per plane, full planes one range in all.
"""
from __future__ import annotations

import numpy as np


def box_ranges(shape, lo, hi) -> np.ndarray:
    """{first element, count} pairs (uint64, shape (n, 2)) of the C-order sub-box [lo, hi) of a field of `shape`,
    in the order numpy's `field[lo0:hi0, lo1:hi1, ...]` lists the elements.  Every extent must be non-empty and
    inside the field."""
    shape = tuple(int(s) for s in shape)
    lo = tuple(int(v) for v in lo)
    hi = tuple(int(v) for v in hi)
    if not (len(shape) == len(lo) == len(hi)) or not shape:
        raise ValueError(f"shape {shape}, lo {lo} and hi {hi} must have the same, non-zero number of axes")
    for ax, (s, a, b) in enumerate(zip(shape, lo, hi)):
        if not 0 <= a < b <= s:
            raise ValueError(f"axis {ax}: [{a}, {b}) is empty or leaves [0, {s})")
    # the trailing axes the box covers whole, plus the first one it cuts, form one contiguous run per index of the
    # axes before them
    k = len(shape) - 1
    while k > 0 and lo[k] == 0 and hi[k] == shape[k]:
        k -= 1
    inner = int(np.prod(shape[k + 1:], dtype=np.int64))
    strides = [int(np.prod(shape[i + 1:], dtype=np.int64)) for i in range(len(shape))]
    first = np.zeros(1, dtype=np.uint64)
    for i in range(k):
        first = (first[:, None] + np.arange(lo[i], hi[i], dtype=np.uint64)[None, :] * np.uint64(strides[i])).reshape(-1)
    first = first + np.uint64(lo[k] * strides[k])
    out = np.empty((first.size, 2), dtype=np.uint64)
    out[:, 0] = first
    out[:, 1] = (hi[k] - lo[k]) * inner
    return out
