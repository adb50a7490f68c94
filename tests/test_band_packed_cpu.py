"""Stage 2 from band storage, host side: the diagonal range the packed working layout relies on, and the band storage
convention of pack_upper_band.

The packed layout keeps 3c diagonals per row, -(c-1) .. 2c-1 (csrc/stage2_common.cuh, Layout).  That holds every element
the chase reads or writes only because every window of either schedule lies inside those diagonals; the first test
proves it by brute force over the window lists (the same lists tests/test_stage2_head.py checks the sweep head on)."""
import numpy as np
import pytest

from svdsolver_b200.capi import pack_upper_band
from test_stage2_head import _ops_complete, _ops_reference


def _diagonal_range(ops, n, c):
    lo, hi = None, None
    for i in range(n - 1):
        for w in ops(i, n, c):
            if not w or w[1] <= w[0] or w[3] <= w[2]:
                continue
            r0, r1, c0, c1 = w
            a, b = c0 - (r1 - 1), (c1 - 1) - r0       # lowest / highest diagonal col - row the window touches
            lo = a if lo is None else min(lo, a)
            hi = b if hi is None else max(hi, b)
    return lo, hi


@pytest.mark.parametrize("complete", [0, 1])
@pytest.mark.parametrize("c", [1, 2, 4, 7, 13, 32, 64])
def test_windows_lie_in_3c_diagonals(c, complete):
    """Every window of both schedules lies in diagonals -(c-1) .. 2c-1, and the bounds are reached once the matrix has room
    for a full RIGHT(0) (rows i .. i+c) and LEFT(0) (columns up to i+2c)."""
    ops = _ops_complete if complete else _ops_reference
    for n in (2, 3, 5, 64, 65, 66, 67, 96, 97, 100, 129, 130, 200, 331, 1000):
        lo, hi = _diagonal_range(ops, n, c)
        assert -(c - 1) <= lo and hi <= 2 * c - 1, (n, lo, hi)
        if n >= 2 * c + 1:
            assert (lo, hi) == (-(c - 1), 2 * c - 1), (n, lo, hi)


@pytest.mark.parametrize("n,band", [(1, 1), (5, 1), (8, 3), (10, 4), (33, 32), (64, 7), (100, 13), (5, 8)])
def test_pack_upper_band_is_scipy_ab_transposed(n, band):
    """pack_upper_band(a, u)[j, t] == scipy's upper ab[t, j] (ab[u + i - j, j] == a[i, j]), n a multiple of the band or not"""
    import scipy.linalg
    rng = np.random.default_rng(n * 131 + band)
    a = np.triu(np.tril(rng.uniform(0.5, 5.0, (n, n)), band)) + np.diag(np.full(n, 5.0 * (band + 1)))   # well conditioned
    ab = pack_upper_band(a, band)
    assert ab.shape == (n, band + 1) and ab.dtype == a.dtype
    ref = np.zeros((band + 1, n))
    for j in range(n):
        for i in range(max(0, j - band), j + 1):
            ref[band + i - j, j] = a[i, j]
    assert np.array_equal(ab.T, ref)
    # scipy reads it the same way: solve_banded((0, u), ab^T, y) solves the upper band system
    y = rng.uniform(-1.0, 1.0, n)
    x = scipy.linalg.solve_banded((0, band), np.ascontiguousarray(ab.T), y)
    np.testing.assert_allclose(a @ x, y, rtol=0, atol=1e-9 * max(1.0, np.abs(y).max()))
    # the entries above the matrix (t < band - j) stay zero, whatever the input holds outside the band
    full = rng.uniform(1.0, 2.0, (n, n))
    abf = pack_upper_band(full, band)
    for j in range(min(n, band)):
        assert not abf[j, : band - j].any()
