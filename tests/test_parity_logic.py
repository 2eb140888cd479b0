"""CPU: the parity checker itself (tests/parity.py) -- a checker that excuses everything proves nothing.  A fake
"GPU" result is derived from the oracle's and perturbed: mismatches at a genuine quantisation-boundary tie must be
accepted and counted, a mismatch away from a boundary, a tie that jumps two bins, or a wrong outlier value must fail."""
import numpy as np
import pytest

from tests import parity, reflib


class FakeCtx:
    """stands in for dctz_b200.Context.dct_blocks: a float32/float64 DCT of the unscaled block by another algorithm"""

    def dct_blocks(self, x, dn=64, inverse=False):
        from scipy.fft import dct

        return dct(x.reshape(-1, dn), type=2, norm="ortho", axis=1).astype(x.dtype).reshape(-1)


def _fake_gpu(orc):
    st = orc["stat"]
    return dict(bin_index=orc["bin_index"].copy(), dc=orc["dc"].copy(), ac=orc["ac"].copy(), qtable=orc["qtable"].copy(),
                info=dict(max_abs=st["max"], min_abs=st["min"], sf=st["sf"], sum=st["sum"], n_outliers=orc["ac"].size, n_qt_dropped=0))


def _field(dtype, boundary_gap):
    """blocks with one AC coefficient placed `boundary_gap` above a bin boundary (sf == 1: values in (1, 10])"""
    from scipy.fft import idct

    eb, nblk = 1e-3, 64
    c = np.zeros((nblk, 64))
    c[:, 0] = 40.0
    c[np.arange(nblk), 1 + np.arange(nblk) % 63] = -255 * eb + 100 * 2 * eb + boundary_gap
    return idct(c, type=2, norm="ortho", axis=-1).reshape(-1).astype(dtype), eb


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_identical_results_pass_and_report_no_ties(dtype):
    x, eb = _field(dtype, 3e-4)
    orc = reflib.oracle_compress(x, eb, False)
    rep = parity.compare_compress(_fake_gpu(orc), orc, x, eb, False, ctx=FakeCtx())
    assert rep["ties"] == 0 and rep["bin_mismatch"] == 0


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_mismatch_away_from_a_boundary_fails(dtype):
    x, eb = _field(dtype, 3e-4)  # 0.15 bins above the boundary: far outside any rounding error
    orc = reflib.oracle_compress(x, eb, False)
    g = _fake_gpu(orc)
    j = 1  # block 0's placed coefficient
    t = parity.ordinal_of(g["bin_index"][j:j + 1], orc["coef"][j:j + 1])[0]
    g["bin_index"][j] = 254 - 2 * (t - 1) if t - 1 <= 127 else 2 * (t - 1 - 127) - 1  # the bin below
    with pytest.raises(AssertionError, match="away from a boundary"):
        parity.compare_compress(g, orc, x, eb, False, ctx=FakeCtx())
    with pytest.raises(AssertionError, match="away from a boundary"):
        parity.compare_compress(g, orc, x, eb, False, ctx=None)  # the 8-ulp fallback window must not excuse it either


def _independent_result(x, orc, eb):
    """a second, independent implementation built like the GPU path: scipy's float32 DCT of the UNSCALED block, the
    division by sf folded in afterwards, the quantiser in exact arithmetic"""
    g = _fake_gpu(orc)
    c = FakeCtx().dct_blocks(x).astype(np.float64) / orc["stat"]["sf"]
    bw, rmin, rmax = parity.quant_consts(eb, np.float32)
    t = np.floor((c - rmin) / bw).astype(np.int64)
    ids = np.where(t <= 127, 254 - 2 * t, 2 * (t - 127) - 1)
    ids[(c < rmin) | (c > rmax) | (t > 254)] = 255
    ids[::64] = 255
    g["bin_index"] = ids.astype(np.uint8)
    g["dc"] = c[::64].astype(np.float32)
    m = (g["bin_index"] == 255) & (np.arange(c.size) % 64 != 0)
    g["ac"] = c[m].astype(np.float32)
    g["info"]["n_outliers"] = int(m.sum())
    return g


def test_genuine_ties_are_accepted_counted_and_limited_to_one_bin():
    from scipy.fft import idct

    eb, nblk = 1e-3, 4096
    rng = np.random.default_rng(8)
    c = np.zeros((nblk, 64))
    c[:, 0] = 40.0
    c[np.arange(nblk), 1 + np.arange(nblk) % 63] = -255 * eb + rng.integers(0, 256, nblk) * 2 * eb  # exactly on boundaries
    x = idct(c, type=2, norm="ortho", axis=-1).reshape(-1).astype(np.float32)
    orc = reflib.oracle_compress(x, eb, False)
    g = _independent_result(x, orc, eb)
    rep = parity.compare_compress(g, orc, x, eb, False, ctx=FakeCtx())
    assert 0 < rep["ties"] <= nblk and rep["tie_window_max"] < 0.02 * 2 * eb, rep  # ties exist; the window is a sliver of a bin
    # the same mismatches moved one bin further are not ties any more
    d = np.nonzero(g["bin_index"] != orc["bin_index"])[0]
    d = d[(g["bin_index"][d] != 255) & (orc["bin_index"][d] != 255)]
    j = d[0]
    tg = int(parity.ordinal_of(g["bin_index"][j:j + 1], orc["coef"][j:j + 1])[0])
    to = int(parity.ordinal_of(orc["bin_index"][j:j + 1], orc["coef"][j:j + 1])[0])
    far = tg + (tg - to)
    g["bin_index"][j] = 254 - 2 * far if far <= 127 else 2 * (far - 127) - 1
    with pytest.raises(AssertionError):
        parity.compare_compress(g, orc, x, eb, False, ctx=FakeCtx())


def test_wrong_outlier_value_fails():
    rng = np.random.default_rng(3)
    x = (3.0 + rng.standard_normal(64 * 50) * 0.5).astype(np.float64)
    orc = reflib.oracle_compress(x, 1e-3, False)
    assert orc["ac"].size > 100
    g = _fake_gpu(orc)
    g["ac"][7] = np.float32(g["ac"][7] * (1 + 1e-5))
    with pytest.raises(AssertionError, match="outlier values differ"):
        parity.compare_compress(g, orc, x, 1e-3, False, ctx=FakeCtx())


class FakeDecoder:
    """stands in for dctz_b200.Context.decompress_core: the oracle's own reconstruction, optionally perturbed"""

    def __init__(self, perturb=None):
        self.perturb = perturb

    def decompress_core(self, bins, dc, ac, n, dtype, eb, sf, qt=False, qtable=None):
        r = reflib.oracle_decompress(bins, dc, ac, qtable, n, eb, sf, qt, dtype)
        return self.perturb(r, sf) if self.perturb else r


def _tiny_field():
    """double field at the bottom of the exponent range (sf = 1e-307): one block of small values among larger ones"""
    t = np.arange(64 * 40, dtype=np.float64)
    x = 3.0 + np.sin(t / 29.0) * 2.0
    x[64 * 7:64 * 8] = 1e-3 * np.cos(t[:64] / 5.0)
    return x * 1e-307


def test_decompress_tolerance_has_no_absolute_floor_and_follows_the_block():
    x = _tiny_field()
    parity.check_decompress(FakeDecoder(), x, 1e-3, False)  # the oracle against itself

    def shift_all(r, sf):  # 1e-9 of sf everywhere: 1e3 times the tolerance, but far below the old 1e-300 floor
        return r + 1e-9 * sf

    with pytest.raises(AssertionError, match="beyond the tolerance"):
        parity.check_decompress(FakeDecoder(shift_all), x, 1e-3, False)

    def shift_small_block(r, sf):  # within RTOL of the FIELD's maximum, far outside RTOL of block 7's
        r = r.copy()
        r[64 * 7 + 3] += 1e-12 * sf
        return r

    with pytest.raises(AssertionError, match="beyond the tolerance"):
        parity.check_decompress(FakeDecoder(shift_small_block), x, 1e-3, False)

    def make_inf(r, sf):
        r = r.copy()
        r[5] = np.inf
        return r

    with pytest.raises(AssertionError, match="non-finite"):
        parity.check_decompress(FakeDecoder(make_inf), x, 1e-3, False)


def test_equal_infinite_sums_agree_and_a_finite_sum_never_matches_an_infinite_one():
    x = np.full(1 << 16, 3e304)  # sum 1.97e309
    orc = reflib.oracle_compress(x, 1e-3, False)
    assert orc["stat"]["sum"] == np.inf  # the reference's running sum overflows
    g = _fake_gpu(orc)
    parity.compare_compress(g, orc, x, 1e-3, False, ctx=FakeCtx())
    g["info"]["sum"] = 1.7e308
    with pytest.raises(AssertionError):
        parity.compare_compress(g, orc, x, 1e-3, False, ctx=FakeCtx())
    g["info"]["sum"] = -np.inf
    with pytest.raises(AssertionError):
        parity.compare_compress(g, orc, x, 1e-3, False, ctx=FakeCtx())
    assert parity.sums_agree(np.inf, np.inf, x, 1e304) and not parity.sums_agree(np.inf, 1e308, x, 1e304)
    assert not parity.sums_agree(1e308, np.inf, x, 1e304)


class OverflowCtx(FakeCtx):
    """a transform that overflowed: every coefficient infinite"""

    def dct_blocks(self, x, dn=64, inverse=False):
        return np.full_like(x, np.inf)


def test_a_non_finite_gpu_coefficient_is_a_failure_not_a_tie():
    x, eb = _field(np.float64, 3e-4)
    orc = reflib.oracle_compress(x, eb, False)
    g = _fake_gpu(orc)
    j = 1
    t = parity.ordinal_of(g["bin_index"][j:j + 1], orc["coef"][j:j + 1])[0]
    g["bin_index"][j] = 254 - 2 * (t - 1) if t - 1 <= 127 else 2 * (t - 1 - 127) - 1  # the bin below
    with pytest.raises(AssertionError, match="non-finite"):
        parity.compare_compress(g, orc, x, eb, False, ctx=OverflowCtx())


def test_a_float_sum_the_reference_could_not_accumulate():
    """2^25 floats near 25: the reference's float running sum stalls near 2^29 (each addend is below half an ulp), so the
    GPU's double sum is judged against the exact sum instead -- and a wrong GPU sum still fails"""
    x = (25.0 + np.sin(np.arange(1 << 25) / 77.0)).astype(np.float32)
    ref = reflib.oracle_stat(x)
    exact = float(np.sum(x[1:].astype(np.float64)))
    assert abs(ref["sum"] - exact) > 0.1 * exact  # the reference's own sum is far off
    assert parity.sums_agree(exact, ref["sum"], x, ref["sf"])
    assert not parity.sums_agree(exact * (1 + 1e-6), ref["sum"], x, ref["sf"])
    assert not parity.sums_agree(ref["sum"] * 1.5, ref["sum"], x, ref["sf"])
    # double data keeps the tight rule alone
    assert not parity.sums_agree(exact, ref["sum"], x.astype(np.float64), ref["sf"])
