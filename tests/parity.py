"""TEST INFRASTRUCTURE: parity checks of the CUDA path (through the C-ABI) against the CPU oracle.

Tolerances are the ones BASELINE.json's north_star states: DCT coefficients within 1e-12 relative
(double) / 1e-5 (float) -- relative to the largest coefficient magnitude of the block --, bin indices
and outlier sets bit-exact except at quantisation-boundary ties, whose count is reported.  A "tie" is a
coefficient that lies closer to a bin boundary (or to the outlier range limit) than the two implementations'
MEASURED coefficient errors against the exact DCT (tie_windows), so that it may legitimately round to either
side; a tie may move by one bin only.
"""
from __future__ import annotations

import numpy as np

from . import reflib

RTOL = {np.dtype(np.float64): 1e-12, np.dtype(np.float32): 1e-5}


def quant_consts(eb, dtype):
    """dctz-comp-lib.c:271-281."""
    dtype = np.dtype(dtype)
    bw, rmin, rmax = eb * 2.0, -255 * eb, 255 * eb
    if dtype == np.float32:
        bw, rmin, rmax = np.float32(bw), np.float32(rmin), np.float32(rmax)
    return float(bw), float(rmin), float(rmax)


def block_max(coef):
    """max |coef| of the 64-block each element belongs to (same shape as coef)."""
    n = coef.size
    nblk = (n + 63) // 64
    pad = np.zeros(nblk * 64, dtype=np.float64)
    pad[:n] = np.abs(coef)
    m = pad.reshape(nblk, 64).max(axis=1)
    return np.repeat(m, 64)[:n]


def boundary_distance(coef, eb, dtype):
    """distance of each coefficient to the nearest bin boundary rmin + t*bw, t = 0..255."""
    bw, rmin, rmax = quant_consts(eb, dtype)
    c = coef.astype(np.float64)
    v = (c - rmin) / bw
    t = np.clip(np.rint(v), 0, 255)
    return np.abs(v - t) * bw


def ulp32(a):
    a = np.abs(a.astype(np.float32))
    return (np.nextafter(a, np.float32(np.inf)) - a).astype(np.float64)


def ordinal_of(ids, coef):
    """inverse of conv_tbl (dctz-comp-lib.c:27-43): stream id -> ordinal bin t (0..254); the outlier marker 255 becomes
    -1 or 255 according to the side of the range the coefficient lies on"""
    ids = ids.astype(np.int64)
    t = np.where(ids % 2 == 0, (254 - ids) // 2, (ids + 255) // 2)
    return np.where(ids == 255, np.where(coef < 0, -1, 255), t)


_DCT_M = {}


def dct_matrix(dn):
    """orthonormal DCT-II matrix in float64 (exact enough to judge float32 coefficients)"""
    if dn not in _DCT_M:
        k = np.arange(dn)[:, None]
        m = np.arange(dn)[None, :]
        M = np.sqrt(2.0 / dn) * np.cos(np.pi * (((2 * m + 1) * k) % (4 * dn)) / (2.0 * dn))
        M[0] /= np.sqrt(2.0)
        _DCT_M[dn] = M
    return _DCT_M[dn]


def exact_coefficients(blocks, dtype):
    """exact DCT-II of scaled blocks [nb, dn]: float64 matrix product for float32 data (1e-16 vs the 6e-8 being judged),
    the oracle's long-double definition-based transform for float64 data"""
    blocks = np.ascontiguousarray(blocks, dtype=np.float64)
    if np.dtype(dtype) == np.float32:
        return blocks @ dct_matrix(blocks.shape[1]).T
    return np.stack([reflib.oracle_dct_exact(b) for b in blocks])


def tie_windows(diff, orc, x, eb, ctx):
    """Distance of the EXACT coefficient to the nearest bin boundary, and the half-width of the tie window, for every
    mismatching element.  The window is the MEASURED error of the two implementations'
    coefficients against the exact DCT of the same scaled block, plus the rounding of the quantiser expression itself
    ((c - range_min)/bin_width evaluated in the element type by the reference, fma(c, kq, 127.5) by the GPU: a few ulps
    of a value up to 255).  Without a GPU context the GPU's coefficient error is bounded by 8 ulps of the block's
    largest coefficient instead."""
    dtype = np.dtype(x.dtype)
    n = x.size
    bw = quant_consts(eb, dtype)[0]
    eps = 2.0 ** -23 if dtype == np.float32 else 2.0 ** -52
    expr = 255.0 * 2.0 * eps * bw
    sf = orc["stat"]["sf"]
    nfull = n // 64
    tol = np.empty(diff.size)
    dist = np.empty(diff.size)
    blocks = diff // 64
    ub = np.unique(blocks)
    groups = [(ub[ub < nfull], 64)]
    if n % 64 and ub.size and ub[-1] == nfull:
        groups.append((ub[-1:], n % 64))
    for ids, dn in groups:
        if ids.size == 0:
            continue
        idx = (ids[:, None] * 64 + np.arange(dn)[None, :])
        ce = exact_coefficients(orc["scaled"][idx], dtype)
        err_o = np.abs(orc["coef"][idx].astype(np.float64) - ce)
        if ctx is not None:  # the kernels transform the UNSCALED block and fold the division into the quantiser
            cg = ctx.dct_blocks(np.ascontiguousarray(x[idx]).reshape(-1), dn=dn).astype(np.float64).reshape(ids.size, dn) / sf
            # an overflowed (or NaN) coefficient would make an infinite window that excuses any mismatch as a "tie"
            assert np.all(np.isfinite(cg)), f"non-finite GPU coefficient in block(s) {ids[~np.all(np.isfinite(cg), axis=1)][:5]}"
            err_g = np.abs(cg - ce) + np.abs(ce) * eps
        else:
            m = np.max(np.abs(ce), axis=1, keepdims=True)
            u = ulp32(m) if dtype == np.float32 else np.spacing(m)
            err_g = np.broadcast_to(8.0 * u, ce.shape)
        win = err_o + err_g + expr
        assert np.all(np.isfinite(win)), "non-finite tie window"
        pos = np.searchsorted(ids, blocks)
        sel = (pos < ids.size) & (ids[np.minimum(pos, ids.size - 1)] == blocks)
        tol[sel] = win[pos[sel], diff[sel] - blocks[sel] * 64]
        dist[sel] = boundary_distance(ce[pos[sel], diff[sel] - blocks[sel] * 64], eb, np.float64)  # of the EXACT coefficient
    return dist, tol


def sums_agree(got, want, x, sf):
    """The GPU's sum of the data (double, another order) against the reference's, compared in the scaled domain (relative to
    sum|x/sf| >= 1, so a tiny sf does not make the check vacuous).  A sum of finite data may overflow: two infinite sums
    agree iff they are the same infinity; a finite sum never agrees with an infinite one."""
    if np.isinf(got) or np.isinf(want):
        if np.dtype(x.dtype) == np.float32 and np.isinf(want) and not np.isinf(got):
            # the reference sums float data in float: it overflows where the GPU's double sum passes FLT_MAX
            return np.sign(got) == np.sign(want) and abs(got) > float(np.finfo(np.float32).max)
        return got == want
    rel = 1e-9 if np.dtype(x.dtype) == np.float64 else 2e-3
    return abs(got / sf - want / sf) <= rel * float(np.sum(np.abs(x.astype(np.float64) / sf)))


def decode_tolerance(want, sf):
    """Per-element bound on |got - want| / sf for a reconstruction `want` (element type) of a stream with scaling factor
    sf: RTOL * 8 of the block's largest |want/sf|, plus two ulps of that maximum in the element type (the rounding of the
    output itself, which near the bottom of the range is subnormal).  No absolute floor: an all-zero block must decode to
    exact zeros."""
    dtype = np.dtype(want.dtype)
    bm = block_max(want.astype(np.float64))
    ulp = ulp32(bm) if dtype == np.float32 else np.spacing(bm)
    return RTOL[dtype] * 8 * (bm / sf) + 2 * ulp / sf


def compare_compress(gpu, orc, x, eb, qt, ctx=None, check_stats=True):
    """gpu: result of Context.compress_core; orc: reflib.oracle_compress (or reference dumps with the
    same keys).  Asserts parity and returns a report.  `ctx` (a dctz_b200.Context) lets the tie criterion use the
    GPU's measured coefficient error (tie_windows).  check_stats=False: `gpu` is a WINDOW of a larger slab that was
    compressed with the field's global statistics (bench.py's per-rank check): only sf must agree."""
    dtype = np.dtype(x.dtype)
    rtol = RTOL[dtype]
    n = x.size
    coef = orc["coef"].astype(np.float64)
    bmax = block_max(coef)
    ctol = rtol * np.maximum(bmax, 1e-300)  # north_star's coefficient tolerance: used for DC / outlier VALUES below
    rep = {}

    # statistics (util.c:12-44): max/min are exact selections, sf must be bit-identical
    st = orc["stat"]
    info = gpu["info"]
    assert info["sf"] == st["sf"], (info["sf"], st["sf"])
    if check_stats:
        assert info["max_abs"] == st["max"], (info["max_abs"], st["max"])
        assert info["min_abs"] == st["min"], (info["min_abs"], st["min"])
        assert sums_agree(info["sum"], st["sum"], x, st["sf"]), (info["sum"], st["sum"])

    # bin indices: bit-exact except at quantisation-boundary ties.  A mismatch is a tie iff the exact coefficient lies
    # within the two implementations' measured errors of a bin boundary; a tie may only move to the neighbouring bin
    # (or in / out of the outlier range at its limit).
    gb, ob = gpu["bin_index"], orc["bin_index"]
    assert gb.shape == ob.shape
    diff = np.nonzero(gb != ob)[0]
    rep["bin_mismatch"] = int(diff.size)
    if diff.size:
        assert diff.size <= max(64, n // 8), f"{diff.size} of {n} bin indices differ: not a tie phenomenon"
        dist, tol = tie_windows(diff, orc, x, eb, ctx)
        not_tie = diff[dist > tol]
        assert not_tie.size == 0, f"{not_tie.size} bin indices differ away from a boundary, first at {not_tie[:5]}: " \
                                  f"gpu {gb[not_tie[:5]]} oracle {ob[not_tie[:5]]} coef {coef[not_tie[:5]]} " \
                                  f"distance {dist[dist > tol][:5]} window {tol[dist > tol][:5]}"
        step = np.abs(ordinal_of(gb[diff], coef[diff]) - ordinal_of(ob[diff], coef[diff]))
        assert step.max() <= 1, f"a tie moved by {int(step.max())} bins at {diff[np.argmax(step)]}"
        rep["tie_window_max"] = float(tol.max())
    rep["ties"] = int(diff.size)
    rep["tie_fraction"] = diff.size / max(n, 1)

    # DC (dctz-comp-lib.c:351): float of the block's first coefficient
    gdc, odc = gpu["dc"].astype(np.float64), orc["dc"].astype(np.float64)
    dc_tol = ctol[::64] + ulp32(orc["dc"])
    bad = np.nonzero(np.abs(gdc - odc) > dc_tol)[0]
    assert bad.size == 0, f"DC differs in {bad.size} blocks, first {bad[:5]}: {gdc[bad[:5]]} vs {odc[bad[:5]]}"

    # outliers: same set (up to ties), same order, same float values
    pos = np.arange(n) % 64
    gmask = (gb == 255) & (pos != 0)
    omask = (ob == 255) & (pos != 0)
    rep["n_outliers"] = int(info["n_outliers"])
    assert gpu["ac"].size == info["n_outliers"]
    # every 255 marker owns exactly one stored outlier: the decoder's serial cursor (dctz-decomp-lib.c:370,402) can never
    # desynchronise.  (The reference would drop a rescaled QT outlier that fell back inside the range, :494-506; the GPU
    # path proves that unreachable and counts it -- DESIGN.md §2.)
    assert info.get("n_qt_dropped", 0) == 0
    assert int(gmask.sum()) == info["n_outliers"], (int(gmask.sum()), info["n_outliers"])
    gval = np.full(n, np.nan)
    oval = np.full(n, np.nan)
    gval[gmask] = gpu["ac"]
    oval[omask] = orc["ac"] if orc["ac"].size == int(omask.sum()) else np.nan
    both = gmask & omask & ~np.isnan(gval) & ~np.isnan(oval)
    if qt:
        # rescaled value = range +- (c/qtable[j]) * 10 eb: sensitivity to c is 10 eb / qtable[j] <= 10 eb
        ac_tol = 10 * eb * ctol[both] + 2 * ulp32(oval[both].astype(np.float32))
    else:
        ac_tol = ctol[both] + ulp32(oval[both].astype(np.float32))
    bad = np.nonzero(np.abs(gval[both] - oval[both]) > ac_tol)[0]
    assert bad.size == 0, f"{bad.size} outlier values differ, e.g. {gval[both][bad[:5]]} vs {oval[both][bad[:5]]}"
    rep["outlier_set_diff"] = int((gmask != omask).sum())
    assert rep["outlier_set_diff"] <= rep["ties"]

    if qt:
        # qtable (dctz-comp-lib.c:371-372, 450-461): a max over existing values -> exact unless a tie changed the set
        gq, oq = gpu["qtable"].astype(np.float64), orc["qtable"].astype(np.float64)
        qtol = rtol * max(1.0, float(np.max(np.abs(coef)))) * 4
        assert np.all(np.abs(gq - oq) <= qtol), (gq, oq)
        rep["qtable_exact"] = bool(np.array_equal(gpu["qtable"][1:], orc["qtable"][1:]))
    return rep


def check_compress(ctx, x, eb, qt):
    gpu = ctx.compress_core(x, eb, qt=qt, want_scaled=True)
    orc = reflib.oracle_compress(x, eb, qt)
    rep = compare_compress(gpu, orc, x, eb, qt, ctx=ctx)
    # the in-place scaling the reference leaves in the caller's buffer: IEEE division, bit-exact
    assert np.array_equal(gpu["scaled"], orc["scaled"]), "x/sf is not bit-identical to the reference's division"
    return rep


def check_decompress(ctx, x, eb, qt):
    """Feed the ORACLE's compressed arrays to the GPU decompressor; compare with the oracle's own
    reconstruction (dctz-decomp-lib.c:358-511)."""
    dtype = np.dtype(x.dtype)
    orc = reflib.oracle_compress(x, eb, qt, want_coef=False)
    sf = orc["stat"]["sf"]
    want = reflib.oracle_decompress(orc["bin_index"], orc["dc"], orc["ac"], orc["qtable"], x.size, eb, sf, qt, dtype)
    got = ctx.decompress_core(orc["bin_index"], orc["dc"], orc["ac"], x.size, dtype, eb, sf, qt=qt, qtable=orc["qtable"])
    return check_reconstruction(got, want, sf)


def check_reconstruction(got, want, sf):
    """got against the oracle's reconstruction of the same stream, in the scaled domain (decode_tolerance)."""
    assert got.dtype == want.dtype and got.shape == want.shape
    assert np.all(np.isfinite(got)), f"{int(np.sum(~np.isfinite(got)))} non-finite values in the reconstruction"
    d = np.abs(got.astype(np.float64) / sf - want.astype(np.float64) / sf)
    tol = decode_tolerance(want, sf)
    bad = np.nonzero(d > tol)[0]
    assert bad.size == 0, f"{bad.size} elements differ beyond the tolerance, first at {bad[:5]}: got {got[bad[:5]]} want {want[bad[:5]]} (sf {sf})"
    scale = float(np.max(np.abs(want))) if want.size else 1.0
    diff = float(np.max(np.abs(got.astype(np.float64) - want.astype(np.float64)))) if want.size else 0.0
    return dict(max_diff=diff, scale=scale, max_scaled_diff=float(d.max()) if d.size else 0.0)
