"""GPU: fields at both ends of the exponent range against the CPU oracle.

The kernels transform the UNSCALED block and fold 1/sf into the quantiser constant kq = 1/(sf*bin_width); decompress
folds *sf into the coefficients before the inverse transform (DESIGN.md §2).  So the GPU arithmetic runs at the
magnitude of the data, and the ends of the range are where it can overflow or lose bits:
- compress admits sf = 1e-302 .. 1e305 (float 1e-32 .. 1e35) and must match the oracle there; outside it every entry
  point fails with DCTZ_GPU_EDEGENERATE (kq or the unscaled transform would overflow);
- decompress must decode every stream the reference can write (sf comes from the stream header): double sf 1e-307 ..
  1e308, float 1e-37 .. 1e38.
Fields are 10^k times patterns that hit the edges of the arithmetic: constant blocks (exactly-zero AC coefficients), smooth
and noisy data, all-zero blocks among non-zero ones, a block of 64 values at the field maximum (the largest DC), a block
alternating +-max (the largest AC coefficients), a single spike, tail blocks of 0, 1, 37 and 63 elements."""
import os

import numpy as np
import pytest
import torch

import dctz_b200
from dctz_b200 import DOUBLE, FLOAT, binding, slabs
from tests import parity, reflib
from tests.test_gpu_device_api import compress_slabs
from tests.test_gpu_ranges import Field, random_ranges

pytestmark = pytest.mark.gpu

EDEGENERATE = -5
EBS = (1e-6, 1e-3, 1e-1)
TAILS = (0, 1, 37, 63)
# decades of sf: every one near both ends of what the reference writes
DECADES = {np.dtype(np.float64): list(range(-307, -294)) + list(range(295, 309)),
           np.dtype(np.float32): list(range(-37, -27)) + list(range(28, 39))}
# the decades compress admits (build_sf_tables)
ADMITTED = {np.dtype(np.float64): (-302, 305), np.dtype(np.float32): (-32, 35)}
ERROR_BOUND = (1 + 63 * np.sqrt(2)) / 8 * 1.01  # times eb: the orthonormal-basis bound of test_roundtrip_error_bound


def _ctx(**env):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        return dctz_b200.Context(0)
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v


@pytest.fixture(scope="module")
def contexts():
    """fused kernels for small fields (the default), streaming with the pre-pass decoder, streaming with count-ahead"""
    cs = dict(fused=_ctx(), prepass=_ctx(DCTZ_FUSED_MAX_MB=0, DCTZ_DECOMP_AHEAD=0), ahead=_ctx(DCTZ_FUSED_MAX_MB=0, DCTZ_DECOMP_AHEAD=1))
    yield cs
    for c in cs.values():
        c.close()


def pattern(tail, seed=3):
    """max|p| == 1 exactly, attained by a whole block, an alternating block and a spike"""
    rng = np.random.default_rng(seed)
    t = np.arange(64, dtype=np.float64)
    blocks = [np.full(64, 0.5), np.full(64, -0.8)]                                    # constant: exactly-zero AC
    blocks += [0.6 + 0.3 * np.sin((t + 64 * i) / 23.0) for i in range(4)]           # smooth
    blocks += [0.5 + 0.1 * rng.standard_normal(64) for _ in range(4)]                 # noisy
    blocks += [np.zeros(64), np.zeros(64), 0.3 * np.cos(t / 5.0), np.zeros(64)]       # zero blocks among non-zero ones
    blocks += [np.ones(64), (-1.0) ** t]                                              # at the maximum; +-max
    spike = np.zeros(64)
    spike[17] = -1.0
    blocks += [spike]
    blocks += [1e-3 * np.sin((t + 64 * i) / 7.0) for i in range(4)]                  # small values next to large ones
    blocks += [0.4 + 0.2 * np.sin(np.arange(tail) / 3.0)]
    p = np.concatenate(blocks)
    assert np.max(np.abs(p)) == 1.0
    return p


def field(dtype, k, tail=None, peak=None):
    """10^k * peak * pattern, multiplied in float64 and cast once: max|x| in (10^k, 10^(k+1)), so sf = 10^k"""
    dtype = np.dtype(dtype)
    tail = TAILS[k % 4] if tail is None else tail
    if peak is None:
        top = float(np.finfo(dtype).max)
        peak = 5.0 if 5.0 * 10.0 ** k < top else 0.9 * top / 10.0 ** k
    return (pattern(tail) * peak * 10.0 ** k).astype(dtype)


def admitted(dtype, sf):
    lo, hi = ADMITTED[np.dtype(dtype)]
    return 10.0 ** lo * (1 - 1e-6) <= sf <= 10.0 ** hi * (1 + 1e-6)


def oracle_stream(x, eb, qt):
    orc = reflib.oracle_compress(x, eb, qt)
    sf = orc["stat"]["sf"]
    want = reflib.oracle_decompress(orc["bin_index"], orc["dc"], orc["ac"], orc["qtable"], x.size, eb, sf, qt, x.dtype)
    return orc, want


def scaled_error(x, r, sf):
    return np.abs(x.astype(np.float64) / sf - r.astype(np.float64) / sf)


def error_bound(bins, dc, ac, eb, r, sf):
    """Oracle-free bound on |x - r| / sf per element of an EC stream: eb * (1 + 63 sqrt 2) / 8 from the bins (as
    test_roundtrip_error_bound), plus what the stream keeps as float -- half a float ulp of the DC and of every outlier of
    the block, through basis functions of at most sqrt(2/dn) (DC: 1/sqrt(dn)) -- plus the arithmetic of the element type:
    64 ulps of the block's largest |r / sf| for the forward and the inverse transform, and the rounding of r itself."""
    n = r.size
    nblk = (n + 63) // 64
    dn = np.full(nblk, 64.0)
    if n % 64:
        dn[-1] = n % 64
    mark = (bins == 255) & (np.arange(n) % 64 != 0)
    kept = np.zeros(nblk)
    np.add.at(kept, np.nonzero(mark)[0] // 64, parity.ulp32(np.asarray(ac, dtype=np.float32)[: int(mark.sum())]) / 2)
    per_blk = kept * np.minimum(1.0, np.sqrt(2 / dn)) + parity.ulp32(dc) / 2 / np.sqrt(dn)
    eps = 2.0 ** -23 if r.dtype == np.float32 else 2.0 ** -52
    rs = np.abs(r.astype(np.float64) / sf)
    arith = 64 * eps * parity.block_max(rs) + (parity.ulp32(r) if r.dtype == np.float32 else np.spacing(np.abs(r.astype(np.float64)))) / 2 / sf
    return (eb * ERROR_BOUND + np.repeat(per_blk, 64)[:n]) * 1.01 + arith


def assert_error_bound(x, r, bins, dc, ac, eb, sf):
    err = scaled_error(x, r, sf)
    bound = error_bound(bins, dc, ac, eb, r, sf)
    bad = np.nonzero(err > bound)[0]
    assert bad.size == 0, f"error bound exceeded at {bad[:5]}: {err[bad[:5]]} > {bound[bad[:5]]} (eb {eb})"


def check_decode(contexts, x, eb, qt, orc, want):
    """the oracle's stream through every decoder: finite, within the scaled tolerance of the oracle, identical bits"""
    sf = orc["stat"]["sf"]
    outs = [c.decompress_core(orc["bin_index"], orc["dc"], orc["ac"], x.size, x.dtype, eb, sf, qt=qt, qtable=orc["qtable"])
            for c in contexts.values()]
    parity.check_reconstruction(outs[0], want, sf)
    for o in outs[1:]:
        assert np.array_equal(o.view(np.uint8), outs[0].view(np.uint8)), "fused / pre-pass / count-ahead decodes differ"
    if not qt:
        assert_error_bound(x, outs[0], orc["bin_index"], orc["dc"], orc["ac"], eb, sf)
    return outs[0]


def check_compress(contexts, x, eb, qt, orc):
    g = contexts["fused"].compress_core(x, eb, qt=qt, want_scaled=True)
    info = g["info"]
    assert info["status"] == 0 and np.all(np.isfinite(g["dc"])) and np.all(np.isfinite(g["ac"]))
    rep = parity.compare_compress(g, orc, x, eb, qt, ctx=contexts["fused"])
    # an "all outliers" stream (kq = inf turns every coefficient into +-inf) must not pass as a legal one
    assert abs(int(info["n_outliers"]) - orc["ac"].size) <= rep["ties"], (info["n_outliers"], orc["ac"].size)
    assert np.array_equal(g["scaled"].view(np.uint8), orc["scaled"].view(np.uint8)), "x/sf is not bit-identical"
    for name in ("prepass", "ahead"):
        s = contexts[name].compress_core(x, eb, qt=qt)
        assert np.array_equal(s["bin_index"], g["bin_index"]) and np.array_equal(s["dc"].view(np.uint32), g["dc"].view(np.uint32))
        assert np.array_equal(s["ac"].view(np.uint32), g["ac"].view(np.uint32)) and s["sf"] == g["sf"], name
        if qt:
            assert np.array_equal(s["qtable"], g["qtable"]), name
    # the GPU's own stream back through every decoder
    outs = [c.decompress_core(g["bin_index"], g["dc"], g["ac"], x.size, x.dtype, eb, g["sf"], qt=qt, qtable=g.get("qtable"))
            for c in contexts.values()]
    assert np.all(np.isfinite(outs[0]))
    for o in outs[1:]:
        assert np.array_equal(o.view(np.uint8), outs[0].view(np.uint8))
    if not qt:
        assert_error_bound(x, outs[0], g["bin_index"], g["dc"], g["ac"], eb, g["sf"])
    return g


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _info(t):
    return binding.GpuInfo.from_buffer_copy(t.cpu().numpy().tobytes()).as_dict()


def _outs(n, tdt):
    return dict(bins=torch.empty(n, dtype=torch.uint8, device="cuda"), dc=torch.empty((n + 63) // 64, dtype=torch.float32, device="cuda"),
                ac=torch.empty(max(n, 1), dtype=torch.float32, device="cuda"), qraw=torch.zeros(64, dtype=tdt, device="cuda"),
                qt=torch.zeros(64, dtype=tdt, device="cuda"), info=torch.zeros(binding.INFO_BYTES, dtype=torch.uint8, device="cuda"))


def two_pass(ctx, x, eb, qt):
    """stats_dev + compress_dev on the whole field"""
    code, tdt = (DOUBLE, torch.float64) if x.dtype == np.float64 else (FLOAT, torch.float32)
    s = torch.cuda.current_stream().cuda_stream
    d, n = _dev(x), x.size
    st = torch.zeros(3, dtype=torch.float64, device="cuda")
    o = _outs(n, tdt)
    ctx.stats_dev(d.data_ptr(), n, code, st.data_ptr(), s)
    ctx.compress_dev(d.data_ptr(), n, n, code, eb, qt, st.data_ptr(), 1, True, o["bins"].data_ptr(), o["dc"].data_ptr(), o["ac"].data_ptr(),
                     o["qraw"].data_ptr(), o["info"].data_ptr(), s)
    if qt:
        ctx.qt_finish_dev(code, eb, o["qraw"].data_ptr(), o["qt"].data_ptr(), o["ac"].data_ptr(), o["info"].data_ptr(), s)
    torch.cuda.synchronize()
    return _result(o)


def single_read(ctx, x, eb, qt):
    """sample_dev -> compress_spec_dev -> compress_spec_finish_dev on the whole field (one rank)"""
    code, tdt = (DOUBLE, torch.float64) if x.dtype == np.float64 else (FLOAT, torch.float32)
    s = torch.cuda.current_stream().cuda_stream
    d, n = _dev(x), x.size
    belief = torch.zeros(3, dtype=torch.float64, device="cuda")
    true3 = torch.zeros(3, dtype=torch.float64, device="cuda")
    o = _outs(n, tdt)
    ctx.sample_dev(d.data_ptr(), n, code, belief.data_ptr(), s)
    ctx.compress_spec_dev(d.data_ptr(), n, n, code, eb, qt, belief.data_ptr(), 1, True, o["bins"].data_ptr(), o["dc"].data_ptr(),
                          o["ac"].data_ptr(), o["qraw"].data_ptr(), o["info"].data_ptr(), true3.data_ptr(), s)
    ctx.compress_spec_finish_dev(d.data_ptr(), n, n, code, eb, qt, true3.data_ptr(), 1, True, o["bins"].data_ptr(), o["dc"].data_ptr(),
                                 o["ac"].data_ptr(), o["qraw"].data_ptr(), o["info"].data_ptr(), s)
    if qt:
        ctx.qt_finish_dev(code, eb, o["qraw"].data_ptr(), o["qt"].data_ptr(), o["ac"].data_ptr(), o["info"].data_ptr(), s)
    torch.cuda.synchronize()
    return _result(o)


def field_dev(ctx, x, eb, qt):
    """compress_field_dev: the single-read path in one call"""
    code, tdt = (DOUBLE, torch.float64) if x.dtype == np.float64 else (FLOAT, torch.float32)
    s = torch.cuda.current_stream().cuda_stream
    d, n = _dev(x), x.size
    o = _outs(n, tdt)
    ctx.compress_field_dev(d.data_ptr(), n, code, eb, qt, o["bins"].data_ptr(), o["dc"].data_ptr(), o["ac"].data_ptr(),
                           o["qt"].data_ptr() if qt else 0, o["qraw"].data_ptr() if qt else 0, o["info"].data_ptr(), s)
    torch.cuda.synchronize()
    return _result(o)


def _result(o):
    i = _info(o["info"])
    return dict(info=i, bins=o["bins"].cpu().numpy(), dc=o["dc"].cpu().numpy(), ac=o["ac"][: i["n_outliers"]].cpu().numpy(),
                qt=o["qt"].cpu().numpy())


def _rejected(call):
    """a compress entry point refuses the field: an error code, or status EDEGENERATE in the device-side info"""
    try:
        r = call()
    except dctz_b200.DctzGpuError as e:
        assert e.code == EDEGENERATE, e
        return
    st = r["info"]["status"] if "info" in r else None
    assert st == EDEGENERATE, r.get("info")


def assert_rejected_everywhere(contexts, x, eb, qt):
    for name, c in contexts.items():
        with pytest.raises(dctz_b200.DctzGpuError) as e:
            c.compress_core(x, eb, qt=qt)
        assert e.value.code == EDEGENERATE, name
    _rejected(lambda: two_pass(contexts["prepass"], x, eb, qt))
    _rejected(lambda: single_read(contexts["prepass"], x, eb, qt))
    _rejected(lambda: field_dev(contexts["prepass"], x, eb, qt))
    parts, xs, stats_all, outs, code = compress_slabs(contexts["prepass"], x, eb, qt, 2)
    torch.cuda.synchronize()
    assert all(_info(o["info"])["status"] == EDEGENERATE for o in outs)


def _cases(dtype):
    return [(np.dtype(dtype), k) for k in DECADES[np.dtype(dtype)]]


@pytest.mark.parametrize("dtype,k", _cases(np.float64) + _cases(np.float32), ids=lambda v: str(v))
def test_decade_against_the_oracle(contexts, dtype, k):
    x = field(dtype, k)
    for eb in EBS:
        for qt in (False, True):
            orc, want = oracle_stream(x, eb, qt)
            sf = orc["stat"]["sf"]
            assert abs(sf / 10.0 ** k - 1) < 1e-6, (sf, k)
            check_decode(contexts, x, eb, qt, orc, want)
            if admitted(dtype, sf):
                assert contexts["fused"].sf_from_max(float(np.max(np.abs(x))), dtype) == sf
                check_compress(contexts, x, eb, qt, orc)
            else:
                assert contexts["fused"].sf_from_max(float(np.max(np.abs(x))), dtype) == 0.0
                assert_rejected_everywhere(contexts, x, eb, qt)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_the_largest_finite_value(contexts, dtype):
    """max|x| == DBL_MAX / FLT_MAX: sf = 1e308 / 1e38, beyond what compress admits; the oracle's stream decodes"""
    x = field(dtype, 0, tail=37, peak=1.0)
    x = (x.astype(np.float64) / np.max(np.abs(x)) * float(np.finfo(dtype).max)).astype(dtype)
    x[np.argmax(np.abs(x))] = np.finfo(dtype).max
    for eb, qt in ((1e-3, False), (1e-6, True)):
        orc, want = oracle_stream(x, eb, qt)
        # the reference's own reconstruction may round past the largest finite value: compare where it is finite
        got = contexts["prepass"].decompress_core(orc["bin_index"], orc["dc"], orc["ac"], x.size, x.dtype, eb, orc["stat"]["sf"], qt=qt,
                                                  qtable=orc["qtable"])
        fin = np.isfinite(want) & np.isfinite(got)
        parity.check_reconstruction(got[fin], want[fin], orc["stat"]["sf"])
        both = ~np.isfinite(want) & ~np.isfinite(got)  # overflowed in both: the same infinity
        assert np.array_equal(got[both], want[both])
        # where only one of the two overflowed, the other lies within the tolerance of the largest finite value
        edge = np.isfinite(want) != np.isfinite(got)
        near = np.where(np.isfinite(want), np.abs(want.astype(np.float64)), np.abs(got.astype(np.float64)))[edge]
        assert np.all(near >= float(np.finfo(dtype).max) * (1 - 8 * parity.RTOL[np.dtype(dtype)])), near
        assert_rejected_everywhere(contexts, x, eb, qt)


def _edge(c, dtype, b):
    """the two adjacent values around the decimal power b between which sf_from_max switches between refusing (0) and
    admitting: (below, above)"""
    it = np.int64 if dtype == np.float64 else np.int32
    ok = lambda u: c.sf_from_max(float(np.array(u, dtype=it).view(dtype)), dtype) != 0.0
    lo, hi = (int(np.array(dtype.type(b * f)).view(it)) for f in (1 - 1e-5, 1 + 1e-5))
    ok_lo = ok(lo)
    assert ok(hi) != ok_lo, "sf_from_max does not switch near the decimal power"
    while hi - lo > 1:  # bisection on the bit pattern
        mid = (lo + hi) // 2
        if ok(mid) == ok_lo:
            lo = mid
        else:
            hi = mid
    v = lambda u: np.array(u, dtype=it).view(dtype)[()]
    return v(lo), v(hi), ok_lo


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_both_limits_of_the_admitted_range(contexts, dtype):
    """the last admitted and the first refused max|x| at each end: inside compresses like the oracle, outside is
    EDEGENERATE on every entry point; both streams of the oracle decode"""
    dtype = np.dtype(dtype)
    lo, hi = ADMITTED[dtype]
    c = contexts["fused"]
    p = field(dtype, 0, tail=1, peak=1.0).astype(np.float64)
    for b, lower_end in ((10.0 ** lo, True), (10.0 ** (hi + 1), False)):
        below, above, below_ok = _edge(c, dtype, b)
        assert below_ok != lower_end  # refused below the lower limit, admitted below the upper one
        for top in (below, above):
            x = (p * float(top)).astype(dtype)
            x[np.argmax(np.abs(x))] = top
            assert float(np.max(np.abs(x))) == float(top)
            orc, want = oracle_stream(x, 1e-6, False)
            check_decode(contexts, x, 1e-6, False, orc, want)
            if c.sf_from_max(float(top), dtype) != 0.0:
                assert c.sf_from_max(float(top), dtype) == orc["stat"]["sf"]
                check_compress(contexts, x, 1e-6, False, orc)
                assert two_pass(contexts["prepass"], x, 1e-6, False)["info"]["status"] == 0
            else:
                assert_rejected_everywhere(contexts, x, 1e-6, False)


@pytest.mark.parametrize("dtype,k", [(np.float64, -302), (np.float64, 305), (np.float32, -32), (np.float32, 35)], ids=str)
@pytest.mark.parametrize("qt", [False, True])
def test_paths_agree_bit_for_bit_at_the_admitted_ends(contexts, dtype, k, qt):
    """single-read vs two-pass vs the host call; two-slab emulation vs the whole field; region decode vs full decode"""
    x = field(dtype, k, tail=37)
    eb = 1e-3
    c = contexts["prepass"]
    ref = two_pass(c, x, eb, qt)
    assert ref["info"]["status"] == 0 and ref["info"]["sf"] == reflib.oracle_stat(x)["sf"]
    for other in (single_read(c, x, eb, qt), field_dev(c, x, eb, qt)):
        assert other["info"]["status"] == 0 and other["info"]["sf"] == ref["info"]["sf"]
        assert np.array_equal(other["bins"], ref["bins"]) and np.array_equal(other["dc"], ref["dc"]) and np.array_equal(other["ac"], ref["ac"])
        if qt:
            assert np.array_equal(other["qt"], ref["qt"])
    host = contexts["fused"].compress_core(x, eb, qt=qt)
    assert np.array_equal(host["bin_index"], ref["bins"]) and np.array_equal(host["ac"], ref["ac"])
    if not qt:  # slabs: the EC emulation of test_gpu_device_api (QT needs the exchange of the per-position maxima)
        parts, xs, stats_all, outs, code = compress_slabs(c, x, eb, False, 2)
        torch.cuda.synchronize()
        infos = [_info(o["info"]) for o in outs]
        assert all(i["status"] == 0 and i["sf"] == ref["info"]["sf"] for i in infos)
        bins = np.concatenate([o["bins"].cpu().numpy() for o in outs])
        ac = np.concatenate([o["ac"][: i["n_outliers"]].cpu().numpy() for o, i in zip(outs, infos)])
        assert np.array_equal(bins, ref["bins"]) and np.array_equal(ac, ref["ac"])


@pytest.mark.parametrize("dtype,k", [(np.float64, -307), (np.float64, -300), (np.float64, 300), (np.float64, 308),
                                     (np.float32, -37), (np.float32, 37), (np.float32, 38)], ids=str)
@pytest.mark.parametrize("qt", [False, True])
def test_region_decode_equals_full_decode(contexts, dtype, k, qt):
    """decompress_ranges_dev against decompress_dev on the oracle's stream, bit for bit, where the decoders rescale sf"""
    x = field(dtype, k, tail=63)
    x = np.tile(x, 24)[: 64 * 32 * 12 + 63]  # several warp tiles
    eb = 1e-3
    orc, want = oracle_stream(x, eb, qt)
    ac = _dev(orc["ac"]) if orc["ac"].size else torch.zeros(4, dtype=torch.float32, device="cuda")
    f = Field(contexts["prepass"], x.size, x.dtype, eb, qt, _dev(orc["bin_index"]), _dev(orc["dc"]), ac, orc["ac"].size,
              _dev(orc["qtable"]) if qt else None, orc["stat"]["sf"])
    torch.cuda.synchronize()
    full = f.full.cpu().numpy()
    parity.check_reconstruction(full, want, orc["stat"]["sf"])
    f.check(random_ranges(np.random.default_rng(k % 97), x.size, 60))


def test_a_finite_field_whose_sum_overflows_compresses(contexts):
    """2^16 values near 3e304: the double sum overflows (as the reference's does); sf = 1e304 is admitted"""
    rng = np.random.default_rng(4)
    x = 3e304 * (1.0 + 0.01 * rng.standard_normal(1 << 16))
    orc, want = oracle_stream(x, 1e-3, False)
    assert orc["stat"]["sum"] == np.inf
    g = check_compress(contexts, x, 1e-3, False, orc)
    assert g["info"]["sum"] == np.inf
    for r in (two_pass(contexts["prepass"], x, 1e-3, False), single_read(contexts["prepass"], x, 1e-3, False)):
        assert r["info"]["status"] == 0 and np.array_equal(r["bins"], g["bin_index"])
    # both signs: partial sums of +inf and -inf would make a NaN sum -- still finite data
    y = x.copy()
    y[1 << 15:] *= -1
    assert contexts["fused"].compress_core(y, 1e-3)["info"]["status"] == 0
    assert two_pass(contexts["prepass"], y, 1e-3, False)["info"]["status"] == 0


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf])
@pytest.mark.parametrize("where", ["block", "tail", "second_slab"])
def test_non_finite_data_is_rejected(contexts, dtype, bad, where):
    """NaN or inf anywhere -- in a full block, in the partial tail block (which the single-read path reads with FP
    arithmetic), in the second of two slabs -- is EDEGENERATE on the single-read and the two-pass path"""
    n = 64 * 32 * 10 + 37
    x = (3.0 + np.sin(np.arange(n) / 17.0)).astype(dtype)
    pos = {"block": 1234, "tail": n - 5, "second_slab": n - 100}[where]
    x[pos] = bad
    c = contexts["prepass"]
    _rejected(lambda: two_pass(c, x, 1e-3, False))
    _rejected(lambda: single_read(c, x, 1e-3, False))
    _rejected(lambda: field_dev(c, x, 1e-3, False))
    for cc in contexts.values():
        with pytest.raises(dctz_b200.DctzGpuError):
            cc.compress_core(x, 1e-3)
    parts, xs, stats_all, outs, code = compress_slabs(c, x, 1e-3, False, 2)
    torch.cuda.synchronize()
    assert all(_info(o["info"])["status"] == EDEGENERATE for o in outs)


@pytest.mark.parametrize("fill", [9.96921e36, 1e36])
def test_float_fill_values(contexts, fill):
    """smooth float data with netCDF / CESM fill values (whole blocks and scattered): sf is beyond what compress admits,
    so compress refuses; the oracle's stream decodes"""
    n = 64 * 200 + 37
    x = (280.0 + 10.0 * np.sin(np.arange(n) / 40.0)).astype(np.float32)
    x[64 * 10:64 * 30] = fill
    x[5::97] = fill
    for eb, qt in ((1e-3, False), (1e-6, False), (1e-3, True)):
        orc, want = oracle_stream(x, eb, qt)
        check_decode(contexts, x, eb, qt, orc, want)
        if admitted(x.dtype, orc["stat"]["sf"]):  # 1e36 in float is 1.00000004e36 < T(36): sf = 1e35
            check_compress(contexts, x, eb, qt, orc)
        else:
            assert_rejected_everywhere(contexts, x, eb, qt)


@pytest.mark.parametrize("dtype,k", [(np.float64, -307), (np.float64, 308), (np.float32, -37), (np.float32, 38)], ids=str)
def test_region_decode_skipped_ranges_and_many_ranges_where_the_output_is_rescaled(contexts, dtype, k):
    """k_scale_ranges: a range outside [0, n) is skipped (its place keeps what was there, bit 1 is set) and the others are
    rescaled; more than 1024 ranges (the chunk offsets), fewer ranges than CTAs (the whole grid per range)"""
    x = np.tile(field(dtype, k, tail=37), 8)
    orc, want = oracle_stream(x, 1e-3, False)
    ac = _dev(orc["ac"]) if orc["ac"].size else torch.zeros(4, dtype=torch.float32, device="cuda")
    f = Field(contexts["prepass"], x.size, x.dtype, 1e-3, False, _dev(orc["bin_index"]), _dev(orc["dc"]), ac, orc["ac"].size, None,
              orc["stat"]["sf"])
    torch.cuda.synchronize()
    parity.check_reconstruction(f.full.cpu().numpy(), want, orc["stat"]["sf"])
    rng = np.random.default_rng(7)
    f.check(np.array([(0, x.size)], dtype=np.uint64))  # one range: the whole grid rescales it
    f.check(random_ranges(rng, x.size, 3000, maxlen=40))  # > 1024 ranges
    ranges = random_ranges(rng, x.size, 50)
    ranges = np.concatenate([ranges[:20], np.array([(x.size - 3, 10)], dtype=np.uint64), ranges[20:]])
    out, corrupt = f.decode(ranges)
    assert corrupt == 2
    counts = ranges[:, 1].astype(np.int64)
    at = np.concatenate([[0], np.cumsum(counts)])
    o = out.cpu().numpy()
    assert np.all(np.isnan(o[at[20]:at[21]]))  # the skipped range's place: untouched (the NaN it was filled with)
    good = np.concatenate([np.arange(at[i], at[i + 1]) for i in range(len(ranges)) if i != 20])
    keep = np.delete(ranges, 20, axis=0)
    assert np.array_equal(o[good].view(np.uint8), f.expected(keep).cpu().numpy().view(np.uint8))


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("belief", ["max", "zero", "nan"])
def test_a_refused_caller_belief_still_gives_the_two_pass_result(contexts, dtype, belief):
    """compress_known_stats_dev with a belief compress refuses (DBL_MAX / FLT_MAX, 0, NaN): the belief pass must still
    gather the true statistics, so that the correcting launch compresses an ordinary field exactly like the two-pass path
    -- also right after another field was compressed on the same context (whose statistics records must not be reused)"""
    c = contexts["prepass"]
    code, tdt = (DOUBLE, torch.float64) if np.dtype(dtype) == np.float64 else (FLOAT, torch.float32)
    s = torch.cuda.current_stream().cuda_stream
    n = 64 * 32 * 40 + 37
    x = (3.0 + 2.0 * np.sin(np.arange(n) / 41.0)).astype(dtype)
    c.compress_core((x * 100).astype(dtype), 1e-3)  # another field first: other sf, other statistics records
    ref = two_pass(c, x, 1e-3, False)
    assert ref["info"]["status"] == 0
    b = {"max": float(np.finfo(dtype).max), "zero": 0.0, "nan": float("nan")}[belief]
    stats = torch.tensor([b, b, 0.0], dtype=torch.float64, device="cuda")
    d = _dev(x)
    o = _outs(n, tdt)
    c.compress_known_stats_dev(d.data_ptr(), n, n, code, 1e-3, False, stats.data_ptr(), 1, True, o["bins"].data_ptr(), o["dc"].data_ptr(),
                               o["ac"].data_ptr(), o["qraw"].data_ptr(), o["info"].data_ptr(), s)
    torch.cuda.synchronize()
    r = _result(o)
    assert r["info"]["status"] == 0 and r["info"]["n_exact_path"] == 1 and r["info"]["sf"] == ref["info"]["sf"], r["info"]
    assert r["info"]["max_abs"] == ref["info"]["max_abs"]
    assert np.array_equal(r["bins"], ref["bins"]) and np.array_equal(r["dc"], ref["dc"]) and np.array_equal(r["ac"], ref["ac"])


@pytest.mark.parametrize("dtype,k", [(np.float64, -306), (np.float64, 307), (np.float32, -36), (np.float32, 37)], ids=str)
def test_quality_matches_the_reference_arithmetic(contexts, dtype, k):
    """k_quality (calc_psnr's double arithmetic, util.c:54-104) at a tiny and a huge decade: min, max and max|a-b| exact,
    the sum of squared errors as a double sum (which under- or overflows there the way the reference's does)"""
    x = field(dtype, k, tail=37)
    orc, want = oracle_stream(x, 1e-3, False)
    q = contexts["fused"].quality(x, want)
    a = x.astype(np.float64)
    e = (x - want).astype(np.float64)  # the difference in the element type, as util.c takes it
    assert q["min"] == a.min() and q["max"] == a.max() and q["maxdiff"] == np.max(np.abs(e))
    ss = float(np.sum(e ** 2))
    if ss == 0.0 or not np.isfinite(ss):
        assert q["sumsq"] == ss
    else:
        assert abs(q["sumsq"] - ss) <= 1e-9 * ss
    psnr = lambda rng, sq: 20 * np.log10(rng) - 10 * np.log10(sq / x.size) if sq > 0 else np.inf
    with np.errstate(all="ignore"):
        pg, pr = psnr(q["max"] - q["min"], q["sumsq"]), psnr(a.max() - a.min(), ss)
    assert (pg == pr) if not np.isfinite(pr) else abs(pg - pr) < 1e-6
