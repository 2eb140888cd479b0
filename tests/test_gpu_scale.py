"""GPU: whole fields past every scheduling threshold of the streaming kernels, against the CPU oracle.

The kernels change how they schedule work as a slab grows (dctz_gpu_launch_plan reports it): tiles are handed out in
batches once every warp has many to go through, the outlier scan runs in chunks of 1024 groups, k_reduce_tiles runs with
one CTA per 4096 tiles, the gathers' CTAs loop over groups, the count-ahead decoder splits its units into super-groups
of 2048, and the single-launch kernels stop at 256 MiB of input.  Each case asserts first that its field reaches the
regime it is meant to test, from the plan of the contexts that run it, and fails (it does not skip) when the device
cannot reach it at this size.

Fields: 2^27 + 64*3 + 37 doubles and 2^28 + 29 floats (1 GiB each), generated on the device with fill_hash_field and
overlaid with stretches of dense outliers, stretches without any and stretches with a few per tile, placed so that
ticket, group, scan-chunk, reduce-CTA, count-ahead group and super-group and slab boundaries fall inside outlier runs
and between them; a run of all-zero tiles; and the global maximum as one spike a decade above the rest, between
k_sample's sample points in the last chunk (the belief is a decade low and every single-read path compresses twice), or
in the partial tail block (which k_sample reads exactly)."""
import numpy as np
import pytest
import torch

from dctz_b200 import slabs
from tests import parity, reflib
from tests.test_gpu_device_api import compress_slabs
from tests.test_gpu_exponent_range import _ctx, _dev, _info, _outs, _result, assert_error_bound, field_dev, single_read, two_pass
from tests.test_gpu_ranges import Field, _bits, random_ranges

pytestmark = pytest.mark.gpu

TILE, GROUP, CHUNK = 2048, 2048 * 32, 2048 * 32 * 1024  # elements per warp tile, per group of 32 tiles, per scan chunk of 1024 groups
N_DOUBLE = (1 << 27) + 64 * 3 + 37
N_FLOAT = (1 << 28) + 29
FUSED_LIMIT = 256 << 20  # bytes: the single-launch kernels' default limit (DCTZ_FUSED_MAX_MB)
SPIKE = 500.0            # the global maximum: sf = 100 where the rest of the field gives sf = 10
WORLDS = (2, 3, 8)


@pytest.fixture(scope="module")
def contexts():
    """the pre-pass and the count-ahead decoder forced; compress runs the same kernels in both"""
    cs = dict(prepass=_ctx(DCTZ_DECOMP_AHEAD=0), ahead=_ctx(DCTZ_DECOMP_AHEAD=1))
    yield cs
    for c in cs.values():
        c.close()


def _dtype_code(dtype):
    return (torch.float64, 8) if np.dtype(dtype) == np.float64 else (torch.float32, 4)


def assert_plan(plan, n, dtype, qt):
    """the streaming regime the scale cases exist for; a plan that misses one names it"""
    print(f"\nplan {np.dtype(dtype).name} {'qt' if qt else 'ec'} n={n}: {plan}")
    want = {
        "compress tiles per ticket > 1": plan["compress_batch"] > 1,
        "decompress (pre-pass) tiles per ticket > 1": plan["decompress_batch"] > 1,
        "count-ahead tiles per ticket > 1": plan["ahead_batch"] > 1,
        "count-ahead super-groups > 1": plan["ahead_super"] > 1,
        "compress scan chunks >= 2": plan["scan_chunks"] >= 2,
        "decompress scan chunks >= 2": plan["decompress_scan_chunks"] >= 2,
        "k_reduce_tiles CTAs >= 2": plan["reduce_ctas"] >= 2,
        "gather grid < groups (every CTA loops)": plan["gather_grid"] < plan["groups"],
        "k_qt_max grid < groups (every CTA loops)": plan["qt_max_grid"] < plan["qt_max_groups"],
        "streaming, not the single-launch kernels": plan["fused_compress_grid"] == 0 and plan["fused_decompress_grid"] == 0,
    }
    missed = [k for k, ok in want.items() if not ok]
    assert not missed, f"this field does not reach the regime it tests: {missed} (plan {plan})"


def boundaries(n, plan):
    """{kind: sorted element positions} of the boundaries the scheduling has at this size (interior ones only)"""
    tb = lambda tiles: tiles * TILE
    kinds = {
        "chunk": range(CHUNK, n, CHUNK),
        "super": range(tb(2048 * plan["ahead_batch"]), n, tb(2048 * plan["ahead_batch"])),
        "reduce": range(tb(4096), n, tb(4096)),
        "group": [GROUP * k for k in (1, 2, 3, 100, 101)] + [n // GROUP * GROUP - GROUP, n // GROUP * GROUP],
        "ahead_group": [tb(64 * plan["ahead_batch"]) * k for k in (1, 2, 7)],
        "ticket": [tb(plan["compress_batch"]) * k for k in (1, 3, 1001)] + [tb(plan["ahead_batch"]) * k for k in (5, 999)],
        "slab": sorted({a for w in WORLDS for a, _ in slabs.partition(n, w)[1:]}),
    }
    return {k: sorted(p for p in v if 0 < p < n) for k, v in kinds.items()}


def make_field(ctx, n, dtype, plan, spike_in_tail, seed=11):
    """the hash field (max|x| about 40) with the overlays of the module docstring; returns (device tensor, spike position)"""
    x = torch.empty(n, dtype=torch.float64, device="cuda")
    ctx.fill_hash_field(x.data_ptr(), 0, n, 2048, 20261018, torch.cuda.current_stream().cuda_stream)
    g = torch.Generator(device="cuda").manual_seed(seed)
    # texture over the whole field: no outliers at eb 1E-3 (its AC coefficients are ~0.4 against a range of 25.5 at sf
    # 100), dense ones at 1E-5 (range 0.255)
    x += 1.5 * (torch.rand(n, generator=g, device="cuda", dtype=torch.float64) - 0.5)

    def dense(a, b):  # outliers in most coefficients at every eb (AC ~ 35 against a range of at most 25.5)
        x[a:b] = 30.0 + 120.0 * (torch.rand(b - a, generator=g, device="cuda", dtype=torch.float64) - 0.5)

    def quiet(a, b):  # constant: no outlier at any eb
        x[a:b] = 25.0

    def sparse(a, b):  # constant with one burst per tile, in the tile's middle: a few outliers per tile
        quiet(a, b)
        for t in range(a // TILE, (b - 1) // TILE + 1):
            c = t * TILE + 1000 + (t % 5) * 64
            if a <= c and c + 8 <= b:
                x[c:c + 8] = 25.0 + 45.0 * torch.tensor([1, -1, 1, -1, 1, -1, 1, -1], dtype=torch.float64, device="cuda")

    # every kind of boundary falls in a dense run, in a stretch without outliers and between sparse outliers, in turn
    styles = (dense, quiet, sparse)
    half = 3 * TILE + 100
    done = set()
    for kind, pos in boundaries(n, plan).items():
        for i, p in enumerate(pos):
            if p not in done:
                done.add(p)
                styles[i % 3](max(0, p - half), min(n - n % 64, p + half))
    zero = 5 * GROUP + 3 * TILE  # 64 all-zero tiles: many candidates for the minimum |x| (k_resolve_extremes)
    x[zero:zero + 64 * TILE] = 0.0
    if spike_in_tail:
        at = n - 5
    else:  # in the full blocks of the last scan chunk, off k_sample's sample points (one 16-byte vector every `stride`)
        es = 8 if np.dtype(dtype) == np.float64 else 4
        vec = 16 // es
        stride = max((n * es // 16) >> 18, 256)
        nfull = n // 64 * 64
        last = (nfull - 1) // CHUNK * CHUNK
        at = last + (nfull - last) // 2 + 1
        if (at // vec) % stride == 0:
            at += vec
        assert (at // vec) % stride != 0 and last <= at < nfull
    x[at] = SPIKE
    if np.dtype(dtype) == np.float32:
        x = x.float()
    torch.cuda.synchronize()
    return x, at


def _same(a, b, qt, what):
    assert a["info"]["sf"] == b["info"]["sf"] and a["info"]["n_outliers"] == b["info"]["n_outliers"], (what, a["info"], b["info"])
    assert a["info"]["max_abs"] == b["info"]["max_abs"] and a["info"]["min_abs"] == b["info"]["min_abs"], what
    assert np.array_equal(a["bins"], b["bins"]), f"{what}: bin ids differ"
    assert np.array_equal(a["dc"].view(np.uint32), b["dc"].view(np.uint32)), f"{what}: DC differs"
    assert np.array_equal(a["ac"].view(np.uint32), b["ac"].view(np.uint32)), f"{what}: AC_exact differs"
    if qt:
        assert np.array_equal(a["qt"], b["qt"]), f"{what}: qtable differs"


def _from_host(r):
    return dict(info=r["info"], bins=r["bin_index"], dc=r["dc"], ac=r["ac"], qt=r.get("qtable"))


def known_stats(ctx, x, eb, qt, belief):
    """compress_known_stats_dev with a caller's belief {max, max, 0}"""
    code = 1 if x.dtype == np.float64 else 0
    tdt = _dtype_code(x.dtype)[0]
    s = torch.cuda.current_stream().cuda_stream
    d, n = _dev(x), x.size
    o = _outs(n, tdt)
    st = torch.tensor([belief, belief, 0.0], dtype=torch.float64, device="cuda")
    ctx.compress_known_stats_dev(d.data_ptr(), n, n, code, eb, qt, st.data_ptr(), 1, True, o["bins"].data_ptr(), o["dc"].data_ptr(),
                                 o["ac"].data_ptr(), o["qraw"].data_ptr(), o["info"].data_ptr(), s)
    if qt:
        ctx.qt_finish_dev(code, eb, o["qraw"].data_ptr(), o["qt"].data_ptr(), o["ac"].data_ptr(), o["info"].data_ptr(), s)
    torch.cuda.synchronize()
    return _result(o)


def slab_compress(ctx, x, eb, qt, world):
    """`world` emulated ranks: EC through compress_slabs; QT with one context per rank (a context holds one call's QT
    scratch) and the table reduced as the NCCL exchange does it (MAX of entries 1..63, entry 0 from the last rank)"""
    code = 1 if x.dtype == np.float64 else 0
    if not qt:
        parts, xs, stats_all, outs, code = compress_slabs(ctx, x, eb, False, world)
        torch.cuda.synchronize()
        del xs
        return parts, outs, [_info(o["info"]) for o in outs], [ctx] * world, []
    tdt = _dtype_code(x.dtype)[0]
    s = torch.cuda.current_stream().cuda_stream
    parts = slabs.partition(x.size, world)
    ranks = [_ctx(DCTZ_DECOMP_AHEAD=0) for _ in range(world)]
    stats_all = torch.zeros(3 * world, dtype=torch.float64, device="cuda")
    xs = [_dev(x[a:a + c]) for a, c in parts]
    for r, (a, c) in enumerate(parts):
        ranks[r].stats_dev(xs[r].data_ptr(), c, code, stats_all[3 * r:].data_ptr(), s)
    outs = []
    for r, (a, c) in enumerate(parts):
        o = _outs(c, tdt)
        ranks[r].compress_dev(xs[r].data_ptr(), c, x.size, code, eb, True, stats_all.data_ptr(), world, r == 0, o["bins"].data_ptr(),
                              o["dc"].data_ptr(), o["ac"].data_ptr(), o["qraw"].data_ptr(), o["info"].data_ptr(), s)
        outs.append(o)
    g = torch.stack([o["qraw"] for o in outs]).max(dim=0).values
    g[0] = outs[-1]["qraw"][0]
    for r, o in enumerate(outs):
        o["qraw"].copy_(g)
        ranks[r].qt_finish_dev(code, eb, o["qraw"].data_ptr(), o["qt"].data_ptr(), o["ac"].data_ptr(), o["info"].data_ptr(), s)
    torch.cuda.synchronize()
    del xs
    return parts, outs, [_info(o["info"]) for o in outs], ranks, ranks


def check_slabs(ctx, x, eb, qt, ref, whole, rng, boundary_ranges):
    """every world: the concatenation equals the single-field result; each slab decodes with decompress_dev to the
    field's decode, and its own outlier index decodes ranges of it, bit for bit"""
    for world in WORLDS:
        parts, outs, infos, rctx, owned = slab_compress(ctx, x, eb, qt, world)
        try:
            assert all(i["status"] == 0 and i["sf"] == ref["info"]["sf"] and i["n_qt_dropped"] == 0 for i in infos), infos
            assert np.array_equal(np.concatenate([o["bins"].cpu().numpy() for o in outs]), ref["bins"]), f"world {world}: bin ids"
            assert np.array_equal(np.concatenate([o["dc"].cpu().numpy() for o in outs]).view(np.uint32), ref["dc"].view(np.uint32)), world
            ac = np.concatenate([o["ac"][: i["n_outliers"]].cpu().numpy() for o, i in zip(outs, infos)])
            assert np.array_equal(ac.view(np.uint32), ref["ac"].view(np.uint32)), f"world {world}: AC_exact"
            if qt:
                assert all(np.array_equal(o["qt"].cpu().numpy(), ref["qt"]) for o in outs), f"world {world}: qtable"
            for (a, c), o, i, rc in zip(parts, outs, infos, rctx):
                slab = Field(rc, c, x.dtype, eb, qt, o["bins"], o["dc"], o["ac"], i["n_outliers"], o["qt"] if qt else None, ref["info"]["sf"])
                torch.cuda.synchronize()
                assert int(slab.index_count.item()) == i["n_outliers"]
                assert torch.equal(_bits(slab.full), _bits(whole.full[a:a + c])), f"world {world}: slab at {a} decodes differently"
                rg = random_ranges(rng, c, 200, maxlen=20000)
                local = [(p - a - 700, 1400) for p in boundary_ranges if a + 700 <= p <= a + c - 700]
                if local:
                    rg = np.concatenate([rg, np.array(local, dtype=np.uint64)])
                out, corrupt = slab.decode(rg)
                assert corrupt == 0
                shifted = rg.copy()
                shifted[:, 0] += np.uint64(a)
                assert torch.equal(_bits(out), _bits(whole.expected(shifted))), f"world {world}: ranges of the slab at {a}"
                del slab
        finally:
            for c in owned:
                c.close()


def decode_all(contexts, stream, n, dtype, eb, qt):
    """one stream through the pre-pass and the count-ahead decoder: finite and identical bits"""
    outs = [c.decompress_core(stream["bin_index"], stream["dc"], stream["ac"], n, dtype, eb, stream["sf"], qt=qt, qtable=stream.get("qtable"))
            for c in contexts.values()]
    assert np.all(np.isfinite(outs[0])), "non-finite values in the reconstruction"
    assert np.array_equal(outs[0].view(np.uint8), outs[1].view(np.uint8)), "pre-pass and count-ahead decodes differ"
    return outs[0]


def _id(v):
    return np.dtype(v).name if isinstance(v, type) else str(v)


CASES = [(np.float64, False, 1e-3), (np.float64, True, 1e-3), (np.float32, False, 1e-3), (np.float32, True, 1e-3), (np.float64, False, 1e-5)]


@pytest.mark.parametrize("dtype,qt,eb", CASES, ids=_id)
def test_whole_field_past_every_threshold(contexts, dtype, qt, eb):
    dtype = np.dtype(dtype)
    n = N_DOUBLE if dtype == np.float64 else N_FLOAT
    c = contexts["prepass"]
    for ctx in contexts.values():
        assert_plan(ctx.launch_plan(n, dtype, qt), n, dtype, qt)
    plan = c.launch_plan(n, dtype, qt)
    xd, at = make_field(c, n, dtype, plan, spike_in_tail=False)
    x = xd.cpu().numpy()
    del xd
    torch.cuda.empty_cache()
    bounds = boundaries(n, plan)

    # compress: the host call (pageable: the staged pipeline) against the oracle
    orc = reflib.oracle_compress(x, eb, qt)
    assert orc["stat"]["max"] == SPIKE and orc["stat"]["sf"] == 100.0, orc["stat"]
    g = c.compress_core(x, eb, qt=qt, want_scaled=True)
    assert g["info"]["status"] == 0
    rep = parity.compare_compress(g, orc, x, eb, qt, ctx=c)
    assert np.array_equal(g["scaled"].view(np.uint8), orc["scaled"].view(np.uint8)), "x/sf is not bit-identical"
    frac = orc["ac"].size / n
    print(f"outliers {orc['ac'].size} ({frac:.1%}), gpu {g['info']['n_outliers']}, ties {rep['ties']} ({rep['tie_fraction']:.2e})")
    if eb == 1e-5:
        assert frac > 0.2, f"the dense case has only {frac:.1%} outliers"
    del g["scaled"], orc["scaled"], orc["coef"]
    ref = _from_host(g)

    # every other compress path: the same bits
    pinned = torch.empty(n, dtype=_dtype_code(dtype)[0], pin_memory=True)
    pinned.numpy()[:] = x
    _same(_from_host(c.compress_core(pinned.numpy(), eb, qt=qt)), ref, qt, "compress_core, page-locked input")
    del pinned
    _same(two_pass(c, x, eb, qt), ref, qt, "stats_dev + compress_dev")
    sr = single_read(c, x, eb, qt)
    assert sr["info"]["n_exact_path"] == 1, "the belief should be a decade low: the spike lies between the sample points"
    _same(sr, ref, qt, "sample + compress_spec + compress_spec_finish")
    fd = field_dev(c, x, eb, qt)
    assert fd["info"]["n_exact_path"] == 1
    _same(fd, ref, qt, "compress_field_dev")
    ks = known_stats(c, x, eb, qt, SPIKE * 10)
    assert ks["info"]["n_exact_path"] == 1, "a belief a decade high must be corrected"
    _same(ks, ref, qt, "compress_known_stats_dev, belief a decade high")
    del sr, fd, ks

    # decompress: the oracle's stream and the GPU's stream through both decoders
    sf = orc["stat"]["sf"]
    want = reflib.oracle_decompress(orc["bin_index"], orc["dc"], orc["ac"], orc["qtable"], n, eb, sf, qt, dtype)
    got = decode_all(contexts, dict(bin_index=orc["bin_index"], dc=orc["dc"], ac=orc["ac"], qtable=orc["qtable"], sf=sf), n, dtype, eb, qt)
    parity.check_reconstruction(got, want, sf)
    if not qt:
        assert_error_bound(x, got, orc["bin_index"], orc["dc"], orc["ac"], eb, sf)
    del orc, want, got
    stream = dict(bin_index=ref["bins"], dc=ref["dc"], ac=ref["ac"], qtable=ref["qt"], sf=sf)
    got = decode_all(contexts, stream, n, dtype, eb, qt)
    want = reflib.oracle_decompress(ref["bins"], ref["dc"], ref["ac"], ref["qt"] if qt else None, n, eb, sf, qt, dtype)
    parity.check_reconstruction(got, want, sf)
    if not qt:
        assert_error_bound(x, got, ref["bins"], ref["dc"], ref["ac"], eb, sf)
    del want

    # region decode of the whole field, then slabs (compress, per-slab decode, per-slab index)
    ac = _dev(ref["ac"]) if ref["ac"].size else torch.zeros(4, dtype=torch.float32, device="cuda")
    whole = Field(c, n, dtype, eb, qt, _dev(ref["bins"]), _dev(ref["dc"]), ac, ref["ac"].size, _dev(ref["qt"]) if qt else None, sf)
    torch.cuda.synchronize()
    assert int(whole.index_count.item()) == ref["info"]["n_outliers"]
    assert np.array_equal(whole.full.cpu().numpy().view(np.uint8), got.view(np.uint8)), "decompress_dev differs from decompress_core"
    del got
    rng = np.random.default_rng(29)
    straddle = sorted({p for v in bounds.values() for p in v} | {at, n - n % 64})
    rg = random_ranges(rng, n, 2000, maxlen=20000)
    rg = np.concatenate([rg, np.array([(p - 700, 1400) for p in straddle if 700 <= p <= n - 700] + [(n - 3000, 3000)], dtype=np.uint64)])
    whole.check(rg)
    check_slabs(c, x, eb, qt, ref, whole, rng, straddle)


@pytest.mark.parametrize("dtype,qt", [(np.float64, False), (np.float32, True)], ids=_id)
def test_maximum_in_the_partial_tail_block(contexts, dtype, qt):
    """the global maximum in the tail block, which k_sample reads exactly: the belief holds (no second pass), and every
    compress path gives the oracle's result and the same bits"""
    dtype = np.dtype(dtype)
    n = N_DOUBLE if dtype == np.float64 else N_FLOAT
    eb = 1e-3
    c = contexts["prepass"]
    plan = c.launch_plan(n, dtype, qt)
    assert_plan(plan, n, dtype, qt)
    xd, at = make_field(c, n, dtype, plan, spike_in_tail=True, seed=12)
    x = xd.cpu().numpy()
    del xd
    assert at >= n // 64 * 64
    orc = reflib.oracle_compress(x, eb, qt)
    assert orc["stat"]["max"] == SPIKE
    g = c.compress_core(x, eb, qt=qt)
    parity.compare_compress(g, orc, x, eb, qt, ctx=c)
    del orc
    ref = _from_host(g)
    _same(two_pass(c, x, eb, qt), ref, qt, "stats_dev + compress_dev")
    sr = single_read(c, x, eb, qt)
    assert sr["info"]["n_exact_path"] == 0, "k_sample reads the tail block exactly: the belief holds"
    _same(sr, ref, qt, "single-read")
    _same(field_dev(c, x, eb, qt), ref, qt, "compress_field_dev")
    _same(known_stats(c, x, eb, qt, SPIKE / 10), ref, qt, "compress_known_stats_dev, belief a decade low")
    got = decode_all(contexts, dict(bin_index=ref["bins"], dc=ref["dc"], ac=ref["ac"], qtable=ref["qt"], sf=ref["info"]["sf"]), n, dtype, eb, qt)
    if not qt:
        assert_error_bound(x, got, ref["bins"], ref["dc"], ref["ac"], eb, ref["info"]["sf"])


@pytest.fixture(scope="module")
def limit_contexts():
    """the default (single-launch kernels up to 256 MiB) and streaming only"""
    cs = dict(default=_ctx(), streaming=_ctx(DCTZ_FUSED_MAX_MB=0))
    yield cs
    for c in cs.values():
        c.close()


@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=_id)
@pytest.mark.parametrize("qt", [False, True])
def test_the_single_launch_limit(limit_contexts, dtype, qt):
    """N = 256 MiB / element size runs the single-launch kernels, 64 elements more the streaming chain; both give the
    streaming path's bits, and the smaller one the oracle's result"""
    dtype = np.dtype(dtype)
    es = dtype.itemsize
    eb = 1e-3
    d, s = limit_contexts["default"], limit_contexts["streaming"]
    for n, fused in ((FUSED_LIMIT // es, True), (FUSED_LIMIT // es + 64, False)):
        plan = d.launch_plan(n, dtype, qt)
        print(f"\nplan {dtype.name} {'qt' if qt else 'ec'} n={n}: {plan}")
        assert (plan["fused_compress_grid"] > 0) == fused and (plan["fused_decompress_grid"] > 0) == fused, plan
        assert s.launch_plan(n, dtype, qt)["fused_compress_grid"] == 0
        xd = torch.empty(n, dtype=torch.float64, device="cuda")
        d.fill_hash_field(xd.data_ptr(), 0, n, 2048, 20261018, torch.cuda.current_stream().cuda_stream)
        g = torch.Generator(device="cuda").manual_seed(13)
        xd[n // 3: n // 3 + 5 * TILE] = 30.0 + 120.0 * (torch.rand(5 * TILE, generator=g, device="cuda", dtype=torch.float64) - 0.5)  # outliers
        x = (xd if es == 8 else xd.float()).cpu().numpy()
        del xd
        r = field_dev(d, x, eb, qt)
        _same(field_dev(s, x, eb, qt), r, qt, f"n={n}: compress_field_dev, default against streaming")
        h = d.compress_core(x, eb, qt=qt)
        _same(_from_host(h), r, qt, f"n={n}: compress_core, default")
        _same(_from_host(s.compress_core(x, eb, qt=qt)), r, qt, f"n={n}: compress_core, streaming")
        out = [c.decompress_core(r["bins"], r["dc"], r["ac"], n, dtype, eb, r["info"]["sf"], qt=qt, qtable=r["qt"]) for c in (d, s)]
        assert np.all(np.isfinite(out[0])) and np.array_equal(out[0].view(np.uint8), out[1].view(np.uint8)), f"n={n}: decodes differ"
        if fused:
            orc = reflib.oracle_compress(x, eb, qt)
            parity.compare_compress(h, orc, x, eb, qt, ctx=d)
            want = reflib.oracle_decompress(orc["bin_index"], orc["dc"], orc["ac"], orc["qtable"], n, eb, orc["stat"]["sf"], qt, dtype)
            got = d.decompress_core(orc["bin_index"], orc["dc"], orc["ac"], n, dtype, eb, orc["stat"]["sf"], qt=qt, qtable=orc["qtable"])
            parity.check_reconstruction(got, want, orc["stat"]["sf"])
            assert np.array_equal(got.view(np.uint8), s.decompress_core(orc["bin_index"], orc["dc"], orc["ac"], n, dtype, eb, orc["stat"]["sf"],
                                                                         qt=qt, qtable=orc["qtable"]).view(np.uint8))
