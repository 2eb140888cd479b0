"""GPU: region decompression (dctz_gpu_outlier_index_dev + dctz_gpu_decompress_ranges_dev).  Every decoded range must equal
the same elements of dctz_gpu_decompress_dev's output bit for bit, whatever the ranges look like; damaged inputs set the
corrupt bits without reading past the outliers."""
import numpy as np
import pytest
import torch

from dctz_b200 import DOUBLE, FLOAT, DctzGpuError, binding, fields, slabs

pytestmark = pytest.mark.gpu

TILE, GROUP, CHUNK = 2048, 2048 * 32, 2048 * 32 * 1024  # elements per warp tile, per group of tiles, per chunk of groups


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _code(dtype):
    return DOUBLE if np.dtype(dtype) == np.float64 else FLOAT


def _tdt(dtype):
    return torch.float64 if np.dtype(dtype) == np.float64 else torch.float32


def _bits(t):
    return t.view(torch.int64) if t.dtype == torch.float64 else t.view(torch.int32)


class Field:
    """A compressed field on the device, its full decode (decompress_dev) and its outlier index."""

    def __init__(self, ctx, n, dtype, eb, qt, bins, dc, ac, n_outliers, qtab, sf):
        self.ctx, self.n, self.dtype, self.eb, self.qt, self.sf = ctx, n, np.dtype(dtype), eb, qt, sf
        self.bins, self.dc, self.ac, self.n_outliers, self.qtab = bins, dc, ac, int(n_outliers), qtab
        s = _stream()
        self.full = torch.empty(n, dtype=_tdt(dtype), device="cuda")
        ctx.decompress_dev(bins.data_ptr(), dc.data_ptr(), ac.data_ptr() if self.n_outliers else 0, self.n_outliers,
                           qtab.data_ptr() if qt else 0, n, _code(dtype), eb, sf, qt, self.full.data_ptr(), s)
        self.index = self.build_index(n)

    def build_index(self, n):
        self.index_count = torch.full((1,), -1, dtype=torch.int64, device="cuda")
        index = torch.empty(self.ctx.outlier_index_bytes(n), dtype=torch.uint8, device="cuda")
        self.ctx.outlier_index_dev(self.bins.data_ptr(), n, index.data_ptr(), self.index_count.data_ptr(), _stream())
        return index

    def decode(self, ranges, n_outliers=None, index=None, ac=None):
        r = np.ascontiguousarray(ranges, dtype=np.uint64)
        d_r = _dev(r.view(np.int64))
        out = torch.full((max(1, int(r[:, 1].sum())),), float("nan"), dtype=_tdt(self.dtype), device="cuda")
        corrupt = torch.zeros(1, dtype=torch.int32, device="cuda")
        n_out = self.n_outliers if n_outliers is None else n_outliers
        ac = self.ac if ac is None else ac
        self.ctx.decompress_ranges_dev(self.bins.data_ptr(), self.dc.data_ptr(), ac.data_ptr() if n_out else 0, n_out,
                                       self.qtab.data_ptr() if self.qt else 0, self.n, _code(self.dtype), self.eb, self.sf, self.qt,
                                       (self.index if index is None else index).data_ptr(), d_r.data_ptr(), r.shape[0], out.data_ptr(),
                                       _stream(), corrupt.data_ptr())
        torch.cuda.synchronize()
        return out, int(corrupt.item())

    def expected(self, ranges):
        r = np.asarray(ranges, dtype=np.int64)
        counts = r[:, 1]
        starts = np.repeat(r[:, 0] - (np.cumsum(counts) - counts), counts)
        idx = _dev(starts + np.arange(int(counts.sum()), dtype=np.int64))
        return self.full[idx]

    def check(self, ranges):
        out, corrupt = self.decode(ranges)
        assert corrupt == 0
        assert torch.equal(_bits(out), _bits(self.expected(ranges)))


def field_from_host(ctx, x, eb, qt):
    c = ctx.compress_core(x, eb, qt=qt)
    ac = _dev(c["ac"]) if c["ac"].size else torch.zeros(4, dtype=torch.float32, device="cuda")
    qtab = _dev(c["qtable"]) if qt else None
    f = Field(ctx, x.size, x.dtype, eb, qt, _dev(c["bin_index"]), _dev(c["dc"]), ac, c["ac"].size, qtab, c["sf"])
    torch.cuda.synchronize()
    assert int(f.index_count.item()) == c["info"]["n_outliers"]
    return f


def random_ranges(rng, n, k, maxlen=5000):
    """the whole field, the tail block, and k ranges of every kind -- single elements, whole blocks, ranges that start
    and end inside blocks, ranges across tile / group / chunk boundaries -- overlapping, in random order"""
    out = [(0, n)]
    tail0 = n // 64 * 64
    if tail0 < n:
        out += [(tail0, n - tail0), (n - 1, 1), (max(0, tail0 - 100), n - max(0, tail0 - 100))]
    for _ in range(k):
        kind = int(rng.integers(5))
        if kind == 0:
            a, c = int(rng.integers(n)), 1
        elif kind == 1 and n >= 64:
            a, c = int(rng.integers(n // 64)) * 64, 64
        elif kind == 2:
            a, c = int(rng.integers(n)), int(rng.integers(2, maxlen))
        elif kind == 3 and n > 64:
            bounds = [b for b in (64, TILE, GROUP, CHUNK) if b < n]
            b = bounds[int(rng.integers(len(bounds)))]
            a = int(rng.integers(1, n // b + 1)) * b - int(rng.integers(1, 300))
            c = int(rng.integers(2, 700))
        else:
            a = int(rng.integers(n))
            c = int(rng.integers(1, min(n - a, maxlen) + 1))
        a = min(max(a, 0), n - 1)
        out.append((a, max(1, min(c, n - a))))
    out = np.array(out, dtype=np.uint64)
    return out[rng.permutation(len(out))]


CASES = ["tail1", "tail32", "three_blocks_tail37", "tail63_odd", "only_tail", "heavy_outliers", "single_spike", "sf_one", "all_equal", "smooth"]


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("qt", [False, True])
def test_ranges_of_the_small_cases_equal_the_full_decode(ctx, dtype, qt):
    rng = np.random.default_rng(17 + int(qt) + 2 * (dtype == np.float32))
    cases = fields.small_cases(dtype)
    for name in CASES:
        f = field_from_host(ctx, cases[name], 1e-3, qt)
        f.check(random_ranges(rng, f.n, 200))
        f.check(np.array([(i, 1) for i in range(f.n)], dtype=np.uint64)[::-1])  # every element alone, backwards


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("qt", [False, True])
def test_many_ranges_in_one_call(ctx, dtype, qt):
    """>= 10^5 ranges over a field of several groups whose tiles hold from no outliers to more than half of their coefficients"""
    rng = np.random.default_rng(5)
    n = 3 * GROUP + 64 * 7 + 45
    t = np.arange(n)
    amp = np.repeat(rng.choice([0.0, 1e-3, 0.05, 3.0], size=(n + TILE - 1) // TILE), TILE)[:n]
    x = (2.0 + np.sin(t / 300.0) + amp * rng.standard_normal(n)).astype(dtype)
    f = field_from_host(ctx, x, 1e-3, qt)
    f.check(random_ranges(rng, n, 120_000, maxlen=300))


@pytest.mark.parametrize("qt", [False, True])
def test_float_field_across_a_chunk_boundary(ctx, qt):
    """more than 2^26 elements: the ranges cross a chunk_prefix boundary of the index (32 768 tiles)"""
    n = CHUNK + 3 * GROUP + 64 * 3 + 29
    s = _stream()
    xd = torch.empty(n, dtype=torch.float64, device="cuda")
    ctx.fill_hash_field(xd.data_ptr(), 0, n, 2048, fields.SEED, s)
    x = xd.float()
    x[CHUNK - 5000] = 57.0  # outliers on both sides of the boundary
    x[CHUNK + 3000] = -41.0
    del xd
    bins = torch.empty(n, dtype=torch.uint8, device="cuda")
    dc = torch.empty((n + 63) // 64, dtype=torch.float32, device="cuda")
    ac = torch.empty(n, dtype=torch.float32, device="cuda")
    qtab, qraw = torch.zeros(64, dtype=torch.float32, device="cuda"), torch.zeros(64, dtype=torch.float32, device="cuda")
    info = torch.zeros(binding.INFO_BYTES, dtype=torch.uint8, device="cuda")
    ctx.compress_field_dev(x.data_ptr(), n, FLOAT, 1e-3, qt, bins.data_ptr(), dc.data_ptr(), ac.data_ptr(), qtab.data_ptr(), qraw.data_ptr(),
                           info.data_ptr(), s)
    torch.cuda.synchronize()
    i = binding.GpuInfo.from_buffer_copy(info.cpu().numpy().tobytes()).as_dict()
    assert i["status"] == 0 and i["n_outliers"] > 0
    f = Field(ctx, n, np.float32, 1e-3, qt, bins, dc, ac, i["n_outliers"], qtab, i["sf"])
    torch.cuda.synchronize()
    assert int(f.index_count.item()) == i["n_outliers"]
    rng = np.random.default_rng(23)
    r = random_ranges(rng, n, 2000, maxlen=20000)
    r = np.concatenate([r, np.array([(CHUNK - 7000, 14000), (CHUNK - 1, 2), (CHUNK, 1), (n - 2 * GROUP, 2 * GROUP)], dtype=np.uint64)])
    f.check(r)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_per_slab_indices_reproduce_the_single_field_decode(ctx, dtype):
    """two emulated slabs: each has its own index and outlier array; their ranges are the field's elements"""
    x = np.concatenate([fields.small_cases(dtype)["tail32"], fields.small_cases(dtype)["heavy_outliers"] * 0.02 + 3]).astype(dtype)
    eb, world, code = 1e-3, 2, _code(dtype)
    whole = field_from_host(ctx, x, eb, False)
    parts = slabs.partition(x.size, world)
    s = _stream()
    xs = [_dev(x[a:a + c]) for a, c in parts]
    stats_all = torch.zeros(3 * world, dtype=torch.float64, device="cuda")
    for r, (a, c) in enumerate(parts):
        ctx.stats_dev(xs[r].data_ptr(), c, code, stats_all[3 * r:].data_ptr(), s)
    rng = np.random.default_rng(8)
    for r, (a, c) in enumerate(parts):
        bins = torch.empty(c, dtype=torch.uint8, device="cuda")
        dc = torch.empty((c + 63) // 64, dtype=torch.float32, device="cuda")
        ac = torch.empty(c, dtype=torch.float32, device="cuda")
        info = torch.zeros(binding.INFO_BYTES, dtype=torch.uint8, device="cuda")
        ctx.compress_dev(xs[r].data_ptr(), c, x.size, code, eb, False, stats_all.data_ptr(), world, r == 0, bins.data_ptr(), dc.data_ptr(),
                         ac.data_ptr(), 0, info.data_ptr(), s)
        torch.cuda.synchronize()
        i = binding.GpuInfo.from_buffer_copy(info.cpu().numpy().tobytes()).as_dict()
        assert i["sf"] == whole.sf
        slab = Field(ctx, c, dtype, eb, False, bins, dc, ac, i["n_outliers"], None, whole.sf)
        torch.cuda.synchronize()
        assert int(slab.index_count.item()) == i["n_outliers"]
        rg = random_ranges(rng, c, 300)
        out, corrupt = slab.decode(rg)
        assert corrupt == 0
        shifted = rg.copy()
        shifted[:, 0] += np.uint64(a)
        assert torch.equal(_bits(out), _bits(whole.expected(shifted)))


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("qt", [False, True])
def test_fewer_outliers_than_markers_sets_bit_0_and_reads_nothing_past_them(ctx, dtype, qt):
    x = fields.small_cases(dtype)["heavy_outliers"][: 64 * 150 + 21]
    f = field_from_host(ctx, x, 1e-3, qt)
    k = f.n_outliers // 2
    guard = torch.full((f.n_outliers + 8,), float("nan"), dtype=torch.float32, device="cuda")
    guard[:k] = f.ac[:k]  # the readable part, NaN after it: a read past n_outliers shows in the output
    out, corrupt = f.decode(np.array([(0, f.n), (f.n - 3, 3), (100, 50)], dtype=np.uint64), n_outliers=k, ac=guard)
    assert corrupt & 1 and not corrupt & 2
    assert bool(torch.all(torch.isfinite(out)))
    # the ranges that end before the first damaged tile are still exact
    out, corrupt = f.decode(np.array([(5, 100)], dtype=np.uint64), n_outliers=k, ac=guard)
    assert corrupt == 0 and torch.equal(_bits(out), _bits(f.expected([(5, 100)])))


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_bad_ranges_set_bit_1_and_the_others_are_written(ctx, dtype):
    f = field_from_host(ctx, fields.small_cases(dtype)["tail63_odd"], 1e-3, False)
    n = f.n
    good = [(3, 70), (n - 5, 5), (0, n)]
    bad = [(n - 5, 10), (7, 0), (n, 1), (2**63, 4)]
    rg = np.array([good[0], bad[0], good[1], bad[1], bad[2], good[2], bad[3]], dtype=np.uint64)
    out, corrupt = f.decode(rg)
    assert corrupt == 2
    at = np.concatenate([[0], np.cumsum(rg[:, 1].astype(np.int64))])
    for j, (a, c) in enumerate(rg.astype(np.int64)):
        if (a, c) in good:
            assert torch.equal(_bits(out[at[j]:at[j] + c]), _bits(f.expected([(a, c)])))
        elif j != len(rg) - 1:
            assert bool(torch.all(torch.isnan(out[at[j]:at[j + 1]])))  # not written


def test_index_of_another_length_sets_bit_0_and_writes_nothing(ctx):
    f = field_from_host(ctx, fields.small_cases(np.float64)["tail32"], 1e-3, False)
    other = f.build_index(f.n - 64)
    out, corrupt = f.decode(np.array([(0, 100), (f.n - 10, 10)], dtype=np.uint64), index=other)
    assert corrupt == 1 and bool(torch.all(torch.isnan(out)))


def test_argument_errors(ctx):
    f = field_from_host(ctx, fields.small_cases(np.float64)["tail32"], 1e-3, False)
    d_r = _dev(np.array([[0, 10]], dtype=np.int64))
    out = torch.empty(16, dtype=torch.float64, device="cuda")
    s = _stream()

    def call(**kw):
        a = dict(bins=f.bins.data_ptr(), dc=f.dc.data_ptr(), index=f.index.data_ptr(), ranges=d_r.data_ptr(), nranges=1, out=out.data_ptr())
        a.update(kw)
        ctx.decompress_ranges_dev(a["bins"], a["dc"], f.ac.data_ptr(), f.n_outliers, 0, f.n, DOUBLE, 1e-3, f.sf, False, a["index"], a["ranges"],
                                  a["nranges"], a["out"], s)

    call()
    for kw in (dict(nranges=0), dict(ranges=0), dict(index=0), dict(out=0), dict(bins=0), dict(index=f.index.data_ptr() + 8),
               dict(bins=f.bins.data_ptr() + 4), dict(ranges=d_r.data_ptr() + 4), dict(out=out.data_ptr() + 4)):
        with pytest.raises(DctzGpuError) as e:
            call(**kw)
        assert e.value.code == -3, kw
    with pytest.raises(DctzGpuError) as e:
        ctx.outlier_index_dev(f.bins.data_ptr() + 4, f.n, f.index.data_ptr())
    assert e.value.code == -3
    with pytest.raises(DctzGpuError) as e:
        ctx.outlier_index_dev(f.bins.data_ptr(), f.n, 0)
    assert e.value.code == -3
    torch.cuda.synchronize()
