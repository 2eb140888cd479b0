"""Region decompression on the c5 slab: what one plane or one sub-box of a compressed field costs against a full decode.

The slab is 2^30 doubles, a (256, 2048, 2048) block of the 2048^3 hash field (dctz_gpu_fill_hash_field), compressed once
with dctz_gpu_compress_field_dev (EC, eb 1e-3).  CUDA-event times (median over --iters after --warmup calls) of:
the outlier index build, dctz_gpu_decompress_dev of the whole slab, and dctz_gpu_decompress_ranges_dev for one range
covering the slab, a z-plane (one range of 2^22), a y-plane (256 ranges of 2048), an x-plane (2^19 single elements) and a
128^3 sub-box.  Every range output is compared bit for bit with the matching slice of the full decode.  Bin-id bytes
touched counts what the kernels read of bin_index: a range reads the bin ids of every tile it touches from the tile's
start to its last block.  The slab's arrays far exceed the 126 MB L2; the plane and box queries are small enough that
their inputs stay in L2 between timed calls (those times are for a warm L2).

    python tools/roi_bench.py --out DIR      (writes DIR/roi_bench.json)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import dctz_b200  # noqa: E402
from dctz_b200 import DOUBLE, binding, fields  # noqa: E402
from dctz_b200.regions import box_ranges  # noqa: E402

TILE = 2048


def gpu_identity():
    ident = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        ident.update(power_limit_w=float(q[0]), sm_max_mhz=float(q[1]))
    except Exception as e:  # the numbers are still printed, without the power limit
        ident.update(power_limit_w=None, note=f"nvidia-smi: {e}")
    return ident


def bin_bytes_touched(ranges, n):
    """bytes of bin_index the range kernel reads for these ranges (N % 64 == 0 here: no tail block)"""
    a = ranges[:, 0].astype(np.int64)
    b = a + ranges[:, 1].astype(np.int64)
    t0, t1 = a // TILE, (b - 1) // TILE
    last = ((b - 1) // 64 - t1 * 32 + 1) * 64
    return int(np.sum(np.where(t0 == t1, last, (t1 - t0) * TILE + last)))


def timed(fn, warmup, iters):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return dict(median_ms=float(np.median(ms)), min_ms=float(np.min(ms)), max_ms=float(np.max(ms)), n=len(ms))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--planes", type=int, default=256, help="z extent of the slab (2048 x 2048 planes)")
    ap.add_argument("--eb", type=float, default=1e-3)
    args = ap.parse_args()
    if args.iters < 20:
        ap.error("--iters must be at least 20")
    os.makedirs(args.out, exist_ok=True)
    dim = 2048
    shape = (args.planes, dim, dim)
    n = args.planes * dim * dim
    ident = gpu_identity()
    print(f"GPU: {ident}", flush=True)

    ctx = dctz_b200.Context(0)
    s = torch.cuda.current_stream().cuda_stream
    x = torch.empty(n, dtype=torch.float64, device="cuda")
    ctx.fill_hash_field(x.data_ptr(), 0, n, dim, fields.SEED, s)
    bins = torch.empty(n, dtype=torch.uint8, device="cuda")
    dc = torch.empty(n // 64, dtype=torch.float32, device="cuda")
    ac = torch.empty(n, dtype=torch.float32, device="cuda")
    info = torch.zeros(binding.INFO_BYTES, dtype=torch.uint8, device="cuda")
    ctx.compress_field_dev(x.data_ptr(), n, DOUBLE, args.eb, False, bins.data_ptr(), dc.data_ptr(), ac.data_ptr(), 0, 0, info.data_ptr(), s)
    torch.cuda.synchronize()
    del x
    inf = binding.GpuInfo.from_buffer_copy(info.cpu().numpy().tobytes()).as_dict()
    k, sf = inf["n_outliers"], inf["sf"]
    print(f"slab {shape}: N = {n}, outliers = {k}, sf = {sf}", flush=True)

    full = torch.empty(n, dtype=torch.float64, device="cuda")
    index = torch.empty(ctx.outlier_index_bytes(n), dtype=torch.uint8, device="cuda")
    n_idx = torch.zeros(1, dtype=torch.int64, device="cuda")
    results = []

    def record(name, t, elements, bin_bytes, nranges=None, identical=None):
        row = dict(name=name, nranges=nranges, elements=elements, bin_bytes_touched=bin_bytes, **t,
                   elements_per_s=elements / (t["median_ms"] * 1e-3), bit_identical=identical)
        results.append(row)
        print(f"{name:<14} ranges={str(nranges):>7} elements={elements:>11} median={t['median_ms']:8.4f} ms "
              f"({row['elements_per_s'] / 1e9:8.3f} G elem/s) bin bytes={bin_bytes:>11} identical={identical}", flush=True)

    t = timed(lambda: ctx.outlier_index_dev(bins.data_ptr(), n, index.data_ptr(), n_idx.data_ptr(), s), args.warmup, args.iters)
    torch.cuda.synchronize()
    assert int(n_idx.item()) == k, (int(n_idx.item()), k)
    record("index_build", t, n, n)
    t = timed(lambda: ctx.decompress_dev(bins.data_ptr(), dc.data_ptr(), ac.data_ptr(), k, 0, n, DOUBLE, args.eb, sf, False, full.data_ptr(), s),
              args.warmup, args.iters)
    record("decompress_dev", t, n, n)

    z, y, xx = args.planes // 2, 1000, 777
    lo3 = (args.planes // 2 - 64, 960, 960)
    queries = [
        ("whole_range", np.array([[0, n]], dtype=np.uint64), full),
        ("z_plane", box_ranges(shape, (z, 0, 0), (z + 1, dim, dim)), full.view(shape)[z]),
        ("y_plane", box_ranges(shape, (0, y, 0), (args.planes, y + 1, dim)), full.view(shape)[:, y, :]),
        ("x_plane", box_ranges(shape, (0, 0, xx), (args.planes, dim, xx + 1)), full.view(shape)[:, :, xx]),
        ("box_128", box_ranges(shape, lo3, tuple(v + 128 for v in lo3)), full.view(shape)[lo3[0]:lo3[0] + 128, 960:1088, 960:1088]),
    ]
    ok = True
    for name, rg, want in queries:
        d_r = torch.from_numpy(rg.view(np.int64)).cuda()
        m = int(rg[:, 1].sum())
        out = torch.empty(m, dtype=torch.float64, device="cuda")
        corrupt = torch.zeros(1, dtype=torch.int32, device="cuda")
        t = timed(lambda: ctx.decompress_ranges_dev(bins.data_ptr(), dc.data_ptr(), ac.data_ptr(), k, 0, n, DOUBLE, args.eb, sf, False,
                                                    index.data_ptr(), d_r.data_ptr(), rg.shape[0], out.data_ptr(), s, corrupt.data_ptr()),
                  args.warmup, args.iters)
        same = bool(torch.equal(out.view(torch.int64), want.reshape(-1).view(torch.int64))) and int(corrupt.item()) == 0
        ok &= same
        record(name, t, m, bin_bytes_touched(rg, n), rg.shape[0], same)
        del out, d_r

    base = next(r for r in results if r["name"] == "decompress_dev")
    whole = next(r for r in results if r["name"] == "whole_range")
    ratio = whole["elements_per_s"] / base["elements_per_s"]
    print(f"whole-slab range / decompress_dev throughput: {ratio:.3f}", flush=True)
    doc = dict(gpu=ident, slab=dict(shape=shape, n=n, eb=args.eb, n_outliers=k, sf=sf), warmup=args.warmup, iters=args.iters,
               whole_range_vs_decompress_dev=ratio, all_bit_identical=ok, results=results)
    with open(os.path.join(args.out, "roi_bench.json"), "w") as fh:
        json.dump(doc, fh, indent=1)
    ctx.close()
    if not ok:
        print("FAILED: a range output differs from the full decode", flush=True)
        sys.exit(1)


if __name__ == "__main__":
    main()
