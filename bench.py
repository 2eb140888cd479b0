#!/usr/bin/env python3
"""bench.py -- DCTZ hot path (block DCT-II/IDCT + adaptive binning quantiser) on 1..8 B200.

A "step" is one pass of the hot path over one slab of synthetic input: COMPRESS (statistics ->
[NCCL all-gather of 3 doubles per rank] -> fused scale+DCT+quantise+outlier compaction [-> QT: NCCL max-reduction of
the 64-entry table -> rescale]) followed by DECOMPRESS (outlier scan + dequantise + IDCT + de-scale).  The metric is
BASELINE.json's "compress/decompress GB/s of input": input bytes divided by the time of the compress+decompress
round trip, summed over ranks; the two halves are also reported separately.

Default workload (config.workload = "c5-slab"): each rank owns a contiguous block slab of 2^30 doubles (8 GiB) of
BASELINE.json's config[4] field (2048^3 double, error bound 1E-3, EC mode, generated on the device by the exactly
reproducible formula of SURVEY.md §8d).  At --gpus 8 the ranks together hold exactly the 64 GiB field; fewer ranks
hold its first slabs (weak scaling).  `--scaling strong` keeps the field fixed at 2^33 elements instead: it is cut
by dctz_b200.slabs.partition over the ranks and every rank works through its share in sub-slabs of 2^30 elements.
The other BASELINE configs (c1..c4, c3 at its three error bounds) are timed in the `configs` leg of the default
line and alone with --workload c1|c2|c3|c4 [--eb ...].

`--impl reference` times the reference's own CPU implementation of the same path (the unmodified sources compiled
into oracle/_ref, FFTW replaced by the stand-in because FFTW3 is not installed) on the host cores, on a bounded
sample of the same workload.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "compress+decompress round-trip GB/s of input (hot path: stats, scale, block DCT-II/IDCT, binning quantiser)"
UNIT = "GB/s"
SEED = 20261018
HASH_DIM = 2048
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback
FFT_NOTE = "stand-in radix-2 FFT (FFTW3 is not installed; ~43% of dct_t, an FFTW-class transform would make the CPU arm ~1.4x faster)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", choices=["c5-slab", "c1", "c2", "c3", "c4"], default="c5-slab")
    ap.add_argument("--eb", type=float, default=1e-3, help="error bound (config[2] sweeps 1E-3 / 1E-4 / 1E-5)")
    ap.add_argument("--scaling", choices=["weak", "strong"], default="weak",
                    help="c5-slab: weak = 2^slab-log2 elements per rank; strong = the fixed 2^33-element field cut over the ranks")
    ap.add_argument("--field-log2", type=int, default=33, help="--scaling strong: elements of the whole field (2048^3 = 2^33)")
    ap.add_argument("--slab-log2", type=int, default=30, help="elements per rank of the c5 slab / per sub-slab in strong mode (2^30 = 8 GiB)")
    ap.add_argument("--e2e-log2", type=int, default=27, help="elements of the slab pushed through the host-buffer API for e2e")
    ap.add_argument("--cpu-log2", type=int, default=23, help="elements per process of the CPU reference sample")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / quality legs")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-lanes", type=int, default=3, help="independent fields in flight through the host-buffer API (host threads, a context each)")
    ap.add_argument("--no-configs", action="store_true", help="skip the configs leg (c1..c4 beside the headline)")
    ap.add_argument("--f32", action="store_true", help="c5-slab only: cast the slab to float (single-precision path)")
    ap.add_argument("--qt", action="store_true", help="c5-slab: quantiser (QT) mode instead of error-bounded (EC); at N > 1 the qtable is reduced over NCCL")
    ap.add_argument("--noise", type=float, default=0.0, help="c5-slab only: add Gaussian noise of this std (raw units) to study the outlier path")
    ap.add_argument("--two-pass", action="store_true", help="c5-slab: statistics pass + compress pass (two reads of the input) instead of the single-read path")
    ap.add_argument("--no-outlier-leg", action="store_true", help="skip the extra (reported, not headline) measurement with ~5%% outliers")
    ap.add_argument("--watchdog", type=int, default=1500, help="seconds after which a stuck run dumps every thread's Python stack to stderr and exits 3 (0 = off)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step handed back (bin indices, DC, outliers and their "
                                                          "count, [qtable,] scaling factor, reconstruction) as DIR/<name>.npy, rank 0 only")
    return ap.parse_args()


def eb_str(eb):
    """1e-3 -> '1E-3' (the spelling of the reference's command line and file names)"""
    m, e = f"{eb:.0E}".split("E")
    return f"{m}E{int(e)}"


# ------------------------------------------------------------------------------------------------
# CPU reference arm (oracle/_ref = unmodified reference sources + FFTW stand-in; else the oracle port)
# ------------------------------------------------------------------------------------------------
REF_BIN = {False: os.path.join(ROOT, "oracle", "_ref", "dctz-ec-test"), True: os.path.join(ROOT, "oracle", "_ref", "dctz-qt-test")}
_T = r"([0-9.eE+-]+)\(s\)"


def _parse_ref_stdout(txt):
    """Stage timers printed under -DTIME_DEBUG (dctz-comp-lib.c:762-773, dctz-decomp-lib.c:513-528)."""
    m1 = re.search(r"sf_t=" + _T + r", dct_t=" + _T + r", zlib_t\(compress\)=" + _T, txt)
    m2 = re.search(r"sf_t=" + _T + r", idct_t=" + _T + r", zlib_t\(uncompress\)=" + _T, txt)
    if not m1 or not m2:
        raise RuntimeError("cannot parse the reference's stage timers:\n" + txt[-2000:])
    cr = re.search(r"CR = ([0-9.]+)", txt)
    ct = re.search(r"comp_time = ([0-9.eE+-]+) \(s\)", txt)
    dt = re.search(r"decomp_time = ([0-9.eE+-]+) \(s\)", txt)
    return dict(comp_hot=float(m1.group(1)) + float(m1.group(2)), comp_zlib=float(m1.group(3)),
                decomp_hot=float(m2.group(1)) + float(m2.group(2)), cr=float(cr.group(1)) if cr else None,
                comp_api=float(ct.group(1)) if ct else None, decomp_api=float(dt.group(1)) if dt else None)


def run_reference_cli(sample_path, n, is_double, qt, procs, eb):
    """Run `procs` independent copies of the reference's own CLI (one per host thread; its hot path is
    single-threaded, dct.c:18-22 is not re-entrant) on the same sample; returns per-process timers."""
    tmp = tempfile.mkdtemp(prefix="dctz_ref_")
    try:
        ps = []
        for i in range(procs):
            d = os.path.join(tmp, f"p{i}")
            os.makedirs(d)
            os.symlink(sample_path, os.path.join(d, "in.bin"))
            cmd = [REF_BIN[qt], "-d" if is_double else "-f", eb_str(eb), "var", os.path.join(d, "in.bin"), str(n)]
            ps.append(subprocess.Popen(cmd, cwd=d, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
        outs = [p.communicate()[0] for p in ps]
        for p, o in zip(ps, outs):
            if p.returncode != 0:
                raise RuntimeError(f"reference CLI failed ({p.returncode}):\n{o[-2000:]}")
        return [_parse_ref_stdout(o) for o in outs]
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def time_port(x, qt, eb):
    """Fallback when oracle/_ref is absent: the oracle port, single thread."""
    from tests import reflib

    t0 = time.perf_counter()
    o = reflib.oracle_compress(x, eb, qt, want_coef=False)
    t1 = time.perf_counter()
    reflib.oracle_decompress(o["bin_index"], o["dc"], o["ac"], o["qtable"], x.size, eb, o["stat"]["sf"], qt, x.dtype)
    t2 = time.perf_counter()
    return dict(comp_hot=t1 - t0, decomp_hot=t2 - t1, comp_zlib=None, cr=None, comp_api=None, decomp_api=None)


def cpu_reference(sample, qt, procs, eb):
    """Times the CPU implementation on `sample` (numpy array); aggregate GB/s of input over `procs`
    concurrent single-threaded instances."""
    import numpy as np

    n = sample.size
    nbytes = sample.nbytes
    have_ref = os.path.exists(REF_BIN[qt])
    if have_ref:
        tmp = tempfile.mkdtemp(prefix="dctz_sample_")
        try:
            path = os.path.join(tmp, "sample.bin")
            sample.tofile(path)
            res = run_reference_cli(path, n, sample.dtype == np.float64, qt, procs, eb)
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        kind = "reference"
    else:
        procs = 1
        res = [time_port(sample, qt, eb)]
        kind = "port"
    tc = max(r["comp_hot"] for r in res)
    td = max(r["decomp_hot"] for r in res)
    gb = procs * nbytes / 1e9
    out = dict(value=gb / (tc + td), unit=UNIT, cores=procs, kind=kind, compress_gbs=gb / tc, decompress_gbs=gb / td,
               host_cpus=os.cpu_count(), cr=res[0]["cr"], fft=FFT_NOTE if have_ref else "oracle port (same stand-in FFT)",
               sample=f"{procs} concurrent single-thread instance(s), each {n} elements ({nbytes / 2**20:.0f} MiB) of the workload; "
                      f"hot-path stage timers only (sf_t+dct_t, idct_t+sf_t), zlib excluded"
                      + ("; FFTW3 replaced by oracle/fftw_standin" if have_ref else ""))
    if res[0]["comp_api"]:
        ca, da = max(r["comp_api"] for r in res), max(r["decomp_api"] for r in res)
        out["api"] = dict(compress_gbs=gb / ca, decompress_gbs=gb / da, value=gb / (ca + da),
                          note="the reference's own comp_time / decomp_time (whole dctz_compress / dctz_decompress: hot path + zlib + dumps), "
                               f"aggregate of the same {procs} instances")
    return out


def make_host_field(workload):
    import numpy as np

    from dctz_b200 import fields

    if workload == "c1":
        return fields.cesm_like(), False
    if workload == "c2":
        return fields.cesm_like(dtype=np.float32), True
    if workload == "c3":
        return fields.hurricane_like(), False
    if workload == "c4":
        return fields.nyx_like(), False
    raise ValueError(workload)


def make_sample(workload, n):
    import numpy as np

    from dctz_b200 import fields

    if workload == "c5-slab":
        return fields.hash_field(0, n, HASH_DIM, SEED), False
    x, qt = make_host_field(workload)
    return np.ascontiguousarray(x[:n]), qt


DUMP_SAMPLE = 1 << 20  # elements kept of a longer output: at most 8 MiB an array, 20 MiB for the four long ones


def dump_outputs(path, arrays):
    """--dump-outputs: name -> 1-D device tensor.  An array longer than DUMP_SAMPLE is cut to a seeded sample of its
    positions, the same for every array of that length, so that the dumps of two builds compare element for element.
    Floating-point arrays keep their type; the bin indices (uint8) are stored as float32.  An empty array is not written:
    the outliers of a field that has none are absent, and n_outliers.npy holds their count."""
    import numpy as np
    import torch

    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        if t.numel() == 0:
            continue
        if t.numel() > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(SEED).choice(t.numel(), DUMP_SAMPLE, replace=False))
            t = t[torch.from_numpy(idx).to(t.device)]
        a = t.cpu().numpy()
        np.save(os.path.join(path, f"{name}.npy"), a if a.dtype in (np.float32, np.float64) else a.astype(np.float32))


def main_reference(args):
    if args.dump_outputs:
        raise SystemExit("bench.py: --dump-outputs applies to the GPU arm (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    procs = max(1, min(os.cpu_count() or 1, 32))
    n = 1 << args.cpu_log2
    sample, qt = make_sample(args.workload, n)
    qt = qt or (args.workload == "c5-slab" and args.qt)
    if args.f32:
        sample = sample.astype("float32")
    for _ in range(args.warmup):
        cpu_reference(sample, qt, procs, args.eb)
    t0 = time.perf_counter()
    runs = [cpu_reference(sample, qt, procs, args.eb) for _ in range(args.steps)]
    wall = time.perf_counter() - t0
    # aggregate: total bytes / total hot-path time over the K steps
    inv = sum(1.0 / r["value"] for r in runs) / len(runs)
    val = 1.0 / inv
    base = runs[-1]
    base["value"] = val
    line = dict(metric=METRIC, value=val, unit=UNIT, impl="reference", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * wall / args.steps, higher_is_better=True, scaling=args.scaling, vs_baseline=None,
                dtype="f64" if sample.dtype.itemsize == 8 else "f32", data="synthetic",
                config=workload_config(args, args.gpus), cpu_baseline=base,
                e2e=dict(value=val, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    _emit(line)
    return 0


def workload_config(args, world):
    eb = args.eb
    if args.workload == "c5-slab":
        n = 1 << args.slab_log2
        mode = "qt" if getattr(args, "qt", False) else "ec"
        if args.scaling == "strong":
            nt = 1 << args.field_log2
            return dict(workload=f"c5-field: the whole {HASH_DIM}^3 double field of BASELINE config[4] (2^{args.field_log2} elements, "
                                 f"{nt * 8 / 2**30:.0f} GiB) cut into contiguous block slabs over {world} GPU(s), each rank working through its "
                                 f"share in sub-slabs of 2^{args.slab_log2} elements; {mode.upper()} mode, error bound {eb_str(eb)}",
                        mode=mode, error_bound=eb, elements_total=nt, elements_per_gpu=nt // world, block=64,
                        l2="inputs larger than L2 (no flush needed)", parallelism=f"slab{world}")
        if getattr(args, "f32", False):
            return dict(workload=f"c5-slab-f32: per-GPU slab of 2^{args.slab_log2} floats (the {HASH_DIM}^3 field cast to float), {mode.upper()}, eb {eb_str(eb)}",
                        mode=mode, error_bound=eb, elements_per_gpu=n, block=64, l2="inputs larger than L2 (no flush needed)",
                        parallelism=f"slab{world}")
        return dict(workload=f"c5-slab: per-GPU contiguous slab of 2^{args.slab_log2} doubles ({n * 8 / 2**30:.0f} GiB) of the "
                             f"{HASH_DIM}^3 double field (BASELINE config[4]), {mode.upper()} mode, error bound {eb_str(eb)}; "
                             f"{world} slab(s) = {world * n * 8 / 2**30:.0f} GiB",
                    mode=mode, error_bound=eb, elements_per_gpu=n, block=64, l2="inputs larger than L2 (no flush needed)",
                    parallelism=f"slab{world}")
    desc = {"c1": "config[0] CESM-ATM-shaped 1800x3600 double, EC", "c2": "config[1] 1800x3600 float, QT",
            "c3": "config[2] Hurricane-shaped 100x500x500 float, EC", "c4": "config[3] NYX-shaped 512^3 double, EC"}[args.workload]
    return dict(workload=f"{args.workload}: {desc}, error bound {eb_str(eb)}, one field per GPU", error_bound=eb, block=64,
                l2="L2 flushed between timed steps (write of a 256 MiB buffer, then a read of another 256 MiB so that the lines are clean)" if args.workload in ("c1", "c2", "c3") else
                   "inputs larger than L2 (no flush needed)", parallelism=f"replica{world}")


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi polled every 20 ms from before the warm-up (its first line takes ~0.2 s to appear); stop() keeps
    the samples whose timestamp falls inside the timed region."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None
        self.t0 = self.t1 = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(prefix="clocks_", suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        import datetime

        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        rows = []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        with open(self.path) as fh:
            for ln in fh:
                p = [x.strip() for x in ln.split(",")]
                if len(p) < 10:
                    continue
                try:
                    ts = datetime.datetime.strptime(p[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    rows.append((ts, float(p[2]), float(p[3]), float(p[4]), [nm for nm, v in zip(names, p[6:10]) if v.lower().startswith("active")]))
                except ValueError:
                    continue
        os.unlink(self.path)
        inside = [r for r in rows if self.t0 is not None and self.t0 - 0.02 <= r[0] <= self.t1 + 0.02]
        use = inside if inside else rows[-3:]
        if not use:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        sm = sorted(r[1] for r in use)
        reasons = sorted({x for r in use for x in r[4]})
        return dict(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(r[2] for r in use), power_w_max=max(r[3] for r in use), samples=len(use),
                    samples_in_timed_region=len(inside), reasons=reasons)


class L2Flush:
    """Between timed steps of a field that fits in L2: write a 256 MiB buffer (the contract's flush), then READ another
    256 MiB -- the cache ends up full of clean foreign lines.  (After the write alone L2 is full of DIRTY lines and the
    next kernel is charged for writing the flush itself back to HBM: ~2x the bytes of a 50 MB field.)"""

    def __init__(self, torch, dev):
        self.w = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        self.r = torch.zeros(64 << 20, dtype=torch.float32, device=dev)

    def __call__(self):
        self.w.zero_()
        self.r.sum()


def bytes_per_element(es, p):
    """SURVEY.md §8d: algorithmic bytes per element of compress (B_c, statistics read included) and decompress (B_d)"""
    return 2 * es + 1 + 4 / 64 + 4 * p, es + 1 + 4 / 64 + 4 * p


def time_field(ctx, torch, binding, x, code, eb, qt, steps, warmup, peak, flush):
    """One whole field resident in HBM through the single-field entry points (what dctz_compress drives: one call per
    direction): dctz_gpu_compress_field_dev / dctz_gpu_decompress_dev, CUDA events on the launching stream."""
    n = x.numel()
    es = x.element_size()
    dev = x.device
    stream = torch.cuda.current_stream()
    sh = stream.cuda_stream
    bins = torch.empty(n, dtype=torch.uint8, device=dev)
    dc = torch.empty((n + 63) // 64, dtype=torch.float32, device=dev)
    ac = torch.empty(n, dtype=torch.float32, device=dev)
    out = torch.empty_like(x)
    qtab = torch.zeros(64, dtype=x.dtype, device=dev)
    qraw = torch.zeros(64, dtype=x.dtype, device=dev)
    info_d = torch.zeros(binding.INFO_BYTES, dtype=torch.uint8, device=dev)

    def comp():
        ctx.compress_field_dev(x.data_ptr(), n, code, eb, qt, bins.data_ptr(), dc.data_ptr(), ac.data_ptr(), qtab.data_ptr(), qraw.data_ptr(),
                               info_d.data_ptr(), sh)

    comp()
    torch.cuda.synchronize()
    info = binding.GpuInfo.from_buffer_copy(info_d.cpu().numpy().tobytes()).as_dict()
    if info["status"] != 0:
        raise SystemExit(f"bench.py: compress failed with status {info['status']}")
    sf, n_out = info["sf"], info["n_outliers"]

    def decomp():
        ctx.decompress_dev(bins.data_ptr(), dc.data_ptr(), ac.data_ptr(), n_out, qtab.data_ptr() if qt else 0, n, code, eb, sf, qt, out.data_ptr(), sh)

    for _ in range(warmup):
        if flush is not None:
            flush()
        comp()
        decomp()
    torch.cuda.synchronize()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    l0 = ctx.launch_count
    for k in range(steps):
        if flush is not None:
            flush()
        ev[k][0].record(stream)
        comp()
        ev[k][1].record(stream)
        decomp()
        ev[k][2].record(stream)
    torch.cuda.synchronize()
    launches = (ctx.launch_count - l0) / steps
    tc = sum(e[0].elapsed_time(e[1]) for e in ev) / 1e3 / steps
    td = sum(e[1].elapsed_time(e[2]) for e in ev) / 1e3 / steps
    med = lambda v: sorted(v)[len(v) // 2]  # noqa: E731  (the means are the reported figures; the medians show a step that a hiccup stretched)
    tc_med, td_med = med([e[0].elapsed_time(e[1]) for e in ev]), med([e[1].elapsed_time(e[2]) for e in ev])
    p = n_out / n
    bc, bd = bytes_per_element(es, p)
    single_read = n * es > (256 << 20)  # whole fields beyond the single-launch kernels' limit take the single-read path
    if single_read:
        bc = bc - es + es * 16.0 / 4096.0
    return dict(elements=n, algorithm="single-read compress (sample + verify)" if single_read else "single launch per direction, two reads (the second from L2)", dtype="f64" if es == 8 else "f32", mode="qt" if qt else "ec", error_bound=eb, outlier_fraction=p,
                ms_compress=1e3 * tc, ms_decompress=1e3 * td, ms_compress_median=tc_med, ms_decompress_median=td_med, compress_gbs=n * es / 1e9 / tc, decompress_gbs=n * es / 1e9 / td,
                compress_frac=bc * n / tc / 1e9 / peak, decompress_frac=bd * n / td / 1e9 / peak, launches_per_step=launches,
                max_abs_err=float((out - x).abs().max().item()), sf=sf), dict(bins=bins, dc=dc, ac=ac, n_out=n_out, sf=sf, qtab=qtab)


def window_parity(ctx, torch, x, res, w0, wn, eb, qt):
    """bin indices / DC / outliers of elements [w0, w0+wn) of a compressed slab against the oracle run on that window
    alone (valid when the window's own scaling factor equals the slab's: checked).  Returns a small report."""
    import numpy as np

    from tests import parity, reflib

    xw = x[w0:w0 + wn].cpu().numpy()
    o = reflib.oracle_compress(xw, eb, qt)
    if o["stat"]["sf"] != res["sf"]:
        return dict(skipped=f"the window's own scaling factor {o['stat']['sf']} differs from the slab's {res['sf']}")
    bins = res["bins"]
    pos = torch.arange(w0 % 64, w0 % 64 + wn, device=bins.device) % 64
    before = int((bins[:w0] == 255).sum().item()) - (w0 + 63) // 64 if w0 else 0
    mine = int(((bins[w0:w0 + wn] == 255) & (pos != 0)).sum().item())
    g = dict(bin_index=bins[w0:w0 + wn].cpu().numpy(), dc=res["dc"][w0 // 64:(w0 + wn + 63) // 64].cpu().numpy(),
             ac=res["ac"][before:before + mine].cpu().numpy(), info=dict(sf=res["sf"], n_outliers=mine, n_qt_dropped=0))
    if qt:
        return dict(skipped="QT windows are not comparable (the table is a property of the whole field)")
    rep = parity.compare_compress(g, o, xw, eb, False, ctx=ctx, check_stats=False)
    return dict(window_start=w0, window_elements=wn, ties=rep["ties"], bin_mismatch=rep["bin_mismatch"], n_outliers=rep["n_outliers"])


def main_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import dctz_b200
    from dctz_b200 import DOUBLE, FLOAT, binding, slabs

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    try:  # run (and allocate pinned host memory) on the CPU cores / NUMA node next to this rank's GPU
        import pynvml

        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local))
    except Exception:
        pass
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ctx = dctz_b200.Context(local)
    stream = torch.cuda.current_stream()
    sh = stream.cuda_stream
    EB = args.eb
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", FALLBACK_HBM_GBS))

    # ---- workload resident in HBM -------------------------------------------------------------
    # The rank's share is a list of sub-slabs (one in the weak mode); in field order over all ranks they are the
    # "ranks" whose statistics dctz_gpu_compress_dev merges.
    qt = False
    strong = args.scaling == "strong"
    if (args.qt or strong) and args.workload != "c5-slab":
        raise SystemExit("bench.py: --qt / --scaling strong apply to the c5-slab workload (c2 is the QT config)")
    if args.workload == "c5-slab":
        qt = bool(args.qt)
        sub = 1 << args.slab_log2
        tdt, code, es = torch.float64, DOUBLE, 8
        if strong:
            n_total = 1 << args.field_log2
            start, n = slabs.partition(n_total, world)[rank]
        else:
            n_total, start, n = sub * world, rank * sub, sub
        x = torch.empty(n, dtype=tdt, device=dev)
        ctx.fill_hash_field(x.data_ptr(), start, n, HASH_DIM, SEED, sh)
        if args.noise > 0:
            gen = torch.Generator(device=dev).manual_seed(SEED + rank)
            x += args.noise * torch.randn(n, generator=gen, device=dev, dtype=torch.float64)
        if args.f32:
            x = x.float()
            tdt, code, es = torch.float32, FLOAT, 4
        pieces = [(a, min(sub, n - a)) for a in range(0, n, sub)]  # (offset in x, elements)
        first = rank == 0
        slabbed = world > 1 or len(pieces) > 1
    else:
        host, qt = make_host_field(args.workload)
        n = host.size
        es = host.dtype.itemsize
        tdt, code = (torch.float64, DOUBLE) if es == 8 else (torch.float32, FLOAT)
        x = torch.from_numpy(host).to(dev)
        n_total, first, pieces, slabbed, start = n, True, [(0, n)], False, 0  # replicas: every rank compresses its own copy of the field
    npiece = len(pieces)
    pmax = max(c for _, c in pieces)
    bins = torch.empty(n, dtype=torch.uint8, device=dev)
    dc = torch.empty((n + 63) // 64, dtype=torch.float32, device=dev)
    ac = torch.empty(pmax if npiece > 1 else n, dtype=torch.float32, device=dev)  # several sub-slabs: their outliers share one buffer (timing only)
    out = torch.empty(pmax if npiece > 1 else n, dtype=tdt, device=dev)
    qtab = torch.zeros(64, dtype=tdt, device=dev)
    qraws = [torch.zeros(64, dtype=tdt, device=dev) for _ in pieces]
    info_d = [torch.zeros(binding.INFO_BYTES, dtype=torch.uint8, device=dev) for _ in pieces]
    stats_mine = torch.zeros(3 * npiece, dtype=torch.float64, device=dev)
    nslab_all = npiece * world if slabbed else 1
    stats_all = torch.zeros(3 * nslab_all, dtype=torch.float64, device=dev) if world > 1 else stats_mine
    flush = L2Flush(torch, dev) if n * es < (200 << 20) else None
    if qt and npiece > 1:
        raise SystemExit("bench.py: QT with several sub-slabs per rank needs one context per sub-slab (a context holds one call's outlier scratch); use --scaling weak")
    last_src = slabs.last_rank_with_data(n_total, world) if world > 1 else 0

    def read_info(k=0):
        raw = info_d[k].cpu().numpy().tobytes()
        return binding.GpuInfo.from_buffer_copy(raw).as_dict()

    two_pass = bool(getattr(args, "two_pass", False))
    # whole fields (c1 .. c4: every rank its own copy) go through the single-field entry point, as dctz_compress does: ONE
    # cooperative launch per direction up to 256 MB, the single-read chain beyond
    whole_field = args.workload != "c5-slab" and not two_pass
    fused_small = whole_field and n * es <= (256 << 20)
    true_mine = torch.zeros(3 * npiece, dtype=torch.float64, device=dev)
    true_all = torch.zeros(3 * nslab_all, dtype=torch.float64, device=dev) if world > 1 else true_mine

    def compress(ev=None):
        """SINGLE-READ path (default): sample -> [all-gather 24 B per slab] -> compress with the believed scaling factor while
        gathering the true statistics -> [all-gather 24 B per slab] -> verdict (a gate launch that leaves at once when the belief
        held) + outlier scan + gather.  --two-pass: statistics pass -> [all-gather] -> compress."""
        if whole_field:
            if ev:
                ev[0].record(stream)
            ctx.compress_field_dev(x.data_ptr(), n, code, EB, qt, bins.data_ptr(), dc.data_ptr(), ac.data_ptr(), qtab.data_ptr(), qraws[0].data_ptr(),
                                   info_d[0].data_ptr(), sh)
            if ev:
                ev[1].record(stream)
            return
        for k, (a, c) in enumerate(pieces):
            if two_pass:
                ctx.stats_dev(x.data_ptr() + a * es, c, code, stats_mine.data_ptr() + 24 * k, sh)
            else:
                ctx.sample_dev(x.data_ptr() + a * es, c, code, stats_mine.data_ptr() + 24 * k, sh)
        if world > 1:
            dist.all_gather_into_tensor(stats_all, stats_mine)  # 24 bytes per slab
        if ev:
            ev[0].record(stream)
        for k, (a, c) in enumerate(pieces):
            args_k = (x.data_ptr() + a * es, c, n_total, code, EB, qt)
            outs_k = (bins.data_ptr() + a, dc.data_ptr() + 4 * (a // 64), ac.data_ptr(), qraws[k].data_ptr(), info_d[k].data_ptr())
            if two_pass:
                ctx.compress_dev(*args_k, stats_all.data_ptr(), nslab_all, first and k == 0, *outs_k, sh)
            else:
                ctx.compress_spec_dev(*args_k, stats_all.data_ptr(), nslab_all, first and k == 0, *outs_k, true_mine.data_ptr() + 24 * k, sh)
        if not two_pass:
            if world > 1:
                dist.all_gather_into_tensor(true_all, true_mine)  # the true statistics: 24 bytes per slab
            for k, (a, c) in enumerate(pieces):
                ctx.compress_spec_finish_dev(x.data_ptr() + a * es, c, n_total, code, EB, qt, true_all.data_ptr(), nslab_all, first and k == 0,
                                             bins.data_ptr() + a, dc.data_ptr() + 4 * (a // 64), ac.data_ptr(), qraws[k].data_ptr(), info_d[k].data_ptr(), sh)
        if ev:
            ev[1].record(stream)
        if qt:
            if world > 1:
                slabs.all_reduce_qtable(qraws[0], rank, world, src_last=last_src)  # 64-value max-reduction + entry 0 from the last slab
            ctx.qt_finish_dev(code, EB, qraws[0].data_ptr(), qtab.data_ptr(), ac.data_ptr(), info_d[0].data_ptr(), sh)

    def decompress(sf, n_outs):
        for k, (a, c) in enumerate(pieces):
            ctx.decompress_dev(bins.data_ptr() + a, dc.data_ptr() + 4 * (a // 64), ac.data_ptr(), n_outs[k], qtab.data_ptr() if qt else 0, c, code, EB, sf,
                               qt, out.data_ptr(), sh)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    compress()
    torch.cuda.synchronize()
    infos = [read_info(k) for k in range(npiece)]
    if any(i["status"] != 0 for i in infos):
        raise SystemExit(f"bench.py: compress failed with status {[i['status'] for i in infos]}")
    info = infos[0]
    sf = info["sf"]
    n_outs = [i["n_outliers"] for i in infos]
    p_out = sum(n_outs) / n
    if npiece > 1 and max(n_outs) > 0:
        # with several sub-slabs per rank the outlier buffer is reused: the last sub-slab's outliers are what it holds
        n_outs = [min(v, n_outs[-1]) for v in n_outs]

    for _ in range(args.warmup):
        if flush is not None:
            flush()
        compress()
        decompress(sf, n_outs)
    barrier()

    E = lambda: torch.cuda.Event(enable_timing=True)
    evs = [[E() for _ in range(5)] for _ in range(args.steps)]
    launches0 = ctx.launch_count
    barrier()
    sampler.mark_begin()
    for k in range(args.steps):
        if flush is not None:
            flush()
        e = evs[k]
        e[0].record(stream)
        compress(ev=(e[1], e[2]))
        e[3].record(stream)
        decompress(sf, n_outs)
        e[4].record(stream)
    barrier()
    sampler.mark_end()
    clocks = sampler.stop() if rank == 0 else None
    launches = ctx.launch_count - launches0
    t_c = sum(e[0].elapsed_time(e[3]) for e in evs) / 1e3
    t_d = sum(e[3].elapsed_time(e[4]) for e in evs) / 1e3
    t_k2 = sum(e[1].elapsed_time(e[2]) for e in evs) / 1e3      # k_finalize (1 thread) + k_compress (+ scan + gather)
    t_k1 = sum(e[0].elapsed_time(e[1]) for e in evs) / 1e3      # k_stats (+ all-gather)
    times = torch.tensor([t_c + t_d, t_c, t_d, t_k2, t_k1], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    t_rt, t_c, t_d, t_k2, t_k1 = [float(v) for v in times.cpu()]
    a_last, c_last = pieces[-1]
    max_err = float((out[:c_last] - x[a_last:a_last + c_last]).abs().max().item())
    if args.dump_outputs and rank == 0:
        # with several sub-slabs per rank the outlier and output buffers hold the last sub-slab's
        dumped = dict(bin_index=bins, dc=dc, ac=ac[:n_outs[-1]], n_outliers=torch.tensor([float(n_outs[-1])], dtype=torch.float64),
                      sf=torch.tensor([sf], dtype=torch.float64), recon=out[:c_last])
        if qt:
            dumped["qtable"] = qtab
        dump_outputs(args.dump_outputs, dumped)
    n_all = n_total if (strong and args.workload == "c5-slab") else n * world  # replicas / weak slabs: every rank's own elements
    gb_all = n_all * es * args.steps / 1e9

    # ---- per-rank parity: every rank checks a window of ITS OWN slab against the oracle (N > 1: slabs at rank > 0
    #      offsets, compressed with the exchanged statistics) -------------------------------------------
    rank_quality = None
    if not args.no_cpu and args.workload == "c5-slab" and not qt:
        compress()  # (the buffers hold the last timed step's result; recompute piece 0's outliers for the window)
        torch.cuda.synchronize()
        wn = min(pieces[0][1], 1 << 23 if world > 1 else 1 << 20)
        w0 = ((pieces[0][1] - wn) // 2 // 64) * 64
        res = dict(bins=bins[:pieces[0][1]], dc=dc, ac=ac, sf=sf)
        if npiece > 1:  # the shared outlier buffer holds the LAST sub-slab's outliers: check that one instead
            res = dict(bins=bins[a_last:a_last + c_last], dc=dc[a_last // 64:], ac=ac, sf=sf)
            wn = min(c_last, wn)
            w0 = ((c_last - wn) // 2 // 64) * 64
            xs = x[a_last:a_last + c_last]
        else:
            xs = x[:pieces[0][1]]
        try:
            rank_quality = window_parity(ctx, torch, xs, res, w0, wn, EB, qt)
            rank_quality.update(rank=rank, slab_start=start + (a_last if npiece > 1 else 0), max_abs_err=max_err)
        except AssertionError as e:
            rank_quality = dict(rank=rank, failed=str(e)[:300])
    quality_per_rank = [rank_quality]
    if world > 1:
        quality_per_rank = [None] * world
        dist.all_gather_object(quality_per_rank, rank_quality)
        if any(q and q.get("failed") for q in quality_per_rank):
            raise SystemExit(f"bench.py: per-rank parity check failed: {quality_per_rank}")

    # ---- end to end through the host-buffer C-ABI (pinned host buffers, copies inside the timing) ----
    # Every step uploads its input from page-locked host memory and brings the result back.  A compress call is upload-
    # heavy and a decompress call download-heavy, and the link is full duplex: `lanes` host threads (a context and a set
    # of host buffers each) keep that many independent fields in flight, the library's per-device link gates put them in
    # step (one uploads while the other downloads).  `serial_value` is one field at a time, as in round 1.
    e2e = None
    if not args.no_e2e:
        import threading

        ne = min(pieces[0][1], 1 << args.e2e_log2)
        nblk_e = (ne + 63) // 64
        np_dt = np.float64 if es == 8 else np.float32
        ksteps = max(1, min(args.steps, 8))
        lanes = max(1, args.e2e_lanes)

        class Lane:
            def __init__(self, c):
                self.ctx = c
                self.hx = binding.PinnedArray((ne,), np_dt)
                self.hout = binding.PinnedArray((ne,), np_dt)
                self.hb = binding.PinnedArray((ne,), np.uint8)
                self.hdc = binding.PinnedArray((nblk_e,), np.float32)
                self.hac = binding.PinnedArray((ne,), np.float32)
                self.pre = dict(bin_index=self.hb.array, dc=self.hdc.array, ac_full=self.hac.array)
                self.err = None
                self.trace = []

            def step(self):
                t0 = time.perf_counter()
                g = self.ctx.compress_core(self.hx.array, EB, qt=qt, out=self.pre)
                t1 = time.perf_counter()
                self.st_c = self.ctx.last_call_stats()
                self.ctx.decompress_core(g["bin_index"], g["dc"], g["ac"], ne, np_dt, EB, g["sf"], qt=qt, qtable=g.get("qtable"), out=self.hout.array)
                t2 = time.perf_counter()
                self.st_d = self.ctx.last_call_stats()
                self.trace.append((t0, t1, t2, self.st_c, self.st_d))

            def run(self, k):
                try:
                    for _ in range(k):
                        self.step()
                except Exception as e:  # noqa: BLE001
                    self.err = e

            def free(self):
                for h in (self.hx, self.hout, self.hb, self.hdc, self.hac):
                    h.free()

        lane_list = [Lane(ctx)]
        for _ in range(lanes - 1):  # (page-locked memory is a limited resource: run with the lanes that could be set up)
            try:
                lane_list.append(Lane(dctz_b200.Context(local)))
            except Exception as e:  # noqa: BLE001
                print(f"bench.py: e2e lane {len(lane_list)} could not be set up ({e}); continuing with {len(lane_list)}", file=sys.stderr)
                break
        lanes = len(lane_list)
        src = x[:ne].cpu().numpy()
        for ln in lane_list:
            ln.hx.array[:] = src
            ln.step()  # warm-up: buffers grown, kernels loaded
        del src

        def timed(active):
            barrier()
            t0 = time.perf_counter()
            if len(active) == 1:
                active[0].run(ksteps)
            else:
                th = [threading.Thread(target=ln.run, args=(ksteps,)) for ln in active]
                for t in th:
                    t.start()
                for t in th:
                    t.join()
            torch.cuda.synchronize()
            te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            for ln in active:
                if ln.err is not None:
                    raise ln.err
            return world * len(active) * ne * es * ksteps / 1e9 / float(te.item())

        v_serial = timed(lane_list[:1])
        for ln in lane_list:
            ln.trace = []
        v_lanes = timed(lane_list) if lanes > 1 else v_serial
        if os.environ.get("DCTZ_BENCH_TRACE"):
            tb = min(t[0] for ln in lane_list for t in ln.trace)
            for i, ln in enumerate(lane_list):
                print(f"e2e lane {i}: " + " | ".join(
                    f"C {1e3 * (a - tb):.1f} (gate +{sc['gate_taken_ms']:.1f}, kernels done +{sc['wall_to_kernels_ms']:.1f}) -{1e3 * (b - tb):.1f} "
                    f"D (gate +{sd['gate_taken_ms']:.1f}, first piece +{sd['first_dominant_piece_ms']:.1f}) -{1e3 * (c - tb):.1f}"
                    for a, b, c, sc, sd in ln.trace), file=sys.stderr)
        l0 = lane_list[0]
        e2e = dict(value=v_lanes, unit=UNIT, serial_value=v_serial, fields_in_flight=lanes,
                   h2d_bytes_per_step=l0.st_c["h2d_bytes"] + l0.st_d["h2d_bytes"], d2h_bytes_per_step=l0.st_c["d2h_bytes"] + l0.st_d["d2h_bytes"],
                   steps=ksteps * lanes,
                   sample=f"a step = the first {ne} elements of the rank's slab through dctz_gpu_compress_core + dctz_gpu_decompress_core (synchronous "
                          f"calls on pinned host buffers, copies included; bytes per step counted by the library); {lanes} host thread(s) with a context "
                          f"each keep {lanes} independent field(s) in flight so that one field's upload overlaps the other's download on the full-duplex "
                          f"link (serial_value: one field at a time); wall clock over {ksteps} step(s) per thread",
                   max_abs_err=float(max(np.max(np.abs(ln.hout.array - ln.hx.array)) for ln in lane_list)))
        for ln in lane_list:
            ln.free()
        for ln in lane_list[1:]:
            ln.ctx.close()

    # (every rank takes part: barrier + max over ranks -- hence before the other ranks leave)
    # Reported beside the headline, never as it: compress with KNOWN statistics (those of the previous step, as a
    # time-stepping simulation would have them) -- dctz_gpu_compress_known_stats_dev reads the input once and verifies
    # the scaling factor on the fly.
    known_leg = None
    if args.workload == "c5-slab" and not qt and npiece == 1 and world == 1:
        # the other way round: the TWO-PASS compress (statistics pass + compress pass), for comparison with the headline's single read
        st2 = torch.zeros(3, dtype=torch.float64, device=dev)
        evk = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

        def two():
            ctx.stats_dev(x.data_ptr(), n, code, st2.data_ptr(), sh)
            ctx.compress_dev(x.data_ptr(), n, n_total, code, EB, False, st2.data_ptr(), 1, True, bins.data_ptr(), dc.data_ptr(), ac.data_ptr(),
                             qraws[0].data_ptr(), info_d[0].data_ptr(), sh)

        for _ in range(2):
            two()
        torch.cuda.synchronize()
        evk[0].record(stream)
        for _ in range(5):
            two()
        evk[1].record(stream)
        torch.cuda.synchronize()
        tk = evk[0].elapsed_time(evk[1]) / 5e3
        known_leg = dict(compress_ms=1e3 * tk, compress_gbs=n * es / 1e9 / tk,
                         note="TWO-PASS compress of the same slab (statistics pass + compress pass, two reads of the input): what the headline's single-read path replaces")

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- roofline: the whole step against the measured HBM copy bandwidth; phases and the dominant kernel below it ----
    bpe_c, bpe_d = bytes_per_element(es, p_out)            # SURVEY.md §8d B_c (statistics read included), B_d
    bpe_c2 = bpe_c                                         # the two-pass model, kept for reference
    if not two_pass and not fused_small:
        bpe_c = bpe_c - es + es * 16.0 / 4096.0            # SINGLE READ: one pass over the input + the 0.4 % sample
    bpe_k2 = es + 1 + 4 / 64 + 4 * p_out                   # transform read + bin index + DC + outliers
    step_bytes = (bpe_c + bpe_d) * n * args.steps
    ach_step = step_bytes / t_rt / 1e9
    traffic = None  # dram__bytes_read+write per element of the step's kernels, from the committed ncu capture, scaled to this slab
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(args.workload, {})
        if tr and es == 8 and not qt and args.noise == 0:
            traffic = dict(step=sum(v["bytes_per_element"] for v in tr.values()) * n,
                           **{k: v["bytes_per_element"] * n for k, v in tr.items()}, source="profiles/traffic.json (ncu --set full, per launch, scaled to this slab)")
    except Exception:
        pass
    frac = lambda b, t: b * n * args.steps / t / 1e9 / peak
    roofline = dict(bound="hbm", scope="whole step (compress + decompress) per GPU", achieved=ach_step, peak=peak, unit="GB/s", frac=ach_step / peak,
                    traffic=traffic["step"] if traffic else None, traffic_detail=traffic,
                    peak_source="measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)",
                    bytes_per_element=bpe_c + bpe_d, elements_per_launch=n, outlier_fraction=p_out,
                    algorithm=("single launch per direction, two reads (the second from L2)" if fused_small else
                               "single-read compress (sample + verify; the input is read once)" if not two_pass else "two-pass compress"),
                    two_pass_model=dict(bytes_per_element=bpe_c2 + bpe_d, frac=(bpe_c2 + bpe_d) * n * args.steps / t_rt / 1e9 / peak,
                                        note="SURVEY.md §8d counts two reads of the input as compulsory; against THAT byte count the step runs above 1"),
                    phases=dict(compress=dict(achieved=frac(bpe_c, t_c) * peak, frac=frac(bpe_c, t_c), bytes_per_element=bpe_c),
                                decompress=dict(achieved=frac(bpe_d, t_d) * peak, frac=frac(bpe_d, t_d), bytes_per_element=bpe_d)),
                    kernels={("k_stats" if two_pass else "k_sample"):
                                 dict(achieved=frac(es if two_pass else es * 16.0 / 4096.0, t_k1) * peak, frac=frac(es if two_pass else es * 16.0 / 4096.0, t_k1),
                                      bytes_per_element=es if two_pass else es * 16.0 / 4096.0,
                                      note="events around the statistics pass (two-pass) / the 0.4 % sample (single-read) + the all-gather at N > 1"),
                             "k_compress<%s,%s>" % ("double" if es == 8 else "float", "QT" if qt else "EC"):
                                 dict(achieved=frac(bpe_k2, t_k2) * peak, frac=frac(bpe_k2, t_k2), bytes_per_element=bpe_k2, dominant=True,
                                      note="events around k_compress (the VERIFY instantiation in the single-read path) + tile-sum reduction + gate launch "
                                           "+ outlier scan + gather")})

    # ---- CPU baseline + quality on a bounded sample (rank 0, N = 1 only) -------------------------
    cpu = None
    quality = dict(max_abs_err=max_err, outlier_fraction=p_out, sf=sf, n_edge=info["n_edge"], n_exact_path=info["n_exact_path"],
                   per_rank=quality_per_rank)
    if world == 1 and not args.no_cpu:
        from tests import parity, reflib

        ns = min(n, 1 << args.cpu_log2)
        sample = x[:ns].cpu().numpy()
        procs = max(1, min(os.cpu_count() or 1, 32))
        cpu = cpu_reference(sample, qt, procs, EB)
        # quality vs the oracle on the same sample: ties, reconstruction difference, ratio with host zlib
        g = ctx.compress_core(sample, EB, qt=qt)
        o = reflib.oracle_compress(sample, EB, qt)
        rep = parity.compare_compress(g, o, sample, EB, qt, ctx=ctx)
        r_gpu = ctx.decompress_core(g["bin_index"], g["dc"], g["ac"], ns, sample.dtype, EB, g["sf"], qt=qt, qtable=g.get("qtable"))
        r_ref = reflib.oracle_decompress(o["bin_index"], o["dc"], o["ac"], o["qtable"], ns, EB, o["stat"]["sf"], qt, sample.dtype)
        zsz = 56 + sum(len(zlib.compress(a.tobytes(), -1)) for a in (g["bin_index"], g["dc"], g["ac"])) + (64 * es if qt else 0)
        quality.update(sample_elements=ns, ties=rep["ties"], bin_mismatch=rep["bin_mismatch"],
                       max_abs_err_vs_ref=float(np.max(np.abs(r_gpu.astype(np.float64) - r_ref.astype(np.float64)))),
                       max_abs_err_sample=float(np.max(np.abs(r_gpu.astype(np.float64) - sample.astype(np.float64)))),
                       max_abs_err_ref_sample=float(np.max(np.abs(r_ref.astype(np.float64) - sample.astype(np.float64)))),
                       ratio=ns * es / zsz)

    # ---- the real drop-in call: dctz_compress() / dctz_decompress() of libdctz_{ec,qt}.so on ordinary (pageable) memory,
    #      in-place scaling, zlib, side files and all -- what a user of the reference's API gets ----
    e2e_api = None
    if world == 1 and not args.no_e2e:
        e2e_api = api_leg(x, min(n, 1 << args.e2e_log2), es, qt, EB)

    outlier_leg = None
    if world == 1 and args.workload == "c5-slab" and not qt and args.noise == 0 and not args.no_outlier_leg and npiece == 1:
        # The headline field is smooth (no AC coefficient leaves the bin range).  Reported beside it, never as the
        # headline: the same slab shape with white noise added so that ~5 % of the coefficients are outliers.
        n2 = min(n, 1 << 28)
        gen = torch.Generator(device=dev).manual_seed(SEED)
        x2 = x[:n2].double() + 1.3 * torch.randn(n2, generator=gen, device=dev, dtype=torch.float64)
        del bins, dc, ac, out
        torch.cuda.empty_cache()

        def noisy(xx, cd, mode_qt):
            r, _ = time_field(ctx, torch, binding, xx, cd, EB, mode_qt, 5, 3, peak, None)
            r["workload"] = f"first 2^{n2.bit_length() - 1} elements of the slab + Gaussian noise (std 1.3), {'QT' if mode_qt else 'EC'} mode, {r['dtype']}"
            r["value"] = n2 * xx.element_size() / 1e9 / ((r["ms_compress"] + r["ms_decompress"]) / 1e3)
            return r

        outlier_leg = noisy(x2, DOUBLE, False)
        outlier_leg["qt_mode"] = noisy(x2, DOUBLE, True)  # the quantiser mode on the same data (not strictly error bounded by design)
        x2f = x2.float()
        del x2
        outlier_leg["f32"] = noisy(x2f, FLOAT, False)
        outlier_leg["f32_qt"] = noisy(x2f, FLOAT, True)
        del x2f

    # ---- the other BASELINE configs beside the headline (N = 1): c1, c2, c3 at its three error bounds, c4 ----
    configs_leg = None
    if world == 1 and args.workload == "c5-slab" and not args.no_configs and not args.f32 and not qt and args.noise == 0:
        del x
        torch.cuda.empty_cache()
        configs_leg = configs(ctx, torch, binding, peak, not args.no_cpu)

    line = dict(metric=METRIC, value=gb_all / t_rt, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * t_rt / args.steps, higher_is_better=True, scaling=args.scaling, vs_baseline=None,
                dtype="f64" if es == 8 else "f32", data="synthetic", config=workload_config(args, world),
                compress_gbs=gb_all / t_c, decompress_gbs=gb_all / t_d, ms_compress=1e3 * t_c / args.steps,
                ms_decompress=1e3 * t_d / args.steps, roofline=roofline, cpu_baseline=cpu, e2e=e2e, e2e_api=e2e_api, quality=quality,
                outlier_leg=outlier_leg, two_pass_leg=known_leg, configs=configs_leg, gpu_launches=int(launches), clocks=clocks, impl="ours")
    _emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


def configs(ctx, torch, binding, peak, with_parity):
    """BASELINE configs[0..3] on one GPU, whole field per call, L2 flushed between steps for the fields that fit in it;
    ties / mismatches against the oracle on a 2^22-element window (the full-size comparisons are tests/test_gpu_parity.py)."""
    import numpy as np

    from dctz_b200 import DOUBLE, FLOAT, fields

    out = {}
    flush = L2Flush(torch, "cuda")
    plan = [("c1", lambda: fields.cesm_like(), False, [1e-3]), ("c2", lambda: fields.cesm_like(dtype=np.float32), True, [1e-3]),
            ("c3", lambda: fields.hurricane_like(), False, [1e-3, 1e-4, 1e-5]), ("c4", lambda: fields.nyx_like(), False, [1e-3])]
    for name, make, qt, ebs in plan:
        host = make()
        x = torch.from_numpy(host).cuda()
        code = DOUBLE if host.dtype == np.float64 else FLOAT
        for eb in ebs:
            r, res = time_field(ctx, torch, binding, x, code, eb, qt, 20, 3, peak, flush if x.numel() * x.element_size() < (200 << 20) else None)
            if with_parity and not qt:
                try:
                    wn = 1 << 22
                    w0 = ((x.numel() - wn) // 2 // 64) * 64
                    r["parity_window"] = window_parity(ctx, torch, x, res, w0, wn, eb, qt)
                except AssertionError as e:
                    r["parity_window"] = dict(failed=str(e)[:300])
            out[name if len(ebs) == 1 else f"{name}@{eb_str(eb)}"] = r
            del res
        del x, host
        torch.cuda.empty_cache()
    return out


def api_leg(x, ne, es, qt, eb):
    """dctz_compress() / dctz_decompress() of the drop-in host library (dctz.h:126-127) on malloc-like memory."""
    import numpy as np

    lib = ctypes.CDLL(os.path.join(ROOT, "dctz_b200", f"libdctz_{'qt' if qt else 'ec'}.so"))

    class TVar(ctypes.Structure):  # dctz.h:49-59
        _fields_ = [("datatype", ctypes.c_int), ("err_bound", ctypes.c_double), ("var_name", ctypes.c_char_p), ("buf", ctypes.c_void_p)]

    np_dt = np.float64 if es == 8 else np.float32
    x0 = x[:ne].cpu().numpy()
    buf = np.empty(ne, np_dt)
    zbuf = np.empty(ne * es + 4096, np.uint8)
    rbuf = np.empty(ne, np_dt)
    code = 1 if es == 8 else 0
    var, var_z, var_r = (TVar(code, eb, b"v", a.ctypes.data) for a in (buf, zbuf, rbuf))
    out = ctypes.c_size_t(0)
    tc, td, reps = [], [], 3
    tmp = tempfile.mkdtemp(prefix="dctz_api_")
    old = os.getcwd()
    os.chdir(tmp)  # the side files bin_index.bin / AC_exact.bin (dctz-comp-lib.c:583-595) are written, as by the reference
    try:
        stats = None
        for it in range(reps + 1):
            buf[:] = x0  # dctz_compress leaves the input scaled: restore it (not timed)
            t0 = time.perf_counter()
            lib.dctz_compress(ctypes.byref(var), ctypes.c_int(ne), ctypes.byref(out), ctypes.byref(var_z), ctypes.c_double(eb))
            t1 = time.perf_counter()
            ms = (ctypes.c_double * 8)()
            h, d = ctypes.c_ulonglong(0), ctypes.c_ulonglong(0)
            lib.dctz_host_last_call_stats(ms, ctypes.byref(h), ctypes.byref(d))
            t2 = time.perf_counter()
            lib.dctz_decompress(ctypes.byref(var_z), ctypes.byref(var_r))
            t3 = time.perf_counter()
            if it:  # the first round pays the one-off costs (context, page-locked staging ring)
                tc.append(t1 - t0)
                td.append(t3 - t2)
            stats = (int(h.value), int(d.value))
    finally:
        os.chdir(old)
        shutil.rmtree(tmp, ignore_errors=True)
    gb = ne * es / 1e9
    return dict(compress_gbs=gb / (sum(tc) / reps), decompress_gbs=gb / (sum(td) / reps), value=gb / ((sum(tc) + sum(td)) / reps), unit=UNIT,
                compressed_bytes=int(out.value), ratio=ne * es / int(out.value), compress_pcie_bytes=dict(h2d=stats[0], d2h=stats[1]),
                compress_pcie_over_input=(stats[0] + stats[1]) / (ne * es), max_abs_err=float(np.max(np.abs(rbuf - x0))),
                sample=f"dctz_compress + dctz_decompress (dctz.h:126-127) of libdctz_{'qt' if qt else 'ec'}.so on {ne} elements of pageable host "
                       f"memory: staged uploads, in-place x/sf by host threads, chunk-parallel zlib overlapped with the downloads, side files written; "
                       f"wall clock, mean of {reps} calls after one warm-up call")


def _emit(line):
    """The contract is ONE JSON line on stdout: everything else any library prints goes to stderr (see __main__)."""
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


if __name__ == "__main__":
    a = parse_args()
    # keep stdout clean: NCCL, torchrun and friends print banners on fd 1; route fd 1 to stderr and keep a private
    # handle on the real stdout for the JSON line
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = sys.stderr
    if a.watchdog > 0:  # a hung collective or kernel must not sit on the GPU box until somebody else's timeout fires
        import faulthandler

        faulthandler.dump_traceback_later(a.watchdog, exit=True)
    sys.exit(main_reference(a) if a.impl == "reference" else main_ours(a))
