"""ctypes binding of include/dctz_gpu.h (libdctz_gpu.so).  One method per C entry point; numpy arrays
for the host-buffer API, raw device pointers (e.g. torch.Tensor.data_ptr()) for the *_dev API."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

FLOAT = 0   # t_datatype, dctz.h:44-47
DOUBLE = 1
BLK = 64
NBINS = 255

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libdctz_gpu.so")

# every symbol include/dctz_gpu.h declares (tests/test_abi.py checks the header against this list)
EXPORTS = [
    "dctz_gpu_create", "dctz_gpu_destroy", "dctz_gpu_last_error", "dctz_gpu_device_count", "dctz_gpu_sm_count",
    "dctz_gpu_host_alloc", "dctz_gpu_host_free", "dctz_gpu_compress_core", "dctz_gpu_decompress_core", "dctz_gpu_stats",
    "dctz_gpu_compress_core_with_stats", "dctz_gpu_quality", "dctz_gpu_quality_dev",
    "dctz_gpu_stats_dev", "dctz_gpu_compress_dev", "dctz_gpu_compress_known_stats_dev", "dctz_gpu_qt_finish_dev", "dctz_gpu_compress_field_dev",
    "dctz_gpu_decompress_dev", "dctz_gpu_scale_dev", "dctz_gpu_dct_blocks", "dctz_gpu_dct64_dev", "dctz_gpu_fp64_rate", "dctz_gpu_fill_hash_field",
    "dctz_gpu_sf_from_max", "dctz_gpu_selftest_division", "dctz_gpu_launch_count", "dctz_gpu_compress_core_cb",
    "dctz_gpu_set_timing", "dctz_gpu_last_call_stats", "dctz_gpu_fused_phase_times", "dctz_gpu_compress_slab_comm",
    "dctz_gpu_sample_dev", "dctz_gpu_compress_spec_dev", "dctz_gpu_compress_spec_finish_dev",
    "dctz_gpu_outlier_index_bytes", "dctz_gpu_outlier_index_dev", "dctz_gpu_decompress_ranges_dev",
]


class DctzGpuError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"dctz_gpu error {code}: {msg}")
        self.code = code


class GpuInfo(C.Structure):  # dctz_gpu_info
    _fields_ = [("sf", C.c_double), ("mean", C.c_double), ("max_abs", C.c_double), ("min_abs", C.c_double),
                ("sum", C.c_double), ("n_outliers", C.c_uint64), ("n_edge", C.c_uint64), ("n_exact_path", C.c_uint64),
                ("n_qt_dropped", C.c_uint64), ("status", C.c_int32), ("scale_mode", C.c_int32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


INFO_BYTES = C.sizeof(GpuInfo)
_lib = None


def load_library():
    """Load libdctz_gpu.so; fails loudly if it has not been built (no fallback of any kind)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DctzGpuError(-1, f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`")
    lib = C.CDLL(LIB_PATH)
    vp, sz, i32, u64, dbl = C.c_void_p, C.c_size_t, C.c_int, C.c_uint64, C.c_double
    sig = {
        "dctz_gpu_create": (i32, [C.POINTER(vp), i32]),
        "dctz_gpu_destroy": (None, [vp]),
        "dctz_gpu_last_error": (C.c_char_p, [vp]),
        "dctz_gpu_device_count": (i32, []),
        "dctz_gpu_sm_count": (i32, [vp]),
        "dctz_gpu_host_alloc": (vp, [sz]),
        "dctz_gpu_host_free": (None, [vp]),
        "dctz_gpu_compress_core": (i32, [vp, vp, sz, i32, dbl, i32, vp, vp, vp, vp, vp, vp, C.POINTER(GpuInfo)]),
        "dctz_gpu_decompress_core": (i32, [vp, vp, vp, vp, u64, vp, sz, i32, dbl, dbl, i32, vp]),
        "dctz_gpu_stats": (i32, [vp, vp, sz, i32, C.POINTER(GpuInfo)]),
        "dctz_gpu_compress_core_with_stats": (i32, [vp, vp, sz, sz, C.POINTER(dbl), i32, i32, dbl, i32, vp, vp, vp, vp, vp, vp, C.POINTER(GpuInfo)]),
        "dctz_gpu_quality": (i32, [vp, vp, vp, sz, i32, C.POINTER(dbl)]),
        "dctz_gpu_quality_dev": (i32, [vp, vp, vp, sz, i32, vp, vp]),
        "dctz_gpu_stats_dev": (i32, [vp, vp, sz, i32, vp, vp]),
        "dctz_gpu_compress_dev": (i32, [vp, vp, sz, sz, i32, dbl, i32, vp, i32, i32, vp, vp, vp, vp, vp, vp]),
        "dctz_gpu_compress_known_stats_dev": (i32, [vp, vp, sz, sz, i32, dbl, i32, vp, i32, i32, vp, vp, vp, vp, vp, vp]),
        "dctz_gpu_qt_finish_dev": (i32, [vp, i32, dbl, vp, vp, vp, vp, vp]),
        "dctz_gpu_sample_dev": (i32, [vp, vp, sz, i32, vp, vp]),
        "dctz_gpu_compress_spec_dev": (i32, [vp, vp, sz, sz, i32, dbl, i32, vp, i32, i32, vp, vp, vp, vp, vp, vp, vp]),
        "dctz_gpu_compress_spec_finish_dev": (i32, [vp, vp, sz, sz, i32, dbl, i32, vp, i32, i32, vp, vp, vp, vp, vp, vp]),
        "dctz_gpu_compress_field_dev": (i32, [vp, vp, sz, i32, dbl, i32, vp, vp, vp, vp, vp, vp, vp]),
        "dctz_gpu_decompress_dev": (i32, [vp, vp, vp, vp, u64, vp, sz, i32, dbl, dbl, i32, vp, vp, vp]),
        "dctz_gpu_outlier_index_bytes": (sz, [sz]),
        "dctz_gpu_outlier_index_dev": (i32, [vp, vp, sz, vp, vp, vp]),
        "dctz_gpu_decompress_ranges_dev": (i32, [vp, vp, vp, vp, u64, vp, sz, i32, dbl, dbl, i32, vp, vp, sz, vp, vp, vp]),
        "dctz_gpu_scale_dev": (i32, [vp, vp, sz, i32, dbl, i32, vp]),
        "dctz_gpu_dct_blocks": (i32, [vp, vp, vp, sz, i32, i32, i32]),
        "dctz_gpu_dct64_dev": (i32, [vp, vp, vp, sz, i32, i32, i32, vp]),
        "dctz_gpu_fp64_rate": (i32, [vp, i32, vp]),
        "dctz_gpu_fill_hash_field": (i32, [vp, vp, u64, u64, C.c_uint32, C.c_uint32, vp]),
        "dctz_gpu_sf_from_max": (dbl, [vp, dbl, i32]),
        "dctz_gpu_selftest_division": (i32, [vp, i32, dbl, u64, C.c_uint32, C.POINTER(u64)]),
        "dctz_gpu_launch_count": (u64, [vp]),
        "dctz_gpu_compress_core_cb": (i32, [vp, vp, sz, i32, dbl, i32, vp, vp, vp, vp, vp, vp, C.POINTER(GpuInfo), vp, vp]),
        "dctz_gpu_set_timing": (i32, [vp, i32]),
        "dctz_gpu_fused_phase_times": (i32, [vp, i32, C.POINTER(dbl)]),
        "dctz_gpu_last_call_stats": (i32, [vp, C.POINTER(dbl), C.POINTER(u64), C.POINTER(u64)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _code(dtype):
    dtype = np.dtype(dtype)
    if dtype == np.float64:
        return DOUBLE
    if dtype == np.float32:
        return FLOAT
    raise TypeError(f"DCTZ handles float32/float64 only, not {dtype}")


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


class PinnedArray:
    """numpy view over page-locked host memory from dctz_gpu_host_alloc."""

    def __init__(self, shape, dtype):
        lib = load_library()
        dtype = np.dtype(dtype)
        n = int(np.prod(shape))
        self._bytes = max(1, n * dtype.itemsize)
        self._ptr = lib.dctz_gpu_host_alloc(self._bytes)
        if not self._ptr:
            raise DctzGpuError(-4, "pinned host allocation failed")
        buf = (C.c_char * self._bytes).from_address(self._ptr)
        self.array = np.frombuffer(buf, dtype=dtype, count=n).reshape(shape)

    def free(self):
        if self._ptr:
            self.array = None
            load_library().dctz_gpu_host_free(self._ptr)
            self._ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Context:
    """dctz_gpu_ctx: one CUDA device, one operation in flight at a time."""

    def __init__(self, device=0):
        self._lib = load_library()
        h = C.c_void_p()
        rc = self._lib.dctz_gpu_create(C.byref(h), int(device))
        if rc != 0:
            raise DctzGpuError(rc, (self._lib.dctz_gpu_last_error(None) or b"").decode())
        self._h = h
        self.device = int(device)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.dctz_gpu_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc):
        if rc != 0:
            raise DctzGpuError(rc, (self._lib.dctz_gpu_last_error(self._h) or b"").decode())

    # ---- queries -------------------------------------------------------------------------
    @property
    def sm_count(self):
        return self._lib.dctz_gpu_sm_count(self._h)

    @property
    def launch_count(self):
        return int(self._lib.dctz_gpu_launch_count(self._h))

    def set_timing(self, on):
        return self._lib.dctz_gpu_set_timing(self._h, int(bool(on)))

    def fused_phase_times(self, kernel):
        """[(earliest, latest)] per phase stamp of the last single-launch kernel (0 compress, 1 decompress), microseconds"""
        t = (C.c_double * 16)()
        self._check(self._lib.dctz_gpu_fused_phase_times(self._h, int(kernel), t))
        n = 6 if kernel == 0 else 4
        return [(t[2 * k], t[2 * k + 1]) for k in range(n)]

    def last_call_stats(self):
        """stage timers (ms) and PCIe bytes of the last host-buffer call"""
        t = (C.c_double * 8)()
        h, d = C.c_uint64(0), C.c_uint64(0)
        self._check(self._lib.dctz_gpu_last_call_stats(self._h, t, C.byref(h), C.byref(d)))
        return dict(upload_ms=t[0], stats_ms=t[1], transform_ms=t[2], wall_to_kernels_ms=t[3], wall_downloads_ms=t[4],
                    gate_taken_ms=t[5], first_dominant_piece_ms=t[6],
                    h2d_bytes=int(h.value), d2h_bytes=int(d.value))

    def sf_from_max(self, max_abs, dtype):
        return self._lib.dctz_gpu_sf_from_max(self._h, float(max_abs), _code(dtype))

    # ---- host-buffer API -----------------------------------------------------------------
    def compress_core(self, x, eb, qt=False, want_scaled=False, out=None):
        """dctz_gpu_compress_core on a 1-D float32/float64 numpy array.  Returns a dict with
        bin_index, dc, ac (trimmed to n_outliers), info and -- in QT mode -- qtable / qtable_raw.
        `out` may carry preallocated (e.g. pinned) arrays under the same keys (ac sized N)."""
        x = np.ascontiguousarray(x)
        code = _code(x.dtype)
        n = x.size
        nblk = (n + BLK - 1) // BLK
        out = out or {}
        bins = out.get("bin_index") if out.get("bin_index") is not None else np.empty(n, np.uint8)
        dc = out.get("dc") if out.get("dc") is not None else np.empty(nblk, np.float32)
        ac = out.get("ac_full") if out.get("ac_full") is not None else np.empty(max(n, 1), np.float32)
        qtable = np.zeros(BLK, x.dtype) if qt else None
        qtable_raw = np.zeros(BLK, x.dtype) if qt else None
        scaled = np.empty_like(x) if want_scaled else None
        info = GpuInfo()
        rc = self._lib.dctz_gpu_compress_core(self._h, _p(x), n, code, float(eb), int(bool(qt)), _p(scaled), _p(bins), _p(dc),
                                              _p(ac), _p(qtable), _p(qtable_raw), C.byref(info))
        self._check(rc)
        res = dict(bin_index=bins, dc=dc, ac=ac[: info.n_outliers], info=info.as_dict(), sf=info.sf, mean=info.mean)
        if qt:
            res["qtable"] = qtable
            res["qtable_raw"] = qtable_raw
        if want_scaled:
            res["scaled"] = scaled
        return res

    def compress_core_with_stats(self, x, n_total, stats3, first_piece, eb, qt=False):
        """one block-aligned piece of a larger data set, scaled by the caller's global statistics"""
        x = np.ascontiguousarray(x)
        n = x.size
        bins, dc, ac = np.empty(n, np.uint8), np.empty((n + BLK - 1) // BLK, np.float32), np.empty(max(n, 1), np.float32)
        qtable = np.zeros(BLK, x.dtype) if qt else None
        info = GpuInfo()
        st = (C.c_double * 3)(*[float(v) for v in stats3])
        self._check(self._lib.dctz_gpu_compress_core_with_stats(self._h, _p(x), n, int(n_total), st, int(bool(first_piece)), _code(x.dtype),
                                                                float(eb), int(bool(qt)), None, _p(bins), _p(dc), _p(ac), _p(qtable), None,
                                                                C.byref(info)))
        res = dict(bin_index=bins, dc=dc, ac=ac[: info.n_outliers], info=info.as_dict(), sf=info.sf, mean=info.mean)
        if qt:
            res["qtable"] = qtable
        return res

    def quality(self, a, b):
        """{min(a), max(a), max|a-b|, sum (a-b)^2}: the core of calc_psnr (util.c:54-104)"""
        a, b = np.ascontiguousarray(a), np.ascontiguousarray(b, dtype=a.dtype)
        out = (C.c_double * 4)()
        self._check(self._lib.dctz_gpu_quality(self._h, _p(a), _p(b), a.size, _code(a.dtype), out))
        return dict(min=out[0], max=out[1], maxdiff=out[2], sumsq=out[3])

    def stats(self, x):
        x = np.ascontiguousarray(x)
        info = GpuInfo()
        self._check(self._lib.dctz_gpu_stats(self._h, _p(x), x.size, _code(x.dtype), C.byref(info)))
        return info.as_dict()

    def decompress_core(self, bin_index, dc, ac, n, dtype, eb, sf, qt=False, qtable=None, out=None):
        dtype = np.dtype(dtype)
        code = _code(dtype)
        bin_index = np.ascontiguousarray(bin_index, dtype=np.uint8)
        dc = np.ascontiguousarray(dc, dtype=np.float32)
        ac = np.ascontiguousarray(ac, dtype=np.float32)
        if qt:
            qtable = np.ascontiguousarray(qtable, dtype=dtype)
        if out is None:
            out = np.empty(n, dtype)
        rc = self._lib.dctz_gpu_decompress_core(self._h, _p(bin_index), _p(dc), _p(ac) if ac.size else None, int(ac.size),
                                                _p(qtable) if qt else None, n, code, float(eb), float(sf), int(bool(qt)), _p(out))
        self._check(rc)
        return out

    def dct_blocks(self, x, dn=BLK, inverse=False):
        x = np.ascontiguousarray(x)
        assert x.size % dn == 0
        out = np.empty_like(x)
        self._check(self._lib.dctz_gpu_dct_blocks(self._h, _p(x), _p(out), x.size // dn, int(dn), _code(x.dtype), int(bool(inverse))))
        return out

    def selftest_division(self, dtype, b, count, seed=1):
        m = C.c_uint64(0)
        self._check(self._lib.dctz_gpu_selftest_division(self._h, _code(dtype), float(b), int(count), int(seed), C.byref(m)))
        return int(m.value)

    # ---- device-resident API (raw device pointers, stream handle as int) -----------------
    def stats_dev(self, d_in, n, code, d_stats3, stream=0):
        self._check(self._lib.dctz_gpu_stats_dev(self._h, d_in, n, code, d_stats3, stream or None))

    def compress_dev(self, d_in, n, n_total, code, eb, qt, d_stats_all, nranks, first_slab, d_bins, d_dc, d_ac, d_qtable_raw,
                     d_info, stream=0):
        self._check(self._lib.dctz_gpu_compress_dev(self._h, d_in, n, n_total, code, float(eb), int(bool(qt)), d_stats_all,
                                                    int(nranks), int(bool(first_slab)), d_bins, d_dc, d_ac,
                                                    d_qtable_raw or None, d_info, stream or None))

    def compress_known_stats_dev(self, d_in, n, n_total, code, eb, qt, d_stats_all, nranks, first_slab, d_bins, d_dc, d_ac,
                                 d_qtable_raw, d_info, stream=0):
        """whole field with a caller-supplied belief about its statistics: one read of the input, a wrong belief is corrected
        on the device (info.n_exact_path = 1)"""
        self._check(self._lib.dctz_gpu_compress_known_stats_dev(self._h, d_in, n, n_total, code, float(eb), int(bool(qt)), d_stats_all,
                                                                int(nranks), int(bool(first_slab)), d_bins, d_dc, d_ac,
                                                                d_qtable_raw or None, d_info, stream or None))

    def sample_dev(self, d_in, n, code, d_belief3, stream=0):
        """single-read path, step 1: max|x| over a 0.4 % sample (+ the exact tail block) -> d_belief3"""
        self._check(self._lib.dctz_gpu_sample_dev(self._h, d_in, n, code, d_belief3, stream or None))

    def compress_spec_dev(self, d_in, n, n_total, code, eb, qt, d_belief_all, nranks, first_slab, d_bins, d_dc, d_ac, d_qtable_raw, d_info, d_true3,
                          stream=0):
        """step 3: compress with the believed scaling factor, gathering the slab's true statistics -> d_true3"""
        self._check(self._lib.dctz_gpu_compress_spec_dev(self._h, d_in, n, n_total, code, float(eb), int(bool(qt)), d_belief_all, int(nranks),
                                                         int(bool(first_slab)), d_bins, d_dc, d_ac, d_qtable_raw or None, d_info, d_true3, stream or None))

    def compress_spec_finish_dev(self, d_in, n, n_total, code, eb, qt, d_true_all, nranks, first_slab, d_bins, d_dc, d_ac, d_qtable_raw, d_info, stream=0):
        """step 5: verdict from the true statistics (re-compress only if the belief was wrong), outlier scan + gather"""
        self._check(self._lib.dctz_gpu_compress_spec_finish_dev(self._h, d_in, n, n_total, code, float(eb), int(bool(qt)), d_true_all, int(nranks),
                                                                int(bool(first_slab)), d_bins, d_dc, d_ac, d_qtable_raw or None, d_info, stream or None))

    def qt_finish_dev(self, code, eb, d_qtable_raw, d_qtable, d_ac, d_info, stream=0):
        self._check(self._lib.dctz_gpu_qt_finish_dev(self._h, code, float(eb), d_qtable_raw, d_qtable, d_ac, d_info, stream or None))

    def compress_field_dev(self, d_in, n, code, eb, qt, d_bins, d_dc, d_ac, d_qtable, d_qtable_raw, d_info, stream=0):
        self._check(self._lib.dctz_gpu_compress_field_dev(self._h, d_in, n, code, float(eb), int(bool(qt)), d_bins, d_dc, d_ac,
                                                          d_qtable or None, d_qtable_raw or None, d_info, stream or None))

    def decompress_dev(self, d_bins, d_dc, d_ac, n_outliers, d_qtable, n, code, eb, sf, qt, d_out, stream=0, d_corrupt=0):
        """n_outliers = readable floats at d_ac; d_corrupt = optional device uint32 set to 1 when the bin indices
        mark more outliers than that"""
        self._check(self._lib.dctz_gpu_decompress_dev(self._h, d_bins, d_dc, d_ac or None, int(n_outliers), d_qtable or None, n, code,
                                                      float(eb), float(sf), int(bool(qt)), d_out, d_corrupt or None, stream or None))

    def outlier_index_bytes(self, n):
        """bytes of the outlier index of an n-element slab"""
        return int(self._lib.dctz_gpu_outlier_index_bytes(int(n)))

    def outlier_index_dev(self, d_bins, n, d_index, d_n_outliers=0, stream=0):
        """build the outlier index of a slab's bin ids into d_index (outlier_index_bytes(n) bytes, 16-byte aligned);
        d_n_outliers = optional device uint64 that receives the number of outliers the bin ids mark"""
        self._check(self._lib.dctz_gpu_outlier_index_dev(self._h, d_bins, int(n), d_index, d_n_outliers or None, stream or None))

    def decompress_ranges_dev(self, d_bins, d_dc, d_ac, n_outliers, d_qtable, n, code, eb, sf, qt, d_index, d_ranges, nranges, d_out,
                              stream=0, d_corrupt=0):
        """decode nranges {first, count} element ranges (uint64 pairs at d_ranges) into d_out, concatenated in range order;
        d_corrupt = optional device uint32: bit 0 as in decompress_dev, bit 1 = a range outside [0, n) or of count 0"""
        self._check(self._lib.dctz_gpu_decompress_ranges_dev(self._h, d_bins, d_dc, d_ac or None, int(n_outliers), d_qtable or None, int(n), code,
                                                             float(eb), float(sf), int(bool(qt)), d_index, d_ranges, int(nranges), d_out,
                                                             d_corrupt or None, stream or None))

    def scale_dev(self, d_x, n, code, sf, multiply, stream=0):
        self._check(self._lib.dctz_gpu_scale_dev(self._h, d_x, n, code, float(sf), int(bool(multiply)), stream or None))

    def fp64_rate(self, kind):
        """measured FP64 rate in TFLOP/s: kind 0 = DFMA on the vector pipe, 1 = DMMA m8n8k4 on the tensor pipe"""
        v = C.c_double(0.0)
        self._check(self._lib.dctz_gpu_fp64_rate(self._h, int(kind), C.byref(v)))
        return v.value

    def dct64_dev(self, d_in, d_out, nblocks, code, inverse=False, variant=0, stream=0):
        self._check(self._lib.dctz_gpu_dct64_dev(self._h, d_in, d_out, int(nblocks), code, int(bool(inverse)), int(variant), stream or None))

    def fill_hash_field(self, d_out, start, count, dim=2048, seed=20261018, stream=0):
        self._check(self._lib.dctz_gpu_fill_hash_field(self._h, d_out, int(start), int(count), int(dim), int(seed), stream or None))
