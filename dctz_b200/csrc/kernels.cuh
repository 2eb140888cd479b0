// kernels.cuh -- hand-written sm_100a kernels of the DCTZ hot path.
//
//   k_stats        K1  max|x|, min|x|, sum(x)                      (util.c:12-44)
//   k_finalize         reduce per-rank statistics, derive sf        (util.c:28/42)
//   k_compress     K2  scale + DCT-II + quantise + ordered outliers (dctz-comp-lib.c:188-217, 318-544)
//   k_tail             the partial last block (rem = N % 64)        (dctz-comp-lib.c:326-336)
//   k_scan_groups / k_gather_ec   ordered outlier compaction        (dctz-comp-lib.c:478-544)
//   k_qt_gather    K2b QT outlier rescale + compaction              (dctz-comp-lib.c:450-533)
//   k_count_bins       outlier markers per tile (decompress pre-pass)
//   k_decompress   K3  dequantise + DCT-III + de-scale              (dctz-decomp-lib.c:389-511)
//
// Mapping: ONE THREAD OWNS ONE 64-ELEMENT BLOCK, all 64 values live in registers and go through
// the generated straight-line transform (dct64_gen.cuh, 592 FP ops, no shuffles, no indexing).
// The kernels are persistent and WARP-AUTONOMOUS: a warp takes tiles of 32 consecutive blocks in batches
// from an atomic ticket counter (TileSeq: requested a batch ahead), a tile arrives by TMA tensor copies
// (-> per-warp mbarrier) into a 128-byte-swizzled, bank-conflict-free shared-memory tile, and the next
// tile's copy is issued as soon as the registers are loaded, so it overlaps the whole compute phase.
// There is no CTA-wide barrier inside the main loops and no waiting between warps: the ordered outlier
// offsets come from per-tile counts + a scan kernel (common.cuh, "Ordered outlier compaction").
#pragma once
#include <cuda.h>  // CUtensorMap (type only; the encoder is fetched from the driver at run time)
#include <type_traits>
#include "common.cuh"
#include "dct64_gen.cuh"

namespace dctz {

// ------------------------------------------------------------------------------------------
// Parameter blocks
// ------------------------------------------------------------------------------------------
struct DevParams {        // written on the device by finalize_params(), read by K2 / tail
  double sf_d, inv_sf_d;  // double path divisor
  float sf_f, inv_sf_f;   // float path divisor
  int scale_iters;        // Divisor::iters for x / sf
  int status;
  double decade_lo, decade_hi;  // sf is right for this data iff decade_lo <= max|x| < decade_hi (util.c:28/42)
};

template <typename T> struct QuantConsts;  // host-computed from the error bound only
template <> struct QuantConsts<double> {
  double bw, rmin, rmax;  // dctz-comp-lib.c:273-275
  double inv_bw;          // RN(1/bw) for the fast path
};
template <> struct QuantConsts<float> {
  float bw, rmin, rmax;   // dctz-comp-lib.c:278-280 (double expressions rounded to float)
  Divisor<float> div;     // exact division by bw
};

struct SfTables {         // host libm results, see build_sf_tables() in dctz_gpu.cu
  const double *thr_d; const double *sf_d; int n_d, kmin_d; double min_d, max_d;  // thr[i] = T_{kmin+i}; admitted: min_d <= max|x| < max_d
  const float *thr_f; const float *sf_f; int n_f, kmin_f; float min_f, max_f;
  int qmax_words;          // 64-bit words of the QT per-position maxima to clear (64 elements of T)
};

struct Info {             // mirrors dctz_gpu_info (include/dctz_gpu.h)
  double sf, mean, max_abs, min_abs, sum;
  unsigned long long n_outliers, n_edge, n_exact_path, n_qt_dropped;
  int status, scale_mode;
};

// ------------------------------------------------------------------------------------------
// K1: statistics.  Persistent CTAs stream 16 KB chunks through shared memory (TMA bulk copies); |x| compared
// as unsigned bit patterns (monotonic for non-negative IEEE values), sum accumulated in double.
// ------------------------------------------------------------------------------------------
struct StatPartial { unsigned long long umax, umin; double sum; };
constexpr int STAT_CHUNK = 16384;   // bytes per TMA bulk copy
constexpr int STAT_STAGES = 4;      // chunks in flight per CTA
constexpr int STAT_SMEM = STAT_CHUNK * STAT_STAGES;

template <typename T> struct AbsBits;
template <> struct AbsBits<double> {
  static __device__ __forceinline__ unsigned long long get(double v) { return (unsigned long long)__double_as_longlong(v) & 0x7FFFFFFFFFFFFFFFull; }
  static __device__ __forceinline__ double back(unsigned long long u) { return __longlong_as_double((long long)u); }
};
template <> struct AbsBits<float> {
  static __device__ __forceinline__ unsigned long long get(float v) { return (unsigned long long)((unsigned)__float_as_int(v) & 0x7FFFFFFFu); }
  static __device__ __forceinline__ double back(unsigned long long u) { return (double)__int_as_float((int)(unsigned)u); }
};

__device__ __forceinline__ void finalize_params(const double *stats_all, int nranks, unsigned long long n_total,
                                                int is_double, double first_value, int first_slab,
                                                const SfTables &tb, DevParams *p, Info *info,
                                                unsigned long long *qmax_zero);

// max(a, b) that returns a NaN operand (fmax drops it): merges of partial maxima must keep a NaN of the data visible to
// finalize_params, which rejects it
__device__ __forceinline__ double max_keep_nan(double a, double b) { return (a > b || a != a) ? a : b; }

template <typename T>
__global__ void __launch_bounds__(256) k_stats(const T *__restrict__ in, size_t n, StatPartial *partials,
                                               unsigned *done_counter, double *stats3 /* max,min,sum */,
                                               int finalize_inline, unsigned long long n_total, int first_slab,
                                               SfTables tb, DevParams *params, Info *info,
                                               unsigned long long *qmax_zero) {
  constexpr int VEC = 16 / (int)sizeof(T);
  unsigned long long umax = 0ull, umin = ~0ull;
  double s0 = 0.0, s1 = 0.0;
  const size_t nvec = n / VEC;
  // The slab streams through shared memory in 16 KB chunks fetched by TMA bulk copies (one thread issues, a
  // STAT_STAGES-deep ring of mbarriers tracks them): the load path costs the SM one instruction per 16 KB
  // instead of 1024 LDG.128, and reaches the bandwidth the TMA-fed transform kernels reach.
  extern __shared__ __align__(128) unsigned char stat_smem[];
  __shared__ __align__(8) unsigned long long s_full[STAT_STAGES];
  const size_t nchunks = (nvec * 16 + STAT_CHUNK - 1) / STAT_CHUNK;
  const unsigned char *src = reinterpret_cast<const unsigned char *>(in);
  auto chunk_bytes = [&](size_t c) -> unsigned {
    const size_t left = nvec * 16 - c * STAT_CHUNK;
    return (unsigned)(left < (size_t)STAT_CHUNK ? left : (size_t)STAT_CHUNK);
  };
  if (threadIdx.x == 0) {
    for (int st = 0; st < STAT_STAGES; st++) mbar_init(smem_u32(&s_full[st]), 1);
    fence_mbar_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int st = 0; st < STAT_STAGES; st++) {
      const size_t c = (size_t)blockIdx.x + (size_t)st * gridDim.x;
      if (c < nchunks) {
        mbar_expect_tx(smem_u32(&s_full[st]), chunk_bytes(c));
        bulk_g2s(smem_u32(stat_smem + st * STAT_CHUNK), src + c * STAT_CHUNK, chunk_bytes(c), smem_u32(&s_full[st]));
      }
    }
  }
  unsigned k = 0;
  for (size_t c = blockIdx.x; c < nchunks; c += gridDim.x, k++) {
    const int st = (int)(k % STAT_STAGES);
    mbar_wait(smem_u32(&s_full[st]), (k / STAT_STAGES) & 1u);
    const uint4 *buf = reinterpret_cast<const uint4 *>(stat_smem + st * STAT_CHUNK);
    const unsigned nv = chunk_bytes(c) / 16;
#pragma unroll
    for (int u = 0; u < STAT_CHUNK / 16 / 256; u++) {
      const unsigned idx = u * 256 + threadIdx.x;
      if (idx < nv) {
        const uint4 v = buf[idx];
        const T *e = reinterpret_cast<const T *>(&v);
#pragma unroll
        for (int q = 0; q < VEC; q++) {
          const unsigned long long a = AbsBits<T>::get(e[q]);
          umax = a > umax ? a : umax;
          umin = a < umin ? a : umin;
          if (q & 1) s1 += (double)e[q]; else s0 += (double)e[q];
        }
      }
    }
    __syncthreads();  // every thread is done with this stage: refill it
    const size_t cn = c + (size_t)STAT_STAGES * gridDim.x;
    if (threadIdx.x == 0 && cn < nchunks) {
      mbar_expect_tx(smem_u32(&s_full[st]), chunk_bytes(cn));
      bulk_g2s(smem_u32(stat_smem + st * STAT_CHUNK), src + cn * STAT_CHUNK, chunk_bytes(cn), smem_u32(&s_full[st]));
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    for (size_t k = nvec * VEC; k < n; k++) {
      const unsigned long long a = AbsBits<T>::get(in[k]);
      umax = a > umax ? a : umax;
      umin = a < umin ? a : umin;
      s0 += (double)in[k];
    }
  }
  double sum = s0 + s1;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long m1 = __shfl_xor_sync(0xFFFFFFFFu, umax, o);
    const unsigned long long m2 = __shfl_xor_sync(0xFFFFFFFFu, umin, o);
    umax = m1 > umax ? m1 : umax;
    umin = m2 < umin ? m2 : umin;
    sum += __shfl_xor_sync(0xFFFFFFFFu, sum, o);
  }
  __shared__ StatPartial sp[8];
  __shared__ bool is_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { sp[warp].umax = umax; sp[warp].umin = umin; sp[warp].sum = sum; }
  __syncthreads();
  if (threadIdx.x == 0) {
    StatPartial r = sp[0];
    for (int w = 1; w < (int)(blockDim.x >> 5); w++) {
      r.umax = sp[w].umax > r.umax ? sp[w].umax : r.umax;
      r.umin = sp[w].umin < r.umin ? sp[w].umin : r.umin;
      r.sum += sp[w].sum;
    }
    partials[blockIdx.x] = r;
    __threadfence();
    const unsigned prev = atomicAdd(done_counter, 1u);
    is_last = (prev == gridDim.x - 1);
  }
  __syncthreads();
  if (!is_last) return;
  // last CTA: deterministic (index-ordered) reduction of the per-CTA partials by warp 0
  if (warp == 0) {
    __threadfence();
    unsigned long long gmax = 0ull, gmin = ~0ull;
    double gsum = 0.0;
    for (unsigned b = lane; b < gridDim.x; b += 32) {
      const StatPartial r = partials[b];
      gmax = r.umax > gmax ? r.umax : gmax;
      gmin = r.umin < gmin ? r.umin : gmin;
      gsum += r.sum;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long m1 = __shfl_xor_sync(0xFFFFFFFFu, gmax, o);
      const unsigned long long m2 = __shfl_xor_sync(0xFFFFFFFFu, gmin, o);
      gmax = m1 > gmax ? m1 : gmax;
      gmin = m2 < gmin ? m2 : gmin;
      gsum += __shfl_xor_sync(0xFFFFFFFFu, gsum, o);
    }
    if (lane == 0) {
      stats3[0] = AbsBits<T>::back(gmax);
      stats3[1] = AbsBits<T>::back(gmin);
      stats3[2] = gsum;
      *done_counter = 0u;  // self-cleaning for the next launch
      if (finalize_inline)
        finalize_params(stats3, 1, n_total, sizeof(T) == 8, (double)in[0], first_slab, tb, params, info, qmax_zero);
    }
  }
}

// sf = pow(10, ceil(log10(max)) - 1) through threshold tables built with the host libm, so the
// result is bit-identical to util.c:28 (double) / util.c:42 (float) without a host round trip.
// Smallest index i with mx < thr[i] (n if none): a linear search from the guess the binary exponent
// gives (log10(mx) ~ 0.30103 * ilogb(mx), off by at most one), i.e. two or three loads instead of ten.
template <typename T> __device__ __forceinline__ int sf_index(T mx, const T *thr, int n, int kmin, int e2) {
  int lo = (int)floorf((float)e2 * 0.30103f) - kmin;
  lo = lo < 0 ? 0 : (lo > n ? n : lo);
  while (lo < n && !(mx < thr[lo])) lo++;
  while (lo > 0 && mx < thr[lo - 1]) lo--;
  return lo;
}
// The same index, its sf and the decade limits thr[idx-1], thr[idx] with ALL table loads issued at once: the guess from
// the binary exponent is off by at most one, so the answer lies in a window of four entries -- one memory latency
// instead of a chain of four (this runs on one thread in the prologue of every compress CTA).
template <typename T> struct SfHit { int idx; T sf, lo, hi; };
template <typename T> __device__ __forceinline__ SfHit<T> sf_window(T mx, const T *__restrict__ thr, const T *__restrict__ sfv, int n, int kmin, int e2) {
  int g = (int)floorf((float)e2 * 0.30103f) - kmin;  // candidate index (smallest i with mx < thr[i]) is within g-1 .. g+1
  g = g < 1 ? 1 : (g > n - 2 ? n - 2 : g);
  T t[4], v[4];
#pragma unroll
  for (int k = 0; k < 4; k++) {  // thr[g-2 .. g+1] (guards at the table ends), sf[g-1 .. g+2]
    const int i = g - 2 + k;
    t[k] = (i >= 0 && i < n) ? __ldg(thr + i) : (i < 0 ? (T)0 : (T)__int_as_float(0x7F800000));
    const int j = g - 1 + k;
    v[k] = __ldg(sfv + (j < 0 ? 0 : (j > n ? n : j)));
  }
  SfHit<T> h;
  if (mx < t[0] || !(mx < t[3])) {  // (never for a consistent table: fall back to the search)
    h.idx = sf_index<T>(mx, thr, n, kmin, e2);
    h.sf = sfv[h.idx];
    h.lo = h.idx > 0 ? thr[h.idx - 1] : (T)0;
    h.hi = h.idx < n ? thr[h.idx] : (T)0;
    return h;
  }
  // smallest i in {g-1, g, g+1} with mx < thr[i]  (thr[g-2] <= mx < thr[g+1] here)
  const int step = (mx < t[1]) ? 0 : ((mx < t[2]) ? 1 : 2);
  h.idx = g - 1 + step;
  h.sf = v[step];
  h.lo = t[step];
  h.hi = t[step + 1];
  return h;
}
__device__ __forceinline__ double sf_lookup_d(double mx, const SfTables &tb) {
  return tb.sf_d[sf_index<double>(mx, tb.thr_d, tb.n_d, tb.kmin_d, ilogb(mx))];
}
__device__ __forceinline__ float sf_lookup_f(float mx, const SfTables &tb) {
  return tb.sf_f[sf_index<float>(mx, tb.thr_f, tb.n_f, tb.kmin_f, ilogbf(mx))];
}

__device__ __forceinline__ void finalize_params(const double *stats_all, int nranks, unsigned long long n_total,
                                                int is_double, double first_value, int first_slab,
                                                const SfTables &tb, DevParams *p, Info *info,
                                                unsigned long long *qmax_zero) {
  if (qmax_zero) for (int j = 0; j < tb.qmax_words; j++) qmax_zero[j] = 0ull;  // QT per-position maxima
  double mx = stats_all[0], mn = stats_all[1], sum = stats_all[2];
  for (int r = 1; r < nranks; r++) {  // rank order => deterministic sum
    mx = max_keep_nan(mx, stats_all[3 * r]);
    mn = fmin(mn, stats_all[3 * r + 1]);
    sum += stats_all[3 * r + 2];
  }
  if (first_slab) sum -= first_value;  // util.c:21-25: the running sum starts at element 1
  // DCTZ_GPU_EDEGENERATE: max|x| is 0, inf or NaN (every statistics pass keeps a NaN in the maximum), or outside the admitted
  // range (build_sf_tables).  The sum of finite data may overflow (the reference's sum and mean become inf as well; the
  // decoder never reads the mean): it is not a test for non-finite data.
  int status = 0;
  double sf = 1.0, mean;
  if (is_double ? !(mx >= tb.min_d && mx < tb.max_d) : !((float)mx >= tb.min_f && (float)mx < tb.max_f)) status = -5;
  p->decade_lo = 0.0;
  p->decade_hi = __longlong_as_double(0x7FF0000000000000ll);
  if (is_double) {
    if (!status) {
      SfHit<double> h = sf_window<double>(mx, tb.thr_d, tb.sf_d, tb.n_d, tb.kmin_d, ilogb(mx));
      sf = h.sf;
      p->decade_lo = h.idx > 0 ? h.lo : tb.min_d;
      if (h.idx < tb.n_d) p->decade_hi = h.hi;
    }
    mean = sum / (double)(long long)n_total;
    const Divisor<double> d = make_divisor(sf);
    p->sf_d = d.b; p->inv_sf_d = d.y; p->scale_iters = d.iters;
    p->sf_f = (float)sf; p->inv_sf_f = 0.f;
  } else {
    float sff = 1.0f;
    if (!status) {
      SfHit<float> h = sf_window<float>((float)mx, tb.thr_f, tb.sf_f, tb.n_f, tb.kmin_f, ilogbf((float)mx));
      sff = h.sf;
      p->decade_lo = (double)(h.idx > 0 ? h.lo : tb.min_f);
      if (h.idx < tb.n_f) p->decade_hi = (double)h.hi;
    }
    sf = (double)sff;
    mean = (double)((float)sum / (float)(long long)n_total);
    const Divisor<float> d = make_divisor(sff);
    p->sf_f = d.b; p->inv_sf_f = d.y; p->scale_iters = d.iters;
    p->sf_d = sf; p->inv_sf_d = 0.0;
  }
  if (!(sf > 0.0)) status = -5;
  p->status = status;
  info->sf = sf; info->mean = mean; info->max_abs = mx; info->min_abs = mn; info->sum = sum;
  info->n_outliers = 0; info->n_edge = 0; info->n_exact_path = 0; info->n_qt_dropped = 0;
  info->status = status; info->scale_mode = p->scale_iters;
}

__global__ void k_finalize(const double *stats_all, int nranks, unsigned long long n_total, int is_double,
                           const void *first_elem, int first_slab, SfTables tb, DevParams *p, Info *info,
                           unsigned long long *qmax_zero) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    double fv = 0.0;
    if (first_slab) fv = is_double ? *(const double *)first_elem : (double)*(const float *)first_elem;
    finalize_params(stats_all, nranks, n_total, is_double, fv, first_slab, tb, p, info, qmax_zero);
  }
}

// ------------------------------------------------------------------------------------------
// Quantiser (dctz-comp-lib.c:363-414).  Returns the stream id 0..254, or 255 for an outlier.
// ------------------------------------------------------------------------------------------
// Exact restatement on a scaled coefficient, used for the rare near-boundary coefficients and by
// the tail kernel.
__device__ __forceinline__ unsigned quant_exact_d(double c, double rmin, double rmax, double bw, unsigned *edge) {
  if (c < rmin || c > rmax) return 255u;
  const double q = __ddiv_rn(__dsub_rn(c, rmin), bw);
  const int t = (int)q;  // (t_bin_id) truncation; q in [0, 255]
  if (t > 254) { (*edge)++; return 255u; }  // item == range_max: conv_tbl[255] is out of bounds in the reference -> outlier (DESIGN.md §2)
  return conv_ordinal(t);
}
__device__ __forceinline__ unsigned quant_exact(double c, const QuantConsts<double> &q, unsigned *edge) {
  return quant_exact_d(c, q.rmin, q.rmax, q.bw, edge);
}
__device__ __forceinline__ unsigned quant_exact_f(float c, float rmin, float rmax, float bw, unsigned *edge) {
  if (c < rmin || c > rmax) return 255u;
  const float q = __fdiv_rn(__fsub_rn(c, rmin), bw);
  const int t = (int)q;
  if (t > 254) { (*edge)++; return 255u; }
  return conv_ordinal(t);
}
__device__ __forceinline__ unsigned quant_exact(float c, const QuantConsts<float> &q, unsigned *edge) {
  return quant_exact_f(c, q.rmin, q.rmax, q.bw, edge);
}

template <typename T> struct BitsOf;
template <> struct BitsOf<double> {
  typedef unsigned long long U;
  static __device__ __forceinline__ U abs_bits(double v) { return (U)__double_as_longlong(v) & 0x7FFFFFFFFFFFFFFFull; }
};
template <> struct BitsOf<float> {
  typedef unsigned U;
  static __device__ __forceinline__ U abs_bits(float v) { return (U)__float_as_int(v) & 0x7FFFFFFFu; }
};

// Per-thread quantiser.  The transform runs on the UNSCALED block (the DCT is linear; dividing afterwards
// instead of before changes a coefficient by ~1 ulp, far inside the coefficient tolerance, and saves the
// per-element division), and the division by sf is folded into one constant kq = 1/(sf*bw):
//     v = c_u*kq + 127.5  ~  (c_u/sf - range_min)/bin_width,   t = floor(v),   0 <= t < 255 or outlier.
// v differs from the exactly rounded reference expression by ~1e-13 (double) / ~1e-5 (float, one ulp of v
// -- the reference's own float evaluation of that expression carries the same error), i.e. by less than the
// difference between two correct DCT implementations, so a different floor() can only happen at a
// quantisation-boundary tie (counted by the parity tests, tests/parity.py).
//   double: the "magic add" 1.5*2^32, rounded DOWN, leaves floor(v) in bits 20.. of the low word; out of
//           range saturates.
//   float : F2I with round-down.
// id = conv_tbl[t] = max(2t-255, 254-2t) = max(b, ~b) with b = 2t-255; t clamped to 255 gives id 255 (outlier).
// t == 255 includes item == range_max exactly, where the reference indexes conv_tbl[255] one past the table (UB):
// every path of this library (this quantiser, quant_exact for the tail block) and the oracle store such a
// coefficient as an outlier.
template <typename T> struct Quantizer;
template <> struct Quantizer<double> {
  double kq;
  Divisor<double> sfdiv;
  __device__ __forceinline__ void init(const DevParams *p, const QuantConsts<double> &qc) {
    sfdiv.b = p->sf_d; sfdiv.y = p->inv_sf_d; sfdiv.iters = p->scale_iters;
    kq = __ddiv_rn(1.0, __dmul_rn(p->sf_d, qc.bw));
  }
  __device__ __forceinline__ double scaled(double c_u) const { return div_exact(c_u, sfdiv); }
  // outliers are stored as float (USE_TRUNCATE): c_u * RN(1/sf) differs from c_u / sf by at most one double ulp,
  // i.e. the float it rounds to differs with probability ~2^-29 -- one multiply instead of the division sequence
  __device__ __forceinline__ float outlier(double c_u) const { return (float)__dmul_rn(c_u, sfdiv.y); }
  // candidate parking of the sparse emission path: what goes into the float-sized candidate array, and what comes out
  __device__ __forceinline__ float park(double c_u) const { return outlier(c_u); }
  __device__ __forceinline__ float unpark(float v) const { return v; }
  __device__ __forceinline__ unsigned quantize(double c_u) const {
    const double v = __fma_rn(c_u, kq, 127.5);
#ifdef DCTZ_QUANT_MAGIC_ADD
    const double z = __dadd_rd(v, 6442450944.0 /* 1.5 * 2^32 */);  // ROUND DOWN: the 2^-20 grid must not round v up past an integer
    const unsigned lo = (unsigned)__double2loint(z), hi = (unsigned)__double2hiint(z);
    const unsigned u = (hi == 0x41F80000u) ? lo : 0xFFFFFFFFu;  // v outside [0, 4096) saturates
    const int b = (int)(2u * min(u >> 20, 255u)) - 255;
#else
    // floor(v) by the conversion instruction (F2I.F64.FLOOR saturates; a negative result wraps to a huge unsigned): three
    // instructions fewer per coefficient than the magic add, the same integer for every finite v
    const int b = (int)(2u * min((unsigned)__double2int_rd(v), 255u)) - 255;
#endif
    return (unsigned)max(b, ~b);
  }
};
template <> struct Quantizer<float> {
  float kq;
  Divisor<float> sfdiv;
  __device__ __forceinline__ void init(const DevParams *p, const QuantConsts<float> &qc) {
    sfdiv.b = p->sf_f; sfdiv.y = p->inv_sf_f; sfdiv.iters = p->scale_iters;
    kq = (float)__ddiv_rn(1.0, __dmul_rn((double)p->sf_f, (double)qc.bw));
  }
  __device__ __forceinline__ float scaled(float c_u) const { return div_exact(c_u, sfdiv); }
  __device__ __forceinline__ float outlier(float c_u) const { return div_exact(c_u, sfdiv); }
  // float: the RAW coefficient is parked (no arithmetic for the 60 coefficients that are no outliers); the exact division
  // is done for the few that are picked up
  __device__ __forceinline__ float park(float c_u) const { return c_u; }
  __device__ __forceinline__ float unpark(float v) const { return div_exact(v, sfdiv); }
  __device__ __forceinline__ unsigned quantize(float c_u) const {
    const int t = __float2int_rd(__fmaf_rn(c_u, kq, 127.5f));
    const int b = (int)(2u * min((unsigned)t, 255u)) - 255;  // negative t wraps to a huge unsigned -> 255
    return (unsigned)max(b, ~b);
  }
};

// ------------------------------------------------------------------------------------------
// Scan of the per-tile outlier counts (shared by K2 / the gather kernels / K3)
// ------------------------------------------------------------------------------------------
// Chunk c = 1024 consecutive groups, one per thread of CTA c.  group_prefix[g] = outliers in the earlier
// groups of the same chunk; the last CTA to finish turns the chunk totals into chunk_prefix[c] and
// writes the grand total to *total.  Consumers add the two: prefix_of_group().
struct ScanOut {
  unsigned long long *group_prefix;  // one per group
  unsigned long long *chunk_prefix;  // one per chunk (first used as chunk totals)
  unsigned *done;                    // CTAs finished; reset by the last one
};
__device__ __forceinline__ unsigned long long prefix_of_group(const unsigned long long *__restrict__ group_prefix,
                                                              const unsigned long long *__restrict__ chunk_prefix, unsigned g) {
  return __ldg(chunk_prefix + (g >> 10)) + __ldg(group_prefix + g);
}
__device__ __forceinline__ unsigned long long block_exclusive_scan_1024(unsigned long long v, unsigned long long *s_warp,
                                                                        unsigned long long *total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long n = __shfl_up_sync(0xFFFFFFFFu, incl, o);
    if (lane >= o) incl += n;
  }
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    const unsigned long long w = (lane < (int)(blockDim.x >> 5)) ? s_warp[lane] : 0ull;  // CTAs smaller than 1024 threads
    unsigned long long wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long n = __shfl_up_sync(0xFFFFFFFFu, wi, o);
      if (lane >= o) wi += n;
    }
    s_warp[lane] = wi - w;
    if (lane == 31) s_warp[32] = wi;
  }
  __syncthreads();
  *total = s_warp[32];
  return s_warp[warp] + incl - v;
}
// For small fields the producer kernel's LAST CTA runs the scan itself (one launch less): ngroups <= 1024, i.e. one
// chunk, so group_prefix holds global prefixes and chunk_prefix[0] = 0.  Executed by every thread of the CTA.
struct FusedScan {
  ScanOut out;
  unsigned long long *total;
  unsigned n_entries;  // 0 = the caller launches k_scan_groups instead
};
__device__ __forceinline__ void cta_scan_small(const unsigned *counts, const FusedScan &f) {
  __shared__ unsigned long long s_w[33];
  __shared__ unsigned long long s_carry;
  const unsigned ngroups = (f.n_entries + 31u) / 32u;
  if (threadIdx.x == 0) s_carry = 0ull;
  __syncthreads();
  for (unsigned base = 0; base < ngroups; base += blockDim.x) {
    const unsigned g = base + threadIdx.x;
    unsigned long long sum = 0;
    if (g < ngroups) {
      const unsigned first = g * 32u;
      if (first + 32u <= f.n_entries) {
        const uint4 *p = reinterpret_cast<const uint4 *>(counts + first);
#pragma unroll
        for (int k = 0; k < 8; k++) { const uint4 v = __ldcg(p + k); sum += (unsigned long long)v.x + v.y + v.z + v.w; }
      } else {
        for (unsigned t = first; t < f.n_entries; t++) sum += __ldcg(counts + t);
      }
    }
    unsigned long long tot;
    const unsigned long long excl = block_exclusive_scan_1024(sum, s_w, &tot);
    const unsigned long long carry = s_carry;
    if (g < ngroups) f.out.group_prefix[g] = carry + excl;
    __syncthreads();
    if (threadIdx.x == 0) s_carry = carry + tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) { f.out.chunk_prefix[0] = 0ull; *f.total = s_carry; }
}

// ------------------------------------------------------------------------------------------
// K2: fused scale + DCT-II + quantise + ordered outlier compaction.
// Shared memory per warp: [ tile: 4 (2) swizzled slabs ][ EC: outlier candidates 63 x 32 floats ][ bin ids 2 KB ]
// ------------------------------------------------------------------------------------------
// QT outlier emission: store value and position and advance both cursors, all under one predicate taken straight from a
// bit of the group mask.  Only the LOW words of the two cursors move: a tile's slots (TILE_SLOT values, TILE_SLOT position
// bytes) are aligned to their own size (QT_RAW_ALIGN / QT_J_ALIGN on the arrays' bases, dctz_gpu.cu), so a cursor inside
// a slot never carries into the high word.  (With two 64-bit cursors and the hit flag taken as a value SASS showed 12.5
// instructions per coefficient position -- 29 % of the instructions of k_compress<double,QT> at 5 % outliers; a 32-bit
// offset from a 64-bit base is no better, ptxas spells the wide multiply-add as four instructions.)
constexpr size_t QT_RAW_ALIGN = (size_t)2048 * 8;  // = TILE_SLOT * sizeof(double) (static_assert below)
constexpr size_t QT_J_ALIGN = 2048;                // = TILE_SLOT
__device__ __forceinline__ void park_if(unsigned &plo, unsigned phi, unsigned &qlo, unsigned qhi, double v, unsigned j, unsigned mg, unsigned bit) {
  asm volatile(
      "{\n.reg .pred q;\n.reg .b32 t;\n.reg .u64 a, b;\n"
      "and.b32 t, %6, %7;\nsetp.ne.u32 q, t, 0;\n"
      "mov.b64 a, {%0, %2};\nmov.b64 b, {%1, %3};\n"
      "@q st.global.f64 [a], %4;\n@q st.global.u8 [b], %5;\n"
      "@q add.u32 %0, %0, 8;\n@q add.u32 %1, %1, 1;\n}\n"
      : "+r"(plo), "+r"(qlo)
      : "r"(phi), "r"(qhi), "d"(v), "r"(j), "r"(mg), "r"(bit)
      : "memory");
}
__device__ __forceinline__ void park_if(unsigned &plo, unsigned phi, unsigned &qlo, unsigned qhi, float v, unsigned j, unsigned mg, unsigned bit) {
  asm volatile(
      "{\n.reg .pred q;\n.reg .b32 t;\n.reg .u64 a, b;\n"
      "and.b32 t, %6, %7;\nsetp.ne.u32 q, t, 0;\n"
      "mov.b64 a, {%0, %2};\nmov.b64 b, {%1, %3};\n"
      "@q st.global.f32 [a], %4;\n@q st.global.u8 [b], %5;\n"
      "@q add.u32 %0, %0, 4;\n@q add.u32 %1, %1, 1;\n}\n"
      : "+r"(plo), "+r"(qlo)
      : "r"(phi), "r"(qhi), "f"(v), "r"(j), "r"(mg), "r"(bit)
      : "memory");
}

template <typename T, bool QT> struct CompressCfg {
  // EC outlier emission: a tile in which some block has more than DENSE_MIN outliers takes the dense form (predicated
  // convert + store per coefficient), sparser tiles the parked-candidates loop.  Measured on B200 (2^28-element slab
  // + white noise, 5% outliers): double 0.848 / 0.832 / 0.815 of roofline at thresholds 3 / 6 / 16, float 0.57 at 6,
  // 0.66 at 16 (its exact-division outliers make the dense form expensive); at 20-40% outliers all thresholds agree.
#ifndef DCTZ_DENSE_MIN_D
#define DCTZ_DENSE_MIN_D 3u
#endif
#ifndef DCTZ_DENSE_MIN_F
#define DCTZ_DENSE_MIN_F 16u
#endif
  static constexpr unsigned DENSE_MIN = (sizeof(T) == 8) ? DCTZ_DENSE_MIN_D : DCTZ_DENSE_MIN_F;
  static constexpr int WARPS = 4;
  static constexpr int THREADS = WARPS * 32;
  static constexpr int CTAS_PER_SM = (sizeof(T) == 8) ? 2 : 3;
  // EC: outlier candidates [63 coefficient positions][32 lanes] as float, written only by tiles that have outliers
  static constexpr int OFF_CAND = WarpTile<T>::BYTES;
  static constexpr int OFF_BINS = OFF_CAND + (QT ? 0 : 63 * WTILE * 4);
  static constexpr int WARP_BYTES = ((OFF_BINS + WTILE * BLK + 1023) / 1024) * 1024;  // tiles need 1 KB alignment (swizzle atom)
  static constexpr int SMEM = WARPS * WARP_BYTES + 1024;                             // + slack to align the base
};

// VERIFY: the statistics behind `params` are the caller's belief (a previous time step, a sample, a bound), not
// a pass over this data.  The kernel then also tracks the true max|x| (exact 64-bit bit-pattern maximum) and
// its last CTA checks that it lies in the decade the scaling factor was derived from; if not, info->status =
// DCTZ_GPU_ESTALE and the outputs are to be discarded.  `verify_lower` = 0 leaves the lower limit to the caller
// (a slab of a larger field need not contain the global maximum).
__device__ __forceinline__ double fabs_t(double v) { return fabs(v); }
__device__ __forceinline__ float fabs_t(float v) { return fabsf(v); }
__device__ __forceinline__ double fmax_t(double a, double b) { return fmax(a, b); }
__device__ __forceinline__ float fmax_t(float a, float b) { return fmaxf(a, b); }
__device__ __forceinline__ double fmin_t(double a, double b) { return fmin(a, b); }
__device__ __forceinline__ float fmin_t(float a, float b) { return fminf(a, b); }

// Out of line: the path of a refused field only, kept out of the register allocation of the compress kernels' tile loop.
__device__ __noinline__ void zero_tile_counts(unsigned *counts, unsigned long long nblk_full) {
  const unsigned long long ntiles = (nblk_full + WTILE - 1) / WTILE;
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < ntiles; i += (unsigned long long)gridDim.x * blockDim.x)
    counts[i] = 0u;
}

// VERIFY: what a thread has seen of the slab's true statistics while compressing with a BELIEF about them.
template <typename T> struct VerifyStat {
  double *tile_sums;  // per-tile sum of x, reduced in tile order afterwards: deterministic
  uint2 *tile_ext;    // per-tile {max, min} of the HIGH 32 bits of |x| (float: of all its bits, i.e. exact)
};

// The tile loop of the compress kernels: one warp, tiles handed out by `seq` (TileSeq: dynamic tickets; RangeSeq: the
// CTA's own contiguous range in the single-launch kernel), `phase` = the parity of the warp's mbarrier.
template <typename T, bool QT, bool VERIFY, class Seq>
__device__ __forceinline__ void compress_tiles(const CUtensorMap *tmap_in, unsigned long long nblk_full, const DevParams *params,
                                               const QuantConsts<T> &qc, uint8_t *__restrict__ bins, float *__restrict__ dc_out,
                                               unsigned *__restrict__ counts, float *__restrict__ ac_slots, T *__restrict__ raw_slots,
                                               uint8_t *__restrict__ j_slots, T *qtable0, unsigned char *wsm, unsigned mb, Seq &seq,
                                               int lane, VerifyStat<T> &vstat, unsigned &phase) {
  typedef typename ArithOf<T>::type A;
  typedef CompressCfg<T, QT> Cfg;
  typedef WarpTile<T> L;
  typedef typename BitsOf<T>::U U;
  constexpr unsigned FULL = 0xFFFFFFFFu;
  const unsigned tile_s = smem_u32(wsm);
  unsigned char *binbuf = wsm + Cfg::OFF_BINS;
  const unsigned ntiles = (unsigned)((nblk_full + WTILE - 1) / WTILE);
  Quantizer<T> qz;
  qz.init(params, qc);

  auto rows_of = [&](unsigned t) -> unsigned {
    const unsigned long long left = nblk_full - (unsigned long long)t * WTILE;
    return left < (unsigned long long)WTILE ? (unsigned)left : (unsigned)WTILE;
  };
  auto issue_tile = [&](unsigned t) {  // one lane: 4 (double) / 2 (float) tensor copies of a [32 rows x 128 B] slab each
    if (lane == 0) {
      mbar_expect_tx(mb, L::BYTES);  // rows beyond the field are zero-filled and still counted
#pragma unroll
      for (int q = 0; q < L::SLABS; q++) tma_load_2d(tile_s + q * L::SLAB_BYTES, tmap_in, q * 128, (int)(t * WTILE), mb);
    }
  };
  unsigned cur = seq.advance(lane);
  if (cur < ntiles) issue_tile(cur);
  unsigned nxt = seq.advance(lane);

  while (cur < ntiles) {
    mbar_wait(mb, phase);
    phase ^= 1u;
    unsigned keep = 0u;  // VERIFY: the low words of the pre-pass, fed into the probe below so that its loads stay 128 bits wide (lds128)
    if constexpr (VERIFY) {
      // The statistics pass folded into this one (util.c:12-44).  max|x| / min|x| are taken on the HIGH WORD of the bit
      // pattern (one integer max and min per element; for float that is the value, for double k_resolve_extremes settles
      // the low words of the few candidates afterwards) -- in a pass of its own over the tile in shared memory, BEFORE the
      // 64 values occupy the registers (folded into the load below it spilled).  The SUM is not taken here at all: it is
      // 8 x the block's DC coefficient, which the transform delivers anyway.
      unsigned hx2[2] = {0u, 0u}, hn2[2] = {0xFFFFFFFFu, 0xFFFFFFFFu};
      const unsigned long long left = nblk_full - (unsigned long long)cur * WTILE;
      if ((unsigned long long)lane < left) {  // rows beyond the field arrive zero-filled: they must not lower the minimum
#pragma unroll
        for (int q = 0; q < L::SLABS; q++) {
#pragma unroll
          for (int c = 0; c < 8; c++) {
            const uint4 v = lds128(tile_s + L::chunk_offset(q, lane, c));  // (see lds128: two narrowed loads cost four times the wavefronts)
            if constexpr (sizeof(T) == 8) {
              const unsigned h0 = v.y & 0x7FFFFFFFu, h1 = v.w & 0x7FFFFFFFu;
              hx2[c & 1] = max(hx2[c & 1], max(h0, h1));
              hn2[c & 1] = min(hn2[c & 1], min(h0, h1));
              keep |= v.x | v.z;
            } else {
              const unsigned h0 = v.x & 0x7FFFFFFFu, h1 = v.y & 0x7FFFFFFFu, h2 = v.z & 0x7FFFFFFFu, h3 = v.w & 0x7FFFFFFFu;
              hx2[c & 1] = max(hx2[c & 1], max(max(h0, h1), max(h2, h3)));
              hn2[c & 1] = min(hn2[c & 1], min(min(h0, h1), min(h2, h3)));
            }
          }
        }
      }
      const unsigned hmax = __reduce_max_sync(FULL, max(hx2[0], hx2[1])), hmin = __reduce_min_sync(FULL, min(hn2[0], hn2[1]));
      if (lane == 0) vstat.tile_ext[cur] = make_uint2(hmax, hmin);
    }
    T x[BLK];
    unsigned probe = keep;
#pragma unroll
    for (int q = 0; q < L::SLABS; q++) {
#pragma unroll
      for (int c = 0; c < 8; c++) {
        const uint4 v = *reinterpret_cast<const uint4 *>(wsm + L::chunk_offset(q, lane, c));
        const T *e = reinterpret_cast<const T *>(&v);
#pragma unroll
        for (int k = 0; k < L::PER_CHUNK; k++) x[(q * 8 + c) * L::PER_CHUNK + k] = e[k];
        probe |= v.x ^ v.w;
      }
    }
    // every lane HOLDS its row in registers (reads_have_landed: completed, not just issued) before the buffer is refilled
    __syncwarp();
    if (reads_have_landed(probe) && nxt < ntiles) issue_tile(nxt);  // overlaps everything below

    const unsigned rows = rows_of(cur);
    const unsigned long long blk = (unsigned long long)cur * WTILE + lane;
    const bool active = (unsigned)lane < rows;
    // (rows beyond the field arrive zero-filled: they quantise to bin 0 and are never stored)

    // ---- orthonormal DCT-II (dct.c:55-103) of the unscaled block; x / sf is folded into the quantiser ----
    dct64_forward<A>(x);
    if constexpr (VERIFY) {  // sum of the block = sqrt(64) x its DC coefficient (orthonormal DCT-II); reduced over the warp in a fixed order
      double ts = active ? 8.0 * (double)x[0] : 0.0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) ts += __shfl_xor_sync(FULL, ts, o);
      if (lane == 0) vstat.tile_sums[cur] = ts;
    }

    // ---- quantise (dctz-comp-lib.c:350-414); the ids go straight to the warp's bin-id buffer in shared
    //      memory (four at a time), which keeps 16 registers free and is where the bulk store reads them ----
    if (lane == 0) bulk_wait_read();  // the previous tile's bin ids have left shared memory
    __syncwarp();
    uint4 *brow = reinterpret_cast<uint4 *>(binbuf + lane * BLK);
    unsigned mlo = 0, mhi = 0;  // bit j: coefficient j is an outlier (bin id 255)
#pragma unroll
    for (int q4 = 0; q4 < 4; q4++) {
      unsigned wq[4];
#pragma unroll
      for (int k = 0; k < 4; k++) {
        unsigned word = (q4 == 0 && k == 0) ? 255u : 0u;  // bin_index[i*64] = NBINS, :361
#pragma unroll
        for (int b = 0; b < 4; b++) {
          const int j = 16 * q4 + 4 * k + b;
          if (j == 0) continue;
          word |= qz.quantize(x[j]) << (8 * b);
        }
        const unsigned nib = (ff_flags(word) * 0x00204081u) >> 28;  // flag (bit 7) of byte b -> bit b: 16 partial products, all at different positions
        if (q4 < 2) mlo |= nib << (16 * q4 + 4 * k); else mhi |= nib << (16 * (q4 - 2) + 4 * k);
        wq[k] = word;
      }
      brow[q4] = make_uint4(wq[0], wq[1], wq[2], wq[3]);
    }
    mlo &= ~1u;  // the DC marker is not an outlier
    if (!active) { mlo = 0; mhi = 0; }
    const unsigned cnt = __popc(mlo) + __popc(mhi);

    const unsigned incl = warp_inclusive_scan(cnt, lane);
    const unsigned tile_total = __shfl_sync(FULL, incl, 31);
    const unsigned my_off = incl - cnt;  // this block's first outlier inside the tile's run
    if (lane == 0) counts[cur] = tile_total;

    // ---- bin ids: one bulk store per tile; DC ----
    fence_async_smem();
    __syncwarp();
    if (lane == 0) {
      bulk_s2g(bins + (unsigned long long)cur * WTILE * BLK, smem_u32(binbuf), rows * BLK);
      bulk_commit();
    }
    const T dcs = qz.scaled(x[0]);
    if (active) {
      dc_out[blk] = (float)dcs;  // :351 (USE_TRUNCATE)
      if (QT && blk == nblk_full - 1) *qtable0 = dcs;  // :357/:359 (a later tail block overwrites it)
    }

    // ---- outliers (dctz-comp-lib.c:478-544): each lane writes its block's outliers, in ascending j, at the block's
    //      offset inside the tile's slot, so the slot holds the tile's outliers packed in their final order;
    //      k_gather_* only has to move whole tile runs ----
    if (tile_total != 0) {
      const unsigned long long run = (unsigned long long)cur * TILE_SLOT + my_off;
      if constexpr (QT) {  // raw (unscaled) coefficient + position; scaled and rescaled by K2b once the global qtable is known
        // The UNSCALED coefficient is parked.  The exact division by sf is done once per outlier by the gather
        // (k_qt_gather), and the per-position maxima (:371-372, 396-397) are taken by k_qt_max over the parked
        // values: here they would cost a look-up and a branch per coefficient POSITION (measured: the branches,
        // not the arithmetic, held this kernel at half its EC speed).  For the same reason the stores are predicated
        // by hand -- the compiler turns the plain `if` into 63 divergent branches.
        static_assert(QT_RAW_ALIGN == (size_t)TILE_SLOT * 8 && QT_J_ALIGN == (size_t)TILE_SLOT, "slot alignment");
        const unsigned long long praw = (unsigned long long)(raw_slots + (unsigned long long)cur * TILE_SLOT + my_off);
        const unsigned long long pj = (unsigned long long)(j_slots + (unsigned long long)cur * TILE_SLOT + my_off);
        unsigned plo = (unsigned)praw, qlo = (unsigned)pj;  // the cursors' low words (see park_if)
        const unsigned phi = (unsigned)(praw >> 32), qhi = (unsigned)(pj >> 32);
        // (coefficient positions in groups of eight: a group in which no block of the tile has an outlier -- the high
        // frequencies of a smooth field -- is skipped by a warp-uniform branch)
#pragma unroll
        for (int g = 0; g < 8; g++) {
          const unsigned mg = ((g < 4) ? (mlo >> (8 * g)) : (mhi >> (8 * (g - 4)))) & 0xFFu;
          if (__any_sync(FULL, mg != 0u)) {
#pragma unroll
            for (int b = 0; b < 8; b++) {
              const int j = 8 * g + b;
              if (j == 0) continue;
              park_if(plo, phi, qlo, qhi, x[j], (unsigned)j, mg, 1u << b);
            }
          }
        }
      } else {
        // Uniform, branch-free part: every lane parks all 63 scaled AC coefficients as float (:537, USE_TRUNCATE) in
        // its own column of the candidate array (conflict-free; register indices stay compile-time).  Then a short
        // loop over the set bits of the lane's outlier mask -- its trip count is the largest per-block count of the
        // warp -- copies the outliers to the block's run.
        const unsigned maxcnt = __reduce_max_sync(FULL, cnt);
        if (maxcnt > Cfg::DENSE_MIN) {
          // Dense tile: one predicated convert + store per coefficient, straight from the registers (no parking, no
          // dependent chain: the stores only share the running offset).
          float *tile_run = ac_slots + (unsigned long long)cur * TILE_SLOT;  // warp-uniform base, 32-bit lane offsets
          unsigned off = my_off;
#pragma unroll
          for (int g = 0; g < 8; g++) {  // (groups of eight positions; an empty group is skipped warp-uniformly, see the QT branch)
            const unsigned mg = ((g < 4) ? (mlo >> (8 * g)) : (mhi >> (8 * (g - 4)))) & 0xFFu;
            if (__any_sync(FULL, mg != 0u)) {
#pragma unroll
              for (int b = 0; b < 8; b++) {
                const int j = 8 * g + b;
                if (j == 0) continue;
                if ((mg >> b) & 1u) tile_run[off++] = qz.outlier(x[j]);
              }
            }
          }
          cur = nxt;
          nxt = seq.advance(lane);
          continue;
        }
        float *cand = reinterpret_cast<float *>(wsm + Cfg::OFF_CAND) + lane;
#pragma unroll
        for (int j = 1; j < BLK; j++) cand[(j - 1) * WTILE] = qz.park(x[j]);
        // two independent chains per trip: the lowest remaining position goes to the front of the run, the highest
        // to its back
        const unsigned trips = (maxcnt + 1u) >> 1;
        float *lo = ac_slots + run, *hi = lo + cnt;
        for (unsigned it = 0; it < trips; it++) {
          if (mlo | mhi) {
            const int j = mlo ? (__ffs(mlo) - 1) : (31 + __ffs(mhi));
            *lo++ = qz.unpark(cand[(j - 1) * WTILE]);
            if (mlo) mlo &= mlo - 1u; else mhi &= mhi - 1u;
          }
          if (mlo | mhi) {
            const int j = mhi ? (63 - __clz(mhi)) : (31 - __clz(mlo));
            *--hi = qz.unpark(cand[(j - 1) * WTILE]);
            if (mhi) mhi &= ~(1u << (j - 32)); else mlo &= ~(1u << j);
          }
        }
      }
    }
    cur = nxt;
    nxt = seq.advance(lane);
  }

}

// Where the scaling factor of a launch comes from.  k_compress derives the parameters in its own prologue (every CTA for
// itself, identically; CTA 0 publishes them and the result block): no separate one-thread launch in front of it.
//   MODE_STATS   stats_all are the TRUE statistics of the field (one triple per rank, merged in rank order)
//   MODE_BELIEF  stats_all are a BELIEF (a sample, the previous time step): the VERIFY instantiation compresses with the
//                scaling factor they give and gathers the true max / min / per-tile sums of the slab on the way
//   MODE_REDO    stats_all are the true statistics gathered by a MODE_BELIEF launch: if they give the scaling factor that
//                launch used, every CTA leaves at once (the normal case: the input has been read ONCE); otherwise the
//                slab is compressed again with the right one
enum { MODE_STATS = 0, MODE_BELIEF = 1, MODE_REDO = 2 };
struct StatSource {
  const double *stats_all;
  int nranks, first_slab, is_double, mode;
  unsigned long long n_total;
  const void *first_elem;       // element 0 of the field (only read by the first slab: util.c:21-25 skips it in the sum)
  SfTables tb;
  DevParams *params;            // published by CTA 0 (the tail kernel and the QT gather read it)
  unsigned long long *qmax_zero;  // QT: the per-position maxima to clear
  double *tile_sums;            // MODE_BELIEF: per-tile sums
  uint2 *tile_ext;              // MODE_BELIEF: per-tile extremes of the high word of |x|
};

template <typename T, bool QT, bool VERIFY>
__global__ void __launch_bounds__(CompressCfg<T, QT>::THREADS, CompressCfg<T, QT>::CTAS_PER_SM)
k_compress(const __grid_constant__ CUtensorMap tmap_in, unsigned long long nblk_full, StatSource src,
           QuantConsts<T> qc, uint8_t *__restrict__ bins, float *__restrict__ dc_out,
           unsigned *__restrict__ counts,                     // outliers per warp tile
           float *__restrict__ ac_slots,                      // EC: outlier scratch, TILE_SLOT entries per tile, packed
           T *__restrict__ raw_slots, uint8_t *__restrict__ j_slots,  // QT: raw outliers + their position j, same layout
           T *qtable0,                                        // QT: entry 0 of the table: the last full block's DC
           TileControl *ctl, Info *info, FusedScan fused, unsigned batch) {
  typedef CompressCfg<T, QT> Cfg;
  extern __shared__ unsigned char smem_raw[];
  __shared__ __align__(8) unsigned long long s_mbar[Cfg::WARPS];
  __shared__ DevParams s_params;
  __shared__ Info s_info;
  __shared__ int s_skip;

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned char *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char *wsm = smem + warp * Cfg::WARP_BYTES;
  const unsigned mb = smem_u32(&s_mbar[warp]);

  if (lane == 0) { mbar_init(mb, 1); fence_mbar_init(); }
  if (threadIdx.x == 0) {  // sf and the quantiser's divisor, from the merged statistics (util.c:28/42)
    double fv = 0.0;
    if (src.first_slab) fv = src.is_double ? __ldg((const double *)src.first_elem) : (double)__ldg((const float *)src.first_elem);
    finalize_params(src.stats_all, src.nranks, src.n_total, src.is_double, fv, src.first_slab, src.tb, &s_params, &s_info,
                    (blockIdx.x == 0 && src.mode != MODE_REDO) ? src.qmax_zero : nullptr);
    if (VERIFY && s_params.status != 0) {
      // A refused BELIEF (0, NaN, inf, or outside the admitted exponent range -- a caller's bound may be DBL_MAX) must not
      // skip the tile loop: the loop is what gathers the true statistics the REDO launch decides on.  Compress with the
      // placeholder belief max|x| = 1 instead; the REDO launch recompresses (or refuses) from the true statistics.
      const double one[3] = {1.0, 1.0, 0.0};
      finalize_params(one, 1, src.n_total, src.is_double, 0.0, 0, src.tb, &s_params, &s_info, nullptr);
    }
    int skip = 0;
    if (src.mode == MODE_REDO) {
      skip = (s_params.status == 0 && s_params.sf_d == *reinterpret_cast<volatile double *>(&ctl->belief_sf)) ? 1 : 0;
      if (!skip) s_info.n_exact_path = 1;  // the belief was wrong: the slab is compressed a second time
    }
    if (s_params.status != 0) skip = 1;  // degenerate statistics (max|x| = 0 / inf / NaN): nothing to compress, the status says why
    s_skip = skip;
    if (blockIdx.x == 0) {
      if (src.mode == MODE_BELIEF) ctl->belief_sf = s_params.sf_d;
      *src.params = s_params;
      *info = s_info;
    }
  }
  __syncthreads();  // the only CTA-wide barrier before the epilogue
  if (s_skip) {
    // degenerate statistics: no tile is compressed, so no tile writes its outlier count -- zero them all, or the scan and
    // gather launched after this kernel would move stale or uninitialised counts' worth of outliers
    if (s_params.status != 0) zero_tile_counts(counts, nblk_full);
    return;
  }

  VerifyStat<T> vstat;
  vstat.tile_sums = src.tile_sums;
  vstat.tile_ext = src.tile_ext;
  unsigned phase = 0;
  TileSeq seq;
  seq.init(&ctl->ticket, blockIdx.x * Cfg::WARPS + warp, gridDim.x * Cfg::WARPS, batch, lane);
  compress_tiles<T, QT, VERIFY>(&tmap_in, nblk_full, &s_params, qc, bins, dc_out, counts, ac_slots, raw_slots, j_slots, qtable0, wsm, mb, seq, lane,
                                vstat, phase);

  // ---- epilogue ----
  bulk_wait_all();
  __syncthreads();
  __shared__ bool s_last;
  __threadfence();  // this thread's counts are visible device-wide before the CTA signs off
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned prev = atomicAdd(&ctl->done, 1u);
    s_last = (prev == gridDim.x - 1);
    if (s_last) {
      ctl->ticket = 0u;
      ctl->done = 0u;
    }
  }
  __syncthreads();
  if (s_last && fused.n_entries) {
    __threadfence();
    cta_scan_small(counts, fused);
  }
}

// MODE_BELIEF, second half: the slab's sum from the per-tile sums, in tile order whatever the tiles' owners were
// (deterministic): CTA c adds tiles [4096 c, 4096 c + 4096) with a fixed tree, the last CTA adds the CTA sums in order --
// and the slab's extreme high words.  spec[0] = max high word, spec[1] = min high word; true3[2] = the sum (+ the tail's).
// For float the high word is the value: true3[0..1] are final here.  For double k_resolve_extremes settles the low words.
struct TileReduce { double *cta_sums; uint2 *cta_ext; unsigned *done; unsigned *hw; /* [2] */ unsigned long long *ext_bits; /* [2] exact |x| patterns */ };
template <typename T>
__global__ void __launch_bounds__(256) k_reduce_tiles(const double *__restrict__ tile_sums, const uint2 *__restrict__ tile_ext, unsigned ntiles, TileReduce r,
                                                      const double *tail3, double *true3) {
  __shared__ double s_w[8];
  __shared__ unsigned s_hx[8], s_hn[8];
  __shared__ bool s_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned first = blockIdx.x * 4096u;
  double s = 0.0;
  unsigned hx = 0u, hn = 0xFFFFFFFFu;
  for (unsigned i = first + threadIdx.x; i < first + 4096u && i < ntiles; i += 256u) {
    s += __ldcg(tile_sums + i);
    const uint2 e = __ldcg(tile_ext + i);
    hx = max(hx, e.x);
    hn = min(hn, e.y);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
  hx = __reduce_max_sync(0xFFFFFFFFu, hx);
  hn = __reduce_min_sync(0xFFFFFFFFu, hn);
  if (lane == 0) { s_w[warp] = s; s_hx[warp] = hx; s_hn[warp] = hn; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    unsigned x = 0u, n = 0xFFFFFFFFu;
    for (int w = 0; w < 8; w++) { t += s_w[w]; x = max(x, s_hx[w]); n = min(n, s_hn[w]); }
    r.cta_sums[blockIdx.x] = t;
    r.cta_ext[blockIdx.x] = make_uint2(x, n);
    __threadfence();
    s_last = (atomicAdd(r.done, 1u) == gridDim.x - 1);
  }
  __syncthreads();
  if (!s_last || threadIdx.x != 0) return;
  __threadfence();
  double t = 0.0;
  unsigned x = 0u, n = 0xFFFFFFFFu;
  for (unsigned c = 0; c < gridDim.x; c++) {
    t += __ldcg(r.cta_sums + c);
    const uint2 e = __ldcg(r.cta_ext + c);
    x = max(x, e.x);
    n = min(n, e.y);
  }
  if (tail3) t += tail3[2];
  true3[2] = t;
  if (sizeof(T) == 4) {  // float: the "high word" is the whole pattern -- exact
    double mx = (double)__int_as_float((int)x), mn = (double)__int_as_float((int)n);
    if (tail3) { mx = max_keep_nan(mx, tail3[0]); mn = fmin(mn, tail3[1]); }
    true3[0] = mx; true3[1] = mn;
  } else {
    r.hw[0] = x; r.hw[1] = n;
    r.ext_bits[0] = 0ull; r.ext_bits[1] = ~0ull;
  }
  *r.done = 0u;
}

// double: exact max|x| / min|x| among the elements whose high word equals the slab's extreme high word.  Only the tiles
// that recorded that high word are read again (usually one or two; a constant field: all of them -- a second pass, as
// the two-pass path always makes).  The last CTA merges the tail block and publishes true3[0..1].
__global__ void __launch_bounds__(256) k_resolve_extremes(const double *__restrict__ in, unsigned long long nblk_full, const uint2 *__restrict__ tile_ext,
                                                          unsigned ntiles, TileReduce r, unsigned *done2, const double *tail3, double *true3) {
  const unsigned hx = __ldcg(r.hw), hn = __ldcg(r.hw + 1);
  const int lane = threadIdx.x & 31;
  const unsigned wpg = (gridDim.x * blockDim.x) >> 5;
  unsigned long long bmax = 0ull, bmin = ~0ull;
  for (unsigned t0 = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * 32u; t0 < ntiles; t0 += wpg * 32u) {  // 32 tile records per warp and trip
    const unsigned tl = t0 + (unsigned)lane;
    uint2 e = make_uint2(0xFFFFFFFFu, 0u);
    if (tl < ntiles) e = __ldcg(tile_ext + tl);
    unsigned hit = __ballot_sync(0xFFFFFFFFu, tl < ntiles && (e.x == hx || e.y == hn));
    while (hit) {  // re-read the (few) tiles that hold a candidate
      const unsigned t = t0 + (unsigned)(__ffs(hit) - 1);
      hit &= hit - 1u;
      const unsigned long long first = (unsigned long long)t * (WTILE * BLK);
      unsigned long long last = first + WTILE * BLK;
      if (last > nblk_full * BLK) last = nblk_full * BLK;
      // 16-byte vectors, eight loads in flight per lane (a lone warp walking a tile element by element took 36 us: the
      // whole launch waited for it); slabs start 16-byte aligned and tiles are 16 KB, so the vectors are aligned
      const uint4 *pv = reinterpret_cast<const uint4 *>(in + first);
      const unsigned nvec = (unsigned)((last - first) >> 1);
      for (unsigned i0 = 0; i0 < nvec; i0 += 256) {
        uint4 v[8];
#pragma unroll
        for (int u = 0; u < 8; u++) { const unsigned i = i0 + 32 * u + lane; v[u] = i < nvec ? __ldg(pv + i) : make_uint4(0u, 0u, 0u, 0u); }
#pragma unroll
        for (int u = 0; u < 8; u++) {
          if (i0 + 32 * u + lane >= nvec) continue;
          const unsigned long long a0 = (((unsigned long long)v[u].y << 32) | v[u].x) & 0x7FFFFFFFFFFFFFFFull;
          const unsigned long long a1 = (((unsigned long long)v[u].w << 32) | v[u].z) & 0x7FFFFFFFFFFFFFFFull;
          const unsigned h0 = (unsigned)(a0 >> 32), h1 = (unsigned)(a1 >> 32);
          if (h0 == hx) bmax = a0 > bmax ? a0 : bmax;
          if (h0 == hn) bmin = a0 < bmin ? a0 : bmin;
          if (h1 == hx) bmax = a1 > bmax ? a1 : bmax;
          if (h1 == hn) bmin = a1 < bmin ? a1 : bmin;
        }
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long m1 = __shfl_xor_sync(0xFFFFFFFFu, bmax, o), m2 = __shfl_xor_sync(0xFFFFFFFFu, bmin, o);
    bmax = m1 > bmax ? m1 : bmax;
    bmin = m2 < bmin ? m2 : bmin;
  }
  if (lane == 0) {
    if (bmax != 0ull) atomicMax(r.ext_bits, bmax);
    if (bmin != ~0ull) atomicMin(r.ext_bits + 1, bmin);
  }
  __shared__ bool s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(done2, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!s_last || threadIdx.x != 0) return;
  __threadfence();
  double mx = __longlong_as_double((long long)*reinterpret_cast<volatile unsigned long long *>(r.ext_bits));
  double mn = __longlong_as_double((long long)*reinterpret_cast<volatile unsigned long long *>(r.ext_bits + 1));
  if (tail3) { mx = max_keep_nan(mx, tail3[0]); mn = fmin(mn, tail3[1]); }
  true3[0] = mx; true3[1] = mn;
  *done2 = 0u;
}

// The BELIEF: max|x| over a sample of the slab -- one 16-byte vector of every 4 KB (0.4 % of the bytes) -- plus the
// exact {max, min, sum} of the partial tail block, which the tile loop never sees.  belief3 = {max, max, 0}: only the
// decade of the maximum matters (util.c:28), the true statistics replace it after the compress pass.
constexpr unsigned SAMPLE_STRIDE_VECS = 256;  // at least this many 16-byte vectors between two samples (4 KB); large slabs: ~256 K samples in all
template <typename T>
__global__ void __launch_bounds__(256) k_sample(const T *__restrict__ in, size_t n, size_t stride_vecs, unsigned long long *max_bits, unsigned *done_counter,
                                                double *belief3, double *tail3) {
  constexpr int VEC = 16 / (int)sizeof(T);
  const size_t nfull = (n / BLK) * BLK, nvec = nfull / VEC, nsamp = (nvec + stride_vecs - 1) / stride_vecs;
  const uint4 *p = reinterpret_cast<const uint4 *>(in);
  T vmax = (T)0;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < nsamp; i0 += 4 * stride) {
    uint4 v[4];
#pragma unroll
    for (int u = 0; u < 4; u++) { const size_t i = i0 + u * stride; v[u] = i < nsamp ? __ldg(p + i * stride_vecs) : make_uint4(0u, 0u, 0u, 0u); }
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const T *e = reinterpret_cast<const T *>(&v[u]);
#pragma unroll
      for (int q = 0; q < VEC; q++) { const T a = e[q] < (T)0 ? -e[q] : e[q]; vmax = a > vmax ? a : vmax; }
    }
  }
  double m = (double)vmax;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(max_bits, (unsigned long long)__double_as_longlong(m));
  __shared__ bool s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(done_counter, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!s_last || threadIdx.x != 0) return;
  __threadfence();
  double mx = __longlong_as_double((long long)atomicExch(max_bits, 0ull));
  const double inf = __longlong_as_double(0x7FF0000000000000ll);
  double tmax = 0.0, tmin = inf, tsum = 0.0;
  for (size_t k = nfull; k < n; k++) {  // the partial tail block, exactly
    const double v = (double)in[k], a = fabs(v);
    tmax = max_keep_nan(tmax, a); tmin = fmin(tmin, a); tsum += v;  // (a NaN stays in the maximum: finalize_params rejects it)
  }
  tail3[0] = tmax; tail3[1] = tmin; tail3[2] = tsum;
  mx = fmax(mx, tmax);
  if (!(mx > 0.0) || !(mx < inf)) mx = 1.0;  // a sample of zeros (or a NaN): any belief will do, the true statistics decide afterwards
  belief3[0] = mx; belief3[1] = mx; belief3[2] = 0.0;
  *done_counter = 0u;
}

// ------------------------------------------------------------------------------------------
// Generic orthonormal DCT-II / DCT-III of one block of length dn (1..64) by the definition, in
// double, with exact cospi arguments.  One warp; used for the partial tail block (any dn,
// including odd ones: dct.c:59-72 / 144-164) and by dctz_gpu_dct_blocks for dn != 64.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
  return v;
}
// coef[k] for k = lane, lane+32 (kept in two registers)
__device__ __forceinline__ void generic_dct(const double *xs /* shared, dn values */, int dn, int lane, double out[2]) {
  const double scale = sqrt(2.0 / (double)dn);
#pragma unroll
  for (int h = 0; h < 2; h++) {
    const int k = lane + 32 * h;
    double s = 0.0;
    if (k < dn) {
      for (int n = 0; n < dn; n++) {
        const int idx = ((2 * n + 1) * k) % (4 * dn);
        s = __fma_rn(xs[n], cospi((double)idx / (double)(2 * dn)), s);
      }
      s *= scale;
      if (k == 0) s *= 0.70710678118654752440;
    }
    out[h] = s;
  }
}
__device__ __forceinline__ void generic_idct(const double *cs /* shared, dn coefficients */, int dn, int lane, double out[2]) {
  const double scale = sqrt(2.0 / (double)dn);
#pragma unroll
  for (int h = 0; h < 2; h++) {
    const int n = lane + 32 * h;
    double s = 0.0;
    if (n < dn) {
      s = cs[0] * 0.70710678118654752440;
      for (int k = 1; k < dn; k++) {
        const int idx = ((2 * n + 1) * k) % (4 * dn);
        s = __fma_rn(cs[k], cospi((double)idx / (double)(2 * dn)), s);
      }
      s *= scale;
    }
    out[h] = s;
  }
}

// Partial last block of the compress path: it is warp tile number `slot_tile` of the scratch layout.
template <typename T, bool QT>
__global__ void __launch_bounds__(32) k_tail_compress(const T *__restrict__ in /* start of the tail block */, int rem,
                                                      unsigned long long blk_index, unsigned slot_tile,
                                                      const DevParams *params, QuantConsts<T> qc, uint8_t *bins,
                                                      float *dc_out, unsigned *counts, float *ac_slots,
                                                      T *raw_slots, uint8_t *j_slots, typename BitsOf<T>::U *qmax_bits,
                                                      T *qtable0, Info *info) {
  __shared__ double xs[BLK];
  const int lane = threadIdx.x;
  if (params->status != 0) {  // degenerate statistics: nothing is compressed; the scan and gather that follow see no outliers
    if (lane == 0) counts[slot_tile] = 0u;
    return;
  }
  const T sf = (sizeof(T) == 8) ? (T)params->sf_d : (T)params->sf_f;
  for (int n = lane; n < rem; n += 32) {
    T v = in[n];
    if (sf != (T)1) v = v / sf;  // IEEE division (no fast-math)
    xs[n] = (double)v;
  }
  __syncwarp();
  double c2[2];
  generic_dct(xs, rem, lane, c2);
  const unsigned long long slot = (unsigned long long)slot_tile * TILE_SLOT;
  unsigned base = 0;
  unsigned edge = 0;
  for (int h = 0; h < 2; h++) {
    const int j = lane + 32 * h;
    const T c = (T)c2[h];  // float path: double result rounded once to float
    unsigned id = 0;
    bool valid = j < rem;
    if (valid) {
      if (j == 0) {
        id = 255u;
        dc_out[blk_index] = (float)c;
        if (QT) *qtable0 = c;
      } else {
        id = quant_exact(c, qc, &edge);
      }
      bins[blk_index * BLK + j] = (uint8_t)id;
    }
    const bool outl = valid && j > 0 && id == 255u;
    const unsigned m = __ballot_sync(0xFFFFFFFFu, outl);
    if (outl) {
      const unsigned p = base + __popc(m & ((1u << lane) - 1u));
      if (QT) {
        raw_slots[slot + p] = c; j_slots[slot + p] = (uint8_t)j;
        atomicMax(&qmax_bits[j], BitsOf<T>::abs_bits(c));
      } else {
        ac_slots[slot + p] = (float)c;
      }
    }
    base += __popc(m);
  }
  edge = (unsigned)warp_sum((double)edge);
  if (lane == 0) { counts[slot_tile] = base; if (edge) info->n_edge += edge; }
}

// ------------------------------------------------------------------------------------------
// Scan + gather: per-tile counts -> exclusive prefix per group of 32 tiles -> final AC_exact order.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) k_scan_groups(const unsigned *__restrict__ counts, unsigned ntiles, ScanOut out,
                                                     unsigned long long *total) {
  __shared__ unsigned long long s_warp[33];
  __shared__ bool s_last;
  const unsigned ngroups = (ntiles + 31u) / 32u;
  const unsigned g = blockIdx.x * 1024u + threadIdx.x;
  unsigned long long sum = 0;
  if (g < ngroups) {  // the 32 counts of a group are one 128-byte line
    const unsigned first = g * 32u;
    if (first + 32u <= ntiles) {
      const uint4 *p = reinterpret_cast<const uint4 *>(counts + first);
      uint4 v[8];
#pragma unroll
      for (int k = 0; k < 8; k++) v[k] = __ldg(p + k);
#pragma unroll
      for (int k = 0; k < 8; k++) sum += (unsigned long long)v[k].x + v[k].y + v[k].z + v[k].w;
    } else {
      for (unsigned t = first; t < ntiles; t++) sum += counts[t];
    }
  }
  unsigned long long chunk_total;
  const unsigned long long excl = block_exclusive_scan_1024(sum, s_warp, &chunk_total);
  if (g < ngroups) out.group_prefix[g] = excl;
  if (threadIdx.x == 0) {
    out.chunk_prefix[blockIdx.x] = chunk_total;
    __threadfence();
    s_last = (atomicAdd(out.done, 1u) == gridDim.x - 1);
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  // last CTA: exclusive scan of the chunk totals (any number of chunks, 1024 at a time)
  unsigned long long carry = 0;
  for (unsigned c0 = 0; c0 < gridDim.x; c0 += 1024u) {
    const unsigned c = c0 + threadIdx.x;
    const unsigned long long v = (c < gridDim.x) ? *(volatile unsigned long long *)(out.chunk_prefix + c) : 0ull;
    unsigned long long tot;
    __syncthreads();
    const unsigned long long e = block_exclusive_scan_1024(v, s_warp, &tot);
    if (c < gridDim.x) out.chunk_prefix[c] = carry + e;
    carry += tot;
  }
  if (threadIdx.x == 0) { *total = carry; *out.done = 0u; }
}

// Gather: a tile's packed run goes to prefix_of_group + (totals of the earlier tiles of its group).
__global__ void __launch_bounds__(256) k_gather_ec(const unsigned *__restrict__ counts, const unsigned long long *__restrict__ group_prefix,
                                                   const unsigned long long *__restrict__ chunk_prefix, unsigned ntiles,
                                                   const float *__restrict__ ac_slots, float *__restrict__ ac_out,
                                                   const unsigned long long *__restrict__ n_total) {
  if (__ldg(n_total) == 0ull) return;  // nothing to move (the scan has counted)
  // One CTA per GROUP of 32 tiles: every warp scans the group's 32 counts itself (the same 128 bytes, one per lane; no
  // shared memory, no barrier) and copies the packed runs of tiles warp, warp + 8, ... to their final place with up to
  // eight independent loads in flight per lane.  (A warp per tile was bound by the latency of its three dependent
  // loads; a flat element index with a per-element search of the scanned counts was bound by its instructions.)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned ngroups = (ntiles + 31u) >> 5;
  for (unsigned g = blockIdx.x; g < ngroups; g += gridDim.x) {
    const unsigned t0 = g * 32u + (unsigned)lane;
    const unsigned c = (t0 < ntiles) ? __ldg(counts + t0) : 0u;
    const unsigned incl = warp_inclusive_scan(c, lane);
    if (__shfl_sync(0xFFFFFFFFu, incl, 31) == 0u) continue;
    float *gdst = ac_out + prefix_of_group(group_prefix, chunk_prefix, g);
    const float *gsrc = ac_slots + (unsigned long long)g * 32u * TILE_SLOT;
    // the warp's four runs (tiles warp, warp + 8, ...): the first 128 outliers of ALL of them are requested before any is stored
    // (one run at a time, the warp sat out the load latency four times per group); longer runs finish in the loop below
    unsigned n4[4], off4[4];
    float v4[4][4];
#pragma unroll
    for (int q = 0; q < 4; q++) {
      n4[q] = __shfl_sync(0xFFFFFFFFu, c, warp + 8 * q);
      off4[q] = __shfl_sync(0xFFFFFFFFu, incl - c, warp + 8 * q);
      const float *src = gsrc + (unsigned)(warp + 8 * q) * TILE_SLOT;
#pragma unroll
      for (int k = 0; k < 4; k++) { const unsigned i = 32u * k + lane; v4[q][k] = (i < n4[q]) ? __ldg(src + i) : 0.f; }
    }
#pragma unroll
    for (int q = 0; q < 4; q++) {
      float *dst = gdst + off4[q];
#pragma unroll
      for (int k = 0; k < 4; k++) { const unsigned i = 32u * k + lane; if (i < n4[q]) dst[i] = v4[q][k]; }
    }
    for (int q = 0; q < 4; q++) {
      const unsigned n = n4[q];
      const float *src = gsrc + (unsigned)(warp + 8 * q) * TILE_SLOT;
      float *dst = gdst + off4[q];
      for (unsigned i0 = 128u; i0 < n; i0 += 256u) {
        float v[8];
#pragma unroll
        for (int k = 0; k < 8; k++) { const unsigned i = i0 + 32u * k + lane; v[k] = (i < n) ? __ldg(src + i) : 0.f; }
#pragma unroll
        for (int k = 0; k < 8; k++) { const unsigned i = i0 + 32u * k + lane; if (i < n) dst[i] = v[k]; }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// K2b (QT): rescale the ordered raw outliers with the global per-position table
// (dctz-comp-lib.c:450-461 clamp, 485-533 rescale).  An entry whose rescaled value falls back inside
// the bin range would be dropped by the reference (its bin_index stays 255; :494-506); see qt_rescale_one
// for why that cannot happen -- such entries are only counted (info->n_qt_dropped).
// ------------------------------------------------------------------------------------------
template <typename T> __device__ __forceinline__ Divisor<T> sf_divisor(const DevParams *p);
template <> __device__ __forceinline__ Divisor<double> sf_divisor<double>(const DevParams *p) {
  Divisor<double> d;
  d.b = p->sf_d; d.y = p->inv_sf_d; d.iters = p->scale_iters;
  return d;
}
template <> __device__ __forceinline__ Divisor<float> sf_divisor<float>(const DevParams *p) {
  Divisor<float> d;
  d.b = p->sf_f; d.y = p->inv_sf_f; d.iters = p->scale_iters;
  return d;
}
// QT: per-position maxima of |coefficient| over the parked outliers of the full tiles (dctz-comp-lib.c:371-372, 396-397),
// as bit patterns (non-negative floats order like unsigned integers).  One CTA per group of 32 tiles, a warp per tile
// run; per-CTA maxima in shared memory, looked at before the atomic (they stop moving quickly), flushed once.
template <typename T>
__global__ void __launch_bounds__(256) k_qt_max(const unsigned *__restrict__ counts, unsigned ntiles /* full tiles only */,
                                                const T *__restrict__ raw_slots, const uint8_t *__restrict__ j_slots,
                                                typename BitsOf<T>::U *qmax_bits, const DevParams *__restrict__ params,
                                                unsigned *done_counter) {
  typedef typename BitsOf<T>::U U;
  __shared__ U s_max[BLK];
  __shared__ bool s_last;
  if (threadIdx.x < BLK) s_max[threadIdx.x] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned ngroups = (ntiles + 31u) >> 5;
  for (unsigned g = blockIdx.x; g < ngroups; g += gridDim.x) {
    const unsigned t0 = g * 32u + (unsigned)lane;
    const unsigned c = (t0 < ntiles) ? __ldg(counts + t0) : 0u;
    for (int s = warp; s < 32; s += 8) {
      const unsigned n = __shfl_sync(0xFFFFFFFFu, c, s);
      const unsigned long long src = (unsigned long long)(g * 32u + (unsigned)s) * TILE_SLOT;
      for (unsigned i0 = 0; i0 < n; i0 += 128u) {
        U a[4];
        unsigned jj[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const unsigned i = i0 + 32u * u + lane;
          a[u] = 0; jj[u] = 1u;
          if (i < n) { a[u] = BitsOf<T>::abs_bits(__ldg(raw_slots + src + i)); jj[u] = __ldg(j_slots + src + i); }
        }
#pragma unroll
        for (int u = 0; u < 4; u++)
          if (a[u] > *reinterpret_cast<volatile U *>(&s_max[jj[u]])) atomicMax(&s_max[jj[u]], a[u]);
      }
    }
  }
  __syncthreads();
  if (threadIdx.x >= 1 && threadIdx.x < BLK && s_max[threadIdx.x] != 0) atomicMax(&qmax_bits[threadIdx.x], s_max[threadIdx.x]);
  // The maxima are those of the UNSCALED coefficients; the last CTA turns them into the maxima of the scaled ones:
  // max |c| / sf == max |c / sf| (exact division is monotone).  The tail block's kernel, whose values are scaled
  // already, runs after this one.
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    s_last = (atomicAdd(done_counter, 1u) == gridDim.x - 1);
    if (s_last) *done_counter = 0u;
  }
  __syncthreads();
  if (s_last && threadIdx.x >= 1 && threadIdx.x < BLK) {
    __threadfence();
    volatile T *t = reinterpret_cast<volatile T *>(qmax_bits);
    const T v = t[threadIdx.x];
    t[threadIdx.x] = div_exact(v, sf_divisor<T>(params));
  }
}

template <typename T> struct QtConsts {
  double eb;        // error_bound (double in both paths)
  T rmin, rmax;     // compress-side range (dctz-comp-lib.c:274-275 / 279-280)
  T d_rmin, d_rmax; // decompress-side range (dctz-decomp-lib.c:373-374 / 378-379)
  double den;       // error_bound * qt_factor  (dctz-decomp-lib.c:405,450)
  Divisor<double> den_div;  // exact division by it without the division instruction sequence (common.cuh)
};

// The branch is chosen by the SIGN of the coefficient, not by re-testing it against the range: the element IS an outlier
// (its bin id says so), and the fast quantiser's verdict may differ from an exact `item > range_max` at a
// quantisation-boundary tie.  Wherever the reference's own tests (:488/:490, :514/:516) fire, the sign test picks the
// same branch; at a tie it keeps the outlier an outlier (range_max + something positive), so the stream never desyncs.
// Returns false if the rescaled value fell back inside the range (the reference would then drop it although its bin
// id stays 255, :494-506).  That cannot happen for valid input: it needs |c|/qtable[j] * 10 eb <= ulp(255 eb)/2, i.e.
// qtable[j] >= 168 (float; far more for double) while |c_j| <= sqrt(2/64)*64*10 = 113 for data scaled into (1,10]
// (DESIGN.md §2); the count is kept as a diagnostic (info->n_qt_dropped, always 0).
__device__ __forceinline__ bool qt_rescale_one(double item, double q, const QtConsts<double> &k, float *out) {
  if (item < 0.0) item = __dadd_rn(__dmul_rn(__dmul_rn(__ddiv_rn(item, q), k.eb), 10.0), k.rmin);  // :489
  else item = __dadd_rn(__dmul_rn(__dmul_rn(__ddiv_rn(item, q), k.eb), 10.0), k.rmax);            // :491
  *out = (float)item;  // :497 USE_TRUNCATE
  return (item < k.rmin || item > k.rmax);
}
__device__ __forceinline__ bool qt_rescale_one(float item, float q, const QtConsts<float> &k, float *out) {
  // (float/float) in float, then promoted to double by error_bound; qt_factor.f = 10.0f; result stored to float
  if (item < 0.0f) item = (float)__dadd_rn(__dmul_rn(__dmul_rn((double)__fdiv_rn(item, q), k.eb), (double)10.0f), (double)k.rmin);  // :515
  else item = (float)__dadd_rn(__dmul_rn(__dmul_rn((double)__fdiv_rn(item, q), k.eb), (double)10.0f), (double)k.rmax);             // :517
  *out = item;
  return (item < k.rmin || item > k.rmax);
}

// QT gather: rescale while moving to the final place.
template <typename T>
__global__ void __launch_bounds__(256) k_qt_gather(const unsigned *__restrict__ counts, const unsigned long long *__restrict__ group_prefix,
                                                   const unsigned long long *__restrict__ chunk_prefix, unsigned ntiles,
                                                   const T *__restrict__ raw_slots, const uint8_t *__restrict__ j_slots,
                                                   const T *__restrict__ qraw /* global maxima, [0] = last DC */,
                                                   T *__restrict__ qtable_out, QtConsts<T> k, float *__restrict__ ac_out, Info *info,
                                                   const DevParams *__restrict__ params, unsigned tail_tile /* its values are scaled already */) {
  __shared__ T qt[BLK];
  const Divisor<T> sfdiv = sf_divisor<T>(params);
  if (threadIdx.x < BLK) {
    T v = qraw[threadIdx.x];
    if (threadIdx.x >= 1 && v < (T)1.0) v = (T)1.0;  // :450-461
    qt[threadIdx.x] = v;
    if (blockIdx.x == 0 && qtable_out) qtable_out[threadIdx.x] = v;
  }
  __syncthreads();
  // one CTA per group of 32 tiles, whole packed runs per warp (as k_gather_ec)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned ngroups = (ntiles + 31u) >> 5;
  unsigned dropped = 0;
  for (unsigned g = blockIdx.x; g < ngroups; g += gridDim.x) {
    const unsigned t0 = g * 32u + (unsigned)lane;
    const unsigned c = (t0 < ntiles) ? __ldg(counts + t0) : 0u;
    const unsigned incl = warp_inclusive_scan(c, lane);
    if (__shfl_sync(0xFFFFFFFFu, incl, 31) == 0u) continue;
    float *gdst = ac_out + prefix_of_group(group_prefix, chunk_prefix, g);
    for (int s = warp; s < 32; s += 8) {
      const unsigned n = __shfl_sync(0xFFFFFFFFu, c, s);
      const unsigned off = __shfl_sync(0xFFFFFFFFu, incl - c, s);
      const unsigned long long src = (unsigned long long)(g * 32u + (unsigned)s) * TILE_SLOT;
      const bool unscaled = (g * 32u + (unsigned)s) != tail_tile;
      float *dst = gdst + off;
      for (unsigned i0 = 0; i0 < n; i0 += 128u) {
        T r[4];
        unsigned jj[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const unsigned i = i0 + 32u * u + lane;
          r[u] = (T)0; jj[u] = 1u;
          if (i < n) { r[u] = __ldg(raw_slots + src + i); jj[u] = __ldg(j_slots + src + i); }
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const unsigned i = i0 + 32u * u + lane;
          if (i < n) {
            float o;
            if (!qt_rescale_one(unscaled ? div_exact(r[u], sfdiv) : r[u], qt[jj[u]], k, &o)) dropped++;
            dst[i] = o;
          }
        }
      }
    }
  }
  if (dropped) atomicAdd(&info->n_qt_dropped, (unsigned long long)dropped);
}

__constant__ int c_l2_hints;  // DCTZ_L2_HINTS: 1 = bin ids read with evict_last by the pre-pass, reconstruction stored with evict_first

// Decompress pre-pass: number of 255 markers at positions j >= 1 per warp tile (32 blocks = 2 KB of bin ids).
__global__ void __launch_bounds__(256) k_count_bins(const uint8_t *__restrict__ bins, unsigned long long nblk_full,
                                                    unsigned *__restrict__ counts, unsigned *done_counter, FusedScan fused) {
  const int lane = threadIdx.x & 31;
  const unsigned ntiles = (unsigned)((nblk_full + WTILE - 1) / WTILE);
  const unsigned wpg = (gridDim.x * blockDim.x) >> 5;
  const int hints = c_l2_hints;
  const unsigned long long pol_last = policy_evict_last();
  // two tiles per warp and trip: eight independent 16-byte loads in flight per lane
  for (unsigned t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; t < ntiles; t += 2 * wpg) {
    uint4 v[2][4];
    unsigned rows[2];
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const unsigned th = t + h * wpg;
      rows[h] = 0;
      if (th < ntiles) {
        const unsigned long long first = (unsigned long long)th * WTILE;
        rows[h] = (nblk_full - first < (unsigned long long)WTILE) ? (unsigned)(nblk_full - first) : (unsigned)WTILE;
        const uint4 *p = reinterpret_cast<const uint4 *>(bins + first * BLK);
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const unsigned chunk = i * 32 + lane;  // 16-byte chunk of the tile; 4 chunks per block
          v[h][i] = (chunk < rows[h] * 4u) ? (hints ? ldg_hint(p + chunk, pol_last) : __ldg(p + chunk)) : make_uint4(0u, 0u, 0u, 0u);
        }
      }
    }
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const unsigned th = t + h * wpg;
      if (th >= ntiles) break;
      unsigned cnt = 0;
#pragma unroll
      for (int i = 0; i < 4; i++) {
        const unsigned chunk = i * 32 + lane;
        if (chunk < rows[h] * 4u) {
          const unsigned x0 = (chunk & 3u) ? v[h][i].x : (v[h][i].x & 0xFFFFFF00u);  // byte 0 of a block is the DC marker
          cnt += __popc(ff_flags(x0)) + __popc(ff_flags(v[h][i].y)) + __popc(ff_flags(v[h][i].z)) + __popc(ff_flags(v[h][i].w));
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xFFFFFFFFu, cnt, o);
      if (lane == 0) counts[th] = cnt;
    }
  }
  if (!fused.n_entries) return;
  __shared__ bool s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    s_last = (atomicAdd(done_counter, 1u) == gridDim.x - 1);
    if (s_last) *done_counter = 0u;
  }
  __syncthreads();
  if (s_last) {
    __threadfence();
    cta_scan_small(counts, fused);
  }
}

// ------------------------------------------------------------------------------------------
// K3: dequantise + DCT-III + de-scale (dctz-decomp-lib.c:389-511).
// Shared memory: static [ centre table 256 T ] + dynamic, per warp [ tile: swizzled slabs ][ outlier stage: 8 KB (double) /
// 4 KB (float) ][ bin ids 2 KB ][ DC 128 B ]
// ------------------------------------------------------------------------------------------
template <typename T, bool QT> struct DecompressCfg {
  static constexpr int WARPS = 4;
  static constexpr int THREADS = WARPS * 32;
  static constexpr int CTAS_PER_SM = (sizeof(T) == 8) ? 2 : 3;
  // Every warp has its own outlier stage: the next tile's outliers are PREFETCHED by TMA together with its bin ids.
  // The stage holds FAST_MAX finished coefficients of type T (half of a tile's coefficients).  double: it also
  // holds the raw floats of ANY tile (2048 >= 3 + 63*32).  float: a tile with more than FAST_MAX outliers does not
  // fit (a bigger stage would cost the third resident CTA); such a tile loads its outliers late, into the tile
  // buffer, which is dead until the inverse transform writes it.
  static constexpr int FAST_MAX = 1024;
  static constexpr int STAGE_BYTES = FAST_MAX * (int)sizeof(T);
  static constexpr int OFF_STAGE = WarpTile<T>::BYTES;
  static constexpr int OFF_BINS = OFF_STAGE + STAGE_BYTES;
  static constexpr int OFF_DC = OFF_BINS + WTILE * BLK;
  static constexpr int WARP_BYTES = ((OFF_DC + WTILE * 4 + 1023) / 1024) * 1024;  // tiles need 1 KB alignment (swizzle atom)
  static constexpr int SMEM = WARPS * WARP_BYTES + 1024;                         // + slack to align the base (the centre table is static)
  static_assert(WarpTile<T>::BYTES >= 63 * WTILE * 4, "the tile must hold a full tile of outliers");
  static_assert(sizeof(T) == 4 || STAGE_BYTES >= (3 + 63 * WTILE + 3) * 4, "double: the stage must hold a full tile of raw outliers");
};

// Rebuild one coefficient of a tile that has outliers: `idb` = bin id * sizeof(T) (byte offset into the centre table);
// the marker 255 redirects the load to the lane's next finished outlier (`spd` = its shared address minus the
// marker's table address) and advances it.  Five instructions, no branch, one load either way.
__device__ __forceinline__ void pick_coefficient(double &x, unsigned &spd, unsigned idb /* by value: clobbered */, unsigned center_s) {
  asm volatile(
      "{\n.reg .pred q;\n.reg .u32 a;\n"
      "setp.eq.u32 q, %2, 0x7f8;\n"
      "@q add.u32 %2, %2, %1;\n"
      "add.u32 a, %2, %3;\n"
      "ld.shared.f64 %0, [a];\n"
      "@q add.u32 %1, %1, 8;\n}\n"
      : "=d"(x), "+r"(spd), "+r"(idb)
      : "r"(center_s)
      : "memory");
}
__device__ __forceinline__ void pick_coefficient(float &x, unsigned &spd, unsigned idb, unsigned center_s) {
  asm volatile(
      "{\n.reg .pred q;\n.reg .u32 a;\n"
      "setp.eq.u32 q, %2, 0x3fc;\n"
      "@q add.u32 %2, %2, %1;\n"
      "add.u32 a, %2, %3;\n"
      "ld.shared.f32 %0, [a];\n"
      "@q add.u32 %1, %1, 4;\n}\n"
      : "=f"(x), "+r"(spd), "+r"(idb)
      : "r"(center_s)
      : "memory");
}
// byte offset of bin id number b (0..3) of the word w in a table of T
template <typename T> __device__ __forceinline__ unsigned id_offset(unsigned w, int b) {
  constexpr int SH = (sizeof(T) == 8) ? 3 : 2;
  constexpr unsigned MASK = 0xFFu << SH;
  return (8 * b >= SH) ? ((w >> (8 * b - SH)) & MASK) : ((w << (SH - 8 * b)) & MASK);
}

__device__ __forceinline__ double qt_unscale_one(float acf, double q, const QtConsts<double> &k) {
  const double v = (double)acf;  // :402
  if (v > 0) return __dmul_rn(div_exact(__dsub_rn(v, k.d_rmax), k.den_div), q);  // :405 (IEEE quotient by den, see Divisor)
  return __dmul_rn(div_exact(__dsub_rn(v, k.d_rmin), k.den_div), q);             // :408
}
__device__ __forceinline__ float qt_unscale_one(float acf, float q, const QtConsts<float> &k) {
  // :450-454 -- float subtraction, double division and product, stored to float
  if (acf > 0) return (float)__dmul_rn(div_exact((double)__fsub_rn(acf, k.d_rmax), k.den_div), (double)q);
  return (float)__dmul_rn(div_exact((double)__fsub_rn(acf, k.d_rmin), k.den_div), (double)q);
}

template <typename T> __device__ __forceinline__ T mul_rn(T a, T b);
template <> __device__ __forceinline__ double mul_rn<double>(double a, double b) { return __dmul_rn(a, b); }
template <> __device__ __forceinline__ float mul_rn<float>(float a, float b) { return __fmul_rn(a, b); }

// The coefficients of a full block, already multiplied by sf (dctz-decomp-lib.c:392-416; the de-scale of :494-511 is folded
// in).  Every decoder of full blocks -- the tile loops (decompress_tiles) and the range kernel (ranges.cuh) -- forms them
// through these three, so that a block decodes to the same bits whichever way it is reached.
// Bin centre of id (gen_bins / gen_bins_f, binning.c:19-22, 39-42).  Entry 255 is a dummy that an outlier replaces.
template <typename T> __device__ __forceinline__ T center_coefficient(unsigned id, T bin_width, T sf) {
  return mul_rn<T>(mul_rn<T>((T)center_multiple(id), bin_width), sf);
}
// Outlier `a` of AC_exact at coefficient position j, q = qtable[j] (only read in QT mode, :402-409 / :450-454).
template <typename T, bool QT> __device__ __forceinline__ T outlier_coefficient(float a, T q, const QtConsts<T> &qk, T sf) {
  T v;
  if (QT) v = qt_unscale_one(a, q, qk); else v = (T)a;
  return mul_rn<T>(v, sf);
}
template <typename T> __device__ __forceinline__ T dc_coefficient(float dc, T sf) { return mul_rn<T>((T)dc, sf); }  // :392

// The partial last block (rem < 64 elements): coefficients by the definition, in double, through generic_idct; element n
// (n < rem) is handed to store(n, value) by lane n % 32.  `base` = offset of the block's first outlier; a marker at or
// past n_limit is a corrupt stream: the coefficient is 0 and on_corrupt() is called.  Used by k_tail_decompress and by
// the range kernel.
template <typename T, bool QT, class OnCorrupt, class Store>
__device__ __forceinline__ void tail_block_decode(const uint8_t *__restrict__ bins, const float *__restrict__ dc_in, const float *__restrict__ ac_in,
                                                  const T *__restrict__ qtable, int rem, unsigned long long blk_index, T bin_width, T sf,
                                                  const QtConsts<T> &qk, unsigned long long base, unsigned long long n_limit,
                                                  const OnCorrupt &on_corrupt, const Store &store, double *cs /* shared, BLK */, int lane) {
  for (int h = 0; h < 2; h++) {
    const int j = lane + 32 * h;
    const bool valid = j < rem;
    const unsigned id = valid ? bins[blk_index * BLK + j] : 0u;
    const bool outl = valid && j > 0 && id == 255u;
    const unsigned m = __ballot_sync(0xFFFFFFFFu, outl);
    if (valid) {
      T v;
      if (j == 0) v = (T)dc_in[blk_index];
      else if (outl) {
        const unsigned long long at = base + __popc(m & ((1u << lane) - 1u));
        float a = 0.f;
        if (at < n_limit) a = ac_in[at]; else on_corrupt();  // more markers than outliers: corrupt stream
        if (QT) v = (T)qt_unscale_one(a, qtable[j], qk); else v = (T)a;
      } else {
        if (sizeof(T) == 8) v = (T)__dmul_rn((double)center_multiple(id), (double)bin_width);
        else v = (T)__fmul_rn((float)center_multiple(id), (float)bin_width);
      }
      cs[j] = (double)v;
    }
    base += __popc(m);
  }
  __syncwarp();
  double r2[2];
  generic_idct(cs, rem, lane, r2);
  for (int h = 0; h < 2; h++) {
    const int n = lane + 32 * h;
    if (n < rem) {
      T v = (T)r2[h];
      if (sf != (T)1) v = v * sf;
      store(n, v);
    }
  }
}

// Outlier extent of a tile (warp-uniform): where its run starts in AC_exact and how long it is.  The loads (load) and
// the warp reduction that consumes them (finish) are a whole iteration apart, so their latency is never waited for.
struct Extent { unsigned long long base; unsigned total; bool bad; };  // bad: the run would leave the caller's AC_exact array
struct ExtentRaw { unsigned long long gp, cp; unsigned c; unsigned k; };  // loaded values, untouched until finish()
// Extents from the scan of the pre-pass (k_count_bins + k_scan_groups): offset of the first outlier = scanned group prefix
// + the counts of the earlier tiles of its group; the size is the tile's count.
struct ScannedExtents {
  typedef ExtentRaw Raw;
  static __device__ __forceinline__ Raw none() { Raw r; r.gp = 0; r.cp = 0; r.c = 0; r.k = 0; return r; }
  const unsigned *__restrict__ counts;
  const unsigned long long *__restrict__ group_prefix, *__restrict__ chunk_prefix;
  unsigned long long n_limit;
  unsigned *corrupt_flag;
  __device__ __forceinline__ ExtentRaw load(unsigned t, int lane) const {
    ExtentRaw r;
    r.k = t & 31u;
    r.c = ((unsigned)lane <= r.k) ? __ldg(counts + (t & ~31u) + lane) : 0u;  // lanes < k: earlier tiles of the group; lane k: the tile
    r.gp = __ldg(group_prefix + (t >> 5));
    r.cp = __ldg(chunk_prefix + (t >> 15));  // prefix_of_group(), its addition left to finish()
    return r;
  }
  __device__ __forceinline__ Extent finish(ExtentRaw &r, int lane) const {
    Extent e;
    r.c = pin_here(r.c);  // first use of the loaded values: here, at the end of the iteration
    r.gp = pin_here(r.gp);
    r.cp = pin_here(r.cp);
    e.total = __shfl_sync(0xFFFFFFFFu, r.c, (int)r.k);
    unsigned before = ((unsigned)lane < r.k) ? r.c : 0u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xFFFFFFFFu, before, o);
    e.base = r.gp + r.cp + before;
    // A stream whose bin indices mark more outliers than AC_exact holds (n_limit: its length as the caller states it)
    // is corrupt: such a tile decodes without its outliers and the launch is flagged; nothing is read out of bounds.
    e.bad = e.base + e.total > n_limit;
    if (e.bad) { e.total = 0u; *corrupt_flag = 1u; }
    return e;
  }
};

// ------------------------------------------------------------------------------------------
// Decompress WITHOUT the pre-pass (k_count_bins + k_scan_groups), warp-specialised: k_decompress<T, QT, true> runs two
// warpgroups per CTA.
//   count  (warps 4-7): take units (a ticket's batch of tiles) in increasing order from a count ticket of their own, load
//          the units' bin ids with the evict_last hint (the decode warps' bulk copies then find them in L2), count the
//          markers and PUBLISH them:
//              counts[t]   the tile's outliers                                   (flag bit 31 | count)
//              agg[u]      the unit's outliers                                   (flag bit 31 | count)
//              S[u / 64]   sum over the group of 64 units, by atomic addition    (contributions << 48 | sum)
//              T[u / 2048] sum over the super-group of 32 groups, likewise       (contributions << 48 | sum)
//          Every entry carries its own completion mark on a buffer the host zeroes before the launch, so a publish needs no
//          fence and a reader no acquire: a value is either marked complete or read again.
//   decode (warps 0-3): the tile loop of the pre-pass kernel (decompress_tiles) over units from the decode ticket, with the
//          extents of CountedExtents: a unit's first outlier is a pure READ (complete super-groups below it + complete
//          groups of its super-group below it + the units of its group below it -- five coalesced loads), a tile's is that
//          plus the counts of the earlier tiles of its unit, and both are loaded one iteration before they are used.
// The counting thereby leaves the decode warps' dependent chain, and setmaxnreg hands the registers the count warps do not
// need (COUNT_REGS) to the decode warps (DECODE_REGS).
// Deadlock freedom.  Counters wait only for the decode TICKET (unit u is counted once u < decode tickets taken + COUNT_LEAD),
// never for a decode to complete; decoders wait only for counts.  Both tickets are taken only by running warps, in
// increasing order.  Let D be the number of decode tickets taken.  A decoder waits only for units below its own, i.e. below
// D.  A counter holding a unit below D + COUNT_LEAD never waits; a counter that waits holds a unit >= D + COUNT_LEAD, so
// the count ticket has passed every unit below D, and each of those belongs to a running counter that does not wait: every
// unit below D is published, no decoder waits for ever, and D grows until it passes the last unit, which releases every
// counter.  A CTA that is not resident holds no ticket of either kind, so two such kernels of two contexts sharing the
// device (neither fully resident) cannot wait for each other's missing CTAs.
// ------------------------------------------------------------------------------------------
#ifndef DCTZ_COUNT_LEAD
#define DCTZ_COUNT_LEAD 384u
#endif
// units the count ticket may run ahead of the decode ticket: 384 units of 4 tiles = 3 MB of counted bin ids beyond the
// units the decode warps hold (up to two a warp, 19 MB on a B200); 8 GiB slab on a B200: 1.57-1.58 ms at 192 and 384,
// 1.58-1.59 at 1024, 1.62 at 2048 units (profiles/README.md)
constexpr unsigned COUNT_LEAD = DCTZ_COUNT_LEAD;
struct SplitCfg {
  static constexpr int DECODE_WARPS = 4, COUNT_WARPS = 4;
  static constexpr int THREADS = (DECODE_WARPS + COUNT_WARPS) * 32;
  static constexpr int CTAS_PER_SM = 2;
  // (DECODE_REGS + COUNT_REGS) * 128 threads * 2 CTAs = 65536 = the register file; the launch gives every thread 128
  static constexpr unsigned DECODE_REGS = 216, COUNT_REGS = 40;
};
static_assert((SplitCfg::DECODE_REGS + SplitCfg::COUNT_REGS) * 128 * SplitCfg::CTAS_PER_SM == 65536, "the register split must fill the register file");
template <unsigned N> __device__ __forceinline__ void setmaxnreg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;\n" ::"n"(N)); }
template <unsigned N> __device__ __forceinline__ void setmaxnreg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" ::"n"(N)); }
#ifdef DCTZ_WAIT_STATS
// diagnostic build (-DDCTZ_WAIT_STATS): [0] decode-warp re-reads of counts not yet published, [1] count-warp looks at a
// closed lead window, [2] units counted; printed by dctz_gpu_destroy
__device__ unsigned long long g_wait_stats[3];
#endif

struct AheadBufs { unsigned *counts, *agg; unsigned long long *S, *T; };
__device__ __forceinline__ unsigned ld_volatile(const unsigned *p) {
  unsigned v;
  asm volatile("ld.volatile.global.u32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long ld_volatile(const unsigned long long *p) {
  unsigned long long v;
  asm volatile("ld.volatile.global.u64 %0, [%1];\n" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
  return v;
}
constexpr unsigned long long AHEAD_LOW48 = 0xFFFFFFFFFFFFull;

// The count warpgroup's loop (one warp).  Returns when the count ticket has passed the last unit.
__device__ __forceinline__ void count_units(const uint8_t *__restrict__ bins, unsigned long long nblk_full, unsigned ntiles, unsigned batch,
                                            unsigned nunits, AheadBufs b, unsigned *count_ticket, const unsigned *decode_ticket, int lane) {
  const unsigned long long pol = policy_evict_last();
  unsigned lead_end = 0;  // units below it may be counted: decode tickets taken (as last read) + COUNT_LEAD
#ifdef DCTZ_WAIT_STATS
  unsigned long long n_wait = 0, n_units = 0;
#endif
  for (;;) {
    unsigned u = 0;
    if (lane == 0) u = ticket_next(count_ticket);
    u = __shfl_sync(0xFFFFFFFFu, u, 0);
    if (u >= nunits) break;
    while (u >= lead_end) {
      lead_end = ld_volatile(decode_ticket) + COUNT_LEAD;
      if (u < lead_end) break;
#ifdef DCTZ_WAIT_STATS
      n_wait++;
#endif
      // the decoders take ~90 units per microsecond on a B200; sleep about as long as the window needs to open, so
      // that a thousand waiting warps do not hammer the decode ticket's line
      const unsigned short_by = u + 1u - lead_end;
      __nanosleep(short_by < 256u ? 64u + 16u * short_by : 4096u);
    }
    const unsigned t0 = u * batch, t1 = (t0 + batch < ntiles) ? t0 + batch : ntiles;
    unsigned sum = 0;
    for (unsigned t = t0; t < t1; t++) {
      const unsigned long long first = (unsigned long long)t * WTILE;
      const unsigned rows = (nblk_full - first < (unsigned long long)WTILE) ? (unsigned)(nblk_full - first) : (unsigned)WTILE;
      const uint4 *p = reinterpret_cast<const uint4 *>(bins + first * BLK);
      uint4 v[4];
#pragma unroll
      for (int i = 0; i < 4; i++) {
        const unsigned chunk = i * 32 + lane;  // 16-byte chunk of the tile; 4 chunks per block
        v[i] = (chunk < rows * 4u) ? ldg_hint(p + chunk, pol) : make_uint4(0u, 0u, 0u, 0u);  // (zero words hold no marker)
      }
      unsigned cnt = 0;
#pragma unroll
      for (int i = 0; i < 4; i++) {
        const unsigned x0 = (lane & 3) ? v[i].x : (v[i].x & 0xFFFFFF00u);  // byte 0 of a block is the DC marker (chunk & 3 == lane & 3)
        cnt += __popc(ff_flags(x0)) + __popc(ff_flags(v[i].y)) + __popc(ff_flags(v[i].z)) + __popc(ff_flags(v[i].w));
      }
      cnt = __reduce_add_sync(0xFFFFFFFFu, cnt);
      if (lane == 0) asm volatile("st.volatile.global.u32 [%0], %1;\n" ::"l"(b.counts + t), "r"(0x80000000u | cnt) : "memory");
      sum += cnt;
    }
    if (lane == 0) {
      asm volatile("st.volatile.global.u32 [%0], %1;\n" ::"l"(b.agg + u), "r"(0x80000000u | sum) : "memory");
      const unsigned long long contrib = (1ull << 48) | (unsigned long long)sum;
      atomicAdd(b.S + (u >> 6), contrib);
      atomicAdd(b.T + (u >> 11), contrib);
    }
#ifdef DCTZ_WAIT_STATS
    n_units++;
#endif
  }
#ifdef DCTZ_WAIT_STATS
  if (lane == 0) { atomicAdd(&g_wait_stats[1], n_wait); atomicAdd(&g_wait_stats[2], n_units); }
#endif
}

// The decode warpgroup's tile sequence (advance) and extent source (load / finish) for decompress_tiles.  Units come from
// the decode ticket, the first one too (a statically assigned first unit could belong to a CTA that is not resident yet).
// Unit u is tiles [u * batch, (u + 1) * batch); a warp takes its units whole and in increasing order, so the extent of a
// unit's first tile is finished before those of its other tiles, and the super-group sums it has added up stay valid.
struct CountedExtents {
  struct Raw { unsigned c, k, u, a0, a1; unsigned long long s, t; };  // loaded values, untouched until finish()
  static __device__ __forceinline__ Raw none() {
    Raw r;
    r.c = 0x80000000u; r.k = 0; r.u = 0; r.a0 = r.a1 = 0x80000000u; r.s = r.t = 0ull;
    return r;
  }
  AheadBufs b;
  unsigned long long n_limit;
  unsigned *corrupt_flag, *counter;
  unsigned ntiles, batch, nunits;
  unsigned pend, next, end;          // sequence: lane 0 holds the ticket requested for the unit after [next, end)
  unsigned long long u_base;         // first outlier of the unit whose extents are being finished
  unsigned t_upto;                   // super-groups [0, t_upto) are complete and summed in t_sum
  unsigned long long t_sum;
#ifdef DCTZ_WAIT_STATS
  unsigned long long n_spin;
#endif

  __device__ __forceinline__ void init(unsigned ntiles_, unsigned batch_, AheadBufs bufs, unsigned long long n_limit_, unsigned *corrupt_flag_,
                                       unsigned *ticket_counter, int lane) {
    b = bufs; ntiles = ntiles_; batch = batch_; nunits = (ntiles_ + batch_ - 1) / batch_;
    n_limit = n_limit_; corrupt_flag = corrupt_flag_; counter = ticket_counter;
    u_base = 0ull; t_upto = 0; t_sum = 0ull;
#ifdef DCTZ_WAIT_STATS
    n_spin = 0;
#endif
    pend = 0;
    if (lane == 0) pend = ticket_next(counter);
    next = end = 0;
  }
  __device__ __forceinline__ unsigned advance(int lane) {  // warp-uniform: the next tile to process
    if (next >= end) {
      const unsigned start = __shfl_sync(0xFFFFFFFFu, pin_here(pend), 0) * batch;
      if (start >= ntiles) { next = end = ntiles; return 0xFFFFFFFFu; }  // (no further ticket)
      if (lane == 0) pend = ticket_next(counter);
      next = start;
      end = start + batch;
    }
    if (next >= ntiles) return 0xFFFFFFFFu;
    return next++;
  }
  // what unit u's offset needs: lanes hold the units of its group below it, the groups of its super-group below its
  // group, and a window of the not yet summed super-groups below its super-group
  __device__ __forceinline__ void load_lookback(Raw &r, unsigned u, unsigned w0, int lane) const {
    const unsigned g = u >> 6, h = u >> 11;
    const unsigned i0 = (g << 6) + (unsigned)lane, i1 = i0 + 32u, gi = (h << 5) + (unsigned)lane, wi = w0 + (unsigned)lane;
    r.a0 = (i0 < u) ? ld_volatile(b.agg + i0) : 0x80000000u;
    r.a1 = (i1 < u) ? ld_volatile(b.agg + i1) : 0x80000000u;
    r.s = (gi < g) ? ld_volatile(b.S + gi) : 0ull;
    r.t = (wi < h) ? ld_volatile(b.T + wi) : 0ull;
  }
  __device__ __forceinline__ bool lookback_complete(const Raw &r, unsigned u, unsigned w0, int lane) const {
    const unsigned g = u >> 6, h = u >> 11;
    const unsigned gi = (h << 5) + (unsigned)lane, wi = w0 + (unsigned)lane;
    bool ok = (r.a0 >> 31) && (r.a1 >> 31);
    if (gi < g) { const unsigned want = nunits - (gi << 6) < 64u ? nunits - (gi << 6) : 64u; ok = ok && (unsigned)(r.s >> 48) == want; }
    if (wi < h) { const unsigned want = nunits - (wi << 11) < 2048u ? nunits - (wi << 11) : 2048u; ok = ok && (unsigned)(r.t >> 48) == want; }
    return __all_sync(0xFFFFFFFFu, ok);
  }
  __device__ __forceinline__ void load_counts(Raw &r, int lane) const {  // lanes < k: earlier tiles of the unit; lane k: the tile
    r.c = ((unsigned)lane <= r.k) ? ld_volatile(b.counts + r.u * batch + (unsigned)lane) : 0x80000000u;
  }
  __device__ __forceinline__ Raw load(unsigned t, int lane) const {
    Raw r = none();
    r.u = t / batch;
    r.k = t - r.u * batch;
    load_counts(r, lane);
    if (r.k == 0) load_lookback(r, r.u, t_upto, lane);  // the tile starts a unit: the unit's offset is looked up
    return r;
  }
  __device__ __forceinline__ Extent finish(Raw &r, int lane) {
    r.c = pin_here(r.c);  // first use of the loaded values: here, at the end of the iteration
    if (r.k == 0) {
      const unsigned u = r.u, h = u >> 11;
      r.a0 = pin_here(r.a0);
      for (;;) {  // (complete at the first look unless the counters have fallen behind)
        while (!lookback_complete(r, u, t_upto, lane)) load_lookback(r, u, t_upto, lane);
        if (t_upto + 32u >= h) break;
        t_sum += warp_sum_u64(r.t & AHEAD_LOW48);  // more than 32 new super-groups (a very large slab's first look): next window
        t_upto += 32u;
        load_lookback(r, u, t_upto, lane);
      }
      t_sum += warp_sum_u64(r.t & AHEAD_LOW48);
      t_upto = h;
      const unsigned within = __reduce_add_sync(0xFFFFFFFFu, (r.a0 & 0x7FFFFFFFu) + (r.a1 & 0x7FFFFFFFu));
      u_base = t_sum + warp_sum_u64(r.s & AHEAD_LOW48) + within;
    }
    while (!__all_sync(0xFFFFFFFFu, r.c >> 31)) {  // a count not yet published
#ifdef DCTZ_WAIT_STATS
      n_spin++;
#endif
      load_counts(r, lane);
    }
    Extent e;
    e.total = __shfl_sync(0xFFFFFFFFu, r.c, (int)r.k) & 0x7FFFFFFFu;
    e.base = u_base + __reduce_add_sync(0xFFFFFFFFu, ((unsigned)lane < r.k) ? (r.c & 0x7FFFFFFFu) : 0u);
    e.bad = e.base + e.total > n_limit;
    if (e.bad) { e.total = 0u; *corrupt_flag = 1u; }
    return e;
  }
};

// The tile loop of the decompress kernels: one warp, tiles handed out by `seq`, outlier extents by `ext`.
template <typename T, bool QT, class Seq, class Ext>
__device__ __forceinline__ void decompress_tiles(const uint8_t *__restrict__ bins, const float *__restrict__ dc_in, const float *__restrict__ ac_in,
                                                 unsigned long long nblk_full, T sf, const QtConsts<T> &qk, const CUtensorMap *tmap_out,
                                                 unsigned long long n_ac /* end of the readable part of AC_exact */, int dc_aligned16,
                                                 unsigned char *wsm, unsigned mb, const T *center, const T *s_qt, Seq &seq, Ext &ext,
                                                 int lane, unsigned &phase, int l2_hints = 0) {
  typedef typename ArithOf<T, QT>::type A;  // double: constants from the table in QT mode, literals in EC mode (same-box A/B, common.cuh)
  typedef DecompressCfg<T, QT> Cfg;
  typedef WarpTile<T> L;
  constexpr bool WIDE = (sizeof(T) == 8);
  constexpr unsigned FAST_MAX = (unsigned)Cfg::FAST_MAX;
  float *stage = reinterpret_cast<float *>(wsm + Cfg::OFF_STAGE);
  unsigned char *binbuf = wsm + Cfg::OFF_BINS;
  float *dcbuf = reinterpret_cast<float *>(wsm + Cfg::OFF_DC);
  const unsigned ntiles = (unsigned)((nblk_full + WTILE - 1) / WTILE);
  // l2_hints: bit 0 = the reconstruction is stored with evict_first, bit 1 = the bin ids are fetched with evict_first (both
  // so that lines somebody still needs -- the bin ids the count-ahead path has touched -- outlive the streaming traffic)
  const unsigned long long pol_first = policy_evict_first();
  auto rows_of = [&](unsigned t) -> unsigned {
    const unsigned long long left = nblk_full - (unsigned long long)t * WTILE;
    return left < (unsigned long long)WTILE ? (unsigned)left : (unsigned)WTILE;
  };
  // Stage layout: the stage mirrors the 16-byte granules of AC_exact that hold the tile's run: outlier i lives at
  // stage[fofs + lead + i], lead = (elements between the previous 16-byte boundary and the run's first element), so ONE
  // bulk copy of the aligned superset of the run fetches everything (up to 3 foreign floats on either side are copied
  // and ignored).  Only where the superset would leave the array -- before AC_exact[0] when the array itself is not
  // 16-byte aligned, or past the last outlier of the field -- the copy is clipped to whole granules inside the array
  // and the at most 3 + 3 ragged elements are fetched by plain loads.
  struct Plan { unsigned lead, kend, fofs; bool fits, prefetch; };  // warp-uniform, a function of the extent alone
  auto plan_of = [&](const Extent &e) -> Plan {
    Plan p;
    p.lead = (unsigned)(((unsigned long long)(uintptr_t)(ac_in + e.base) & 15ull) >> 2);
    p.kend = p.lead + e.total;
    p.fits = p.kend <= FAST_MAX;
    p.prefetch = e.total != 0u && (WIDE || p.fits);
    p.fofs = (WIDE && p.fits) ? FAST_MAX : 0u;  // double: raw floats in the upper half, expanded downwards
    return p;
  };
  // The ragged elements are LOADED when the tile's copies are issued and STORED to the stage only at the end of the
  // iteration (park_ragged), so the global-load latency hides behind the inverse transform.
  struct Ragged { float v; int idx; };
  auto issue_tile = [&](unsigned t, const Extent &e) -> Ragged {  // bin ids (2 KB) + DC (128 B) [+ outliers] of tile t
    const unsigned rows = rows_of(t);
    // the DC slice is 4*rows bytes: bulk copies need a multiple of 16 bytes at a 16-byte aligned address, so partial
    // tiles -- and slabs whose DC pointer is only float-aligned (a slice of a concatenated DC array) -- load DC directly
    const bool dc_bulk = (rows == WTILE) && dc_aligned16;
    const Plan pl = plan_of(e);
    unsigned k0 = 0, k1 = 0;  // stage indices: the bulk copy covers [k0, k1), the run is [lead, kend)
    if (pl.prefetch) {
      k0 = (e.base < (unsigned long long)pl.lead) ? 4u : 0u;                                 // would start before AC_exact[0]
      k1 = (pl.kend + 3u) & ~3u;
      if (e.base + (unsigned long long)(k1 - pl.lead) > n_ac) k1 = pl.kend & ~3u;            // would end past the last outlier
      if (k1 < k0) k1 = k0;
    }
    if (lane == 0) {
      mbar_expect_tx(mb, rows * BLK + (dc_bulk ? WTILE * 4 : 0) + (k1 - k0) * 4u);
      if (l2_hints & 2) bulk_g2s_hint(smem_u32(binbuf), bins + (unsigned long long)t * WTILE * BLK, rows * BLK, mb, pol_first);
      else bulk_g2s(smem_u32(binbuf), bins + (unsigned long long)t * WTILE * BLK, rows * BLK, mb);
      if (dc_bulk) bulk_g2s(smem_u32(dcbuf), dc_in + (unsigned long long)t * WTILE, WTILE * 4, mb);
      if (k1 > k0) bulk_g2s(smem_u32(stage) + (pl.fofs + k0) * 4u, ac_in + e.base + k0 - pl.lead, (k1 - k0) * 4u, mb);
    }
    Ragged r;
    r.v = 0.f; r.idx = -1;
    if (pl.prefetch) {
      const unsigned kh = pl.lead + (unsigned)lane;      // head: stage indices lead .. k0-1 (k0 = 4 only)
      const unsigned kt = (k1 > pl.lead ? k1 : pl.lead) + (unsigned)(lane - 8);  // tail: stage indices max(k1, lead) .. kend-1 (at most 3), lanes 8..10
      if (kh < k0 && kh < pl.kend) { r.idx = (int)(pl.fofs + kh); r.v = __ldg(ac_in + e.base + lane); }
      else if (lane >= 8 && lane < 12 && kt < pl.kend) { r.idx = (int)(pl.fofs + kt); r.v = __ldg(ac_in + e.base + (kt - pl.lead)); }
    }
    return r;
  };
  auto park_ragged = [&](const Ragged &r) { if (r.idx >= 0) stage[r.idx] = r.v; };
  // Tiles are known three ahead (there is no ordering between tiles): `nxt` and its outlier extent are known when an
  // iteration starts, so all of its loads are issued as soon as the current tile's inputs are consumed; the counts
  // behind the extent of the tile after it (`nn`) are loaded at the top of the iteration and reduced at its end.
  unsigned cur = seq.advance(lane);
  unsigned nxt = seq.advance(lane);
  unsigned nn = seq.advance(lane);
  Extent ext_cur, ext_nxt;
  ext_cur.base = 0; ext_cur.total = 0; ext_cur.bad = false;
  ext_nxt = ext_cur;
  if (cur < ntiles) { typename Ext::Raw r0 = ext.load(cur, lane); ext_cur = ext.finish(r0, lane); park_ragged(issue_tile(cur, ext_cur)); }
  if (nxt < ntiles) { typename Ext::Raw r1 = ext.load(nxt, lane); ext_nxt = ext.finish(r1, lane); }

  while (cur < ntiles) {
    typename Ext::Raw raw_nn = Ext::none();
    if (nn < ntiles) raw_nn = ext.load(nn, lane);  // loads in flight for the whole iteration
    const unsigned rows = rows_of(cur);
    const unsigned long long blk = (unsigned long long)cur * WTILE + lane;
    const bool active = (unsigned)lane < rows;
    mbar_wait(mb, phase);
    phase ^= 1u;
    __syncwarp();  // the ragged outlier elements were stored by other lanes
    unsigned w[16];
    {
      const uint4 *bp = reinterpret_cast<const uint4 *>(binbuf + lane * BLK);
#pragma unroll
      for (int q = 0; q < 4; q++) {
        const uint4 v = bp[q];
        w[4 * q] = v.x; w[4 * q + 1] = v.y; w[4 * q + 2] = v.z; w[4 * q + 3] = v.w;
      }
    }
    float dcv = (rows == WTILE && dc_aligned16) ? dcbuf[lane] : (active ? __ldg(dc_in + blk) : 0.f);
    if (!active) {
#pragma unroll
      for (int q = 0; q < 16; q++) w[q] = 0;
    }
    unsigned cnt = 0;
#pragma unroll
    for (int q = 0; q < 16; q++) cnt += __popc(ff_flags(q == 0 ? (w[0] & 0xFFFFFF00u) : w[q]));  // position 0 is the DC marker
    const unsigned my_off = warp_inclusive_scan(cnt, lane) - cnt;
    const Plan pl = plan_of(ext_cur);

    // ---- the tile's outliers: finished coefficients at rdy[0..total) (`ready`), or raw floats at raw[0..total) ----
    bool ready = false;  // warp-uniform
    const T *rdy = reinterpret_cast<const T *>(stage);
    const float *raw = stage + pl.fofs + pl.lead;
    if (!WIDE && ext_cur.total != 0u && !pl.fits) {
      // float, more than FAST_MAX outliers: nothing was prefetched; load them now (coalesced) into the tile buffer
      if (lane == 0) bulk_wait_read();  // the previous tile's output has left shared memory
      __syncwarp();
      float *tb = reinterpret_cast<float *>(wsm);
      if (QT) {
        for (unsigned i = lane; i < ext_cur.total; i += 32) tb[i] = __ldg(ac_in + ext_cur.base + i);
        raw = tb;
      } else {
        for (unsigned i = lane; i < ext_cur.total; i += 32) tb[i] = __fmul_rn(__ldg(ac_in + ext_cur.base + i), (float)sf);
        rdy = reinterpret_cast<const T *>(tb);
        ready = true;
      }
      __syncwarp();
    } else if (ext_cur.total != 0u && pl.fits) {
      // QT: an outlier is rescaled with the table entry of its coefficient position (dctz-decomp-lib.c:404-409,
      // 450-454).  Every lane first notes the positions of its block's outliers, in order, in the bin-id buffer
      // (every lane holds its bin ids in registers by now; the buffer is dead until the next tile's copy), so that
      // the cooperative pass below finds outlier i of the tile next to its position.
      uint8_t *jpos = binbuf;
      if constexpr (QT) {
        __syncwarp();  // all lanes have read their bin ids
        unsigned p = my_off;
#pragma unroll
        for (int j = 1; j < BLK; j++) {
          if (((w[j >> 2] >> (8 * (j & 3))) & 0xFFu) == 255u) jpos[p++] = (uint8_t)j;
        }
        __syncwarp();
      }
      if constexpr (WIDE) {
        // in-place expansion float -> double: batch b reads floats [32b, 32b+32) of the upper half and writes doubles
        // [32b, 32b+32) from the bottom; a write only ever lands on floats of batches <= b (8i+8 <= 4096+4(32b+32)
        // for i < 32b+32 <= 1024), which every lane has read once the batch's __syncwarp is passed.
        // (four batches per barrier: the same argument holds for the union of the batches)
        T *dst = reinterpret_cast<T *>(stage);
        for (unsigned i0 = 0; i0 < ext_cur.total; i0 += 128) {
          float a[4];
#pragma unroll
          for (int k = 0; k < 4; k++) { const unsigned i = i0 + 32 * k + lane; a[k] = (i < ext_cur.total) ? raw[i] : 0.f; }
          __syncwarp();
#pragma unroll
          for (int k = 0; k < 4; k++) {
            const unsigned i = i0 + 32 * k + lane;
            if (i < ext_cur.total) dst[i] = outlier_coefficient<T, QT>(a[k], QT ? s_qt[jpos[i]] : (T)0, qk, sf);
          }
        }
      } else {
        float *f = stage + pl.lead;
        for (unsigned i = lane; i < ext_cur.total; i += 32) f[i] = outlier_coefficient<T, QT>(f[i], QT ? s_qt[jpos[i]] : (T)0, qk, sf);
        rdy = reinterpret_cast<const T *>(f);
      }
      fence_async_smem();  // the stage was written through the generic proxy; TMA writes it next
      __syncwarp();
      ready = true;
    }

    // ---- rebuild coefficients (dctz-decomp-lib.c:392-416), already multiplied by sf ----
    T x[BLK];
    x[0] = dc_coefficient<T>(dcv, sf);
    if (ready && ext_cur.total != 0) {
      // marker 255 -> next finished outlier of this block, anything else -> its bin centre: one load either way
      const unsigned center_s = smem_u32(center);
      unsigned spd = smem_u32(rdy) + my_off * (unsigned)sizeof(T) - 255u * (unsigned)sizeof(T) - center_s;
#pragma unroll
      for (int j = 1; j < BLK; j++) pick_coefficient(x[j], spd, id_offset<T>(w[j >> 2], j & 3), center_s);
    } else {
#pragma unroll
      for (int j = 1; j < BLK; j++)
        x[j] = *reinterpret_cast<const T *>(reinterpret_cast<const unsigned char *>(center) + id_offset<T>(w[j >> 2], j & 3));  // entry 255 is a dummy, fixed below
    }
    if (!ready && !ext_cur.bad && cnt != 0) {
      // eight coefficients at a time: the (predicated) stage loads first, the conversions after them, so the
      // shared-memory latency is paid once per group and not once per outlier
      unsigned p = my_off;
#pragma unroll
      for (int g = 0; g < 8; g++) {
        unsigned m0 = ff_bytes(w[2 * g]);
        const unsigned m1 = ff_bytes(w[2 * g + 1]);
        if (g == 0) m0 &= ~1u;  // the DC marker
        if (m0 | m1) {
          float a[8];
#pragma unroll
          for (int b = 0; b < 8; b++) {
            const bool hit = ((b < 4 ? m0 >> (8 * b) : m1 >> (8 * (b - 4))) & 1u) != 0u;
            a[b] = 0.f;
            if (hit) a[b] = raw[p++];  // :402-403
          }
#pragma unroll
          for (int b = 0; b < 8; b++) {
            const int j = 8 * g + b;
            const bool hit = ((b < 4 ? m0 >> (8 * b) : m1 >> (8 * (b - 4))) & 1u) != 0u;
            if (hit) x[j] = outlier_coefficient<T, QT>(a[b], QT ? s_qt[j] : (T)0, qk, sf);
          }
        }
      }
    }
    // bin ids, DC and the stage are consumed by every lane: their loads have COMPLETED (reads_have_landed), the next
    // tile's copies may overwrite the buffers
    unsigned probe = w[0] ^ w[15];
    if constexpr (sizeof(T) == 8) {
#pragma unroll
      for (int j = 0; j < BLK; j++) probe |= (unsigned)__double2hiint((double)x[j]) ^ (unsigned)__double2loint((double)x[j]);
    } else {
#pragma unroll
      for (int j = 0; j < BLK; j++) probe |= (unsigned)__float_as_int((float)x[j]);
    }
    Ragged rag;
    rag.v = 0.f; rag.idx = -1;
    __syncwarp();
    if (reads_have_landed(probe) && nxt < ntiles) rag = issue_tile(nxt, ext_nxt);  // overlaps the inverse transform and the stores

    // ---- orthonormal DCT-III (dct.c:115-205) ----
    dct64_inverse<A>(x);

    // ---- registers -> own row of the swizzled tile -> TMA tensor stores (rows beyond the field are clipped) ----
    if (lane == 0) bulk_wait_read();  // the previous tile's output has left shared memory
    __syncwarp();
#pragma unroll
    for (int q = 0; q < L::SLABS; q++) {
#pragma unroll
      for (int c = 0; c < 8; c++) {
        uint4 v;
        T *e = reinterpret_cast<T *>(&v);
#pragma unroll
        for (int k = 0; k < L::PER_CHUNK; k++) e[k] = x[(q * 8 + c) * L::PER_CHUNK + k];
        *reinterpret_cast<uint4 *>(wsm + L::chunk_offset(q, lane, c)) = v;
      }
    }
    fence_async_smem();
    __syncwarp();
    if (lane == 0) {
      if (l2_hints & 1) {
#pragma unroll
        for (int q = 0; q < L::SLABS; q++) tma_store_2d_hint(tmap_out, q * 128, (int)(cur * WTILE), smem_u32(wsm) + q * L::SLAB_BYTES, pol_first);
      } else {
#pragma unroll
        for (int q = 0; q < L::SLABS; q++) tma_store_2d(tmap_out, q * 128, (int)(cur * WTILE), smem_u32(wsm) + q * L::SLAB_BYTES);
      }
      bulk_commit();
    }
    park_ragged(rag);
    cur = nxt;
    ext_cur = ext_nxt;
    nxt = nn;
    ext_nxt = ext.finish(raw_nn, lane);
    nn = seq.advance(lane);
  }
}

// AHEAD = false: extents from the pre-pass (k_count_bins + k_scan_groups), `counts` are its per-tile counts.  AHEAD = true: no
// pre-pass, a count warpgroup publishes the counts while the decode warpgroup runs the tile loop (count_units /
// CountedExtents); `counts`, `unit_counts`, `group_prefix` and `chunk_prefix` then carry AheadBufs' counts / agg / S / T
// (zeroed by the host before the launch) and the last CTA writes the number of outliers the full blocks hold to
// `n_outliers_total` (the tail block's offset).
template <typename T, bool QT, bool AHEAD>
__global__ void __launch_bounds__(AHEAD ? SplitCfg::THREADS : DecompressCfg<T, QT>::THREADS, AHEAD ? SplitCfg::CTAS_PER_SM : DecompressCfg<T, QT>::CTAS_PER_SM)
k_decompress(const uint8_t *__restrict__ bins, const float *__restrict__ dc_in, const float *__restrict__ ac_in,
             const T *__restrict__ qtable, unsigned long long nblk_full, T bin_width, T sf, QtConsts<T> qk,
             const __grid_constant__ CUtensorMap tmap_out, unsigned *counts, unsigned *unit_counts,
             unsigned long long *group_prefix, unsigned long long *chunk_prefix,
             unsigned long long *n_outliers_total, unsigned long long n_limit, TileControl *ctl,
             unsigned *corrupt_flag, int dc_aligned16, unsigned batch, int l2_hints) {
  typedef DecompressCfg<T, QT> Cfg;
  constexpr int THREADS = AHEAD ? SplitCfg::THREADS : Cfg::THREADS;
  extern __shared__ unsigned char smem_raw[];
  __shared__ __align__(8) unsigned long long s_mbar[Cfg::WARPS];
  __shared__ T s_qt[QT ? BLK : 1];

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool decoder = warp < Cfg::WARPS;  // AHEAD: warps Cfg::WARPS.. are the count warpgroup
  unsigned char *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  __shared__ __align__(16) T center[256];  // static: its address is an immediate of the lookups
  unsigned char *wsm = smem + warp * Cfg::WARP_BYTES;
  // (decompress_tiles) EC: a tile's outliers are turned into coefficients (converted to T, times sf) ONCE, cooperatively and
  // conflict-free, before the lanes pick them up -- the per-coefficient work of a lane is then a select between two
  // shared-memory addresses (pick_coefficient).  double: the converted values need 8 bytes each, so the prefetched
  // floats are put in the upper half of the stage and expanded in place from the bottom.  Tiles with more than
  // FAST_MAX outliers (double) and QT tiles (whose outliers are rescaled with a per-position table entry,
  // dctz-decomp-lib.c:404-409) take the per-lane conversion path.
  const unsigned mb = smem_u32(&s_mbar[decoder ? warp : 0]);

  // bin centres: gen_bins / gen_bins_f (binning.c:19-22, 39-42): centre = (int multiple) * bin_width.  The de-scale
  // (x * sf, dctz-decomp-lib.c:494-511) is folded into the coefficients -- the inverse transform is linear, the
  // result moves by ~1 ulp -- so the table holds centre * sf.
  for (int i = threadIdx.x; i < 256; i += THREADS) center[i] = center_coefficient<T>((unsigned)i, bin_width, sf);
  if (QT && threadIdx.x < BLK) s_qt[threadIdx.x] = qtable[threadIdx.x];
  if (decoder && lane == 0) { mbar_init(mb, 1); fence_mbar_init(); }
  __syncthreads();  // the only CTA-wide barrier before the epilogue

  unsigned phase = 0;
  const unsigned ntiles = (unsigned)((nblk_full + WTILE - 1) / WTILE);
  if constexpr (AHEAD) {
    AheadBufs ab;
    ab.counts = counts; ab.agg = unit_counts; ab.S = group_prefix; ab.T = chunk_prefix;
    const unsigned nunits = (ntiles + batch - 1) / batch;
    if (!decoder) {
      setmaxnreg_dec<SplitCfg::COUNT_REGS>();
      count_units(bins, nblk_full, ntiles, batch, nunits, ab, &ctl->count_ticket, &ctl->ticket, lane);
    } else {
      setmaxnreg_inc<SplitCfg::DECODE_REGS>();
      CountedExtents ce;
      ce.init(ntiles, batch, ab, n_limit, corrupt_flag, &ctl->ticket, lane);
      decompress_tiles<T, QT>(bins, dc_in, ac_in, nblk_full, sf, qk, &tmap_out, n_limit, dc_aligned16, wsm, mb, center, s_qt, ce, ce, lane, phase,
                              l2_hints);
      bulk_wait_all();
      if (lane == 0) (void)pin_here(ce.pend);  // (as below)
#ifdef DCTZ_WAIT_STATS
      if (lane == 0) atomicAdd(&g_wait_stats[0], ce.n_spin);
#endif
    }
  } else {
    const unsigned long long n_scan = __ldg(n_outliers_total);
    ScannedExtents ext;
    ext.counts = counts; ext.group_prefix = group_prefix; ext.chunk_prefix = chunk_prefix; ext.n_limit = n_limit; ext.corrupt_flag = corrupt_flag;
    TileSeq seq;
    // l2_hints bit 2: from the last tile down -- what the pre-pass read last (with evict_last) is what L2 still holds
    seq.init(&ctl->ticket, blockIdx.x * Cfg::WARPS + warp, gridDim.x * Cfg::WARPS, batch, lane, (l2_hints & 4) ? ntiles - 1u : 0u);
    decompress_tiles<T, QT>(bins, dc_in, ac_in, nblk_full, sf, qk, &tmap_out, n_scan < n_limit ? n_scan : n_limit, dc_aligned16, wsm, mb, center,
                            s_qt, seq, ext, lane, phase, l2_hints);
    bulk_wait_all();
    // every warp still has one look-ahead ticket request outstanding (TileSeq::advance): its result is consumed here, so
    // the increment has been performed before this thread's fence and therefore before the last CTA resets the counter
    if (lane == 0) (void)pin_here(seq.pend);
  }
  __threadfence();
  __syncthreads();
  __shared__ bool s_last;
  if (threadIdx.x == 0) {
    const unsigned prev = atomicAdd(&ctl->done, 1u);
    s_last = (prev == gridDim.x - 1);
    if (s_last) { ctl->ticket = 0u; ctl->count_ticket = 0u; ctl->done = 0u; }
  }
  if constexpr (AHEAD) {
    __syncthreads();
    if (s_last && warp == 0) {  // every unit has been published: the full blocks' outliers = the sum over the super-groups
      __threadfence();
      const unsigned nunits = (ntiles + batch - 1) / batch, nsuper = (nunits + 2047u) >> 11;
      unsigned long long tot = 0ull;
      for (unsigned w = lane; w < nsuper; w += 32) tot += ld_volatile(chunk_prefix + w) & AHEAD_LOW48;
      tot = warp_sum_u64(tot);
      if (lane == 0) *n_outliers_total = tot;
    }
  }
}

// Partial last block of the decompress path.
template <typename T, bool QT>
__global__ void __launch_bounds__(32) k_tail_decompress(const uint8_t *__restrict__ bins, const float *__restrict__ dc_in,
                                                        const float *__restrict__ ac_in, const T *__restrict__ qtable,
                                                        int rem, unsigned long long blk_index, T bin_width, T sf,
                                                        QtConsts<T> qk, T *out, const unsigned long long *n_consumed,
                                                        unsigned long long pos0_if_no_full_blocks, unsigned long long n_limit,
                                                        unsigned *corrupt_flag) {
  __shared__ double cs[BLK];
  const int lane = threadIdx.x;
  const unsigned long long base = n_consumed ? *n_consumed : pos0_if_no_full_blocks;
  tail_block_decode<T, QT>(bins, dc_in, ac_in, qtable, rem, blk_index, bin_width, sf, qk, base, n_limit, [&] { *corrupt_flag = 1u; },
                           [&](int n, T v) { out[blk_index * BLK + n] = v; }, cs, lane);
}

// ------------------------------------------------------------------------------------------
// Small utility kernels
// ------------------------------------------------------------------------------------------
// x <- x / sf (IEEE division; dctz-comp-lib.c:193-216) or x <- x * sf (dctz-test.c:186-210), 128-bit accesses, four
// independent vectors in flight per thread; the ragged head/tail around the 16-byte-aligned body is done by CTA 0.
template <typename T>
__global__ void __launch_bounds__(256) k_scale(T *x, size_t n, T sf, int multiply) {
  constexpr int VEC = 16 / (int)sizeof(T);
  const size_t head = ((16 - ((uintptr_t)x & 15)) & 15) / sizeof(T);  // elements before the first 16-byte boundary
  const size_t h = head < n ? head : n;
  uint4 *body = reinterpret_cast<uint4 *>(x + h);
  const size_t nvec = (n - h) / VEC;
  auto op = [&](T v) -> T { return multiply ? v * sf : v / sf; };  // IEEE mul / div (no fast-math, nothing to contract)
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += 4 * stride) {
    uint4 v[4];
#pragma unroll
    for (int u = 0; u < 4; u++) if (i + u * stride < nvec) v[u] = body[i + u * stride];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      if (i + u * stride < nvec) {
        T *e = reinterpret_cast<T *>(&v[u]);
#pragma unroll
        for (int q = 0; q < VEC; q++) e[q] = op(e[q]);
        body[i + u * stride] = v[u];
      }
    }
  }
  if (blockIdx.x == 0) {
    for (size_t k = threadIdx.x; k < h; k += blockDim.x) x[k] = op(x[k]);
    for (size_t k = h + nvec * VEC + threadIdx.x; k < n; k += blockDim.x) x[k] = op(x[k]);
  }
}

// ------------------------------------------------------------------------------------------
// Transform-only kernels on device buffers (dctz_gpu_dct64_dev): the butterfly-vs-DMMA comparison
// of BASELINE config[3].  Both are persistent and warp-autonomous with the same TMA tile movement as
// K2/K3 (read 8 B + write 8 B per element), so the only difference is the arithmetic:
//   k_dct64_tile      one block per lane, generated 592-op flow graph on the FP64 vector pipe;
//   k_dct64_dmma      matrix form Y = D * X on the FP64 tensor pipe: mma.sync.m8n8k4.f64, 8 blocks per
//                     MMA column tile, 64x64 matrix = 8 m-tiles x 16 k-steps = 128 DMMA per 8 blocks
//                     (64 FMA per element instead of 9.25 operations).
// ------------------------------------------------------------------------------------------
template <typename T> struct DctOnlyCfg {
  static constexpr int WARPS = 4;
  static constexpr int THREADS = WARPS * 32;
  static constexpr int SMEM = WARPS * WarpTile<T>::BYTES + 1024;
};

template <typename T, bool INVERSE>
__global__ void __launch_bounds__(DctOnlyCfg<T>::THREADS, (sizeof(T) == 8 ? 2 : 3))
k_dct64_tile(const __grid_constant__ CUtensorMap tmap_in, const __grid_constant__ CUtensorMap tmap_out, unsigned long long nblk) {
  typedef typename ArithOf<T>::type A;
  typedef WarpTile<T> L;
  extern __shared__ unsigned char smem_raw[];
  __shared__ __align__(8) unsigned long long s_mbar[DctOnlyCfg<T>::WARPS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned char *wsm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u) + warp * L::BYTES;
  const unsigned mb = smem_u32(&s_mbar[warp]);
  const unsigned ntiles = (unsigned)((nblk + WTILE - 1) / WTILE);
  if (lane == 0) { mbar_init(mb, 1); fence_mbar_init(); }
  __syncthreads();
  unsigned phase = 0;
  for (unsigned t = blockIdx.x * DctOnlyCfg<T>::WARPS + warp; t < ntiles; t += gridDim.x * DctOnlyCfg<T>::WARPS) {
    if (lane == 0) {
      bulk_wait_read();  // the previous tile's stores have read the buffer
      mbar_expect_tx(mb, L::BYTES);
#pragma unroll
      for (int q = 0; q < L::SLABS; q++) tma_load_2d(smem_u32(wsm) + q * L::SLAB_BYTES, &tmap_in, q * 128, (int)(t * WTILE), mb);
    }
    mbar_wait(mb, phase);
    phase ^= 1u;
    T x[BLK];
#pragma unroll
    for (int q = 0; q < L::SLABS; q++) {
#pragma unroll
      for (int c = 0; c < 8; c++) {
        const uint4 v = *reinterpret_cast<const uint4 *>(wsm + L::chunk_offset(q, lane, c));
        const T *e = reinterpret_cast<const T *>(&v);
#pragma unroll
        for (int k = 0; k < L::PER_CHUNK; k++) x[(q * 8 + c) * L::PER_CHUNK + k] = e[k];
      }
    }
    if (INVERSE) dct64_inverse<A>(x); else dct64_forward<A>(x);
#pragma unroll
    for (int q = 0; q < L::SLABS; q++) {
#pragma unroll
      for (int c = 0; c < 8; c++) {
        uint4 v;
        T *e = reinterpret_cast<T *>(&v);
#pragma unroll
        for (int k = 0; k < L::PER_CHUNK; k++) e[k] = x[(q * 8 + c) * L::PER_CHUNK + k];
        *reinterpret_cast<uint4 *>(wsm + L::chunk_offset(q, lane, c)) = v;
      }
    }
    fence_async_smem();
    __syncwarp();
    if (lane == 0) {
#pragma unroll
      for (int q = 0; q < L::SLABS; q++) tma_store_2d(&tmap_out, q * 128, (int)(t * WTILE), smem_u32(wsm) + q * L::SLAB_BYTES);
      bulk_commit();
    }
  }
  bulk_wait_all();
}

__device__ __forceinline__ void dmma_m8n8k4(double &d0, double &d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};\n" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// dfrag: the 64x64 transform matrix pre-arranged as MMA A-fragments, dfrag[(i*16 + s)*32 + lane] =
// M[8i + lane/4][4s + lane%4], M = orthonormal DCT-II matrix (forward) or its transpose (inverse).
__global__ void __launch_bounds__(DctOnlyCfg<double>::THREADS, 2)
k_dct64_dmma(const __grid_constant__ CUtensorMap tmap_in, const __grid_constant__ CUtensorMap tmap_out, unsigned long long nblk,
             const double *__restrict__ dfrag) {
  typedef WarpTile<double> L;
  extern __shared__ unsigned char smem_raw[];
  __shared__ __align__(8) unsigned long long s_mbar[DctOnlyCfg<double>::WARPS];
  __shared__ __align__(16) double s_d[BLK * BLK];  // 32 KB, fragment order
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned char *wsm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u) + warp * L::BYTES;
  const unsigned mb = smem_u32(&s_mbar[warp]);
  const unsigned ntiles = (unsigned)((nblk + WTILE - 1) / WTILE);
  for (int i = threadIdx.x; i < BLK * BLK; i += blockDim.x) s_d[i] = dfrag[i];
  if (lane == 0) { mbar_init(mb, 1); fence_mbar_init(); }
  __syncthreads();
  unsigned phase = 0;
  const int brow = lane >> 2, kk = lane & 3;  // B fragment: block (column) brow of the group, sample 4s + kk
  for (unsigned t = blockIdx.x * DctOnlyCfg<double>::WARPS + warp; t < ntiles; t += gridDim.x * DctOnlyCfg<double>::WARPS) {
    if (lane == 0) {
      bulk_wait_read();
      mbar_expect_tx(mb, L::BYTES);
#pragma unroll
      for (int q = 0; q < L::SLABS; q++) tma_load_2d(smem_u32(wsm) + q * L::SLAB_BYTES, &tmap_in, q * 128, (int)(t * WTILE), mb);
    }
    mbar_wait(mb, phase);
    phase ^= 1u;
    double acc[4][8][2];
#pragma unroll
    for (int g = 0; g < 4; g++)
#pragma unroll
      for (int i = 0; i < 8; i++) acc[g][i][0] = acc[g][i][1] = 0.0;
#pragma unroll
    for (int s = 0; s < 16; s++) {
      double bf[4];
#pragma unroll
      for (int g = 0; g < 4; g++) {  // element n = 4s + kk of block 8g + brow: chunk (4s+kk)/2 of the row
        const int n = 4 * s + kk, c = n >> 1, r = 8 * g + brow;
        bf[g] = *reinterpret_cast<const double *>(wsm + L::chunk_offset(c >> 3, r, c & 7) + (n & 1) * 8);
      }
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const double af = s_d[(i * 16 + s) * 32 + lane];
#pragma unroll
        for (int g = 0; g < 4; g++) dmma_m8n8k4(acc[g][i][0], acc[g][i][1], af, bf[g]);
      }
    }
    __syncwarp();  // every lane has consumed the input tile
#pragma unroll
    for (int g = 0; g < 4; g++)
#pragma unroll
      for (int i = 0; i < 8; i++)
#pragma unroll
        for (int e = 0; e < 2; e++) {  // C fragment: row k = 8i + lane/4, column (block) 2*(lane%4) + e
          const int k = 8 * i + brow, c = k >> 1, r = 8 * g + 2 * kk + e;
          *reinterpret_cast<double *>(wsm + L::chunk_offset(c >> 3, r, c & 7) + (k & 1) * 8) = acc[g][i][e];
        }
    fence_async_smem();
    __syncwarp();
    if (lane == 0) {
#pragma unroll
      for (int q = 0; q < L::SLABS; q++) tma_store_2d(&tmap_out, q * 128, (int)(t * WTILE), smem_u32(wsm) + q * L::SLAB_BYTES);
      bulk_commit();
    }
  }
  bulk_wait_all();
}

// The matrix form with the even/odd split: x -> (s, d) = (x[i] + x[63-i], x[i] - x[63-i]), i < 32; the even coefficients are
// a 32x32 matrix times s, the odd ones a 32x32 matrix times d (the rows of the DCT-II matrix are symmetric / antisymmetric
// about the middle): 64 instead of 128 flop per element, 256 instead of 512 DMMA per tile.  Inverse: u = E^T X_even,
// v = O^T X_odd, x[i] = u[i] + v[i], x[63-i] = u[i] - v[i].
// dfrag2[m][(i*8 + s)*32 + lane] = M_m[8i + lane/4][4s + lane%4]; forward: M_0[k][i] = C[2k][i], M_1[k][i] = C[2k+1][i]
// (C = orthonormal DCT-II matrix); inverse: their transposes.
template <bool INVERSE>
__global__ void __launch_bounds__(DctOnlyCfg<double>::THREADS, 2)
k_dct64_dmma_split(const __grid_constant__ CUtensorMap tmap_in, const __grid_constant__ CUtensorMap tmap_out, unsigned long long nblk,
                   const double *__restrict__ dfrag2) {
  typedef WarpTile<double> L;
  extern __shared__ unsigned char smem_raw[];
  __shared__ __align__(8) unsigned long long s_mbar[DctOnlyCfg<double>::WARPS];
  __shared__ __align__(16) double s_d[2 * 32 * 32];  // 16 KB, fragment order
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned char *wsm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u) + warp * L::BYTES;
  const unsigned mb = smem_u32(&s_mbar[warp]);
  const unsigned ntiles = (unsigned)((nblk + WTILE - 1) / WTILE);
  for (int i = threadIdx.x; i < 2 * 32 * 32; i += blockDim.x) s_d[i] = dfrag2[i];
  if (lane == 0) { mbar_init(mb, 1); fence_mbar_init(); }
  __syncthreads();
  unsigned phase = 0;
  const int brow = lane >> 2, kk = lane & 3;
  auto elem = [&](int r, int n) -> double * {  // element n of block row r of the swizzled tile
    const int c = n >> 1;
    return reinterpret_cast<double *>(wsm + L::chunk_offset(c >> 3, r, c & 7) + (n & 1) * 8);
  };
  for (unsigned t = blockIdx.x * DctOnlyCfg<double>::WARPS + warp; t < ntiles; t += gridDim.x * DctOnlyCfg<double>::WARPS) {
    if (lane == 0) {
      bulk_wait_read();
      mbar_expect_tx(mb, L::BYTES);
#pragma unroll
      for (int q = 0; q < L::SLABS; q++) tma_load_2d(smem_u32(wsm) + q * L::SLAB_BYTES, &tmap_in, q * 128, (int)(t * WTILE), mb);
    }
    mbar_wait(mb, phase);
    phase ^= 1u;
    double a0[4][4][2], a1[4][4][2];  // [block group g][row group i][C fragment element]: matrix 0 / matrix 1
#pragma unroll
    for (int g = 0; g < 4; g++)
#pragma unroll
      for (int i = 0; i < 4; i++) a0[g][i][0] = a0[g][i][1] = a1[g][i][0] = a1[g][i][1] = 0.0;
#pragma unroll
    for (int s = 0; s < 8; s++) {
      double b0[4], b1[4];
#pragma unroll
      for (int g = 0; g < 4; g++) {
        const int n = 4 * s + kk, r = 8 * g + brow;
        if (INVERSE) {  // X[2n], X[2n+1]: one 16-byte chunk
          const double2 v = *reinterpret_cast<const double2 *>(elem(r, 2 * n));
          b0[g] = v.x; b1[g] = v.y;
        } else {
          const double p = *elem(r, n), q = *elem(r, BLK - 1 - n);
          b0[g] = __dadd_rn(p, q); b1[g] = __dsub_rn(p, q);
        }
      }
#pragma unroll
      for (int i = 0; i < 4; i++) {
        const double f0 = s_d[(i * 8 + s) * 32 + lane], f1 = s_d[1024 + (i * 8 + s) * 32 + lane];
#pragma unroll
        for (int g = 0; g < 4; g++) {
          dmma_m8n8k4(a0[g][i][0], a0[g][i][1], f0, b0[g]);
          dmma_m8n8k4(a1[g][i][0], a1[g][i][1], f1, b1[g]);
        }
      }
    }
    __syncwarp();  // every lane has consumed the input tile
#pragma unroll
    for (int g = 0; g < 4; g++)
#pragma unroll
      for (int i = 0; i < 4; i++)
#pragma unroll
        for (int e = 0; e < 2; e++) {  // C fragment: row m = 8i + lane/4, column (block) 2*(lane%4) + e
          const int m = 8 * i + brow, r = 8 * g + 2 * kk + e;
          if (INVERSE) {
            *elem(r, m) = __dadd_rn(a0[g][i][e], a1[g][i][e]);
            *elem(r, BLK - 1 - m) = __dsub_rn(a0[g][i][e], a1[g][i][e]);
          } else {
            *reinterpret_cast<double2 *>(elem(r, 2 * m)) = make_double2(a0[g][i][e], a1[g][i][e]);
          }
        }
    fence_async_smem();
    __syncwarp();
    if (lane == 0) {
#pragma unroll
      for (int q = 0; q < L::SLABS; q++) tma_store_2d(&tmap_out, q * 128, (int)(t * WTILE), smem_u32(wsm) + q * L::SLAB_BYTES);
      bulk_commit();
    }
  }
  bulk_wait_all();
}

// FP64 issue-rate probes (the denominators of the butterfly / DMMA comparison): kind 0 = independent DFMA chains on the vector
// pipe, kind 1 = mma.sync.m8n8k4.f64 on the tensor pipe.  `iters` x 32 operations per thread; the result keeps the
// compiler honest.
__global__ void __launch_bounds__(256) k_fp64_rate(int kind, int iters, double seed, double *sink) {
  double a[16];
#pragma unroll
  for (int i = 0; i < 16; i++) a[i] = seed + (double)(threadIdx.x + i);
  const double m = 1.0000001, c = 1e-9;
  if (kind == 0) {
    for (int it = 0; it < iters; it++) {
#pragma unroll
      for (int r = 0; r < 2; r++)
#pragma unroll
        for (int i = 0; i < 16; i++) a[i] = __fma_rn(a[i], m, c);
    }
  } else {
    for (int it = 0; it < iters; it++) {
#pragma unroll
      for (int r = 0; r < 4; r++)
#pragma unroll
        for (int i = 0; i < 8; i++) dmma_m8n8k4(a[2 * i], a[2 * i + 1], m, c);
    }
  }
  double t = 0.0;
#pragma unroll
  for (int i = 0; i < 16; i++) t += a[i];
  if (t == 123.456) sink[0] = t;
}

// DCT-only kernels behind dctz_gpu_dct_blocks (dct.h:17-27 equivalents)
constexpr int DCT_ONLY_THREADS = 128;
template <typename T, bool INVERSE>
__global__ void __launch_bounds__(DCT_ONLY_THREADS) k_dct64_blocks(const T *__restrict__ in, T *__restrict__ out, size_t nblocks) {
  typedef typename ArithOf<T>::type A;
  const size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nblocks) return;
  T x[BLK];
#pragma unroll
  for (int j = 0; j < BLK; j++) x[j] = in[b * BLK + j];
  if (INVERSE) dct64_inverse<A>(x); else dct64_forward<A>(x);
#pragma unroll
  for (int j = 0; j < BLK; j++) out[b * BLK + j] = x[j];
}
template <typename T, bool INVERSE>
__global__ void __launch_bounds__(32) k_dct_generic_blocks(const T *__restrict__ in, T *__restrict__ out, int dn) {
  __shared__ double xs[BLK];
  const int lane = threadIdx.x;
  const size_t b = blockIdx.x;
  for (int n = lane; n < dn; n += 32) xs[n] = (double)in[b * dn + n];
  __syncwarp();
  double r[2];
  if (INVERSE) generic_idct(xs, dn, lane, r); else generic_dct(xs, dn, lane, r);
  for (int h = 0; h < 2; h++) if (lane + 32 * h < dn) out[b * dn + lane + 32 * h] = (T)r[h];
}

// Quality metrics of a reconstruction against the original (util.c:54-104 calc_psnr): min, max of the
// original, max |a-b| and sum (a-b)^2 (float data: the difference is formed in float like util.c:88).
struct QualityPartial { double vmin, vmax, maxdiff, sumsq; };
template <typename T>
__global__ void __launch_bounds__(256) k_quality(const T *__restrict__ a, const T *__restrict__ b, size_t n, QualityPartial *partials,
                                                 unsigned *done_counter, QualityPartial *out) {
  constexpr int VEC = 16 / (int)sizeof(T);
  const double inf = __longlong_as_double(0x7FF0000000000000ll);
  double vmin = inf, vmax = -inf, md = 0.0, ss = 0.0;
  auto acc = [&](T va, T vb) {
    const double e = (double)(T)(va - vb);
    vmin = fmin(vmin, (double)va);
    vmax = fmax(vmax, (double)va);
    md = fmax(md, fabs(e));
    ss = __fma_rn(e, e, ss);
  };
  // 128-bit loads when both arrays are 16-byte aligned (two vectors of each in flight per thread), scalar otherwise
  const bool vec_ok = ((((uintptr_t)a) | ((uintptr_t)b)) & 15) == 0;
  const size_t nvec = vec_ok ? n / VEC : 0;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  const uint4 *a4 = reinterpret_cast<const uint4 *>(a), *b4 = reinterpret_cast<const uint4 *>(b);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += 2 * stride) {
    uint4 va[2], vb[2];
#pragma unroll
    for (int u = 0; u < 2; u++) if (i + u * stride < nvec) { va[u] = __ldg(a4 + i + u * stride); vb[u] = __ldg(b4 + i + u * stride); }
#pragma unroll
    for (int u = 0; u < 2; u++) {
      if (i + u * stride < nvec) {
        const T *ea = reinterpret_cast<const T *>(&va[u]), *eb = reinterpret_cast<const T *>(&vb[u]);
#pragma unroll
        for (int q = 0; q < VEC; q++) acc(ea[q], eb[q]);
      }
    }
  }
  for (size_t i = nvec * VEC + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) acc(a[i], b[i]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    vmin = fmin(vmin, __shfl_xor_sync(0xFFFFFFFFu, vmin, o));
    vmax = fmax(vmax, __shfl_xor_sync(0xFFFFFFFFu, vmax, o));
    md = fmax(md, __shfl_xor_sync(0xFFFFFFFFu, md, o));
    ss += __shfl_xor_sync(0xFFFFFFFFu, ss, o);
  }
  __shared__ QualityPartial sp[8];
  __shared__ bool is_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { sp[warp].vmin = vmin; sp[warp].vmax = vmax; sp[warp].maxdiff = md; sp[warp].sumsq = ss; }
  __syncthreads();
  if (threadIdx.x == 0) {
    QualityPartial r = sp[0];
    for (int w = 1; w < 8; w++) { r.vmin = fmin(r.vmin, sp[w].vmin); r.vmax = fmax(r.vmax, sp[w].vmax); r.maxdiff = fmax(r.maxdiff, sp[w].maxdiff); r.sumsq += sp[w].sumsq; }
    partials[blockIdx.x] = r;
    __threadfence();
    is_last = (atomicAdd(done_counter, 1u) == gridDim.x - 1);
  }
  __syncthreads();
  if (!is_last || threadIdx.x != 0) return;
  __threadfence();
  QualityPartial r = partials[0];  // index order: deterministic
  for (unsigned k = 1; k < gridDim.x; k++) {
    const QualityPartial q = partials[k];
    r.vmin = fmin(r.vmin, q.vmin); r.vmax = fmax(r.vmax, q.vmax); r.maxdiff = fmax(r.maxdiff, q.maxdiff); r.sumsq += q.sumsq;
  }
  *out = r;
  *done_counter = 0u;
}

// Exactly reproducible synthetic field (config C5, SURVEY.md §8d); host twin in dctz_b200/fields.py.
__device__ __forceinline__ unsigned hash32(unsigned h) {
  h ^= h >> 16; h *= 0x7FEB352Du; h ^= h >> 15; h *= 0x846CA68Bu; h ^= h >> 16;
  return h;
}
__global__ void __launch_bounds__(256) k_fill_hash_field(double *out, unsigned long long start, unsigned long long count,
                                                         unsigned dim, unsigned seed) {
  for (unsigned long long k = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; k < count;
       k += (unsigned long long)gridDim.x * blockDim.x) {
    const unsigned long long i = start + k;
    const double inv = 1.0 / (double)dim;  // dim is a power of two: exact
    const double x = (double)(i % dim) * inv, y = (double)((i / dim) % dim) * inv, z = (double)(i / ((unsigned long long)dim * dim)) * inv;
    const double tx = 1.0 - fabs(__dsub_rn(__dmul_rn(2.0, x), 1.0));
    const double ty = 1.0 - fabs(__dsub_rn(__dmul_rn(2.0, y), 1.0));
    const double tz = 1.0 - fabs(__dsub_rn(__dmul_rn(2.0, z), 1.0));
    const double h = (double)hash32((unsigned)(i ^ (unsigned long long)seed));
    const double noise = __dmul_rn(__dsub_rn(__dmul_rn(h, 1.0 / 4294967296.0), 0.5), 1.0 / 1024.0);
    double v = __dadd_rn(20.0, __dmul_rn(15.0, __dmul_rn(tx, ty)));
    v = __dadd_rn(v, __dmul_rn(5.0, tz));
    out[k] = __dadd_rn(v, noise);
  }
}

template <typename T>
__global__ void __launch_bounds__(256) k_selftest_division(T b, unsigned long long count, unsigned seed,
                                                           unsigned long long *mismatches) {
  const Divisor<T> d = make_divisor(b);
  unsigned bad = 0;
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < count;
       i += (unsigned long long)gridDim.x * blockDim.x) {
    const unsigned h1 = hash32((unsigned)i ^ seed), h2 = hash32((unsigned)(i >> 32) + h1 + 0x9E3779B9u);
    T a;
    if (sizeof(T) == 8) {
      // random sign and mantissa, exponent spread over [2^-40, 2^40)
      const unsigned long long mant = (((unsigned long long)h1 << 32) | h2) & 0xFFFFFFFFFFFFFull;
      const unsigned long long e = 1023ull - 40ull + (hash32(h2 ^ 0x51ED270Bu) % 80u);
      a = (T)__longlong_as_double((long long)(((unsigned long long)(h1 & 1u) << 63) | (e << 52) | mant));
    } else {
      const unsigned mant = h2 & 0x7FFFFFu;
      const unsigned e = 127u - 30u + (hash32(h2 ^ 0x51ED270Bu) % 60u);
      a = (T)__int_as_float((int)(((h1 & 1u) << 31) | (e << 23) | mant));
    }
    const T q1 = div_exact(a, d);
    const T q2 = a / b;
    if (q1 != q2) bad++;
  }
  if (bad) atomicAdd(mismatches, (unsigned long long)bad);
}

}  // namespace dctz
