// fused.cuh -- ONE launch per direction for fields that fit (or nearly fit) in L2.
//
// The BASELINE configs c1..c3 are 26..100 MB.  At that size the kernels of the streaming path (kernels.cuh) each run for
// 5-30 us and the 4-6 dependent launches of a direction cost as much as the work; the second read of the input (the
// scaling factor is a function of the whole field, util.c:28, so the data must be read twice) could come out of the
// 126 MB L2 instead of HBM.  These kernels are launched cooperatively (all CTAs co-resident) and separate their phases
// by grid barriers instead of kernel boundaries:
//
//   k_compress_fused    statistics | barrier | every CTA derives sf itself, compresses ITS OWN contiguous range of warp
//                       tiles (the range it has just read: from the top down, so that what the statistics pass read last
//                       -- and L2 still holds -- is transformed first) [QT: per-position maxima] | barrier | exclusive
//                       prefix of the CTA totals, gather (QT: rescale) of its own tiles' outliers into AC_exact
//   k_decompress_fused  outlier markers of its own tiles counted (the bin ids then sit in L2) | barrier | prefix of
//                       the CTA totals, dequantise + inverse DCT of its own tiles
//
// The tile loops are the ones of the streaming kernels (compress_tiles / decompress_tiles), so the results are the same
// bit for bit; only the tile order, the source of the outlier offsets and the launch count differ.
#pragma once
#include "kernels.cuh"

namespace dctz {

// Tiles [lo, hi) of a CTA, dealt to its warps round robin, upwards or from the top down.
struct RangeSeq {
  long long cur, lo, hi;
  int step;
  __device__ __forceinline__ void init_up(unsigned lo_, unsigned hi_, int warp, int nwarps) { lo = lo_; hi = hi_; cur = (long long)lo_ + warp; step = nwarps; }
  __device__ __forceinline__ void init_down(unsigned lo_, unsigned hi_, int warp, int nwarps) { lo = lo_; hi = hi_; cur = (long long)hi_ - 1 - warp; step = -nwarps; }
  __device__ __forceinline__ unsigned advance(int) {
    if (cur < lo || cur >= hi) return 0xFFFFFFFFu;
    const unsigned t = (unsigned)cur;
    cur += step;
    return t;
  }
};

__device__ __forceinline__ void cta_tile_range(unsigned ntiles, unsigned *t0, unsigned *t1) {
  const unsigned per = ntiles / gridDim.x, extra = ntiles % gridDim.x, b = blockIdx.x;
  *t0 = b * per + (b < extra ? b : extra);
  *t1 = *t0 + per + (b < extra ? 1u : 0u);
}

// All CTAs of a cooperative launch meet here.  `counter` only ever grows; the host hands every launch the value it
// will have reached before the launch's first barrier, so nothing has to be reset.
__device__ __forceinline__ void grid_barrier(unsigned long long *counter, unsigned long long target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long v;
    __threadfence();  // (cumulative: the CTA's writes, made visible to this thread by the barrier above)
    asm volatile("red.release.gpu.global.add.u64 [%0], 1;\n" ::"l"(counter) : "memory");
    do {
      asm volatile("ld.acquire.gpu.global.u64 %0, [%1];\n" : "=l"(v) : "l"(counter) : "memory");
    } while (v < target);
    __threadfence();
  }
  __syncthreads();
}
// a CTA that leaves early still owes the later barriers its arrivals (the host advances the base by the full count)
__device__ __forceinline__ void grid_arrive_only(unsigned long long *counter) {
  if (threadIdx.x == 0) asm volatile("red.release.gpu.global.add.u64 [%0], 1;\n" ::"l"(counter) : "memory");
}

// Phase timestamps (ns, %globaltimer) of every CTA of a single-launch kernel: dbg[8 * blockIdx.x + k]; read back by
// dctz_gpu_fused_phase_times (profiles/: where the microseconds of a small field go).
__device__ __forceinline__ void stamp(unsigned long long *dbg, int k) {
  if (dbg && threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(t));
    dbg[8 * blockIdx.x + k] = t;
  }
}

constexpr unsigned FUSED_MAX_TILES_PER_CTA = 2048;  // the per-CTA scratch (counts + offsets) lives in the idle tile buffers

// exclusive scan of s_cnt[0..nt) into s_off by warp 0; returns the total in every lane of warp 0
__device__ __forceinline__ unsigned long long warp0_scan_counts(const unsigned *s_cnt, unsigned *s_off, unsigned nt, int lane) {
  unsigned long long carry = 0;
  for (unsigned i0 = 0; i0 < nt; i0 += 32) {
    const unsigned i = i0 + (unsigned)lane;
    const unsigned c = i < nt ? s_cnt[i] : 0u;
    const unsigned incl = warp_inclusive_scan(c, lane);
    if (i < nt) s_off[i] = (unsigned)carry + incl - c;
    carry += __shfl_sync(0xFFFFFFFFu, incl, 31);
  }
  return carry;
}

// sum of cta_totals[0..blockIdx.x) and of all of them, by warp 0 (plain loads: written by other CTAs before the barrier)
__device__ __forceinline__ void warp0_cta_prefix(const unsigned long long *cta_totals, int lane, unsigned long long *base, unsigned long long *total) {
  unsigned long long b = 0, t = 0;
  for (unsigned i = lane; i < gridDim.x; i += 32) {
    const unsigned long long v = __ldcg(cta_totals + i);
    t += v;
    if (i < blockIdx.x) b += v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    b += __shfl_xor_sync(0xFFFFFFFFu, b, o);
    t += __shfl_xor_sync(0xFFFFFFFFu, t, o);
  }
  *base = b;
  *total = t;
}

// (Handing the tiles of the compress phase out by dynamic tickets instead -- counts then complete only after one more
// barrier -- was measured too: c1 41.5 us against 38.8, c3 75 against 71; only the 75 %-outlier case gained, 198 vs 207.)
// (A single-read variant of this kernel -- belief from a sample, true statistics gathered while compressing, as the
// streaming path does for large slabs -- was built and measured: c1 46 us against 39 us, c3 79 against 73.  At this size
// the second read comes out of L2 anyway, and the extra barrier-separated steps cost more than the read they save.)
constexpr int FUSED_COMPRESS_BARRIERS = 2;  // arrivals every CTA makes per launch (the host advances the base by this many per CTA)

template <typename T, bool QT>
__global__ void __launch_bounds__(CompressCfg<T, QT>::THREADS, CompressCfg<T, QT>::CTAS_PER_SM)
k_compress_fused(const __grid_constant__ CUtensorMap tmap_in, const T *__restrict__ in, unsigned long long nblk_full, QuantConsts<T> qc,
                 QtConsts<T> qk, uint8_t *__restrict__ bins, float *__restrict__ dc_out, unsigned *counts, float *ac_slots, T *raw_slots,
                 uint8_t *j_slots, float *__restrict__ ac_out, T *qtable_out, T *qtable_raw, typename BitsOf<T>::U *qmax_scratch,
                 StatPartial *partials, unsigned long long *cta_totals, SfTables tb, DevParams *params_out, Info *info,
                 unsigned long long *barrier, unsigned long long barrier_base, unsigned long long *dbg) {
  typedef CompressCfg<T, QT> Cfg;
  typedef typename BitsOf<T>::U U;
  constexpr int VEC = 16 / (int)sizeof(T);
  constexpr unsigned FULL = 0xFFFFFFFFu;
  extern __shared__ unsigned char smem_raw[];
  __shared__ __align__(8) unsigned long long s_mbar[Cfg::WARPS];
  __shared__ __align__(8) unsigned long long s_mbar2[Cfg::WARPS];  // statistics phase: the second half-buffer's barrier
  __shared__ DevParams s_params;
  __shared__ Info s_info;
  __shared__ StatPartial s_sp[Cfg::WARPS];
  __shared__ double s_stats3[3];
  __shared__ unsigned long long s_base, s_total;

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned char *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char *wsm = smem + warp * Cfg::WARP_BYTES;
  const unsigned mb = smem_u32(&s_mbar[warp]);
  const unsigned ntiles = (unsigned)((nblk_full + WTILE - 1) / WTILE);
  unsigned t0, t1;
  cta_tile_range(ntiles, &t0, &t1);
  const unsigned nt = t1 - t0;
  const unsigned mb2 = smem_u32(&s_mbar2[warp]);
  if (lane == 0) { mbar_init(mb, 1); mbar_init(mb2, 1); fence_mbar_init(); }
  if (QT && blockIdx.x == 0 && threadIdx.x < BLK) qmax_scratch[threadIdx.x] = 0;  // ordered before every use by the first barrier

  stamp(dbg, 0);
  // ---- phase 1: statistics of the CTA's own range (util.c:12-44).  Every warp streams chunks of HALF a tile buffer through
  //      the two halves of its own buffer with TMA bulk copies (one instruction per 8 / 4 KB instead of hundreds of LDG.128):
  //      while one half is looked at the other is on its way (one whole-buffer chunk at a time left the warp with nothing in
  //      flight while it computed: 2.7 round trips per warp set the phase's length) ----
  unsigned phase = 0;  // parity of the warp's mbarrier, carried on into the compress loop
  __syncthreads();     // (the mbarriers are initialised)
  {
    typedef WarpTile<T> L;
    constexpr unsigned CH = (unsigned)L::BYTES / 2;
    constexpr int NV = (int)(CH / 16 / 32);  // 128-bit vectors per lane and chunk
    const unsigned long long e0 = (unsigned long long)t0 * (WTILE * BLK);
    unsigned long long e1 = (unsigned long long)t1 * (WTILE * BLK);
    if (e1 > nblk_full * BLK) e1 = nblk_full * BLK;
    const unsigned char *src = reinterpret_cast<const unsigned char *>(in + e0);
    const unsigned long long bytes = (e1 - e0) * sizeof(T);  // a multiple of 64 elements: of 16 bytes
    const unsigned nchunks = (unsigned)((bytes + CH - 1) / CH);
    auto len_of = [&](unsigned c) -> unsigned { const unsigned long long left = bytes - (unsigned long long)c * CH; return left < CH ? (unsigned)left : CH; };
    auto issue = [&](unsigned c, unsigned half) {
      if (lane == 0) {
        const unsigned bar = half ? mb2 : mb;
        mbar_expect_tx(bar, len_of(c));
        bulk_g2s(smem_u32(wsm) + half * CH, src + (unsigned long long)c * CH, len_of(c), bar);
      }
    };
    unsigned long long umax = 0ull, umin = ~0ull;
    double s0 = 0.0, s1 = 0.0;
    unsigned c = (unsigned)warp, half = 0, phase2 = 0;
    if (c < nchunks) issue(c, 0);
    if (c + Cfg::WARPS < nchunks) issue(c + Cfg::WARPS, 1);
    while (c < nchunks) {
      if (half) { mbar_wait(mb2, phase2); phase2 ^= 1u; } else { mbar_wait(mb, phase); phase ^= 1u; }
      const unsigned nv = len_of(c) / 16;
      const uint4 *buf = reinterpret_cast<const uint4 *>(wsm + half * CH);
      unsigned probe = 0;
      uint4 v[NV];
#pragma unroll
      for (int u = 0; u < NV; u++) { const unsigned i = (unsigned)u * 32u + lane; v[u] = i < nv ? buf[i] : make_uint4(0u, 0u, 0u, 0u); }
#pragma unroll
      for (int u = 0; u < NV; u++) probe |= v[u].x ^ v[u].w;
      // the half is in registers (completed, not just issued): the chunk after the next one may overwrite it
      const unsigned cn = c + 2u * Cfg::WARPS;
      __syncwarp();
      if (reads_have_landed(probe) && cn < nchunks) issue(cn, half);
#pragma unroll
      for (int u = 0; u < NV; u++) {
        if ((unsigned)u * 32u + lane < nv) {
          const T *e = reinterpret_cast<const T *>(&v[u]);
#pragma unroll
          for (int q = 0; q < VEC; q++) {
            const unsigned long long a = AbsBits<T>::get(e[q]);
            umax = a > umax ? a : umax;
            umin = a < umin ? a : umin;
            if (q & 1) s1 += (double)e[q]; else s0 += (double)e[q];
          }
        }
      }
      c += Cfg::WARPS;
      half ^= 1u;
    }
    double sum = s0 + s1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long m1 = __shfl_xor_sync(FULL, umax, o), m2 = __shfl_xor_sync(FULL, umin, o);
      umax = m1 > umax ? m1 : umax;
      umin = m2 < umin ? m2 : umin;
      sum += __shfl_xor_sync(FULL, sum, o);
    }
    if (lane == 0) { s_sp[warp].umax = umax; s_sp[warp].umin = umin; s_sp[warp].sum = sum; }
    __syncthreads();
    if (threadIdx.x == 0) {
      StatPartial r = s_sp[0];
      for (int w = 1; w < Cfg::WARPS; w++) {
        r.umax = s_sp[w].umax > r.umax ? s_sp[w].umax : r.umax;
        r.umin = s_sp[w].umin < r.umin ? s_sp[w].umin : r.umin;
        r.sum += s_sp[w].sum;
      }
      partials[blockIdx.x] = r;
    }
  }
  stamp(dbg, 1);
  grid_barrier(barrier, barrier_base + gridDim.x);
  stamp(dbg, 2);

  // ---- phase 2: every CTA reduces the partials in index order (deterministic) and derives sf for itself ----
  if (warp == 0) {
    unsigned long long gmax = 0ull, gmin = ~0ull;
    double gsum = 0.0;
    for (unsigned b = lane; b < gridDim.x; b += 32) {
      StatPartial r;
      r.umax = __ldcg(&partials[b].umax); r.umin = __ldcg(&partials[b].umin); r.sum = __ldcg(&partials[b].sum);
      gmax = r.umax > gmax ? r.umax : gmax;
      gmin = r.umin < gmin ? r.umin : gmin;
      gsum += r.sum;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long m1 = __shfl_xor_sync(FULL, gmax, o), m2 = __shfl_xor_sync(FULL, gmin, o);
      gmax = m1 > gmax ? m1 : gmax;
      gmin = m2 < gmin ? m2 : gmin;
      gsum += __shfl_xor_sync(FULL, gsum, o);
    }
    if (lane == 0) {
      s_stats3[0] = AbsBits<T>::back(gmax);
      s_stats3[1] = AbsBits<T>::back(gmin);
      s_stats3[2] = gsum;
      finalize_params(s_stats3, 1, nblk_full * BLK, sizeof(T) == 8, (double)__ldg(in), 1, tb, &s_params, &s_info, nullptr);
    }
  }
  __syncthreads();
  if (blockIdx.x == 0 && threadIdx.x == 0) { *params_out = s_params; *info = s_info; }
  if (s_params.status != 0) {  // the same decision in every CTA: nobody is left waiting at the second barrier
    grid_arrive_only(barrier);
    return;
  }

  // ---- phase 3: scale + DCT + quantise + outliers of the CTA's own tiles, from the top down ----
  {
    RangeSeq seq;
    seq.init_down(t0, t1, warp, Cfg::WARPS);
    VerifyStat<T> vs;
    vs.tile_sums = nullptr; vs.tile_ext = nullptr;
    compress_tiles<T, QT, false>(&tmap_in, nblk_full, &s_params, qc, bins, dc_out, counts, ac_slots, raw_slots, j_slots, qtable_raw, wsm, mb, seq,
                                 lane, vs, phase);
  }
  bulk_wait_all();
  __syncthreads();  // the tile buffers are idle from here on: they hold the CTA's scratch now

  unsigned *s_cnt = reinterpret_cast<unsigned *>(smem);           // [FUSED_MAX_TILES_PER_CTA]
  unsigned *s_off = s_cnt + FUSED_MAX_TILES_PER_CTA;              // [FUSED_MAX_TILES_PER_CTA]
  U *s_max = reinterpret_cast<U *>(s_off + FUSED_MAX_TILES_PER_CTA);  // [BLK] QT per-position maxima of this CTA
  T *s_qt = reinterpret_cast<T *>(s_max + BLK);                   // [BLK] QT: the global table
  for (unsigned i = threadIdx.x; i < nt; i += Cfg::THREADS) s_cnt[i] = __ldcg(counts + t0 + i);
  if (QT && threadIdx.x < BLK) s_max[threadIdx.x] = 0;
  __syncthreads();
  if (warp == 0) {
    const unsigned long long tot = warp0_scan_counts(s_cnt, s_off, nt, lane);
    if (lane == 0) { s_total = tot; cta_totals[blockIdx.x] = tot; }
  }
  if constexpr (QT) {
    // per-position maxima of |coefficient| over the parked (unscaled) outliers (dctz-comp-lib.c:371-372, 396-397): a warp per
    // tile run, the CTA's maxima in shared memory, looked at before the atomic
    for (unsigned i = warp; i < nt; i += Cfg::WARPS) {
      const unsigned n = s_cnt[i];
      const unsigned long long src = (unsigned long long)(t0 + i) * TILE_SLOT;
      for (unsigned k0 = 0; k0 < n; k0 += 128u) {
        U a[4];
        unsigned jj[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const unsigned k = k0 + 32u * u + lane;
          a[u] = 0; jj[u] = 1u;
          if (k < n) { a[u] = BitsOf<T>::abs_bits(__ldcg(raw_slots + src + k)); jj[u] = __ldcg(j_slots + src + k); }
        }
#pragma unroll
        for (int u = 0; u < 4; u++)
          if (a[u] > *reinterpret_cast<volatile U *>(&s_max[jj[u]])) atomicMax(&s_max[jj[u]], a[u]);
      }
    }
    __syncthreads();
    if (threadIdx.x >= 1 && threadIdx.x < BLK && s_max[threadIdx.x] != 0) atomicMax(&qmax_scratch[threadIdx.x], s_max[threadIdx.x]);
  }
  stamp(dbg, 3);
  grid_barrier(barrier, barrier_base + 2ull * gridDim.x);
  stamp(dbg, 4);

  // ---- phase 4: the CTA's outliers go to their final place (dctz-comp-lib.c:478-544) ----
  if (warp == 0) {
    unsigned long long base, total;
    warp0_cta_prefix(cta_totals, lane, &base, &total);
    if (lane == 0) {
      s_base = base;
      if (blockIdx.x == gridDim.x - 1) info->n_outliers = total;
    }
  }
  if constexpr (QT) {
    if (threadIdx.x < BLK) {
      // max |c| / sf == max |c / sf| (exact division is monotone); entry 0 is the last block's (scaled) DC, :357/:359
      const Divisor<T> sfdiv = sf_divisor<T>(&s_params);
      T v;
      if (threadIdx.x == 0) v = *reinterpret_cast<volatile T *>(qtable_raw);
      else {
        const U bits = __ldcg(qmax_scratch + threadIdx.x);
        T raw;
        if constexpr (sizeof(T) == 8) raw = __longlong_as_double((long long)bits); else raw = __int_as_float((int)bits);
        v = div_exact(raw, sfdiv);
        if (blockIdx.x == 0) qtable_raw[threadIdx.x] = v;  // (read by nobody else: entry 0 is the only one the CTAs load)
        if (v < (T)1.0) v = (T)1.0;  // :450-461
      }
      s_qt[threadIdx.x] = v;
      if (blockIdx.x == 0) qtable_out[threadIdx.x] = v;
    }
  }
  __syncthreads();
  const unsigned long long base = s_base;
  unsigned dropped = 0;
  for (unsigned i = warp; i < nt; i += Cfg::WARPS) {
    const unsigned n = s_cnt[i];
    float *dst = ac_out + base + s_off[i];
    const unsigned long long slot = (unsigned long long)(t0 + i) * TILE_SLOT;
    if constexpr (QT) {
      const Divisor<T> sfdiv = sf_divisor<T>(&s_params);
      for (unsigned k0 = 0; k0 < n; k0 += 128u) {
        T r[4];
        unsigned jj[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const unsigned k = k0 + 32u * u + lane;
          r[u] = (T)0; jj[u] = 1u;
          if (k < n) { r[u] = __ldcg(raw_slots + slot + k); jj[u] = __ldcg(j_slots + slot + k); }
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const unsigned k = k0 + 32u * u + lane;
          if (k < n) {
            float o;
            if (!qt_rescale_one(div_exact(r[u], sfdiv), s_qt[jj[u]], qk, &o)) dropped++;
            dst[k] = o;
          }
        }
      }
    } else {
      const float *src = ac_slots + slot;
      for (unsigned k0 = 0; k0 < n; k0 += 256u) {
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; u++) { const unsigned k = k0 + 32u * u + lane; v[u] = (k < n) ? __ldcg(src + k) : 0.f; }
#pragma unroll
        for (int u = 0; u < 8; u++) { const unsigned k = k0 + 32u * u + lane; if (k < n) dst[k] = v[u]; }
      }
    }
  }
  if (QT && dropped) atomicAdd(&info->n_qt_dropped, (unsigned long long)dropped);
  stamp(dbg, 5);
}

// Extents of the single-launch decompress kernel: the tile's count and its offset inside the CTA's range (both written
// by this CTA before the barrier: plain, L2-coherent loads) + the CTA's base.
struct LocalExtents {
  typedef ExtentRaw Raw;
  static __device__ __forceinline__ Raw none() { Raw r; r.gp = 0; r.cp = 0; r.c = 0; r.k = 0; return r; }
  const unsigned *counts, *tile_off;
  unsigned long long base, n_limit;
  unsigned *corrupt_flag;
  __device__ __forceinline__ ExtentRaw load(unsigned t, int) const {
    ExtentRaw r;
    r.c = __ldcg(counts + t);
    r.gp = (unsigned long long)__ldcg(tile_off + t);
    r.cp = 0ull;
    r.k = 0u;
    return r;
  }
  __device__ __forceinline__ Extent finish(ExtentRaw &r, int) const {
    Extent e;
    r.c = pin_here(r.c);
    r.gp = pin_here(r.gp);
    e.total = r.c;
    e.base = base + r.gp;
    e.bad = e.base + e.total > n_limit;
    if (e.bad) { e.total = 0u; *corrupt_flag = 1u; }
    return e;
  }
};

template <typename T, bool QT>
__global__ void __launch_bounds__(DecompressCfg<T, QT>::THREADS, DecompressCfg<T, QT>::CTAS_PER_SM)
k_decompress_fused(const uint8_t *__restrict__ bins, const float *__restrict__ dc_in, const float *__restrict__ ac_in,
                   const T *__restrict__ qtable, unsigned long long nblk_full, T bin_width, T sf, QtConsts<T> qk,
                   const __grid_constant__ CUtensorMap tmap_out, unsigned *counts, unsigned *tile_off, unsigned long long *cta_totals,
                   unsigned long long n_limit, unsigned *corrupt_flag, int dc_aligned16, unsigned long long *barrier,
                   unsigned long long barrier_base, unsigned long long *dbg) {
  typedef DecompressCfg<T, QT> Cfg;
  extern __shared__ unsigned char smem_raw[];
  __shared__ __align__(8) unsigned long long s_mbar[Cfg::WARPS];
  __shared__ T s_qt[QT ? BLK : 1];
  __shared__ __align__(16) T center[256];
  __shared__ unsigned long long s_base, s_total;

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned char *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char *wsm = smem + warp * Cfg::WARP_BYTES;
  const unsigned mb = smem_u32(&s_mbar[warp]);
  const unsigned ntiles = (unsigned)((nblk_full + WTILE - 1) / WTILE);
  unsigned t0, t1;
  cta_tile_range(ntiles, &t0, &t1);
  const unsigned nt = t1 - t0;
  for (int i = threadIdx.x; i < 256; i += Cfg::THREADS) center[i] = center_coefficient<T>((unsigned)i, bin_width, sf);
  if (QT && threadIdx.x < BLK) s_qt[threadIdx.x] = qtable[threadIdx.x];
  if (lane == 0) { mbar_init(mb, 1); fence_mbar_init(); }

  stamp(dbg, 0);
  // ---- phase 1: 255 markers at positions j >= 1 of the CTA's own tiles (a warp per tile, two tiles per trip) ----
  unsigned *s_cnt = reinterpret_cast<unsigned *>(smem);  // the tile buffers are idle until the barrier
  unsigned *s_off = s_cnt + FUSED_MAX_TILES_PER_CTA;
  for (unsigned i = warp; i < nt; i += 2 * Cfg::WARPS) {
    uint4 v[2][4];
    unsigned rows[2];
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const unsigned ih = i + h * Cfg::WARPS;
      rows[h] = 0;
      if (ih < nt) {
        const unsigned long long first = (unsigned long long)(t0 + ih) * WTILE;
        rows[h] = (nblk_full - first < (unsigned long long)WTILE) ? (unsigned)(nblk_full - first) : (unsigned)WTILE;
        const uint4 *p = reinterpret_cast<const uint4 *>(bins + first * BLK);
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const unsigned chunk = k * 32 + lane;  // 16-byte chunk of the tile; 4 chunks per block
          v[h][k] = (chunk < rows[h] * 4u) ? __ldg(p + chunk) : make_uint4(0u, 0u, 0u, 0u);
        }
      }
    }
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const unsigned ih = i + h * Cfg::WARPS;
      if (ih >= nt) break;
      unsigned cnt = 0;
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const unsigned chunk = k * 32 + lane;
        if (chunk < rows[h] * 4u) {
          const unsigned x0 = (chunk & 3u) ? v[h][k].x : (v[h][k].x & 0xFFFFFF00u);  // byte 0 of a block is the DC marker
          cnt += __popc(ff_flags(x0)) + __popc(ff_flags(v[h][k].y)) + __popc(ff_flags(v[h][k].z)) + __popc(ff_flags(v[h][k].w));
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xFFFFFFFFu, cnt, o);
      if (lane == 0) { s_cnt[ih] = cnt; counts[t0 + ih] = cnt; }
    }
  }
  __syncthreads();
  if (warp == 0) {
    const unsigned long long tot = warp0_scan_counts(s_cnt, s_off, nt, lane);
    if (lane == 0) cta_totals[blockIdx.x] = tot;
  }
  __syncthreads();
  for (unsigned i = threadIdx.x; i < nt; i += Cfg::THREADS) tile_off[t0 + i] = s_off[i];
  stamp(dbg, 1);
  grid_barrier(barrier, barrier_base + gridDim.x);
  stamp(dbg, 2);

  // ---- phase 2: dequantise + inverse DCT + de-scale of the CTA's own tiles ----
  if (warp == 0) {
    unsigned long long base, total;
    warp0_cta_prefix(cta_totals, lane, &base, &total);
    if (lane == 0) { s_base = base; s_total = total; }
  }
  __syncthreads();
  LocalExtents ext;
  ext.counts = counts; ext.tile_off = tile_off; ext.base = s_base; ext.n_limit = n_limit; ext.corrupt_flag = corrupt_flag;
  const unsigned long long n_scan = s_total;
  RangeSeq seq;
  seq.init_up(t0, t1, warp, Cfg::WARPS);
  unsigned phase = 0;
  decompress_tiles<T, QT>(bins, dc_in, ac_in, nblk_full, sf, qk, &tmap_out, n_scan < n_limit ? n_scan : n_limit, dc_aligned16, wsm, mb, center, s_qt,
                          seq, ext, lane, phase);
  bulk_wait_all();
  __syncthreads();
  stamp(dbg, 3);
}

}  // namespace dctz
