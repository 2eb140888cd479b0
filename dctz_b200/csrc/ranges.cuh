// ranges.cuh -- region decompression (DESIGN.md §4.4): decode element ranges of a device-resident slab.
//
//   k_index_finish       completes the outlier index (header, tail-block markers) after k_count_bins + k_scan_groups
//   k_range_plan         per range: pieces (tiles touched) and output offset, scanned; validates the ranges
//   k_decompress_ranges  persistent warps take pieces from a ticket counter and decode their element windows
//
// The outlier index is the decompress pre-pass kept instead of discarded: the per-tile marker counts of k_count_bins and
// the two-level prefix k_scan_groups makes of them.  A tile's first outlier is then prefix_of_group() + the counts of the
// earlier tiles of its group (as ScannedExtents computes it), and a block's first outlier that plus the markers of the
// tile's blocks before it -- which the warp counts from the bin ids it loads anyway.
#pragma once
#include "kernels.cuh"

namespace dctz {

constexpr unsigned REGION_INDEX_MAGIC = 0x495a4344u;            // "DCZI"
constexpr unsigned long long TILE_ELEMS = (unsigned long long)WTILE * BLK;  // 2048 elements per warp tile
constexpr unsigned long long PIECE_LIMIT = 0xFFFFF000ull;       // pieces are numbered by 32-bit tickets (TileSeq)

struct RegionIndexHdr {                 // first bytes of an index (the layout is private to the library)
  unsigned long long n;                 // elements of the slab it was built for
  unsigned long long n_full_outliers;   // markers in the full blocks = offset of the tail block's first outlier
  unsigned ntiles, magic;
};
struct RegionIndex {  // device view of an index
  const RegionIndexHdr *hdr;
  const unsigned *counts;
  const unsigned long long *group_prefix, *chunk_prefix;
};
struct RangeCtl { unsigned long long pieces; unsigned done, ticket; };  // done: plan CTAs finished; ticket: TileSeq counter
struct RangePlan {
  unsigned long long *piece_at, *out_at;        // per range: first piece / first output element, relative to its chunk of 1024 ranges
  unsigned long long *chunk_piece, *chunk_out;  // per chunk: exclusive prefixes (first written as chunk totals)
  RangeCtl *ctl;
};

// Header + the markers of the partial tail block; d_n_outliers = full blocks + tail = what a stream header must state.
__global__ void __launch_bounds__(32) k_index_finish(const uint8_t *__restrict__ bins, unsigned long long n, unsigned ntiles, RegionIndexHdr *hdr,
                                                     unsigned long long *n_outliers) {
  const int lane = threadIdx.x;
  const unsigned long long tail0 = n / BLK * BLK;
  const int rem = (int)(n - tail0);
  unsigned c = 0;
  for (int j = 1 + lane; j < rem; j += 32) c += (bins[tail0 + j] == 255u) ? 1u : 0u;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
  if (lane == 0) {
    const unsigned long long full = ntiles ? hdr->n_full_outliers : 0ull;  // written by the scan (nothing to scan without full blocks)
    hdr->n = n;
    hdr->n_full_outliers = full;
    hdr->ntiles = ntiles;
    hdr->magic = REGION_INDEX_MAGIC;
    if (n_outliers) *n_outliers = full + c;
  }
}

// Number of pieces of range [a, b): the warp tiles it touches among the full blocks (which end at element `full`), plus one
// for the partial tail block.
__device__ __forceinline__ unsigned long long full_pieces(unsigned long long a, unsigned long long b, unsigned long long full) {
  return a < full ? ((b < full ? b : full) - 1) / TILE_ELEMS - a / TILE_ELEMS + 1 : 0ull;
}

// One thread per range, one CTA per chunk of 1024 ranges; the last CTA scans the chunk totals (the k_scan_groups pattern).
// It also checks that the index was built for this N, and resets the decode kernel's ticket counter.
__global__ void __launch_bounds__(1024) k_range_plan(const unsigned long long *__restrict__ ranges, unsigned long long nranges, unsigned long long n,
                                                     const RegionIndexHdr *__restrict__ hdr, RangePlan plan, unsigned *corrupt_flag) {
  __shared__ unsigned long long s_wp[33], s_wo[33];
  __shared__ bool s_last;
  const unsigned long long r = (unsigned long long)blockIdx.x * 1024u + threadIdx.x;
  const unsigned long long full = n / BLK * BLK;
  unsigned long long pieces = 0, count = 0;
  if (r < nranges) {
    const unsigned long long a = ranges[2 * r], c = ranges[2 * r + 1];
    count = c;  // the output keeps the place of every range, written or not
    if (c == 0 || a >= n || c > n - a) atomicOr(corrupt_flag, 2u);  // this range is not written
    else pieces = full_pieces(a, a + c, full) + (a + c > full ? 1ull : 0ull);
  }
  unsigned long long tp, to;
  const unsigned long long ep = block_exclusive_scan_1024(pieces, s_wp, &tp);
  const unsigned long long eo = block_exclusive_scan_1024(count, s_wo, &to);
  if (r < nranges) { plan.piece_at[r] = ep; plan.out_at[r] = eo; }
  if (threadIdx.x == 0) {
    plan.chunk_piece[blockIdx.x] = tp;
    plan.chunk_out[blockIdx.x] = to;
    __threadfence();
    s_last = (atomicAdd(&plan.ctl->done, 1u) == gridDim.x - 1);
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  unsigned long long carry_p = 0, carry_o = 0;
  for (unsigned c0 = 0; c0 < gridDim.x; c0 += 1024u) {
    const unsigned c = c0 + threadIdx.x;
    const unsigned long long vp = (c < gridDim.x) ? *(volatile unsigned long long *)(plan.chunk_piece + c) : 0ull;
    const unsigned long long vo = (c < gridDim.x) ? *(volatile unsigned long long *)(plan.chunk_out + c) : 0ull;
    unsigned long long sp, so;
    __syncthreads();
    const unsigned long long xp = block_exclusive_scan_1024(vp, s_wp, &sp);
    const unsigned long long xo = block_exclusive_scan_1024(vo, s_wo, &so);
    if (c < gridDim.x) { plan.chunk_piece[c] = carry_p + xp; plan.chunk_out[c] = carry_o + xo; }
    carry_p += sp;
    carry_o += so;
  }
  if (threadIdx.x == 0) {
    const bool index_ok = hdr->magic == REGION_INDEX_MAGIC && hdr->n == n;
    if (!index_ok) atomicOr(corrupt_flag, 1u);
    if (carry_p > PIECE_LIMIT) atomicOr(corrupt_flag, 2u);
    plan.ctl->pieces = (index_ok && carry_p <= PIECE_LIMIT) ? carry_p : 0ull;  // 0: the decode kernel writes nothing
    plan.ctl->ticket = 0u;
    plan.ctl->done = 0u;
  }
}

// out *= s over the places of the ranges k_decompress_ranges wrote (those inside [0, n)): the second half of a decode with
// a rescaled sf (dctz_gpu.cu: decode_exponent).  The places of skipped ranges stay untouched.  Fewer ranges than CTAs (a
// few long ranges, e.g. one whole field): the whole grid strides over each range in turn; else one CTA per range.
template <typename T>
__global__ void __launch_bounds__(256) k_scale_ranges(T *__restrict__ out, const unsigned long long *__restrict__ ranges, unsigned long long nranges,
                                                      unsigned long long n, RangePlan plan, T s) {
  if (__ldg(&plan.ctl->pieces) == 0ull) return;  // the decode kernel wrote nothing
  const bool whole_grid = nranges < gridDim.x;
  const unsigned long long first = whole_grid ? 0ull : blockIdx.x, step = whole_grid ? 1ull : gridDim.x;
  const unsigned long long t0 = whole_grid ? (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x : threadIdx.x;
  const unsigned long long ts = whole_grid ? (unsigned long long)gridDim.x * blockDim.x : blockDim.x;
  for (unsigned long long r = first; r < nranges; r += step) {
    const unsigned long long a = __ldg(ranges + 2 * r), c = __ldg(ranges + 2 * r + 1);
    if (c == 0 || a >= n || c > n - a) continue;
    T *dst = out + __ldg(plan.out_at + r) + __ldg(plan.chunk_out + (r >> 10));
    for (unsigned long long i = t0; i < c; i += ts) dst[i] = dst[i] * s;
  }
}

template <typename T> struct RangeCfg {
  static constexpr int WARPS = 4;
  static constexpr int THREADS = WARPS * 32;
  static constexpr int PER_CHUNK = 16 / (int)sizeof(T);
  // staging rows of 64 T, 16 bytes of padding between them: the 16-byte stores of the 8 lanes of a quarter-warp (one row
  // each, same chunk) fall into 8 different bank groups
  static constexpr int ROW = BLK * (int)sizeof(T) + 16;
  static constexpr int WARP_BYTES = WTILE * ROW;
  static constexpr int SMEM = WARPS * WARP_BYTES;
};

// Elements [lo, hi) of warp tile t (lo, hi inside the tile), stored to dst[e - lo].  Lane i handles block i of the tile; lanes
// before the window's first block only count their markers, which place the first outlier of every block after them.
template <typename T, bool QT>
__device__ __forceinline__ void decode_tile_window(const uint8_t *__restrict__ bins, const float *__restrict__ dc_in, const float *__restrict__ ac_in,
                                                   const RegionIndex &idx, unsigned long long n_limit, unsigned t, unsigned long long lo,
                                                   unsigned long long hi, T sf, const QtConsts<T> &qk, const T *center, const T *s_qt,
                                                   unsigned char *stage, T *__restrict__ dst, unsigned *corrupt_flag, int lane) {
  typedef typename ArithOf<T, QT>::type A;  // the instantiation decompress_tiles uses
  typedef RangeCfg<T> Cfg;
  const unsigned long long blk0 = (unsigned long long)t * WTILE;
  const int first = (int)(lo / BLK - blk0), last = (int)((hi - 1) / BLK - blk0);
  // the tile's outlier extent, as ScannedExtents computes it
  const unsigned k = t & 31u;
  const unsigned c = ((unsigned)lane <= k) ? __ldg(idx.counts + (t & ~31u) + lane) : 0u;
  const unsigned total = __shfl_sync(0xFFFFFFFFu, c, (int)k);
  unsigned before = ((unsigned)lane < k) ? c : 0u;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xFFFFFFFFu, before, o);
  const unsigned long long base = prefix_of_group(idx.group_prefix, idx.chunk_prefix, t >> 5) + before;
  // a tile whose run would leave the caller's AC_exact decodes without its outliers, as in decompress_tiles
  const bool bad = base + total > n_limit;
  if (bad && lane == 0) atomicOr(corrupt_flag, 1u);

  unsigned w[16];
  if (lane <= last) {
    const uint4 *bp = reinterpret_cast<const uint4 *>(bins + (blk0 + lane) * BLK);
#pragma unroll
    for (int q = 0; q < 4; q++) {
      const uint4 v = __ldg(bp + q);
      w[4 * q] = v.x; w[4 * q + 1] = v.y; w[4 * q + 2] = v.z; w[4 * q + 3] = v.w;
    }
  } else {
#pragma unroll
    for (int q = 0; q < 16; q++) w[q] = 0u;
  }
  unsigned cnt = 0;
#pragma unroll
  for (int q = 0; q < 16; q++) cnt += __popc(ff_flags(q == 0 ? (w[0] & 0xFFFFFF00u) : w[q]));  // position 0 is the DC marker
  const unsigned my_off = warp_inclusive_scan(cnt, lane) - cnt;

  const bool mine = lane >= first && lane <= last;
  T x[BLK];
  if (mine) {
    x[0] = dc_coefficient<T>(__ldg(dc_in + blk0 + lane), sf);
    unsigned long long at = base + my_off;
#pragma unroll
    for (int j = 1; j < BLK; j++) {
      const unsigned id = (w[j >> 2] >> (8 * (j & 3))) & 0xFFu;
      if (id == 255u && !bad) x[j] = outlier_coefficient<T, QT>(__ldg(ac_in + at++), QT ? s_qt[j] : (T)0, qk, sf);
      else x[j] = center[id];  // a bad tile's markers take the dummy entry 255, as in decompress_tiles
    }
  } else {
#pragma unroll
    for (int j = 0; j < BLK; j++) x[j] = (T)0;
  }
  dct64_inverse<A>(x);

  // registers -> own staging row -> coalesced stores of the window (outputs are not tile-aligned: no TMA tile maps)
  __syncwarp();  // the previous piece's reads of the stage are done
  if (mine) {
#pragma unroll
    for (int c16 = 0; c16 < BLK / Cfg::PER_CHUNK; c16++) {
      uint4 v;
      T *e = reinterpret_cast<T *>(&v);
#pragma unroll
      for (int i = 0; i < Cfg::PER_CHUNK; i++) e[i] = x[c16 * Cfg::PER_CHUNK + i];
      *reinterpret_cast<uint4 *>(stage + lane * Cfg::ROW + c16 * 16) = v;
    }
  }
  __syncwarp();
  const unsigned o0 = (unsigned)(lo - blk0 * BLK), o1 = (unsigned)(hi - blk0 * BLK);
  for (unsigned o = o0 + lane; o < o1; o += 32) dst[o - o0] = *reinterpret_cast<const T *>(stage + (o / BLK) * Cfg::ROW + (o % BLK) * sizeof(T));
}

template <typename T, bool QT>
__global__ void __launch_bounds__(RangeCfg<T>::THREADS) k_decompress_ranges(const uint8_t *__restrict__ bins, const float *__restrict__ dc_in,
                                                                           const float *__restrict__ ac_in, const T *__restrict__ qtable,
                                                                           unsigned long long n, T bin_width, T sf, QtConsts<T> qk, RegionIndex idx,
                                                                           unsigned long long n_outliers, const unsigned long long *__restrict__ ranges,
                                                                           unsigned long long nranges, RangePlan plan, T *__restrict__ out,
                                                                           unsigned *corrupt_flag) {
  typedef RangeCfg<T> Cfg;
  extern __shared__ __align__(16) unsigned char smem_ranges[];
  __shared__ __align__(16) T center[256];
  __shared__ T s_qt[QT ? BLK : 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned char *stage = smem_ranges + warp * Cfg::WARP_BYTES;
  for (int i = threadIdx.x; i < 256; i += Cfg::THREADS) center[i] = center_coefficient<T>((unsigned)i, bin_width, sf);
  if (QT && threadIdx.x < BLK) s_qt[threadIdx.x] = qtable[threadIdx.x];
  __syncthreads();

  const unsigned long long npieces = __ldg(&plan.ctl->pieces);
  if (npieces == 0ull) return;
  const unsigned long long full = n / BLK * BLK;
  const unsigned long long n_full_out = __ldg(&idx.hdr->n_full_outliers);
  const unsigned long long lim = n_full_out < n_outliers ? n_full_out : n_outliers;  // as k_decompress bounds the full blocks
  const unsigned nwarps = gridDim.x * Cfg::WARPS;
  TileSeq seq;
  seq.init(&plan.ctl->ticket, blockIdx.x * Cfg::WARPS + warp, nwarps, npieces >= 16ull * nwarps ? 4u : 1u, lane);
  auto piece_start = [&](unsigned long long r) { return __ldg(plan.piece_at + r) + __ldg(plan.chunk_piece + (r >> 10)); };
  for (unsigned p = seq.advance(lane); p < npieces; p = seq.advance(lane)) {
    // the range of piece p: the last one whose first piece is <= p (a range without pieces starts where its successor
    // does).  32-way search: every step narrows the candidates 32-fold (four steps for 2^19 ranges).
    unsigned long long r = 0, span = nranges;
    while (span > 1) {
      const unsigned long long step = (span + 31) / 32;
      const unsigned long long i = r + (unsigned long long)lane * step;
      const unsigned m = __ballot_sync(0xFFFFFFFFu, i < r + span && piece_start(i) <= p);  // lane 0 always (piece_start(r) <= p)
      const unsigned long long kk = (unsigned long long)(31 - __clz(m));
      r += kk * step;
      span = (span - kk * step < step) ? span - kk * step : step;
    }
    const unsigned long long a = __ldg(ranges + 2 * r), b = a + __ldg(ranges + 2 * r + 1);
    const unsigned long long j = p - piece_start(r);
    T *dst = out + __ldg(plan.out_at + r) + __ldg(plan.chunk_out + (r >> 10));  // element a of the range
    if (j < full_pieces(a, b, full)) {
      const unsigned long long t = a / TILE_ELEMS + j;
      const unsigned long long lo = a > t * TILE_ELEMS ? a : t * TILE_ELEMS;
      unsigned long long hi = (t + 1) * TILE_ELEMS < full ? (t + 1) * TILE_ELEMS : full;
      if (b < hi) hi = b;
      decode_tile_window<T, QT>(bins, dc_in, ac_in, idx, lim, (unsigned)t, lo, hi, sf, qk, center, s_qt, stage, dst + (lo - a), corrupt_flag, lane);
    } else {  // the partial tail block, with k_tail_decompress's arithmetic
      const unsigned long long lo = a > full ? a : full;
      __syncwarp();  // the previous piece's reads of the stage are done
      tail_block_decode<T, QT>(bins, dc_in, ac_in, qtable, (int)(n - full), n / BLK, bin_width, sf, qk, n_full_out, n_outliers,
                               [&] { atomicOr(corrupt_flag, 1u); },
                               [&](int e, T v) {
                                 const unsigned long long g = full + (unsigned long long)e;
                                 if (g >= lo && g < b) dst[g - a] = v;
                               },
                               reinterpret_cast<double *>(stage), lane);
    }
  }
}

}  // namespace dctz
