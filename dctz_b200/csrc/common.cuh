// common.cuh -- arithmetic policies, exact division, TMA / mbarrier wrappers, tile scheduling and scan helpers shared by
// the sm_100a kernels of the DCTZ hot path.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "dct64_gen.cuh"  // (global scope) the generated transform and its constant table ::dct64_kd

namespace dctz {

constexpr int BLK = 64;            // BLK_SZ, dctz.h:28

// ------------------------------------------------------------------------------------------
// Arithmetic policies for the generated DCT (dct64_gen.cuh).  Only *_rn intrinsics: nvcc never
// contracts or re-associates them, so the flow graph is executed exactly as generated.
// ------------------------------------------------------------------------------------------
struct ArithD {
  typedef double V;
  // entry i of the constant table: ptxas then feeds the DMUL / DFMA a constant-bank operand; a double LITERAL costs two UMOVs
  // (its two 32-bit halves into a uniform register pair) per use, ~250 instructions of the 592-operation transform
  static __device__ __forceinline__ double cst(int i, double) { return ::dct64_kd[i]; }
  static __device__ __forceinline__ V add(V a, V b) { return __dadd_rn(a, b); }
  static __device__ __forceinline__ V sub(V a, V b) { return __dsub_rn(a, b); }
  static __device__ __forceinline__ V mul(V a, double k) { return __dmul_rn(a, k); }
  static __device__ __forceinline__ V fma(V a, double k, V b) { return __fma_rn(a, k, b); }
  static __device__ __forceinline__ V fms(V a, double k, V b) { return __fma_rn(a, k, -b); }
  static __device__ __forceinline__ V neg(V a) { return -a; }
};

// The same with the constants as literals: what the EC decompress kernels use.  Same-box A/B on B200 (tools/probes/ab.sh): with the
// table the compress kernels gain 1-2 % (5 % outlier slab, c4), QT compress 4 % and QT decompress 5 %; the count-ahead EC
// decompress of the 8 GiB slab LOSES 7 % (1.70 -> 1.82 ms) and the pre-pass EC decompress 1 %, so those keep the literals.
struct ArithDLit : ArithD {
  static __device__ __forceinline__ constexpr double cst(int, double k) { return k; }
};

struct ArithF {
  typedef float V;
  static __device__ __forceinline__ constexpr float cst(int, double k) { return (float)k; }  // an immediate of the FMUL / FFMA
  static __device__ __forceinline__ V add(V a, V b) { return __fadd_rn(a, b); }
  static __device__ __forceinline__ V sub(V a, V b) { return __fsub_rn(a, b); }
  static __device__ __forceinline__ V mul(V a, float k) { return __fmul_rn(a, k); }
  static __device__ __forceinline__ V fma(V a, float k, V b) { return __fmaf_rn(a, k, b); }
  static __device__ __forceinline__ V fms(V a, float k, V b) { return __fmaf_rn(a, k, -b); }
  static __device__ __forceinline__ V neg(V a) { return -a; }
};

template <typename T, bool TABLE = true> struct ArithOf;
template <> struct ArithOf<double, true> { typedef ArithD type; };
template <> struct ArithOf<double, false> { typedef ArithDLit type; };
template <bool TABLE> struct ArithOf<float, TABLE> { typedef ArithF type; };

// ------------------------------------------------------------------------------------------
// Exact division by a loop-invariant divisor b with y = RN(1/b) precomputed.
//   q0 = RN(a*y); r = a - q0*b (exact, FMA); q1 = RN(q0 + r*y)
// Markstein's theorem: if y is the correctly rounded reciprocal and q0 is a faithful rounding of
// a/b, then q1 == RN(a/b) (b's significand not all ones; no under/overflow).  q0 is faithful when
// the relative error rho of y is <= 2^-(p+1): then |a*y - a/b| < ulp(a/b)/2 strictly, so RN(a*y) is one
// of the two neighbours of a/b; otherwise one more correction step makes it so.
// The host / finalize kernel measures rho EXACTLY (y*b - 1 is a multiple of 2^-105 (2^-47 for float)
// and, near 2^-54 (2^-25), exactly representable, so the single-rounding fma returns it exactly)
// and picks `iters` (see make_divisor()).  sf = 10 and sf = 0.1 both have rho == 2^-54 exactly.
//   iters: 0 -> b == 1 (identity), 1, 2 -> FMA corrections, 3 -> IEEE division (degenerate b).
// Deviation window (documented in DESIGN.md): |a| below 2^-969 (double) / 2^-102 (float) lets r
// underflow, where the last bit of the quotient may differ from IEEE division.
// ------------------------------------------------------------------------------------------
template <typename T> struct Divisor { T b, y; int iters; };

// The degenerate case is a CALL: inlined, the IEEE division sequence (with its slow path) stood 135 times in k_decompress<double,QT>
// and 77 times in k_compress<float,EC> -- 10 256 and 6 376 SASS instructions, and ncu showed the warps waiting for instructions
// (stall no_instruction 0.43 per issue against 0.12 in the EC kernel of a third the size).
__device__ __noinline__ double div_ieee(double a, double b) { return __ddiv_rn(a, b); }
__device__ __noinline__ float div_ieee(float a, float b) { return __fdiv_rn(a, b); }

__device__ __forceinline__ double div_exact(double a, const Divisor<double> &d) {
  if (d.iters == 3) return div_ieee(a, d.b);  // degenerate divisor: kernel-uniform branch
  double q = __dmul_rn(a, d.y);
  double r = __fma_rn(-q, d.b, a);
  q = __fma_rn(r, d.y, q);
  if (d.iters == 2) {
    r = __fma_rn(-q, d.b, a);
    q = __fma_rn(r, d.y, q);
  }
  return q;
}
__device__ __forceinline__ float div_exact(float a, const Divisor<float> &d) {
  if (d.iters == 3) return div_ieee(a, d.b);
  float q = __fmul_rn(a, d.y);
  float r = __fmaf_rn(-q, d.b, a);
  q = __fmaf_rn(r, d.y, q);
  if (d.iters == 2) {
    r = __fmaf_rn(-q, d.b, a);
    q = __fmaf_rn(r, d.y, q);
  }
  return q;
}

__host__ __device__ inline Divisor<double> make_divisor(double b) {
  Divisor<double> d;
  d.b = b;
#ifdef __CUDA_ARCH__
  d.y = __drcp_rn(b);
  const double rho = fabs(__fma_rn(d.y, b, -1.0));
  const unsigned long long m = (unsigned long long)__double_as_longlong(b) & 0xFFFFFFFFFFFFFull;
#else
  d.y = 1.0 / b;
  const double rho = fabs(fma(d.y, b, -1.0));
  unsigned long long bits; memcpy(&bits, &b, 8);
  const unsigned long long m = bits & 0xFFFFFFFFFFFFFull;
#endif
  if (b == 1.0) d.iters = 0;
  else if (!(b == b) || b == 0.0 || m == 0xFFFFFFFFFFFFFull || !(rho < 1.0)) d.iters = 3;
  else d.iters = (rho <= 5.5511151231257827e-17 /* 2^-54, exact */) ? 1 : 2;
  return d;
}
__host__ __device__ inline Divisor<float> make_divisor(float b) {
  Divisor<float> d;
  d.b = b;
#ifdef __CUDA_ARCH__
  d.y = __frcp_rn(b);
  const float rho = fabsf(__fmaf_rn(d.y, b, -1.0f));
  const unsigned m = (unsigned)__float_as_int(b) & 0x7FFFFFu;
#else
  d.y = 1.0f / b;
  const float rho = fabsf(fmaf(d.y, b, -1.0f));
  unsigned bits; memcpy(&bits, &b, 4);
  const unsigned m = bits & 0x7FFFFFu;
#endif
  if (b == 1.0f) d.iters = 0;
  else if (!(b == b) || b == 0.0f || m == 0x7FFFFFu || !(rho < 1.0f)) d.iters = 3;
  else d.iters = (rho <= 2.98023223876953125e-08f /* 2^-25, exact */) ? 1 : 2;
  return d;
}

// ------------------------------------------------------------------------------------------
// conv_tbl (dctz-comp-lib.c:27-43) in closed form: ordinal t (0..254) -> centre-out id,
// conv(t) = (t <= 127) ? 254 - 2t : 2t - 255 = max(254 - 2t, 2t - 255).
// Its inverse is the identity conv_tbl_i (dctz-decomp-lib.c:23-39) followed by gen_bins'
// centre(id) = ((id & 1) ? id/2 + 1 : -(id/2)) * bin_width (binning.c:19-22).
// ------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ unsigned conv_ordinal(int t) {
  const int a = 254 - 2 * t, b = 2 * t - 255;
  return (unsigned)(a > b ? a : b);
}
__host__ __device__ __forceinline__ int center_multiple(unsigned id) {
  return (id & 1u) ? (int)(id >> 1) + 1 : -(int)(id >> 1);
}

// ------------------------------------------------------------------------------------------
// Warp tiles and TMA.  The hot kernels are WARP-AUTONOMOUS: each warp owns a tile of 32 consecutive
// 64-element blocks (one block per lane) and its own slice of shared memory, and never meets the
// other warps of its CTA at a barrier.
//
// A tile moves global <-> shared with TMA TENSOR copies (cp.async.bulk.tensor.2d, SASS UTMALDG /
// UTMASTG) issued by one lane.  The field is described to the TMA unit as a 2-D byte tensor
// [blocks][64*sizeof(T)]; a tile is fetched as SLABS of [32 blocks][128 bytes] with the 128-byte
// swizzle, i.e. slab q holds bytes [128q, 128q+128) of each of the 32 rows, row r at offset 128 r,
// its 16-byte chunk c stored at chunk position c ^ (r & 7).  A lane reading chunk c of "its" row r
// therefore hits bank group c ^ (r & 7): the 8 lanes of a quarter-warp touch 8 different bank
// groups -- conflict-free 128-bit shared loads with compile-time register indices.  Rows beyond the
// end of the field are zero-filled on load and clipped on store by the TMA unit, so partial tiles
// need no special path.  (Per-lane cp.async.bulk row copies were tried first: UBLKCP takes uniform
// operands, so the compiler serialises them into a 32-trip loop, ~10% of the kernel's instructions.)
// ------------------------------------------------------------------------------------------
constexpr int WTILE = 32;  // blocks per warp tile (one per lane)
template <typename T> struct WarpTile {
  static constexpr int ROW_BYTES = BLK * (int)sizeof(T);
  static constexpr int SLABS = ROW_BYTES / 128;     // 4 (double) or 2 (float)
  static constexpr int SLAB_BYTES = WTILE * 128;    // 4 KB
  static constexpr int BYTES = SLABS * SLAB_BYTES;  // 16 KB / 8 KB, must sit at a 1024-byte aligned address
  static constexpr int PER_CHUNK = 16 / (int)sizeof(T);
  // byte offset of 16-byte chunk `c` (0..7) of slab `q` of row (lane) `r`
  static __device__ __forceinline__ unsigned chunk_offset(int q, int r, int c) {
    return (unsigned)(q * SLAB_BYTES + r * 128 + ((c ^ (r & 7)) << 4));
  }
};

__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned mb, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(mb), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(unsigned mb, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(mb), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(unsigned mb, unsigned parity) {
  unsigned ok;
  asm volatile(
      "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
      : "=r"(ok)
      : "r"(mb), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(unsigned mb, unsigned parity) {
  while (!mbar_try_wait(mb, parity)) {}
}
// global -> shared, completion counted in bytes on the mbarrier
__device__ __forceinline__ void bulk_g2s(unsigned dst, const void *src, unsigned bytes, unsigned mb) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(dst), "l"(src),
               "r"(bytes), "r"(mb)
               : "memory");
}
// shared -> global, tracked by the thread's bulk async-group
__device__ __forceinline__ void bulk_s2g(void *dst, unsigned src, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
}
// TMA tensor copies: 2-D box {128 bytes, 32 rows} at byte column c0, row c1 of the tensor map
__device__ __forceinline__ void tma_load_2d(unsigned dst, const void *tmap, int c0, int c1, unsigned mb) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n" ::"r"(dst),
               "l"(tmap), "r"(c0), "r"(c1), "r"(mb)
               : "memory");
}
__device__ __forceinline__ void tma_store_2d(const void *tmap, int c0, int c1, unsigned src) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%1, %2}], [%3];\n" ::"l"(tmap), "r"(c0), "r"(c1), "r"(src)
               : "memory");
}
// L2 eviction-priority hints (experiment switch: DCTZ_L2_HINTS, see c_l2_hints)
__device__ __forceinline__ unsigned long long policy_evict_last() {
  unsigned long long p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;\n" : "=l"(p));
  return p;
}
__device__ __forceinline__ unsigned long long policy_evict_first() {
  unsigned long long p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;\n" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint4 ldg_hint(const uint4 *ptr, unsigned long long pol) {
  uint4 v;
  asm volatile("ld.global.nc.L2::cache_hint.v4.u32 {%0, %1, %2, %3}, [%4], %5;\n" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(ptr), "l"(pol));
  return v;
}
__device__ __forceinline__ void tma_store_2d_hint(const void *tmap, int c0, int c1, unsigned src, unsigned long long pol) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group.L2::cache_hint [%0, {%1, %2}], [%3], %4;\n" ::"l"(tmap), "r"(c0), "r"(c1),
               "r"(src), "l"(pol)
               : "memory");
}
__device__ __forceinline__ void bulk_g2s_hint(unsigned dst, const void *src, unsigned bytes, unsigned mb, unsigned long long pol) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;\n" ::"r"(dst), "l"(src),
               "r"(bytes), "r"(mb), "l"(pol)
               : "memory");
}
// 128-bit shared-memory load the compiler may not narrow: asked for a uint4 of which only two words are used it emits two
// 32-bit LDS, and a 32-bit access by the 32 lanes of a warp to "own row, swizzled chunk" addresses is a 4-way bank conflict
// (rows r, r+8, r+16, r+24 share their banks), where the 128-bit form -- served per quarter-warp -- has none.
__device__ __forceinline__ uint4 lds128(unsigned addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];\n" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory"); }
// generic-proxy shared-memory writes -> visible to the async proxy (TMA) that reads them next
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }

// ------------------------------------------------------------------------------------------
// Ordered outlier compaction WITHOUT an in-kernel ordered chain.
//
// AC_exact must be in (block, j) order (dctz-comp-lib.c:478-544; the decoder consumes it with a serial
// cursor, dctz-decomp-lib.c:370,402).  A single-pass decoupled look-back was measured first and
// rejected: every warp tile has to wait for all earlier tiles to be counted, which turns the
// persistent kernel into an in-order pipeline that runs at the pace of its slowest warp (2.5-6x
// slower than the same kernel without the chain; profiles/README.md).  Instead:
//   compress:   K2 writes each tile's outliers, packed in their final order, to a tile-strided scratch
//               slot (TILE_SLOT floats per tile) plus the tile's count; k_scan_groups turns the counts into
//               exclusive prefixes per group of 32 tiles; k_gather moves the runs to their final
//               place (8 bytes of traffic per outlier -- nothing when there are none);
//   decompress: k_count_bins counts the 255 markers per tile (1 byte/element of extra reads), the
//               same scan follows, and K3 starts every tile with its offset already known.
// No kernel ever waits for another warp.
// ------------------------------------------------------------------------------------------
constexpr int TILE_SLOT = 2048;  // scratch entries per warp tile (>= 63 * 32 = 2016 outliers worst case), packed in final order

// Control block shared by all CTAs of a persistent kernel.
struct TileControl {
  unsigned ticket;   // next tile index (dynamic scheduling)
  unsigned done;     // CTAs that have exited; the last one resets the fields for the next launch
  unsigned long long max_bits;  // VERIFY variant of K2: largest |x| bit pattern seen so far
  unsigned corrupt;  // K3: set when the bin indices mark more outliers than the caller's AC_exact array holds
  unsigned count_ticket;  // K3 without the pre-pass: next unit to count
  unsigned long long min_bits;  // VERIFY: smallest |x| bit pattern (kept at ~0 between launches)
  double belief_sf;             // the scaling factor the VERIFY launch compressed with (read by the REDO launch)
};

// Keep the first USE of a long-latency result (a ticket atomic, a prefetched global load) where the source puts it:
// the volatile move cannot be hoisted above the other volatile statements of the loop body (barrier waits, bulk
// copies), so the consumer lands in the last basic block of the iteration instead of right behind the request --
// where the warp would sit out the whole round trip.
__device__ __forceinline__ unsigned pin_here(unsigned v) {
  unsigned r;
  asm volatile("mov.u32 %0, %1;\n" : "=r"(r) : "r"(v) : "memory");
  return r;
}
__device__ __forceinline__ unsigned long long pin_here(unsigned long long v) {
  unsigned long long r;
  asm volatile("mov.u64 %0, %1;\n" : "=l"(r) : "l"(v) : "memory");
  return r;
}

// Ticket counter increment by ONE lane.  atomicAdd() -- also as a bare PTX `atom.add` -- under `if (lane == 0)` is
// turned by ptxas into the warp-aggregated form (leader election + atomic + SHFL of the result to the "other"
// lanes): that shuffle consumes the atomic's result immediately and stalls the warp for the whole L2 round trip.
// `atom.inc` (old + 1, wrapping at the bound) is not aggregated; with a bound no ticket ever reaches it is a plain increment (ptxas turns the bound 2^32-1 back into an add).
__device__ __forceinline__ unsigned ticket_next(unsigned *counter) {
  unsigned r;
  asm volatile("atom.global.inc.u32 %0, [%1], 0xfffffff0;\n" : "=r"(r) : "l"(counter) : "memory");
  return r;
}

// The sequence of tiles a warp works on: batches of `batch` consecutive tiles.  The first batch is the warp's own
// index; later ones come from the shared ticket counter (dynamic scheduling: a warp that drew tiles full of outliers
// simply takes fewer batches).  The ticket for the batch after the current one is requested when the current one
// is entered, so the atomic's round trip has `batch` iterations to complete; and one atomic per `batch` tiles keeps
// the single counter far from its throughput limit (at one ticket per tile a 2^30-element slab issues 375 M same-
// address atomics per second -- measured: the whole kernel slows down by 25%).  Small fields use batch = 1.
struct TileSeq {
  unsigned next, end, pend, base, batch;
  unsigned *counter;
  unsigned flip;  // 0: tiles in ascending order; ntiles - 1: the sequence runs from the LAST tile down (advance returns flip - index)
  __device__ __forceinline__ void init(unsigned *ticket_counter, unsigned warp_global, unsigned nwarps_grid, unsigned batch_, int lane,
                                       unsigned flip_ = 0u) {
    counter = ticket_counter;
    batch = batch_;
    base = nwarps_grid;
    next = warp_global * batch;
    end = next + batch;
    pend = 0;
    flip = flip_;
    if (lane == 0) pend = ticket_next(counter);
  }
  __device__ __forceinline__ unsigned map(unsigned idx) const {  // an index past the end stays past the end
    return (flip == 0u) ? idx : (idx <= flip ? flip - idx : 0xFFFFFFFFu);
  }
  __device__ __forceinline__ unsigned advance(int lane) {  // warp-uniform
    if (next < end) return map(next++);
    const unsigned start = (base + __shfl_sync(0xFFFFFFFFu, pin_here(pend), 0)) * batch;
    if (lane == 0) pend = ticket_next(counter);
    next = start + 1u;
    end = start + batch;
    return map(start);
  }
};

// A shared-memory buffer that TMA refills may only be re-armed once every lane's READS of it have COMPLETED -- not merely
// been issued: a generic-proxy load still queued in the memory pipeline is not ordered against an async-proxy write
// (__syncwarp orders issue, not completion).  With the load/store unit backed up by thousands of scattered outlier
// stores and the next tile hot in L2 the refill did overtake such loads (float fields at small error bounds: blocks
// transformed from a mix of two tiles).  `probe` is an OR over (a word of) every value loaded from the buffer: the
// vote cannot issue before all of them have arrived in every lane's registers, and the caller makes the TMA issue
// depend on its result (it is true unless all 32 probes hit one magic value at once).
__device__ __forceinline__ bool reads_have_landed(unsigned probe) {
  return __ballot_sync(0xFFFFFFFFu, probe == 0x7F4A7C15u) != 0xFFFFFFFFu;
}

// inclusive warp scan of one small count per lane
__device__ __forceinline__ unsigned warp_inclusive_scan(unsigned v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned n = __shfl_up_sync(0xFFFFFFFFu, v, o);
    if (lane >= o) v += n;
  }
  return v;
}

// per 32-bit word of four bin ids: 0x80 in every byte that equals 0xFF (the outlier marker) -- three instructions: the low
// seven bits + 1 carry into bit 7 exactly when they are all ones (never beyond it), and bit 7 itself must be set
__device__ __forceinline__ unsigned ff_flags(unsigned w) { return ((w & 0x7F7F7F7Fu) + 0x01010101u) & w & 0x80808080u; }
// per 32-bit word of four bin ids: 0x01 in every byte that equals 0xFF (the outlier marker)
__device__ __forceinline__ unsigned ff_bytes(unsigned w) {
  unsigned y = w & (w >> 4);
  y &= y >> 2;
  y &= y >> 1;
  return y & 0x01010101u;
}

}  // namespace dctz
