/* dctz_gpu.h -- C-ABI boundary of the B200-native DCTZ hot path (libdctz_gpu.so).
 *
 * Plain C: opaque handle, raw pointers, sizes.  No CUDA or C++ types appear in any signature
 * (streams travel as void*), so the reference's C host code -- or any FFI -- can bind it directly.
 *
 * What it replaces in the reference (swson/DCTZ v0.2.2), i.e. where a maintainer cuts the seam:
 *   compress:   dctz-comp-lib.c:186-217  calc_data_stat + in-place scale          (util.c:12-44)
 *               dctz-comp-lib.c:271-281  quantiser parameters
 *               dctz-comp-lib.c:318-420  per-block DCT (dct.c:55-103 / dct-float.c:56-104),
 *                                        DC, bin indices, qtable maxima
 *               dctz-comp-lib.c:443-476  qtable clamp / qt_factor
 *               dctz-comp-lib.c:478-544  ordered outlier ("AC_exact") compaction, QT rescale
 *   decompress: dctz-decomp-lib.c:358-386 bin centres (binning.c:12-50), ranges
 *               dctz-decomp-lib.c:389-483 dequantise + per-block inverse DCT (dct.c:115-205)
 *               dctz-decomp-lib.c:494-511 de-scale
 * Everything else of dctz_compress()/dctz_decompress() (allocation, debug dumps, the three zlib
 * streams, header and stream assembly) stays host C and calls these entry points; see
 * INTEGRATION.md for the exact edit and dctz_b200/csrc/host/ for a host library that does it.
 *
 * Conventions
 *   - datatype uses the reference's t_datatype values (dctz.h:44-47): 0 = FLOAT, 1 = DOUBLE.
 *   - mode_qt: 0 = error-controlled build ("ec", default), 1 = -DUSE_QTABLE build ("qt").
 *   - every function returns 0 on success or a negative DCTZ_GPU_E* code;
 *     dctz_gpu_last_error() gives the message.  There is NO CPU fallback: without a usable
 *     CUDA device every call fails with DCTZ_GPU_ENODEV.
 *   - N may exceed 2^31 (the reference's `int N` limit is a property of its stream header, not of
 *     this layer); outlier counts are 64-bit.
 *   - *_dev entry points take device pointers, enqueue on the given stream and do not
 *     synchronise; host-buffer entry points are synchronous.
 *   - a context owns scratch (tile tickets, outlier slots, scan prefixes) that every call uses:
 *     ONE operation in flight per context.  Calls on one context must be issued on one stream (or
 *     be ordered by the caller); use one context per concurrent stream / host thread.
 */
#ifndef DCTZ_GPU_H
#define DCTZ_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DCTZ_GPU_FLOAT 0
#define DCTZ_GPU_DOUBLE 1

#define DCTZ_GPU_OK 0
#define DCTZ_GPU_ENODEV (-1)    /* no CUDA device / driver */
#define DCTZ_GPU_ECUDA (-2)     /* a CUDA call failed */
#define DCTZ_GPU_EINVAL (-3)    /* bad argument (eb < 1e-6 like dctz-comp-lib.c:135, alignment, ...) */
#define DCTZ_GPU_ENOMEM (-4)
#define DCTZ_GPU_EDEGENERATE (-5) /* max|x| is 0, inf or NaN (the reference computes sf = 0/NaN, util.c:28), or outside
                                     the exponent range compress admits (sf 1e-302..1e305, float 1e-32..1e35: DESIGN.md §2) */
#define DCTZ_GPU_ESTALE (-6)      /* (no longer returned: a wrong belief about the statistics is corrected on the device) */
#define DCTZ_GPU_ECORRUPT (-7)    /* decompress_core: bin_index marks more outliers than AC_exact holds */

#define DCTZ_GPU_BLK 64    /* BLK_SZ, dctz.h:28 */
#define DCTZ_GPU_NBINS 255 /* NBINS,  dctz.h:66 */

typedef struct dctz_gpu_ctx dctz_gpu_ctx;

/* Result block of one compress call (device-resident in the *_dev API, copied out by the host API). */
typedef struct dctz_gpu_info {
  double sf;        /* scaling factor, util.c:28/42 (float path: the float value, widened)          */
  double mean;      /* util.c:27/41; order-dependent in the reference -> compare with a tolerance   */
  double max_abs;   /* bs.max */
  double min_abs;   /* bs.min */
  double sum;       /* sum over x[1..N-1] (util.c:21-25 skips element 0)                            */
  uint64_t n_outliers; /* tot_AC_exact_count, dctz-comp-lib.c:323                                   */
  uint64_t n_edge;     /* partial tail block only: coefficients at ordinal 255 although item <= range_max
                          (the reference indexes conv_tbl[255] out of bounds there); every path stores
                          such a coefficient as an outlier (DESIGN.md §2), the tail kernel also counts it */
  uint64_t n_exact_path; /* single-read path: 1 if the belief gave the wrong scaling factor and the slab was
                            compressed a second time, else 0                                                 */
  uint64_t n_qt_dropped; /* QT diagnostic, always 0: rescaled outliers that fell back inside the bin range
                            (dctz-comp-lib.c:494-506 would drop them; unreachable, DESIGN.md §2)        */
  int32_t status;      /* 0, or DCTZ_GPU_EDEGENERATE                                                */
  int32_t scale_mode;  /* 0: sf == 1 (no scaling), 1/2: exact reciprocal division iterations, 3: IEEE div */
} dctz_gpu_info;

/* ---- lifetime ---------------------------------------------------------------------------- */
int dctz_gpu_create(dctz_gpu_ctx **ctx, int device);
void dctz_gpu_destroy(dctz_gpu_ctx *ctx);
const char *dctz_gpu_last_error(const dctz_gpu_ctx *ctx); /* ctx may be NULL (creation errors) */
int dctz_gpu_device_count(void);
int dctz_gpu_sm_count(const dctz_gpu_ctx *ctx);

/* pinned host memory for callers that want full-speed PCIe copies */
void *dctz_gpu_host_alloc(size_t bytes);
void dctz_gpu_host_free(void *p);

/* ---- host-buffer API: the drop-in seam ------------------------------------------------------
 * compress_core: `in` holds N elements (float or double).  Outputs, all caller-allocated host
 * memory: bin_index[N]; DC[ceil(N/64)]; AC_exact[capacity N floats]; qtable / qtable_raw[64
 * elements of the data type, may be NULL unless mode_qt] = the table after / before the >= 1.0
 * clamp (stream trailer / qtable.bin dump).  If scaled_out is non-NULL it receives x[i]/sf, the
 * value the reference leaves in the caller's input buffer (dctz-comp-lib.c:198,213); passing
 * scaled_out == in reproduces the in-place mutation (an IEEE division done by host threads on the
 * caller's buffer: nothing travels back over PCIe for it).  Pageable buffers are staged through a
 * page-locked ring by the library; page-locked ones (dctz_gpu_host_alloc) are copied directly.  */
int dctz_gpu_compress_core(dctz_gpu_ctx *ctx, const void *in, size_t N, int datatype, double error_bound,
                           int mode_qt, void *scaled_out, uint8_t *bin_index, float *DC, float *AC_exact,
                           void *qtable, void *qtable_raw, dctz_gpu_info *info);

/* compress_core_cb: compress_core that reports its outputs piecewise.  on_ready(user, section, offset, bytes) is
 * called on the calling thread as soon as bytes [offset, offset+bytes) of section 0 = bin_index, 1 = DC,
 * 2 = AC_exact are valid in the caller's buffer (in ascending order, every section at least once; AC_exact with
 * bytes == 0 when there are no outliers), so that the host code can start deflating while the rest is still on
 * its way over PCIe.  `info` is complete before the first call.                                              */
typedef void (*dctz_gpu_section_cb)(void *user, int section, size_t offset, size_t bytes);
int dctz_gpu_compress_core_cb(dctz_gpu_ctx *ctx, const void *in, size_t N, int datatype, double error_bound,
                              int mode_qt, void *scaled_out, uint8_t *bin_index, float *DC, float *AC_exact,
                              void *qtable, void *qtable_raw, dctz_gpu_info *info, dctz_gpu_section_cb on_ready,
                              void *user);

/* decompress_core: inverse of the above; `out` receives N reconstructed elements.
 * qtable (64 elements, clamped table from the stream trailer) is only read when mode_qt.      */
int dctz_gpu_decompress_core(dctz_gpu_ctx *ctx, const uint8_t *bin_index, const float *DC,
                             const float *AC_exact, uint64_t n_outliers, const void *qtable, size_t N,
                             int datatype, double error_bound, double sf, int mode_qt, void *out);

/* stats: the GPU-backed equivalent of calc_data_stat() (util.c:12-44) on a host buffer; fills
 * info->max_abs / min_abs / sum / mean / sf (the other fields are zero).                        */
int dctz_gpu_stats(dctz_gpu_ctx *ctx, const void *in, size_t N, int datatype, dctz_gpu_info *info);

/* compress_core_with_stats: like compress_core, but the scaling factor comes from the caller's statistics
 * {max|x|, min|x|, sum} of the WHOLE data set this buffer is a block-aligned piece of (N_total elements;
 * `first_piece` != 0 for the piece holding element 0).  This is what frames a field beyond the reference's
 * `int N` limit as several standard DCTZ streams that share one global scaling factor (SURVEY.md §8e/§8f-2). */
int dctz_gpu_compress_core_with_stats(dctz_gpu_ctx *ctx, const void *in, size_t N, size_t N_total, const double stats3[3],
                                      int first_piece, int datatype, double error_bound, int mode_qt, void *scaled_out,
                                      uint8_t *bin_index, float *DC, float *AC_exact, void *qtable, void *qtable_raw,
                                      dctz_gpu_info *info);

/* quality: the GPU-backed core of calc_psnr() (util.c:54-104) on host buffers: out4 = {min(a), max(a),
 * max|a-b|, sum (a-b)^2}.                                                                          */
int dctz_gpu_quality(dctz_gpu_ctx *ctx, const void *a, const void *b, size_t N, int datatype, double out4[4]);
/* same on device buffers (d_out4: 4 doubles on the device), asynchronous on `stream`                */
int dctz_gpu_quality_dev(dctz_gpu_ctx *ctx, const void *d_a, const void *d_b, size_t N, int datatype, double *d_out4, void *stream);

/* ---- device-resident API (benchmarks, multi-GPU slabs, pipelines) ---------------------------
 * All pointers are device pointers on ctx's device; `stream` is a cudaStream_t passed as void*
 * (NULL = default stream).  Input/outputs must be 16-byte aligned.
 *
 * Split phases so that a multi-GPU caller can exchange the global statistics between them
 * (SURVEY.md §8e): stats_dev -> [all-gather 3 doubles per rank] -> compress_dev.               */

/* Phase 1: local statistics of a slab.  d_stats3 receives {max|x|, min|x|, sum(x)} as doubles. */
int dctz_gpu_stats_dev(dctz_gpu_ctx *ctx, const void *d_in, size_t N, int datatype, double *d_stats3,
                       void *stream);

/* Phase 2: scale + DCT + quantise + ordered outlier compaction of a slab of `N` elements that is
 * part of a field of `N_total` elements.  d_stats_all holds `nranks` triples from phase 1 in rank
 * order (nranks = 1: the slab's own).  `first_slab` != 0 for the slab that contains element 0 of
 * the field (its value is excluded from the sum like util.c:21-25 does).  Only the last slab may
 * have N % 64 != 0.  In QT mode the outliers are left un-rescaled in internal scratch and
 * d_qtable_raw receives this slab's per-position maxima; call dctz_gpu_qt_finish_dev afterwards.
 * d_AC_exact needs room for N floats.  d_info receives the result block.                       */
int dctz_gpu_compress_dev(dctz_gpu_ctx *ctx, const void *d_in, size_t N, size_t N_total, int datatype,
                          double error_bound, int mode_qt, const double *d_stats_all, int nranks,
                          int first_slab, uint8_t *d_bin_index, float *d_DC, float *d_AC_exact,
                          void *d_qtable_raw, dctz_gpu_info *d_info, void *stream);

/* ---- the SINGLE-READ path: the input is read once instead of twice -------------------------------------------
 * The scaling factor only depends on the DECADE of max|x| (sf = 10^(ceil(log10 max)-1), util.c:28), and a sample of
 * 0.4 % of a slab almost always finds it.  So: (1) sample_dev takes max|x| over one 16-byte vector of every 4 KB (and
 * the exact statistics of a partial tail block) -> d_belief3; (2) [all-gather the beliefs of all ranks];
 * (3) compress_spec_dev compresses with the scaling factor the beliefs give and gathers the slab's TRUE {max|x|,
 * min|x|, sum} on the way (FP max/min per element, per-tile sums reduced in tile order: deterministic) -> d_true3;
 * (4) [all-gather the true statistics]; (5) compress_spec_finish_dev derives the scaling factor from them: if it is the
 * one step 3 used -- the normal case -- its gate launch leaves at once and only the outlier scan + gather run; if not,
 * the slab is compressed again with the right factor (d_info->n_exact_path = 1).  Either way the outputs are exactly
 * those of stats_dev + compress_dev.  Same argument meanings as dctz_gpu_compress_dev; N >= 64.  In QT mode call
 * dctz_gpu_qt_finish_dev afterwards as usual.  dctz_gpu_compress_field_dev uses this path for whole fields
 * (DCTZ_SINGLE_READ=0 in the environment at context creation selects the two-pass path).                      */
int dctz_gpu_sample_dev(dctz_gpu_ctx *ctx, const void *d_in, size_t N, int datatype, double *d_belief3, void *stream);
int dctz_gpu_compress_spec_dev(dctz_gpu_ctx *ctx, const void *d_in, size_t N, size_t N_total, int datatype,
                               double error_bound, int mode_qt, const double *d_belief_all, int nranks, int first_slab,
                               uint8_t *d_bin_index, float *d_DC, float *d_AC_exact, void *d_qtable_raw,
                               dctz_gpu_info *d_info, double *d_true3, void *stream);
int dctz_gpu_compress_spec_finish_dev(dctz_gpu_ctx *ctx, const void *d_in, size_t N, size_t N_total, int datatype,
                                      double error_bound, int mode_qt, const double *d_true_all, int nranks,
                                      int first_slab, uint8_t *d_bin_index, float *d_DC, float *d_AC_exact,
                                      void *d_qtable_raw, dctz_gpu_info *d_info, void *stream);

/* The same with a belief supplied by the CALLER (the previous time step of a simulation, an analytic bound) instead
 * of a sample: steps 3 + 5 for a whole field (nranks must be 1, N_total == N, N >= 64).  d_stats_all = the believed
 * {max|x|, min|x|, sum}; only the maximum matters.  The result is always that of the two-pass path; a wrong belief
 * costs a second compress pass (d_info->n_exact_path = 1).                                                    */
int dctz_gpu_compress_known_stats_dev(dctz_gpu_ctx *ctx, const void *d_in, size_t N, size_t N_total, int datatype,
                                      double error_bound, int mode_qt, const double *d_stats_all, int nranks,
                                      int first_slab, uint8_t *d_bin_index, float *d_DC, float *d_AC_exact,
                                      void *d_qtable_raw, dctz_gpu_info *d_info, void *stream);

/* Phase 3 (QT only): d_qtable_raw now holds the GLOBAL maxima (after the caller's all-reduce;
 * entry 0 = DC of the field's last block).  Writes the clamped table to d_qtable, rescales the
 * slab's outliers into d_AC_exact and finalises d_info->n_outliers.                            */
int dctz_gpu_qt_finish_dev(dctz_gpu_ctx *ctx, int datatype, double error_bound, const void *d_qtable_raw,
                           void *d_qtable, float *d_AC_exact, dctz_gpu_info *d_info, void *stream);

/* Phases 1+2(+3) of ONE RANK of a multi-GPU job, with the exchange between them done inside the library over the
 * caller's NCCL communicator (`nccl_comm` is an ncclComm_t passed as void*): statistics -> ncclAllGather of
 * {max, min, sum} (24 bytes per rank) -> compress [-> QT: ncclAllReduce(max) of the 64-entry table, entry 0
 * broadcast from `last_rank_with_data` (the rank whose slab ends the field) -> rescale].  Everything is enqueued
 * on `stream`; the call does not synchronise with the host.  Every rank calls it with its own slab (N > 0; slabs
 * are contiguous runs of whole blocks in rank order, only the last may end with a partial block) -- this is what
 * a C / MPI caller uses where bench.py uses torch.distributed.  NCCL is looked up in the process at run time
 * (DCTZ_GPU_ENODEV if there is none); the library does not link it.                                    */
int dctz_gpu_compress_slab_comm(dctz_gpu_ctx *ctx, void *nccl_comm, int rank, int nranks, int last_rank_with_data,
                                const void *d_in, size_t N, size_t N_total, int datatype, double error_bound,
                                int mode_qt, uint8_t *d_bin_index, float *d_DC, float *d_AC_exact, void *d_qtable,
                                void *d_qtable_raw, dctz_gpu_info *d_info, void *stream);

/* Convenience: phases 1+2(+3) for a whole field on one GPU, nothing leaves the device.          */
int dctz_gpu_compress_field_dev(dctz_gpu_ctx *ctx, const void *d_in, size_t N, int datatype,
                                double error_bound, int mode_qt, uint8_t *d_bin_index, float *d_DC,
                                float *d_AC_exact, void *d_qtable, void *d_qtable_raw,
                                dctz_gpu_info *d_info, void *stream);

/* Dequantise + inverse DCT + de-scale of a slab.  d_AC_exact points at the slab's first outlier and holds
 * n_outliers readable floats (the slab's own count, or everything up to the end of the field's array): the
 * kernels never read past them.  If the bin indices mark more outliers than that (a truncated or damaged
 * stream) the affected tiles decode without their outliers and *d_corrupt (a 32-bit word on the device, may be
 * NULL; the caller clears it beforehand) is set to 1.  d_DC needs float alignment only (a slab's slice of a
 * concatenated DC array is fine); d_bin_index and d_out must be 16-byte aligned.                          */
int dctz_gpu_decompress_dev(dctz_gpu_ctx *ctx, const uint8_t *d_bin_index, const float *d_DC,
                            const float *d_AC_exact, uint64_t n_outliers, const void *d_qtable, size_t N,
                            int datatype, double error_bound, double sf, int mode_qt, void *d_out,
                            uint32_t *d_corrupt, void *stream);

/* ---- region decompression: element ranges of a slab without decoding the rest (DESIGN.md §4.4) ------------------
 * The offset of a block's first outlier in AC_exact is the number of 255 markers in every block before it.  The outlier
 * index holds that count per tile of 32 blocks, scanned, so that any block can be decoded on its own.  It is about
 * 0.2 % of bin_index; its layout is private to the library.  A slab of a multi-GPU field gets its own index. */

/* Bytes of the outlier index of an N-element slab (a function of N only). */
size_t dctz_gpu_outlier_index_bytes(size_t N);

/* Build the index of a slab's bin ids into the caller's device buffer d_index (16-byte aligned,
 * outlier_index_bytes(N) bytes).  It is the same pre-pass decompress runs (k_count_bins + k_scan_groups),
 * kept instead of discarded.  d_n_outliers (may be NULL): the number of outliers the bin ids mark
 * (full blocks + tail), i.e. what a stream header's tot_AC_exact_count must say.  The index stays valid for as
 * long as the bin ids do not change. */
int dctz_gpu_outlier_index_dev(dctz_gpu_ctx *ctx, const uint8_t *d_bin_index, size_t N, void *d_index,
                               uint64_t *d_n_outliers, void *stream);

/* Decode nranges element ranges of the slab.  d_ranges = nranges pairs {first element, count} (uint64, device).
 * The ranges may come in any order and may overlap.  d_out receives their elements concatenated in range order
 * (sum of counts elements; element-aligned).  Other arguments as in dctz_gpu_decompress_dev; the values are
 * bit-identical to the same elements of dctz_gpu_decompress_dev's output.  d_index: built by
 * dctz_gpu_outlier_index_dev for these bin ids and this N.
 * *d_corrupt (may be NULL, cleared by the caller): bit 0 is set as in decompress_dev (more markers than outliers,
 * or an index not built for this N: then nothing is written); bit 1 is set when a range leaves [0, N) or has
 * count 0; that range's part of d_out (its stated count) is not written, the others are.  Bit 1 is also set, and nothing written, when the ranges touch more than
 * 2^32 - 4096 tiles in all.  A range decodes every 64-element block it touches and reads the bin ids of its
 * tile (2048 elements) from the tile's start: narrow ranges cost more per element than wide ones.          */
int dctz_gpu_decompress_ranges_dev(dctz_gpu_ctx *ctx, const uint8_t *d_bin_index, const float *d_DC,
                                   const float *d_AC_exact, uint64_t n_outliers, const void *d_qtable, size_t N,
                                   int datatype, double error_bound, double sf, int mode_qt, const void *d_index,
                                   const uint64_t *d_ranges, size_t nranges, void *d_out, uint32_t *d_corrupt,
                                   void *stream);

/* x[i] <- x[i] / sf with IEEE division (the reference's in-place scaling, dctz-comp-lib.c:193-216),
 * and its inverse x[i] <- x[i] * sf (dctz-test.c:186-210, dctz-decomp-lib.c:494-511).          */
int dctz_gpu_scale_dev(dctz_gpu_ctx *ctx, void *d_x, size_t N, int datatype, double sf, int multiply,
                       void *stream);

/* ---- thin GPU-backed equivalents of the reference's DCT entry points (dct.h:17-27) -----------
 * nblocks contiguous blocks of dn elements each (dn = 64 uses the register-resident kernels,
 * any other 1 <= dn <= 64 the generic tail kernel).  Host buffers, synchronous.                */
int dctz_gpu_dct_blocks(dctz_gpu_ctx *ctx, const void *in, void *out, size_t nblocks, int dn, int datatype,
                        int inverse);

/* Transform only, device buffers: nblocks blocks of 64 elements, d_in -> d_out (may be the same buffer).
 * variant 0 = register-resident butterfly (the kernel the codec uses), 1 = matrix form on the FP64 tensor
 * pipe (mma.sync m8n8k4, double only), 2 = the matrix form with the even/odd split (two 32x32 products, half
 * the flops; double only) -- the comparison BASELINE config[3] asks for.                                */
int dctz_gpu_dct64_dev(dctz_gpu_ctx *ctx, const void *d_in, void *d_out, size_t nblocks, int datatype, int inverse,
                       int variant, void *stream);
/* Measured FP64 issue rate of the device in TFLOP/s: kind 0 = fused multiply-adds on the vector pipe,
 * 1 = mma.sync.m8n8k4.f64 on the tensor pipe (the denominators of that comparison).  Synchronous.        */
int dctz_gpu_fp64_rate(dctz_gpu_ctx *ctx, int kind, double *tflops);

/* ---- utilities ----------------------------------------------------------------------------- */
/* Elements [start, start+count) of the exactly reproducible synthetic 3-D field of SURVEY.md §8d
 * (config C5), written as doubles to d_out; host twin: dctz_b200/fields.py:hash_field.          */
int dctz_gpu_fill_hash_field(dctz_gpu_ctx *ctx, double *d_out, uint64_t start, uint64_t count, uint32_t dim,
                             uint32_t seed, void *stream);
/* sf exactly as the host libm computes it (util.c:28/42) but through the device-side threshold
 * tables; exported so the tables can be verified against libm on the CPU.                       */
double dctz_gpu_sf_from_max(const dctz_gpu_ctx *ctx, double max_abs, int datatype);
/* Self-test of the exact reciprocal division used by the kernels: compares a/b computed by the
 * FMA sequence with IEEE division for `count` pseudo-random a; returns the mismatch count.      */
int dctz_gpu_selftest_division(dctz_gpu_ctx *ctx, int datatype, double b, uint64_t count, uint32_t seed,
                               uint64_t *mismatches);
/* Number of kernels launched by this context so far (bench.py's gpu_launches).                  */
uint64_t dctz_gpu_launch_count(const dctz_gpu_ctx *ctx);
/* Stage timers of the host-buffer calls (the reference prints sf_t / dct_t / idct_t under -DTIME_DEBUG,
 * dctz-comp-lib.c:762-773, dctz-decomp-lib.c:513-528).  set_timing(1) makes compress_core / decompress_core run
 * upload, statistics and transform strictly one after the other with CUDA events between them (the default
 * overlaps them); returns the previous setting.  last_call_stats: times_ms[0] upload, [1] statistics,
 * [2] transform kernels (CUDA events, only with timing on), [3] wall clock until the kernels were done,
 * [4] wall clock of the downloads + host-side scaling; and the PCIe bytes the call moved.          */
int dctz_gpu_set_timing(dctz_gpu_ctx *ctx, int on);
/* Where the microseconds of a small field go: phase boundaries of the last single-launch kernel (kernel 0 =
 * compress: start, statistics done, past barrier 1, compress done, past barrier 2, end; 1 = decompress: start,
 * markers counted, past the barrier, end).  For stamp k the earliest CTA is out_us[2k], the latest out_us[2k+1],
 * in microseconds after the first CTA started.  Synchronises the device.                              */
int dctz_gpu_fused_phase_times(dctz_gpu_ctx *ctx, int kernel, double out_us[16]);
int dctz_gpu_last_call_stats(const dctz_gpu_ctx *ctx, double times_ms[8], uint64_t *h2d_bytes, uint64_t *d2h_bytes);

#ifdef __cplusplus
}
#endif
#endif /* DCTZ_GPU_H */
