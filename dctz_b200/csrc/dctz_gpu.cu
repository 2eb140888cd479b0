// dctz_gpu.cu -- C-ABI of the B200-native DCTZ hot path (include/dctz_gpu.h).
//
// Host side of the kernels in kernels.cuh: context / scratch management, launch configuration,
// the sf threshold tables (built with the host libm so that the device reproduces util.c:28/42
// bit for bit without a host round trip), and the host-buffer entry points that the reference's
// dctz_compress()/dctz_decompress() call at the seam described in include/dctz_gpu.h.
//
// There is no CPU fallback anywhere in this file: every entry point needs a CUDA device.
#include <cuda.h>
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <new>
#include <thread>
#include <vector>

#include "../../include/dctz_gpu.h"
#include "fused.cuh"
#include "ranges.cuh"

using namespace dctz;

static_assert(sizeof(Info) == sizeof(dctz_gpu_info), "Info must mirror dctz_gpu_info");
static_assert(DCTZ_GPU_BLK == BLK, "block size");

static thread_local char g_err[512] = "";

struct DevBuf {  // grow-only device allocation
  void *p = nullptr;
  size_t cap = 0;
};

// ------------------------------------------------------------------------------------------
// Host worker threads of the host-buffer API: staging copies between the caller's pageable memory and
// the pinned ring, and the caller-visible x/sf (IEEE division) that the reference leaves in its input
// buffer.  One job at a time; parts are handed out by an atomic counter.
// ------------------------------------------------------------------------------------------
class HostPool {
  struct Job {  // immutable per start(): a straggler that still holds the previous job can never touch the next one
    std::function<void(int)> fn;
    int nparts = 0;
    std::atomic<int> next{0};
    int pending = 0;  // guarded by mu_
  };

 public:
  explicit HostPool(int nthreads) {
    for (int t = 0; t < nthreads; t++) workers_.emplace_back([this] { loop(); });
  }
  ~HostPool() {
    {
      std::lock_guard<std::mutex> lk(mu_);
      stop_ = true;
    }
    cv_.notify_all();
    for (auto &w : workers_) w.join();
  }
  int size() const { return (int)workers_.size(); }
  // fn(part) for part in [0, nparts): start() returns at once, wait() joins (the calling thread works too)
  void start(int nparts, std::function<void(int)> fn) {
    auto j = std::make_shared<Job>();
    j->fn = std::move(fn);
    j->nparts = nparts;
    j->pending = nparts;
    {
      std::lock_guard<std::mutex> lk(mu_);
      job_ = j;
      gen_++;
    }
    cv_.notify_all();
  }
  void wait() {
    std::shared_ptr<Job> j;
    {
      std::lock_guard<std::mutex> lk(mu_);
      j = job_;
    }
    if (!j) return;
    run_parts(*j);
    std::unique_lock<std::mutex> lk(mu_);
    done_cv_.wait(lk, [&] { return j->pending == 0; });
    if (job_ == j) job_.reset();
  }
  void parallel_for(int nparts, std::function<void(int)> fn) {
    start(nparts, std::move(fn));
    wait();
  }

 private:
  void run_parts(Job &j) {
    for (;;) {
      const int i = j.next.fetch_add(1);
      if (i >= j.nparts) return;
      j.fn(i);
      std::lock_guard<std::mutex> lk(mu_);
      if (--j.pending == 0) done_cv_.notify_all();
    }
  }
  void loop() {
    unsigned long seen = 0;
    for (;;) {
      std::shared_ptr<Job> j;
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] { return stop_ || gen_ != seen; });
        if (stop_) return;
        seen = gen_;
        j = job_;
      }
      if (j) run_parts(*j);
    }
  }
  std::vector<std::thread> workers_;
  std::mutex mu_;
  std::condition_variable cv_, done_cv_;
  std::shared_ptr<Job> job_;
  unsigned long gen_ = 0;
  bool stop_ = false;
};

constexpr size_t STAGE_BYTES = (size_t)16 << 20;  // one slot of the pinned staging ring
constexpr int NSTAGE = 3;
constexpr size_t PINNED_CHUNK = (size_t)64 << 20;  // copy granularity when the caller's memory is already page-locked
constexpr size_t GATE_BYTES = (size_t)64 << 20;    // transfers of at least this size take their direction's link gate

// One PCIe link per device, full duplex.  A compress call is upload-heavy, a decompress call download-heavy; two host
// threads with a context each that would run in phase (both uploading, then both downloading) use one direction at a
// time.  The direction-dominant transfer of a call therefore holds its direction's gate: concurrent callers fall into
// step with one uploading while the other downloads.  The other call's SHORT transfer in the gated direction must not
// queue behind the long one: a copy engine stays with a stream for as long as that stream has another copy queued
// (tools/probes/link_interleave.cu: 128 MiB submitted beside a 1 GiB transfer kept 2-3 pieces deep completes after
// 17 ms, beside one kept ONE piece deep after 2.5 ms), so while a second host-buffer call is active on the device a
// dominant transfer submits its next piece only when the previous one has landed.  DCTZ_LINK_GATES=0: gates off.
struct LinkGate { std::mutex up, down; std::atomic<int> busy{0}; };
static LinkGate g_gate[64];
struct BusyMark {  // a host-buffer call in progress on the device
  explicit BusyMark(int dev) : g(dev >= 0 && dev < 64 ? &g_gate[dev] : nullptr) { if (g) g->busy.fetch_add(1); }
  ~BusyMark() { if (g) g->busy.fetch_sub(1); }
  LinkGate *g;
};
static bool link_contended(int dev) { return dev >= 0 && dev < 64 && g_gate[dev].busy.load(std::memory_order_relaxed) > 1; }
static bool link_gates_enabled() {
  static const bool on = [] { const char *e = getenv("DCTZ_LINK_GATES"); return !(e && atoi(e) == 0); }();
  return on;
}

struct dctz_gpu_ctx {
  int device = 0;
  int sm_count = 0;
  cudaStream_t stream = nullptr;  // used by the host-buffer API (kernels)
  cudaStream_t copy_stream = nullptr;  // host-buffer API: H2D / D2H copies, overlapped with the kernels through events
  cudaEvent_t ev_chain = nullptr, ev_time[4] = {nullptr, nullptr, nullptr, nullptr};
  void *stage[NSTAGE] = {nullptr, nullptr, nullptr};  // pinned staging ring (allocated on first use with pageable memory)
  cudaEvent_t stage_ev[NSTAGE] = {nullptr, nullptr, nullptr};
  HostPool *pool = nullptr;
  DevBuf chunk_stats;  // {max,min,sum} per chunk of a pipelined upload
  int timing = 0;      // stage timers requested (dctz_gpu_set_timing): the stages then run one after the other
  double times[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  std::chrono::steady_clock::time_point t_call;  // start of the current host-buffer call (times[5..7] count from here)
  uint64_t h2d_bytes = 0, d2h_bytes = 0;  // PCIe traffic of the last host-buffer call
  char err[512] = "";
  uint64_t launches = 0;

  // small fixed scratch
  StatPartial *d_partials = nullptr;
  int stat_grid = 0;
  unsigned *d_done = nullptr;
  double *d_stats3 = nullptr;
  DevParams *d_params = nullptr;
  Info *d_info = nullptr;
  TileControl *d_ctl = nullptr;
  unsigned long long *d_nconsumed = nullptr;
  unsigned long long *d_mismatch = nullptr;
  QualityPartial *d_qpartials = nullptr;  // [stat_grid] + 1 result slot
  double *d_stats_host3 = nullptr;        // 3 doubles for compress_core_with_stats
  DevBuf status;        // [group_prefix: u64 per 32 tiles][counts: u32 per warp tile]
  DevBuf slots;         // EC: tile-strided outlier scratch (TILE_SLOT floats per warp tile)
  DevBuf qt_raw, qt_j;  // QT: tile-strided un-rescaled outliers + their coefficient position
  unsigned qt_entries = 0;  // tiles (incl. the tail slot) of the last QT compress call
  unsigned qt_tail_tile = 0xFFFFFFFFu;  // index of that tail slot (its raw values are scaled already), none = ~0

  // sf tables: host copies + device copies
  std::vector<double> thr_d, sfv_d;
  std::vector<float> thr_f, sfv_f;
  double min_d = 0;
  float min_f = 0;
  SfTables tb{};

  // buffers of the host-buffer API
  DevBuf in, bins, dc, ac, qt, qtraw, out;
  double *d_dfrag[2] = {nullptr, nullptr};  // DMMA A-fragments of the DCT matrix (forward, inverse)
  double *d_dfrag2[2] = {nullptr, nullptr}; // ... of its even / odd halves (k_dct64_dmma_split)
  int occ[2][2][2] = {};  // resident CTAs/SM per [kernel][datatype][qt]
  int occ_ahead[2][2] = {};  // ... of the count-ahead decompress kernel [datatype][qt]
  int decomp_ahead = -1;     // DCTZ_DECOMP_AHEAD: 1 = streaming decompress always without the pre-pass, 0 = never, unset = double where the stated outlier density is below 1/128, float never (DESIGN.md 4.3)
  int l2_hints = -1;         // DCTZ_L2_HINTS: bit 0 stores evict_first, bit 1 bin-id copies evict_first, bit 2 pre-pass path: tiles from the last one down; -1 = 3 for the count-ahead path, 0 otherwise
  DevBuf ahead_buf;          // decompress without the pre-pass: counts[t] | agg[u] | S[u/64] | T[u/2048], zeroed before every launch
  // single-launch kernels for small fields (fused.cuh)
  int occ_fused[2][2][2] = {};
  size_t fused_max_bytes = (size_t)256 << 20;  // fields up to this size take the single-launch path (DCTZ_FUSED_MAX_MB, 0 = never)
  int coop = 0;                                // cooperative launches supported
  int single_read = 1;                         // whole fields take the single-read (sample + verify) path (DCTZ_SINGLE_READ=0: two passes)
  unsigned long long *d_barrier = nullptr;     // [0] compress, [1] decompress: grid-barrier arrival counters (monotonic)
  unsigned long long barrier_base[2] = {0, 0}; // what the counters will have reached when the next launch starts
  unsigned long long *d_cta_totals = nullptr;  // outliers per CTA (two halves: compress, decompress)
  unsigned long long *d_qmax_scratch = nullptr;  // QT: 64 per-position maxima (bit patterns)
  DevBuf tile_off;                             // decompress: offset of every tile's run inside its CTA's range
  double *d_tail3 = nullptr;                   // exact {max, min, sum} of the partial tail block (k_sample)
  double *d_spec3 = nullptr;                   // [0..2] belief, [3..5] true statistics of the single-read path (whole fields)
  unsigned long long *d_sample_bits = nullptr; // k_sample: running maximum (bit pattern)
  DevBuf tile_sums;                            // per-tile sums + per-4096-tile partials (MODE_BELIEF)
  unsigned long long *d_dbg = nullptr;         // phase timestamps of the last single-launch kernels: [2][sm_count * 4][8]
  int dbg_grid[2] = {0, 0};
  int fused_stamps = 0;                        // DCTZ_FUSED_STAMPS=1: the single-launch kernels record their phase boundaries (dctz_gpu_fused_phase_times)
  // region decompression (ranges.cuh)
  int occ_ranges[2][2] = {};  // resident CTAs/SM of k_decompress_ranges [datatype][qt]
  DevBuf region;              // [RangeCtl][piece_at, out_at: u64 per range][chunk_piece, chunk_out: u64 per 1024 ranges]
};

// ------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------
static int fail(dctz_gpu_ctx *ctx, int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  snprintf(g_err, sizeof g_err, "%s", buf);
  if (ctx) snprintf(ctx->err, sizeof ctx->err, "%s", buf);
  return code;
}
#define CU(call)                                                                                          \
  do {                                                                                                    \
    cudaError_t e_ = (call);                                                                              \
    if (e_ != cudaSuccess)                                                                                \
      return fail(ctx, e_ == cudaErrorMemoryAllocation ? DCTZ_GPU_ENOMEM : DCTZ_GPU_ECUDA, "%s: %s (%s:%d)", \
                  #call, cudaGetErrorString(e_), __FILE__, __LINE__);                                     \
  } while (0)
#define TRY(call)            \
  do {                       \
    int r_ = (call);         \
    if (r_ != DCTZ_GPU_OK) return r_; \
  } while (0)

// The QT outlier slots start at the first address of their allocation that is a multiple of a slot's size (park_if, kernels.cuh)
static void *qt_raw_slots(const dctz_gpu_ctx *ctx) { return (void *)(((uintptr_t)ctx->qt_raw.p + QT_RAW_ALIGN - 1) / QT_RAW_ALIGN * QT_RAW_ALIGN); }
static uint8_t *qt_j_slots(const dctz_gpu_ctx *ctx) { return (uint8_t *)(((uintptr_t)ctx->qt_j.p + QT_J_ALIGN - 1) / QT_J_ALIGN * QT_J_ALIGN); }

static int grow(dctz_gpu_ctx *ctx, DevBuf &b, size_t bytes, bool zero = false) {
  if (bytes <= b.cap) return DCTZ_GPU_OK;
  if (b.p) { CU(cudaFree(b.p)); b.p = nullptr; b.cap = 0; }
  size_t want = bytes + bytes / 8 + 256;
  CU(cudaMalloc(&b.p, want));
  b.cap = want;
  if (zero) CU(cudaMemset(b.p, 0, want));
  return DCTZ_GPU_OK;
}

// ------------------------------------------------------------------------------------------
// sf threshold tables.  sf = pow(10, ceil(log10(max)) - 1) (util.c:28); float: powf(10,
// ceil(log10f(max)) - 1) (util.c:42).  T_k := smallest value whose libm log10 exceeds k, found by
// bisection on the bit pattern around 10^k; then ceil(log10(max)) == k  <=>  T_{k-1} <= max < T_k.
// ------------------------------------------------------------------------------------------
static double bits_to_d(uint64_t u) { double d; memcpy(&d, &u, 8); return d; }
static uint64_t d_to_bits(double d) { uint64_t u; memcpy(&u, &d, 8); return u; }
static float bits_to_f(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
static uint32_t f_to_bits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }

static double threshold_d(int k) {
  const double c = pow(10.0, (double)k);
  uint64_t lo = d_to_bits(c * (1.0 - 1e-9)), hi = d_to_bits(c * (1.0 + 1e-9));  // log10(lo) <= k < log10(hi)
  while (hi - lo > 1) {
    const uint64_t mid = lo + (hi - lo) / 2;
    if (log10(bits_to_d(mid)) > (double)k) hi = mid; else lo = mid;
  }
  return bits_to_d(hi);
}
static float threshold_f(int k) {
  const float c = powf(10.0f, (float)k);
  uint32_t lo = f_to_bits(c * (1.0f - 1e-4f)), hi = f_to_bits(c * (1.0f + 1e-4f));
  while (hi - lo > 1) {
    const uint32_t mid = lo + (hi - lo) / 2;
    if (log10f(bits_to_f(mid)) > (float)k) hi = mid; else lo = mid;
  }
  return bits_to_f(hi);
}

// Compress admits max|x| in [T_{kmin-1}, T_kmax), i.e. sf = 10^(k-1) for k = kmin..kmax (DESIGN.md §2, "admitted exponent
// range"): the kernels transform the UNSCALED block and quantise with kq = 1/(sf*bin_width), so below sf = 1e-302 (float
// 1e-32) kq overflows at eb = 1E-6, and above sf = 1e305 (float 1e35) the unscaled transform overflows: the butterflies sum
// all 64 values of a constant block before the factor 1/8, so 64 * max|x| must stay finite.
// sfv holds one entry past the table (read, never used, by sf_window at the upper end).
constexpr int SF_KMIN_D = -301, SF_KMAX_D = 306, SF_KMIN_F = -31, SF_KMAX_F = 36;
static void build_sf_tables(dctz_gpu_ctx *c) {
  const int kmin_d = SF_KMIN_D, kmax_d = SF_KMAX_D;
  c->min_d = threshold_d(kmin_d - 1);
  for (int k = kmin_d; k <= kmax_d; k++) {
    c->thr_d.push_back(threshold_d(k));
    c->sfv_d.push_back(pow(10, (double)k - 1));  // the literal expression of util.c:28 for ceil(.) == k
  }
  c->sfv_d.push_back(pow(10, (double)(kmax_d + 1) - 1));
  const int kmin_f = SF_KMIN_F, kmax_f = SF_KMAX_F;
  c->min_f = threshold_f(kmin_f - 1);
  for (int k = kmin_f; k <= kmax_f; k++) {
    c->thr_f.push_back(threshold_f(k));
    c->sfv_f.push_back(powf(10, (double)k - 1));  // util.c:42: powf(10, ceil(..) - 1); the exponent is a double narrowed to float
  }
  c->sfv_f.push_back(powf(10, (double)(kmax_f + 1) - 1));
}

template <typename T> static int host_lookup(const std::vector<T> &thr, T mx) {
  int lo = 0, hi = (int)thr.size();
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (mx < thr[mid]) hi = mid; else lo = mid + 1; }
  return lo;
}

// ------------------------------------------------------------------------------------------
// lifetime
// ------------------------------------------------------------------------------------------
template <typename K> static int kernel_occupancy(K kernel, int threads, size_t smem) {
  int n = 0;
  if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, threads, smem) != cudaSuccess) return 0;
  return n;
}

extern "C" int dctz_gpu_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

extern "C" const char *dctz_gpu_last_error(const dctz_gpu_ctx *ctx) { return ctx ? ctx->err : g_err; }

extern "C" void dctz_gpu_destroy(dctz_gpu_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  void *small[] = {ctx->d_tail3, ctx->d_spec3, ctx->d_sample_bits, ctx->tile_sums.p, ctx->d_dbg, ctx->d_barrier, ctx->d_cta_totals, ctx->d_qmax_scratch, ctx->tile_off.p, ctx->d_partials, ctx->d_done, ctx->d_stats3, ctx->d_params, ctx->d_info, ctx->d_ctl,
                   ctx->d_nconsumed, ctx->d_mismatch, ctx->d_qpartials, ctx->d_stats_host3, (void *)ctx->tb.thr_d, (void *)ctx->tb.sf_d,
                   (void *)ctx->tb.thr_f, (void *)ctx->tb.sf_f};
  for (void *p : small) if (p) cudaFree(p);
  DevBuf *bufs[] = {&ctx->status, &ctx->slots, &ctx->qt_raw, &ctx->qt_j, &ctx->in, &ctx->bins, &ctx->dc, &ctx->ac,
                    &ctx->qt, &ctx->qtraw, &ctx->out, &ctx->region};
  for (DevBuf *b : bufs) if (b->p) cudaFree(b->p);
  for (double *p : ctx->d_dfrag) if (p) cudaFree(p);
  for (double *p : ctx->d_dfrag2) if (p) cudaFree(p);
  if (ctx->chunk_stats.p) cudaFree(ctx->chunk_stats.p);
  if (ctx->ahead_buf.p) cudaFree(ctx->ahead_buf.p);
#ifdef DCTZ_WAIT_STATS
  {
    unsigned long long w[3] = {};
    if (cudaMemcpyFromSymbol(w, g_wait_stats, sizeof w) == cudaSuccess)
      fprintf(stderr, "dctz wait stats: %llu units counted, decode re-reads of unpublished counts %llu, count-warp looks at a closed lead window %llu\n",
              w[2], w[0], w[1]);
  }
#endif
  delete ctx->pool;
  for (int i = 0; i < NSTAGE; i++) {
    if (ctx->stage[i]) cudaFreeHost(ctx->stage[i]);
    if (ctx->stage_ev[i]) cudaEventDestroy(ctx->stage_ev[i]);
  }
  if (ctx->ev_chain) cudaEventDestroy(ctx->ev_chain);
  for (cudaEvent_t e : ctx->ev_time) if (e) cudaEventDestroy(e);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

template <typename T> static int upload_table(dctz_gpu_ctx *ctx, const std::vector<T> &v, const T **dst) {
  void *p = nullptr;
  CU(cudaMalloc(&p, v.size() * sizeof(T)));
  CU(cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  *dst = (const T *)p;
  return DCTZ_GPU_OK;
}

static int ctx_init(dctz_gpu_ctx *ctx, int device) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(ctx, DCTZ_GPU_ENODEV, "no CUDA device available (this library has no CPU path)");
  }
  if (device < 0 || device >= ndev) return fail(ctx, DCTZ_GPU_EINVAL, "device %d out of range [0,%d)", device, ndev);
  ctx->device = device;
  CU(cudaSetDevice(device));
  CU(cudaMemcpyToSymbol(dct64_kd, dct64_kd_host, sizeof(dct64_kd_host)));  // the double transform's constants (dct64_gen.cuh)
  {
    const char *e = getenv("DCTZ_L2_HINTS");
    const int v = e ? (atoi(e) > 0) : 0;  // (the pre-pass reads the bin ids with evict_last)
    CU(cudaMemcpyToSymbol(c_l2_hints, &v, sizeof(int)));
  }
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(ctx, DCTZ_GPU_ENODEV, "device %d is sm_%d%d; this build contains sm_100a code only", device, prop.major, prop.minor);
  ctx->sm_count = prop.multiProcessorCount;
  CU(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  CU(cudaEventCreateWithFlags(&ctx->ev_chain, cudaEventDisableTiming));
  for (cudaEvent_t &e : ctx->ev_time) CU(cudaEventCreate(&e));
  ctx->stat_grid = ctx->sm_count * 8;
  CU(cudaMalloc(&ctx->d_partials, sizeof(StatPartial) * ctx->stat_grid));
  CU(cudaMalloc(&ctx->d_done, 8 * sizeof(unsigned)));  // [0] k_stats, [1] k_scan_groups, [2] k_quality, [3] k_count_bins, [4] k_qt_max, [5] k_sample, [6] k_reduce_tile_sums
  CU(cudaMemset(ctx->d_done, 0, 8 * sizeof(unsigned)));
  CU(cudaMalloc(&ctx->d_tail3, 3 * sizeof(double)));
  CU(cudaMalloc(&ctx->d_spec3, 6 * sizeof(double)));
  CU(cudaMalloc(&ctx->d_sample_bits, 4 * sizeof(unsigned long long)));  // [0] k_sample's running maximum, [1] extreme high words, [2..3] exact extremes
  CU(cudaMemset(ctx->d_sample_bits, 0, 4 * sizeof(unsigned long long)));
  CU(cudaMalloc(&ctx->d_stats3, 3 * sizeof(double)));
  CU(cudaMalloc(&ctx->d_params, sizeof(DevParams)));
  CU(cudaMalloc(&ctx->d_info, sizeof(Info)));
  CU(cudaMalloc(&ctx->d_ctl, 2 * sizeof(TileControl)));
  CU(cudaMemset(ctx->d_ctl, 0, 2 * sizeof(TileControl)));
  {
    const unsigned long long ones = ~0ull;  // the running minimum of |x| (bit pattern) rests at all ones
    CU(cudaMemcpy(&ctx->d_ctl[0].min_bits, &ones, sizeof ones, cudaMemcpyHostToDevice));
  }
  CU(cudaMalloc(&ctx->d_nconsumed, sizeof(unsigned long long)));
  CU(cudaMalloc(&ctx->d_mismatch, sizeof(unsigned long long)));
  CU(cudaMalloc(&ctx->d_qpartials, sizeof(QualityPartial) * (ctx->stat_grid + 1)));
  CU(cudaMalloc(&ctx->d_stats_host3, 3 * sizeof(double)));
  build_sf_tables(ctx);
  TRY(upload_table(ctx, ctx->thr_d, &ctx->tb.thr_d));
  TRY(upload_table(ctx, ctx->sfv_d, &ctx->tb.sf_d));
  TRY(upload_table(ctx, ctx->thr_f, &ctx->tb.thr_f));
  TRY(upload_table(ctx, ctx->sfv_f, &ctx->tb.sf_f));
  ctx->tb.n_d = (int)ctx->thr_d.size();
  ctx->tb.n_f = (int)ctx->thr_f.size();
  ctx->tb.kmin_d = SF_KMIN_D;
  ctx->tb.kmin_f = SF_KMIN_F;
  ctx->tb.min_d = ctx->min_d;
  ctx->tb.min_f = ctx->min_f;
  ctx->tb.max_d = ctx->thr_d.back();
  ctx->tb.max_f = ctx->thr_f.back();
  // kernel attributes + residency (persistent grids are sized from these)
  ctx->occ[0][1][0] = kernel_occupancy(k_compress<double, false, false>, CompressCfg<double, false>::THREADS, CompressCfg<double, false>::SMEM);
  ctx->occ[0][1][1] = kernel_occupancy(k_compress<double, true, false>, CompressCfg<double, true>::THREADS, CompressCfg<double, true>::SMEM);
  ctx->occ[0][0][0] = kernel_occupancy(k_compress<float, false, false>, CompressCfg<float, false>::THREADS, CompressCfg<float, false>::SMEM);
  ctx->occ[0][0][1] = kernel_occupancy(k_compress<float, true, false>, CompressCfg<float, true>::THREADS, CompressCfg<float, true>::SMEM);
  // the VERIFY instantiations (caller-supplied statistics) need the same shared-memory opt-in
  if (kernel_occupancy(k_compress<double, false, true>, CompressCfg<double, false>::THREADS, CompressCfg<double, false>::SMEM) < 1 ||
      kernel_occupancy(k_compress<double, true, true>, CompressCfg<double, true>::THREADS, CompressCfg<double, true>::SMEM) < 1 ||
      kernel_occupancy(k_compress<float, false, true>, CompressCfg<float, false>::THREADS, CompressCfg<float, false>::SMEM) < 1 ||
      kernel_occupancy(k_compress<float, true, true>, CompressCfg<float, true>::THREADS, CompressCfg<float, true>::SMEM) < 1)
    return fail(ctx, DCTZ_GPU_ECUDA, "k_compress<VERIFY> cannot be made resident");
  ctx->occ[1][1][0] = kernel_occupancy(k_decompress<double, false, false>, DecompressCfg<double, false>::THREADS, DecompressCfg<double, false>::SMEM);
  ctx->occ[1][1][1] = kernel_occupancy(k_decompress<double, true, false>, DecompressCfg<double, true>::THREADS, DecompressCfg<double, true>::SMEM);
  ctx->occ[1][0][0] = kernel_occupancy(k_decompress<float, false, false>, DecompressCfg<float, false>::THREADS, DecompressCfg<float, false>::SMEM);
  ctx->occ[1][0][1] = kernel_occupancy(k_decompress<float, true, false>, DecompressCfg<float, true>::THREADS, DecompressCfg<float, true>::SMEM);
  ctx->occ_ahead[1][0] = kernel_occupancy(k_decompress<double, false, true>, SplitCfg::THREADS, DecompressCfg<double, false>::SMEM);
  ctx->occ_ahead[1][1] = kernel_occupancy(k_decompress<double, true, true>, SplitCfg::THREADS, DecompressCfg<double, true>::SMEM);
  ctx->occ_ahead[0][0] = kernel_occupancy(k_decompress<float, false, true>, SplitCfg::THREADS, DecompressCfg<float, false>::SMEM);
  ctx->occ_ahead[0][1] = kernel_occupancy(k_decompress<float, true, true>, SplitCfg::THREADS, DecompressCfg<float, true>::SMEM);
  {
    const char *e = getenv("DCTZ_DECOMP_AHEAD");
    ctx->decomp_ahead = e ? atoi(e) : -1;  // -1: by the outlier density of the call
    e = getenv("DCTZ_FUSED_STAMPS");
    ctx->fused_stamps = e ? atoi(e) : 0;
    e = getenv("DCTZ_L2_HINTS");
    ctx->l2_hints = e ? atoi(e) : -1;  // -1: the path's own default
  }
  ctx->occ_fused[0][1][0] = kernel_occupancy(k_compress_fused<double, false>, CompressCfg<double, false>::THREADS, CompressCfg<double, false>::SMEM);
  ctx->occ_fused[0][1][1] = kernel_occupancy(k_compress_fused<double, true>, CompressCfg<double, true>::THREADS, CompressCfg<double, true>::SMEM);
  ctx->occ_fused[0][0][0] = kernel_occupancy(k_compress_fused<float, false>, CompressCfg<float, false>::THREADS, CompressCfg<float, false>::SMEM);
  ctx->occ_fused[0][0][1] = kernel_occupancy(k_compress_fused<float, true>, CompressCfg<float, true>::THREADS, CompressCfg<float, true>::SMEM);
  ctx->occ_fused[1][1][0] = kernel_occupancy(k_decompress_fused<double, false>, DecompressCfg<double, false>::THREADS, DecompressCfg<double, false>::SMEM);
  ctx->occ_fused[1][1][1] = kernel_occupancy(k_decompress_fused<double, true>, DecompressCfg<double, true>::THREADS, DecompressCfg<double, true>::SMEM);
  ctx->occ_fused[1][0][0] = kernel_occupancy(k_decompress_fused<float, false>, DecompressCfg<float, false>::THREADS, DecompressCfg<float, false>::SMEM);
  ctx->occ_fused[1][0][1] = kernel_occupancy(k_decompress_fused<float, true>, DecompressCfg<float, true>::THREADS, DecompressCfg<float, true>::SMEM);
  ctx->occ_ranges[1][0] = kernel_occupancy(k_decompress_ranges<double, false>, RangeCfg<double>::THREADS, RangeCfg<double>::SMEM);
  ctx->occ_ranges[1][1] = kernel_occupancy(k_decompress_ranges<double, true>, RangeCfg<double>::THREADS, RangeCfg<double>::SMEM);
  ctx->occ_ranges[0][0] = kernel_occupancy(k_decompress_ranges<float, false>, RangeCfg<float>::THREADS, RangeCfg<float>::SMEM);
  ctx->occ_ranges[0][1] = kernel_occupancy(k_decompress_ranges<float, true>, RangeCfg<float>::THREADS, RangeCfg<float>::SMEM);
  for (int b = 0; b < 2; b++)
    for (int c = 0; c < 2; c++)
      if (ctx->occ_ranges[b][c] < 1) return fail(ctx, DCTZ_GPU_ECUDA, "k_decompress_ranges [%d][%d] cannot be made resident", b, c);
  CU(cudaDeviceGetAttribute(&ctx->coop, cudaDevAttrCooperativeLaunch, device));
  CU(cudaMalloc(&ctx->d_barrier, 2 * sizeof(unsigned long long)));
  CU(cudaMemset(ctx->d_barrier, 0, 2 * sizeof(unsigned long long)));
  CU(cudaMalloc(&ctx->d_cta_totals, 2 * (size_t)ctx->sm_count * 4 * sizeof(unsigned long long)));
  CU(cudaMalloc(&ctx->d_qmax_scratch, BLK * sizeof(unsigned long long)));
  CU(cudaMalloc(&ctx->d_dbg, 2 * (size_t)ctx->sm_count * 4 * 8 * sizeof(unsigned long long)));
  if (const char *e = getenv("DCTZ_FUSED_MAX_MB")) ctx->fused_max_bytes = (size_t)atol(e) << 20;
  if (const char *e = getenv("DCTZ_SINGLE_READ")) ctx->single_read = atoi(e) != 0;
  for (int a = 0; a < 2; a++)
    for (int b = 0; b < 2; b++)
      for (int c = 0; c < 2; c++)
        if (ctx->occ[a][b][c] < 1)
          return fail(ctx, DCTZ_GPU_ECUDA, "kernel [%d][%d][%d] cannot be made resident: %s", a, b, c,
                      cudaGetErrorString(cudaGetLastError()));
  return DCTZ_GPU_OK;
}

extern "C" int dctz_gpu_create(dctz_gpu_ctx **out, int device) {
  if (!out) return fail(nullptr, DCTZ_GPU_EINVAL, "ctx pointer is NULL");
  *out = nullptr;
  dctz_gpu_ctx *ctx = new (std::nothrow) dctz_gpu_ctx();
  if (!ctx) return fail(nullptr, DCTZ_GPU_ENOMEM, "out of host memory");
  const int r = ctx_init(ctx, device);
  if (r != DCTZ_GPU_OK) {
    snprintf(g_err, sizeof g_err, "%s", ctx->err);
    dctz_gpu_destroy(ctx);
    return r;
  }
  *out = ctx;
  return DCTZ_GPU_OK;
}

extern "C" int dctz_gpu_sm_count(const dctz_gpu_ctx *ctx) { return ctx ? ctx->sm_count : 0; }
extern "C" uint64_t dctz_gpu_launch_count(const dctz_gpu_ctx *ctx) { return ctx ? ctx->launches : 0; }

extern "C" void *dctz_gpu_host_alloc(size_t bytes) {
  void *p = nullptr;
  if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return p;
}
extern "C" void dctz_gpu_host_free(void *p) { if (p) cudaFreeHost(p); }

extern "C" double dctz_gpu_sf_from_max(const dctz_gpu_ctx *ctx, double max_abs, int datatype) {
  if (!ctx) return 0.0;
  if (datatype == DCTZ_GPU_DOUBLE) {
    if (!(max_abs >= ctx->min_d && max_abs < ctx->thr_d.back())) return 0.0;  // outside the admitted range (also NaN, inf)
    return ctx->sfv_d[host_lookup(ctx->thr_d, max_abs)];
  }
  const float m = (float)max_abs;
  if (!(m >= ctx->min_f && m < ctx->thr_f.back())) return 0.0;
  return (double)ctx->sfv_f[host_lookup(ctx->thr_f, m)];
}

// ------------------------------------------------------------------------------------------
// TMA tensor maps.  A field (or slab) of nblk full blocks is described as a 2-D byte tensor
// [nblk rows][64*sizeof(T) bytes]; the kernels move [32 rows x 128 bytes] boxes with the 128-byte
// swizzle (common.cuh, WarpTile).  The encoder lives in the driver: fetched once through the runtime,
// so the library does not link libcuda.
// ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;

static int make_tile_map(dctz_gpu_ctx *ctx, CUtensorMap *map, const void *base, size_t row_bytes, unsigned long long nrows) {
  static std::once_flag once;
  std::call_once(once, [] {
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess) g_encode = (EncodeTiledFn)fn;
  });
  if (!g_encode) return fail(ctx, DCTZ_GPU_ECUDA, "cuTensorMapEncodeTiled is not available from this driver");
  const cuuint64_t dims[2] = {(cuuint64_t)row_bytes, (cuuint64_t)nrows};
  const cuuint64_t strides[1] = {(cuuint64_t)row_bytes};
  const cuuint32_t box[2] = {128u, (cuuint32_t)WTILE};
  const cuuint32_t estr[2] = {1u, 1u};
  const CUresult r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void *>(base), dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(ctx, DCTZ_GPU_ECUDA, "cuTensorMapEncodeTiled failed with %d (base %p, %llu rows)", (int)r, base, nrows);
  return DCTZ_GPU_OK;
}

// ------------------------------------------------------------------------------------------
// argument checks shared by the entry points
// ------------------------------------------------------------------------------------------
static int check_common(dctz_gpu_ctx *ctx, int datatype, double eb) {
  if (!ctx) return fail(nullptr, DCTZ_GPU_EINVAL, "ctx is NULL");
  if (datatype != DCTZ_GPU_FLOAT && datatype != DCTZ_GPU_DOUBLE) return fail(ctx, DCTZ_GPU_EINVAL, "datatype %d is neither FLOAT(0) nor DOUBLE(1)", datatype);
  if (!(eb >= 1e-6)) return fail(ctx, DCTZ_GPU_EINVAL, "error bound %g is below 1E-6 (dctz-comp-lib.c:135)", eb);
  return DCTZ_GPU_OK;
}
static bool aligned16(const void *p) { return ((uintptr_t)p & 15u) == 0; }

// Tiles per ticket (TileSeq, common.cuh): 4 once every warp has many batches to go through, 1 for small fields, where
// whole batches would leave part of the grid without work.
#ifndef DCTZ_TILE_BATCH_C
#define DCTZ_TILE_BATCH_C 2u  // (measured on one box against 4 and 1: the same on the 8 GiB slab, 1-2 % faster with outliers and on c4)
#endif
#ifndef DCTZ_TILE_BATCH_D
#define DCTZ_TILE_BATCH_D 4u
#endif
static_assert(DCTZ_TILE_BATCH_D <= 32, "CountedExtents holds the counts of a unit's tiles in the lanes of a warp");
static unsigned tile_batch(size_t ntiles, size_t nwarps, bool compress = false) {
  return ntiles >= 16 * nwarps ? (compress ? DCTZ_TILE_BATCH_C : DCTZ_TILE_BATCH_D) : 1u;
}
static size_t scan_chunks(size_t n_entries) { return ((n_entries + 31) / 32 + 1023) / 1024; }  // k_scan_groups CTAs

// Single-launch path (fused.cuh): whole fields of full blocks up to fused_max_bytes, all CTAs co-resident.
static int fused_grid(const dctz_gpu_ctx *ctx, int kernel, size_t N, size_t es, int mode_qt) {
  static const bool dbg = getenv("DCTZ_DEBUG") != nullptr;
  if (dbg)
    fprintf(stderr, "fused_grid: kernel %d N %zu es %zu qt %d coop %d max_bytes %zu occ %d\n", kernel, N, es, mode_qt, ctx->coop, ctx->fused_max_bytes,
            ctx->occ_fused[kernel][es == 8][mode_qt ? 1 : 0]);
  if (!ctx->coop || N % BLK || N == 0 || N * es > ctx->fused_max_bytes) return 0;
  const size_t ntiles = (N / BLK + WTILE - 1) / WTILE;
  const size_t resident = (size_t)ctx->sm_count * ctx->occ_fused[kernel][es == 8][mode_qt ? 1 : 0];
  if (resident == 0) return 0;
  const size_t grid = ntiles < resident ? ntiles : resident;
  if ((ntiles + grid - 1) / grid > FUSED_MAX_TILES_PER_CTA) return 0;
  return (int)grid;
}

// The launch plan of a slab of N elements (dctz_gpu_plan): the streaming launches below take their grids, tiles per
// ticket and scratch partitions from here, and dctz_gpu_launch_plan reports the same values.
static_assert(CompressCfg<double, false>::WARPS == 4 && CompressCfg<double, true>::WARPS == 4 && CompressCfg<float, false>::WARPS == 4 &&
              CompressCfg<float, true>::WARPS == 4 && DecompressCfg<double, false>::WARPS == 4 && DecompressCfg<double, true>::WARPS == 4 &&
              DecompressCfg<float, false>::WARPS == 4 && DecompressCfg<float, true>::WARPS == 4, "make_plan assumes 4 warps per CTA");
constexpr size_t PLAN_WARPS = 4;
static size_t clamp_grid(size_t want, size_t cap) { return want < cap ? want : cap; }
static size_t gather_grid(const dctz_gpu_ctx *ctx, size_t n_entries) {  // one CTA per group of 32 entries, at most 8 per SM
  const size_t groups = (n_entries + 31) / 32;
  return clamp_grid(groups ? groups : 1, (size_t)ctx->sm_count * 8);
}
static dctz_gpu_plan make_plan(const dctz_gpu_ctx *ctx, size_t N, size_t es, int mode_qt) {
  dctz_gpu_plan p = {};
  const int dbl = es == 8, qt = mode_qt ? 1 : 0;
  const size_t sm = (size_t)ctx->sm_count;
  p.fused_compress_grid = (uint64_t)fused_grid(ctx, 0, N, es, qt);
  p.fused_decompress_grid = (uint64_t)fused_grid(ctx, 1, N, es, qt);
  const size_t ntiles = (N / BLK + WTILE - 1) / WTILE, ctas = (ntiles + PLAN_WARPS - 1) / PLAN_WARPS;
  p.ntiles = ntiles;
  p.n_entries = ntiles + (N % BLK ? 1 : 0);  // the partial tail block is one more "tile" of the compress scratch
  p.compress_grid = clamp_grid(ctas, sm * ctx->occ[0][dbl][qt]);
  p.compress_warps = p.compress_grid * PLAN_WARPS;
  p.compress_batch = tile_batch(ntiles, p.compress_warps, true);
  p.reduce_ctas = (ntiles + 4095) / 4096;
  p.groups = (p.n_entries + 31) / 32;
  p.scan_chunks = scan_chunks(p.n_entries);
  p.gather_grid = gather_grid(ctx, p.n_entries);
  p.qt_max_groups = (ntiles + 31) / 32;
  p.qt_max_grid = clamp_grid(p.qt_max_groups, sm * 8);
  p.decompress_grid = clamp_grid(ctas, sm * ctx->occ[1][dbl][qt]);
  p.decompress_batch = tile_batch(ntiles, p.decompress_grid * PLAN_WARPS);
  p.decompress_scan_chunks = scan_chunks(ntiles);
  p.ahead_grid = clamp_grid(ctas, sm * ctx->occ_ahead[dbl][qt]);
  p.ahead_batch = tile_batch(ntiles, p.ahead_grid * PLAN_WARPS);
  p.ahead_units = (ntiles + p.ahead_batch - 1) / p.ahead_batch;
  p.ahead_groups = (p.ahead_units + 63) / 64;
  p.ahead_super = (p.ahead_units + 2047) / 2048;
  return p;
}

extern "C" int dctz_gpu_launch_plan(const dctz_gpu_ctx *ctx, size_t N, int datatype, int mode_qt, dctz_gpu_plan *out) {
  if (!ctx) return fail(nullptr, DCTZ_GPU_EINVAL, "ctx is NULL");
  dctz_gpu_ctx *c = const_cast<dctz_gpu_ctx *>(ctx);  // (for the error message only)
  if (datatype != DCTZ_GPU_FLOAT && datatype != DCTZ_GPU_DOUBLE) return fail(c, DCTZ_GPU_EINVAL, "datatype %d is neither FLOAT(0) nor DOUBLE(1)", datatype);
  if (!out || N == 0) return fail(c, DCTZ_GPU_EINVAL, "launch_plan: NULL pointer or N == 0");
  *out = make_plan(ctx, N, datatype == DCTZ_GPU_DOUBLE ? 8 : 4, mode_qt);
  return DCTZ_GPU_OK;
}

struct ScanBufs { unsigned *counts; ScanOut out; unsigned nchunks; };
static size_t up128(size_t v) { return (v + 127) / 128 * 128; }
static int scan_bufs(dctz_gpu_ctx *ctx, size_t n_entries, ScanBufs *sb) {
  const size_t ngroups = (n_entries + 31) / 32, nchunks = scan_chunks(n_entries);
  TRY(grow(ctx, ctx->status, up128(ngroups * 8) + up128(nchunks * 8) + up128(n_entries * 4)));
  char *p = (char *)ctx->status.p;
  sb->out.group_prefix = (unsigned long long *)p;
  sb->out.chunk_prefix = (unsigned long long *)(p + up128(ngroups * 8));
  sb->out.done = ctx->d_done + 1;
  sb->counts = (unsigned *)(p + up128(ngroups * 8) + up128(nchunks * 8));  // 16-byte aligned for the uint4 loads
  sb->nchunks = (unsigned)nchunks;
  return DCTZ_GPU_OK;
}

template <typename T> static QuantConsts<T> make_quant(double eb);
template <> QuantConsts<double> make_quant<double>(double eb) {
  QuantConsts<double> q;
  const int half = DCTZ_GPU_NBINS / 2;
  q.bw = eb * 2.0 * 1.0;                   // dctz-comp-lib.c:273 (BRSF == 1.0)
  q.rmin = -(half * 2 + 1) * (eb * 1.0);   // :274
  q.rmax = (half * 2 + 1) * (eb * 1.0);    // :275
  q.inv_bw = 1.0 / q.bw;
  return q;
}
template <> QuantConsts<float> make_quant<float>(double eb) {
  QuantConsts<float> q;
  const int half = DCTZ_GPU_NBINS / 2;
  q.bw = (float)(eb * 2.0 * 1.0);                 // :278
  q.rmin = (float)(-(half * 2 + 1) * (eb * 1.0)); // :279
  q.rmax = (float)((half * 2 + 1) * (eb * 1.0));  // :280
  q.div = make_divisor(q.bw);
  return q;
}
template <typename T> static QtConsts<T> make_qt(double eb) {
  QtConsts<T> k;
  const QuantConsts<T> q = make_quant<T>(eb);
  k.eb = eb;
  k.rmin = q.rmin;
  k.rmax = q.rmax;
  k.d_rmax = (T)(eb * DCTZ_GPU_NBINS);   // dctz-decomp-lib.c:373 / 378
  k.d_rmin = (T)(-eb * DCTZ_GPU_NBINS);  // :374 / 379
  k.den = eb * (sizeof(T) == 8 ? 10.0 : (double)10.0f);  // error_bound * qt_factor (:405, :450)
  k.den_div = make_divisor(k.den);
  return k;
}

// ------------------------------------------------------------------------------------------
// phase 1: statistics
// ------------------------------------------------------------------------------------------
template <typename T>
static int launch_stats(dctz_gpu_ctx *ctx, const T *d_in, size_t N, double *d_stats3, int finalize_inline, size_t n_total,
                        void *d_qtable_raw, Info *d_info, cudaStream_t st) {
  const size_t nchunks = (N * sizeof(T) + STAT_CHUNK - 1) / STAT_CHUNK;
  const size_t resident = (size_t)ctx->sm_count * 3;  // 3 CTAs x 64 KB of staging per SM
  int grid = (int)(nchunks < resident ? (nchunks ? nchunks : 1) : resident);
  SfTables tb = ctx->tb;
  tb.qmax_words = (int)(BLK * sizeof(T) / 8);
  CU(cudaFuncSetAttribute(k_stats<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, STAT_SMEM));
  k_stats<T><<<grid, 256, STAT_SMEM, st>>>(d_in, N, ctx->d_partials, ctx->d_done, d_stats3, finalize_inline,
                                           (unsigned long long)n_total, 1, tb, ctx->d_params, d_info,
                                           (unsigned long long *)d_qtable_raw);
  ctx->launches++;
  CU(cudaGetLastError());
  return DCTZ_GPU_OK;
}

extern "C" int dctz_gpu_stats_dev(dctz_gpu_ctx *ctx, const void *d_in, size_t N, int datatype, double *d_stats3, void *stream) {
  TRY(check_common(ctx, datatype, 1.0));
  if (!d_in || !d_stats3 || N == 0) return fail(ctx, DCTZ_GPU_EINVAL, "stats: NULL pointer or N == 0");
  if (!aligned16(d_in)) return fail(ctx, DCTZ_GPU_EINVAL, "stats: input must be 16-byte aligned");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (datatype == DCTZ_GPU_DOUBLE) return launch_stats<double>(ctx, (const double *)d_in, N, d_stats3, 0, N, nullptr, ctx->d_info, st);
  return launch_stats<float>(ctx, (const float *)d_in, N, d_stats3, 0, N, nullptr, ctx->d_info, st);
}

// ------------------------------------------------------------------------------------------
// phase 2: fused compress
// ------------------------------------------------------------------------------------------
struct StatArgs {  // where a compress launch takes its scaling factor from (kernels.cuh: StatSource)
  const double *d_stats_all;
  int nranks, first_slab, mode;
  size_t n_total;
  double *d_true3;  // MODE_BELIEF: receives the slab's true {max, min, sum}
};

// MODE_STATS:  [k_compress] -> [k_qt_max] -> [tail] -> scan -> gather           (true statistics known: the two-pass path)
// MODE_BELIEF: [k_compress<VERIFY>] -> k_reduce_tile_sums                       (first half of the single-read path)
// MODE_REDO:   [k_compress, leaves at once unless the belief was wrong] -> [k_qt_max] -> [tail] -> scan -> gather
template <typename T, bool QT>
static int launch_compress(dctz_gpu_ctx *ctx, const T *d_in, size_t N, double eb, const StatArgs &sa, uint8_t *d_bins, float *d_dc, float *d_ac,
                           void *d_qtable_raw, Info *d_info, cudaStream_t st) {
  typedef CompressCfg<T, QT> Cfg;
  typedef typename BitsOf<T>::U U;
  const unsigned long long nblk_full = N / BLK;
  const int rem = (int)(N % BLK);
  const QuantConsts<T> qc = make_quant<T>(eb);
  const dctz_gpu_plan plan = make_plan(ctx, N, sizeof(T), QT);
  const size_t ntiles = plan.ntiles;
  const size_t n_entries = plan.n_entries;  // the partial tail block is one more "tile" of the scratch layout
  if (n_entries > 0xFFFFF000ull) return fail(ctx, DCTZ_GPU_EINVAL, "slab too large: %zu tiles", n_entries);
  ScanBufs sb;
  TRY(scan_bufs(ctx, n_entries, &sb));
  float *ac_slots = nullptr;
  T *raw = nullptr;
  uint8_t *jpos = nullptr;
  FusedScan fused;
  fused.n_entries = 0;
  if (QT) {
    TRY(grow(ctx, ctx->qt_raw, n_entries * TILE_SLOT * sizeof(T) + QT_RAW_ALIGN));
    TRY(grow(ctx, ctx->qt_j, n_entries * TILE_SLOT + QT_J_ALIGN));
    raw = (T *)qt_raw_slots(ctx);
    jpos = qt_j_slots(ctx);
    ctx->qt_entries = (unsigned)n_entries;
    ctx->qt_tail_tile = rem ? (unsigned)ntiles : 0xFFFFFFFFu;
  } else {
    TRY(grow(ctx, ctx->slots, n_entries * TILE_SLOT * sizeof(float)));
    ac_slots = (float *)ctx->slots.p;
  }
  StatSource src;
  src.stats_all = sa.d_stats_all; src.nranks = sa.nranks; src.first_slab = sa.first_slab; src.is_double = sizeof(T) == 8; src.mode = sa.mode;
  src.n_total = (unsigned long long)sa.n_total; src.first_elem = d_in; src.tb = ctx->tb;
  src.tb.qmax_words = (int)(BLK * sizeof(T) / 8);
  src.params = ctx->d_params;
  src.qmax_zero = QT ? (unsigned long long *)d_qtable_raw : nullptr;
  src.tile_sums = nullptr; src.tile_ext = nullptr;
  const size_t nred = plan.reduce_ctas;  // CTAs of k_reduce_tiles
  if (sa.mode == MODE_BELIEF) {  // scratch: [tile sums][CTA sums][tile extremes][CTA extremes]
    TRY(grow(ctx, ctx->tile_sums, (ntiles + nred + 8) * sizeof(double) + (ntiles + nred + 8) * sizeof(uint2)));
    src.tile_sums = (double *)ctx->tile_sums.p;
    src.tile_ext = (uint2 *)((double *)ctx->tile_sums.p + ntiles + nred + 8);
  }
  if (nblk_full) {
    const int grid = (int)plan.compress_grid;
    CUtensorMap tmap;
    TRY(make_tile_map(ctx, &tmap, d_in, BLK * sizeof(T), nblk_full));
    fused.out = sb.out;
    fused.total = &d_info->n_outliers;
    // small field, true statistics: the last CTA scans (one launch less); the single-read modes scan after the REDO launch
    fused.n_entries = (sa.mode == MODE_STATS && rem == 0 && plan.groups <= 1024) ? (unsigned)n_entries : 0u;
    const unsigned batch = (unsigned)plan.compress_batch;
    if (sa.mode == MODE_BELIEF)
      k_compress<T, QT, true><<<grid, Cfg::THREADS, Cfg::SMEM, st>>>(tmap, nblk_full, src, qc, d_bins, d_dc, sb.counts, ac_slots, raw, jpos,
                                                                     (T *)d_qtable_raw, &ctx->d_ctl[0], d_info, fused, batch);
    else
      k_compress<T, QT, false><<<grid, Cfg::THREADS, Cfg::SMEM, st>>>(tmap, nblk_full, src, qc, d_bins, d_dc, sb.counts, ac_slots, raw, jpos,
                                                                      (T *)d_qtable_raw, &ctx->d_ctl[0], d_info, fused, batch);
    ctx->launches++;
    CU(cudaGetLastError());
    if (sa.mode == MODE_BELIEF) {  // the slab's true statistics from the per-tile records
      TileReduce tr;
      tr.cta_sums = src.tile_sums + ntiles;
      tr.cta_ext = src.tile_ext + ntiles;
      tr.done = ctx->d_done + 6;
      tr.hw = (unsigned *)(ctx->d_sample_bits + 1);
      tr.ext_bits = ctx->d_sample_bits + 2;
      const double *tail3 = rem ? ctx->d_tail3 : nullptr;
      k_reduce_tiles<T><<<(unsigned)nred, 256, 0, st>>>(src.tile_sums, src.tile_ext, (unsigned)ntiles, tr, tail3, sa.d_true3);
      ctx->launches++;
      if (sizeof(T) == 8) {
        const size_t want = (ntiles + 7) / 8;
        const int gr = (int)(want < (size_t)ctx->sm_count * 8 ? want : (size_t)ctx->sm_count * 8);
        k_resolve_extremes<<<gr, 256, 0, st>>>((const double *)d_in, nblk_full, src.tile_ext, (unsigned)ntiles, tr, ctx->d_done + 7, tail3, sa.d_true3);
        ctx->launches++;
      }
      CU(cudaGetLastError());
      return DCTZ_GPU_OK;
    }
    if (QT) {  // per-position maxima of the parked (unscaled) outliers, scaled by the kernel's last CTA (before the tail
               // block adds its own, scaled, values)
      const int gq = (int)plan.qt_max_grid;
      k_qt_max<T><<<gq, 256, 0, st>>>(sb.counts, (unsigned)ntiles, raw, jpos, (U *)d_qtable_raw, ctx->d_params, ctx->d_done + 4);
      ctx->launches++;
    }
  } else {  // a field of one partial block: nothing for k_compress to do, the parameters come from the one-thread kernel
    if (sa.mode == MODE_BELIEF) return fail(ctx, DCTZ_GPU_EINVAL, "internal: the single-read path needs at least one full block");
    k_finalize<<<1, 32, 0, st>>>(sa.d_stats_all, sa.nranks, (unsigned long long)sa.n_total, sizeof(T) == 8, d_in, sa.first_slab, src.tb, ctx->d_params, d_info,
                                 src.qmax_zero);
    ctx->launches++;
  }
  if (rem) {
    k_tail_compress<T, QT><<<1, 32, 0, st>>>(d_in + nblk_full * BLK, rem, nblk_full, (unsigned)ntiles, ctx->d_params, qc, d_bins, d_dc,
                                             sb.counts, ac_slots, raw, jpos, (U *)d_qtable_raw, (T *)d_qtable_raw, d_info);
    ctx->launches++;
    CU(cudaGetLastError());
  }
  if (!fused.n_entries) {
    k_scan_groups<<<sb.nchunks, 1024, 0, st>>>(sb.counts, (unsigned)n_entries, sb.out, &d_info->n_outliers);
    ctx->launches++;
  }
  if (!QT) {
    const int grid = (int)plan.gather_grid;  // one CTA per group of 32 tiles
    k_gather_ec<<<grid, 256, 0, st>>>(sb.counts, sb.out.group_prefix, sb.out.chunk_prefix, (unsigned)n_entries, ac_slots, d_ac, &d_info->n_outliers);
    ctx->launches++;
  }
  CU(cudaGetLastError());
  return DCTZ_GPU_OK;
}

static int compress_dispatch(dctz_gpu_ctx *ctx, const void *d_in, size_t N, int datatype, double eb, int mode_qt, const StatArgs &sa, uint8_t *d_bins,
                             float *d_dc, float *d_ac, void *d_qtable_raw, Info *d_info, cudaStream_t st) {
  if (datatype == DCTZ_GPU_DOUBLE) {
    if (mode_qt) return launch_compress<double, true>(ctx, (const double *)d_in, N, eb, sa, d_bins, d_dc, d_ac, d_qtable_raw, d_info, st);
    return launch_compress<double, false>(ctx, (const double *)d_in, N, eb, sa, d_bins, d_dc, d_ac, d_qtable_raw, d_info, st);
  }
  if (mode_qt) return launch_compress<float, true>(ctx, (const float *)d_in, N, eb, sa, d_bins, d_dc, d_ac, d_qtable_raw, d_info, st);
  return launch_compress<float, false>(ctx, (const float *)d_in, N, eb, sa, d_bins, d_dc, d_ac, d_qtable_raw, d_info, st);
}

static int check_compress_args(dctz_gpu_ctx *ctx, const void *d_in, size_t N, int datatype, double eb, int mode_qt,
                               const void *d_bins, const void *d_dc, const void *d_ac, const void *d_qtable_raw, const void *d_info) {
  TRY(check_common(ctx, datatype, eb));
  if (!d_in || !d_bins || !d_dc || !d_ac || !d_info || N == 0) return fail(ctx, DCTZ_GPU_EINVAL, "compress: NULL pointer or N == 0");
  if (mode_qt && !d_qtable_raw) return fail(ctx, DCTZ_GPU_EINVAL, "compress: QT mode needs d_qtable_raw");
  if (!aligned16(d_in) || !aligned16(d_bins)) return fail(ctx, DCTZ_GPU_EINVAL, "compress: input and bin_index must be 16-byte aligned");
  if (!aligned16(d_ac) || ((uintptr_t)d_dc & 3u)) return fail(ctx, DCTZ_GPU_EINVAL, "compress: AC_exact / DC alignment");
  return DCTZ_GPU_OK;
}

static int compress_dev_impl(dctz_gpu_ctx *ctx, const void *d_in, size_t N, size_t N_total, int datatype, double eb, int mode_qt,
                             const double *d_stats_all, int nranks, int first_slab, uint8_t *d_bins, float *d_dc, float *d_ac,
                             void *d_qtable_raw, dctz_gpu_info *d_info, void *stream, int mode, double *d_true3) {
  TRY(check_compress_args(ctx, d_in, N, datatype, eb, mode_qt, d_bins, d_dc, d_ac, d_qtable_raw, d_info));
  if (!d_stats_all || nranks < 1 || N_total < N) return fail(ctx, DCTZ_GPU_EINVAL, "compress: bad statistics arguments");
  if (mode == MODE_BELIEF && (!d_true3 || N < (size_t)BLK)) return fail(ctx, DCTZ_GPU_EINVAL, "compress_spec: needs d_true3 and at least one full block");
  CU(cudaSetDevice(ctx->device));
  StatArgs sa;
  sa.d_stats_all = d_stats_all; sa.nranks = nranks; sa.first_slab = first_slab; sa.mode = mode; sa.n_total = N_total; sa.d_true3 = d_true3;
  return compress_dispatch(ctx, d_in, N, datatype, eb, mode_qt, sa, d_bins, d_dc, d_ac, d_qtable_raw, (Info *)d_info, (cudaStream_t)stream);
}

extern "C" int dctz_gpu_compress_dev(dctz_gpu_ctx *ctx, const void *d_in, size_t N, size_t N_total, int datatype, double eb,
                                     int mode_qt, const double *d_stats_all, int nranks, int first_slab, uint8_t *d_bins,
                                     float *d_dc, float *d_ac, void *d_qtable_raw, dctz_gpu_info *d_info, void *stream) {
  return compress_dev_impl(ctx, d_in, N, N_total, datatype, eb, mode_qt, d_stats_all, nranks, first_slab, d_bins, d_dc, d_ac, d_qtable_raw,
                           d_info, stream, MODE_STATS, nullptr);
}

// ---- the single-read path: belief (sample) -> compress while gathering the true statistics -> verdict / redo ----
template <typename T> static int launch_sample(dctz_gpu_ctx *ctx, const T *d_in, size_t N, double *d_belief3, cudaStream_t st) {
  // one 16-byte vector of every 4 KB; large slabs: about 256 K samples in all (scattered 32-byte reads cost DRAM far more than
  // their bytes, and the decade of the maximum is found long before that)
  const size_t nvec = N * sizeof(T) / 16;
  size_t stride = nvec >> 18;
  if (stride < SAMPLE_STRIDE_VECS) stride = SAMPLE_STRIDE_VECS;
  const size_t nsamp = (nvec + stride - 1) / stride;
  const size_t want = (nsamp + 256 * 4 - 1) / (256 * 4);
  const int grid = (int)(want < (size_t)ctx->sm_count * 8 ? (want ? want : 1) : (size_t)ctx->sm_count * 8);
  k_sample<T><<<grid, 256, 0, st>>>(d_in, N, stride, ctx->d_sample_bits, ctx->d_done + 5, d_belief3, ctx->d_tail3);
  ctx->launches++;
  CU(cudaGetLastError());
  return DCTZ_GPU_OK;
}

extern "C" int dctz_gpu_sample_dev(dctz_gpu_ctx *ctx, const void *d_in, size_t N, int datatype, double *d_belief3, void *stream) {
  TRY(check_common(ctx, datatype, 1.0));
  if (!d_in || !d_belief3 || N == 0) return fail(ctx, DCTZ_GPU_EINVAL, "sample: NULL pointer or N == 0");
  if (!aligned16(d_in)) return fail(ctx, DCTZ_GPU_EINVAL, "sample: input must be 16-byte aligned");
  CU(cudaSetDevice(ctx->device));
  if (datatype == DCTZ_GPU_DOUBLE) return launch_sample<double>(ctx, (const double *)d_in, N, d_belief3, (cudaStream_t)stream);
  return launch_sample<float>(ctx, (const float *)d_in, N, d_belief3, (cudaStream_t)stream);
}

extern "C" int dctz_gpu_compress_spec_dev(dctz_gpu_ctx *ctx, const void *d_in, size_t N, size_t N_total, int datatype, double eb, int mode_qt,
                                          const double *d_belief_all, int nranks, int first_slab, uint8_t *d_bins, float *d_dc, float *d_ac,
                                          void *d_qtable_raw, dctz_gpu_info *d_info, double *d_true3, void *stream) {
  return compress_dev_impl(ctx, d_in, N, N_total, datatype, eb, mode_qt, d_belief_all, nranks, first_slab, d_bins, d_dc, d_ac, d_qtable_raw, d_info,
                           stream, MODE_BELIEF, d_true3);
}

extern "C" int dctz_gpu_compress_spec_finish_dev(dctz_gpu_ctx *ctx, const void *d_in, size_t N, size_t N_total, int datatype, double eb, int mode_qt,
                                                 const double *d_true_all, int nranks, int first_slab, uint8_t *d_bins, float *d_dc, float *d_ac,
                                                 void *d_qtable_raw, dctz_gpu_info *d_info, void *stream) {
  return compress_dev_impl(ctx, d_in, N, N_total, datatype, eb, mode_qt, d_true_all, nranks, first_slab, d_bins, d_dc, d_ac, d_qtable_raw, d_info,
                           stream, MODE_REDO, nullptr);
}

// One slab (or a whole field) with a caller-supplied belief about its statistics: compress_spec + finish in one call.
extern "C" int dctz_gpu_compress_known_stats_dev(dctz_gpu_ctx *ctx, const void *d_in, size_t N, size_t N_total, int datatype, double eb,
                                                 int mode_qt, const double *d_stats_all, int nranks, int first_slab, uint8_t *d_bins,
                                                 float *d_dc, float *d_ac, void *d_qtable_raw, dctz_gpu_info *d_info, void *stream) {
  if (nranks != 1 || N_total != N) return fail(ctx, DCTZ_GPU_EINVAL, "compress_known_stats: whole fields only (slabs: sample / compress_spec / compress_spec_finish)");
  if (N < (size_t)BLK)  // nothing to speculate on: the two-pass path
    return fail(ctx, DCTZ_GPU_EINVAL, "compress_known_stats: needs at least one full block");
  // the partial tail block's exact statistics come from the sampling kernel (its belief output is not used)
  TRY(dctz_gpu_sample_dev(ctx, d_in, N, datatype, ctx->d_spec3, stream));
  TRY(compress_dev_impl(ctx, d_in, N, N_total, datatype, eb, mode_qt, d_stats_all, 1, first_slab, d_bins, d_dc, d_ac, d_qtable_raw, d_info, stream,
                        MODE_BELIEF, ctx->d_spec3 + 3));
  return compress_dev_impl(ctx, d_in, N, N_total, datatype, eb, mode_qt, ctx->d_spec3 + 3, 1, first_slab, d_bins, d_dc, d_ac, d_qtable_raw, d_info, stream,
                           MODE_REDO, nullptr);
}

template <typename T>
static int launch_qt_finish(dctz_gpu_ctx *ctx, double eb, const T *d_qraw, T *d_qtable, float *d_ac, Info *d_info, cudaStream_t st) {
  const QtConsts<T> k = make_qt<T>(eb);
  const unsigned n_entries = ctx->qt_entries;
  ScanBufs sb;
  TRY(scan_bufs(ctx, n_entries, &sb));  // same layout as in the compress call: nothing is reallocated
  const int grid = (int)gather_grid(ctx, n_entries);  // as planned for the compress call
  k_qt_gather<T><<<grid, 256, 0, st>>>(sb.counts, sb.out.group_prefix, sb.out.chunk_prefix, n_entries, (const T *)qt_raw_slots(ctx), (const uint8_t *)qt_j_slots(ctx),
                                       d_qraw, d_qtable, k, d_ac, d_info, ctx->d_params, ctx->qt_tail_tile);
  ctx->launches++;
  CU(cudaGetLastError());
  return DCTZ_GPU_OK;
}

extern "C" int dctz_gpu_qt_finish_dev(dctz_gpu_ctx *ctx, int datatype, double eb, const void *d_qtable_raw, void *d_qtable,
                                      float *d_ac, dctz_gpu_info *d_info, void *stream) {
  TRY(check_common(ctx, datatype, eb));
  if (!d_qtable_raw || !d_ac || !d_info) return fail(ctx, DCTZ_GPU_EINVAL, "qt_finish: NULL pointer");
  if (!ctx->qt_raw.p || !ctx->qt_entries) return fail(ctx, DCTZ_GPU_EINVAL, "qt_finish: no QT compress call preceded");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (datatype == DCTZ_GPU_DOUBLE)
    return launch_qt_finish<double>(ctx, eb, (const double *)d_qtable_raw, (double *)d_qtable, d_ac, (Info *)d_info, st);
  return launch_qt_finish<float>(ctx, eb, (const float *)d_qtable_raw, (float *)d_qtable, d_ac, (Info *)d_info, st);
}

template <typename T, bool QT>
static int launch_compress_fused(dctz_gpu_ctx *ctx, int grid, const T *d_in, size_t N, double eb, uint8_t *d_bins, float *d_dc, float *d_ac,
                                 void *d_qtable, void *d_qtable_raw, Info *d_info, cudaStream_t st) {
  typedef CompressCfg<T, QT> Cfg;
  typedef typename BitsOf<T>::U U;
  unsigned long long nblk_full = N / BLK;
  const size_t ntiles = (nblk_full + WTILE - 1) / WTILE;
  QuantConsts<T> qc = make_quant<T>(eb);
  QtConsts<T> qk = make_qt<T>(eb);
  ScanBufs sb;
  TRY(scan_bufs(ctx, ntiles, &sb));
  float *ac_slots = nullptr;
  T *raw = nullptr;
  uint8_t *jpos = nullptr;
  if (QT) {
    TRY(grow(ctx, ctx->qt_raw, ntiles * TILE_SLOT * sizeof(T) + QT_RAW_ALIGN));
    TRY(grow(ctx, ctx->qt_j, ntiles * TILE_SLOT + QT_J_ALIGN));
    raw = (T *)qt_raw_slots(ctx);
    jpos = qt_j_slots(ctx);
    ctx->qt_entries = 0;  // nothing is left for dctz_gpu_qt_finish_dev: the kernel rescales itself
  } else {
    TRY(grow(ctx, ctx->slots, ntiles * TILE_SLOT * sizeof(float)));
    ac_slots = (float *)ctx->slots.p;
  }
  CUtensorMap tmap;
  TRY(make_tile_map(ctx, &tmap, d_in, BLK * sizeof(T), nblk_full));
  SfTables tb = ctx->tb;
  tb.qmax_words = 0;
  T *q_out = (T *)d_qtable, *q_raw = (T *)d_qtable_raw;
  U *qmax = (U *)ctx->d_qmax_scratch;
  StatPartial *partials = ctx->d_partials;
  unsigned long long *totals = ctx->d_cta_totals, *bar = ctx->d_barrier;
  unsigned long long base = ctx->barrier_base[0];
  DevParams *params = ctx->d_params;
  unsigned *counts = sb.counts;
  unsigned long long *dbg = ctx->fused_stamps ? ctx->d_dbg : nullptr;  // (six %globaltimer reads per CTA: diagnostics only)
  ctx->dbg_grid[0] = ctx->fused_stamps ? grid : 0;
  void *args[] = {&tmap, &d_in, &nblk_full, &qc, &qk, &d_bins, &d_dc, &counts, &ac_slots, &raw, &jpos, &d_ac, &q_out, &q_raw, &qmax,
                  &partials, &totals, &tb, &params, &d_info, &bar, &base, &dbg};
  CU(cudaLaunchCooperativeKernel((const void *)k_compress_fused<T, QT>, dim3(grid), dim3(Cfg::THREADS), args, Cfg::SMEM, st));
  ctx->barrier_base[0] += (unsigned long long)FUSED_COMPRESS_BARRIERS * (unsigned long long)grid;
  ctx->launches++;
  return DCTZ_GPU_OK;
}

static int compress_fused_dispatch(dctz_gpu_ctx *ctx, int grid, const void *d_in, size_t N, int datatype, double eb, int mode_qt, uint8_t *d_bins,
                                   float *d_dc, float *d_ac, void *d_qtable, void *d_qtable_raw, Info *d_info, cudaStream_t st) {
  if (datatype == DCTZ_GPU_DOUBLE) {
    if (mode_qt) return launch_compress_fused<double, true>(ctx, grid, (const double *)d_in, N, eb, d_bins, d_dc, d_ac, d_qtable, d_qtable_raw, d_info, st);
    return launch_compress_fused<double, false>(ctx, grid, (const double *)d_in, N, eb, d_bins, d_dc, d_ac, d_qtable, d_qtable_raw, d_info, st);
  }
  if (mode_qt) return launch_compress_fused<float, true>(ctx, grid, (const float *)d_in, N, eb, d_bins, d_dc, d_ac, d_qtable, d_qtable_raw, d_info, st);
  return launch_compress_fused<float, false>(ctx, grid, (const float *)d_in, N, eb, d_bins, d_dc, d_ac, d_qtable, d_qtable_raw, d_info, st);
}

// ------------------------------------------------------------------------------------------
// Multi-GPU slabs from C (SURVEY.md §8e): the ONE exchange the path needs, inside the library, for callers that have an
// NCCL communicator (one process or thread per GPU, e.g. under MPI) and no Python around it.  NCCL is resolved at run
// time from the process (the caller created its communicator with some libnccl: that one is used) or from
// libnccl.so.2; the library does not link it.  Only the handful of enum values of nccl.h that the calls need are
// restated here (stable since NCCL 2.0).
// ------------------------------------------------------------------------------------------
typedef int (*NcclAllGatherFn)(const void *, void *, size_t, int, void *, cudaStream_t);
typedef int (*NcclAllReduceFn)(const void *, void *, size_t, int, int, void *, cudaStream_t);
typedef int (*NcclBroadcastFn)(const void *, void *, size_t, int, int, void *, cudaStream_t);
typedef const char *(*NcclErrFn)(int);
static struct { NcclAllGatherFn all_gather; NcclAllReduceFn all_reduce; NcclBroadcastFn broadcast; NcclErrFn err; } g_nccl = {};
constexpr int kNcclFloat = 7, kNcclDouble = 8, kNcclMax = 2;  // ncclFloat32, ncclFloat64, ncclMax (nccl.h)

static int load_nccl(dctz_gpu_ctx *ctx) {
  static std::once_flag once;
  std::call_once(once, [] {
    void *h = RTLD_DEFAULT;  // (a null handle: "whatever the process has loaded")
    bool ok = dlsym(h, "ncclAllGather") != nullptr;
    if (!ok) { h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL); ok = h != nullptr; }
    if (ok) {
      g_nccl.all_gather = (NcclAllGatherFn)dlsym(h, "ncclAllGather");
      g_nccl.all_reduce = (NcclAllReduceFn)dlsym(h, "ncclAllReduce");
      g_nccl.broadcast = (NcclBroadcastFn)dlsym(h, "ncclBroadcast");
      g_nccl.err = (NcclErrFn)dlsym(h, "ncclGetErrorString");
    }
  });
  if (!g_nccl.all_gather || !g_nccl.all_reduce || !g_nccl.broadcast) return fail(ctx, DCTZ_GPU_ENODEV, "NCCL is not available in this process (libnccl.so.2)");
  return DCTZ_GPU_OK;
}
#define NCCL(call)                                                                                                     \
  do {                                                                                                                 \
    const int r_ = (call);                                                                                             \
    if (r_ != 0) return fail(ctx, DCTZ_GPU_ECUDA, "%s: %s", #call, g_nccl.err ? g_nccl.err(r_) : "NCCL error");        \
  } while (0)

extern "C" int dctz_gpu_compress_slab_comm(dctz_gpu_ctx *ctx, void *nccl_comm, int rank, int nranks, int last_rank_with_data,
                                           const void *d_in, size_t N, size_t N_total, int datatype, double eb, int mode_qt, uint8_t *d_bins,
                                           float *d_dc, float *d_ac, void *d_qtable, void *d_qtable_raw, dctz_gpu_info *d_info, void *stream) {
  TRY(check_compress_args(ctx, d_in, N, datatype, eb, mode_qt, d_bins, d_dc, d_ac, d_qtable_raw, d_info));
  if (!nccl_comm || nranks < 1 || rank < 0 || rank >= nranks || last_rank_with_data < 0 || last_rank_with_data >= nranks || N_total < N)
    return fail(ctx, DCTZ_GPU_EINVAL, "compress_slab_comm: bad communicator / rank arguments");
  if (mode_qt && !d_qtable) return fail(ctx, DCTZ_GPU_EINVAL, "compress_slab_comm: QT mode needs d_qtable");
  TRY(load_nccl(ctx));
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t es = datatype == DCTZ_GPU_DOUBLE ? 8 : 4;
  TRY(grow(ctx, ctx->chunk_stats, (size_t)nranks * 3 * sizeof(double) + BLK * 8));
  double *d_all = (double *)ctx->chunk_stats.p;
  // statistics of the slab -> all-gather of {max, min, sum} (24 bytes per rank) -> every rank merges them in rank order
  TRY(dctz_gpu_stats_dev(ctx, d_in, N, datatype, ctx->d_stats3, st));
  NCCL(g_nccl.all_gather(ctx->d_stats3, d_all, 3, kNcclDouble, nccl_comm, st));
  TRY(dctz_gpu_compress_dev(ctx, d_in, N, N_total, datatype, eb, mode_qt, d_all, nranks, rank == 0, d_bins, d_dc, d_ac, d_qtable_raw, d_info, st));
  if (mode_qt) {
    // per-position maxima: MAX over the ranks; entry 0 (the DC of the field's last block, dctz-comp-lib.c:355-360) comes from
    // the last rank that holds data -- saved aside, reduced with the rest, broadcast, put back
    char *keep = (char *)(d_all + 3 * (size_t)nranks);
    CU(cudaMemcpyAsync(keep, d_qtable_raw, es, cudaMemcpyDeviceToDevice, st));
    NCCL(g_nccl.all_reduce(d_qtable_raw, d_qtable_raw, BLK, es == 8 ? kNcclDouble : kNcclFloat, kNcclMax, nccl_comm, st));
    NCCL(g_nccl.broadcast(keep, keep, 1, es == 8 ? kNcclDouble : kNcclFloat, last_rank_with_data, nccl_comm, st));
    CU(cudaMemcpyAsync(d_qtable_raw, keep, es, cudaMemcpyDeviceToDevice, st));
    TRY(dctz_gpu_qt_finish_dev(ctx, datatype, eb, d_qtable_raw, d_qtable, d_ac, d_info, st));
  }
  return DCTZ_GPU_OK;
}

extern "C" int dctz_gpu_compress_field_dev(dctz_gpu_ctx *ctx, const void *d_in, size_t N, int datatype, double eb, int mode_qt,
                                           uint8_t *d_bins, float *d_dc, float *d_ac, void *d_qtable, void *d_qtable_raw,
                                           dctz_gpu_info *d_info, void *stream) {
  TRY(check_compress_args(ctx, d_in, N, datatype, eb, mode_qt, d_bins, d_dc, d_ac, d_qtable_raw, d_info));
  if (mode_qt && !d_qtable) return fail(ctx, DCTZ_GPU_EINVAL, "compress_field: QT mode needs d_qtable");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (const int grid = fused_grid(ctx, 0, N, datatype == DCTZ_GPU_DOUBLE ? 8 : 4, mode_qt))  // small field: one launch for everything
    return compress_fused_dispatch(ctx, grid, d_in, N, datatype, eb, mode_qt, d_bins, d_dc, d_ac, d_qtable, d_qtable_raw, (Info *)d_info, st);
  if (N >= (size_t)BLK && ctx->single_read) {
    // SINGLE-READ path: the scaling factor only depends on the decade of max|x| (util.c:28), and a sample of 0.4 % of the
    // slab almost always finds it.  sample -> compress with that belief while gathering the true statistics -> a gate
    // launch that leaves at once when the belief held (else the slab is compressed again with the right factor).
    TRY(dctz_gpu_sample_dev(ctx, d_in, N, datatype, ctx->d_spec3, stream));
    TRY(dctz_gpu_compress_spec_dev(ctx, d_in, N, N, datatype, eb, mode_qt, ctx->d_spec3, 1, 1, d_bins, d_dc, d_ac, d_qtable_raw, d_info, ctx->d_spec3 + 3, stream));
    TRY(dctz_gpu_compress_spec_finish_dev(ctx, d_in, N, N, datatype, eb, mode_qt, ctx->d_spec3 + 3, 1, 1, d_bins, d_dc, d_ac, d_qtable_raw, d_info, stream));
  } else {  // two passes: statistics, then compress
    TRY(dctz_gpu_stats_dev(ctx, d_in, N, datatype, ctx->d_stats3, stream));
    TRY(dctz_gpu_compress_dev(ctx, d_in, N, N, datatype, eb, mode_qt, ctx->d_stats3, 1, 1, d_bins, d_dc, d_ac, d_qtable_raw, d_info, stream));
  }
  if (mode_qt) TRY(dctz_gpu_qt_finish_dev(ctx, datatype, eb, d_qtable_raw, d_qtable, d_ac, d_info, stream));
  return DCTZ_GPU_OK;
}

// ------------------------------------------------------------------------------------------
// decompress
// ------------------------------------------------------------------------------------------
template <typename T, bool QT>
static int launch_decompress(dctz_gpu_ctx *ctx, const uint8_t *d_bins, const float *d_dc, const float *d_ac, unsigned long long ac_limit,
                             const T *d_qtable, size_t N, double eb, double sf, T *d_out, unsigned *d_corrupt, cudaStream_t st) {
  typedef DecompressCfg<T, QT> Cfg;
  const unsigned long long nblk_full = N / BLK;
  const int rem = (int)(N % BLK);
  const QtConsts<T> qk = make_qt<T>(eb);
  // gen_bins: bin_width = error_bound*2*BRSF (binning.c:16); gen_bins_f receives the bound as float (binning.c:32-36)
  const T bw = (sizeof(T) == 8) ? (T)(eb * 2 * 1.0) : (T)(float)((float)eb * 2 * 1.0);
  const T sfT = (T)sf;
  const dctz_gpu_plan plan = make_plan(ctx, N, sizeof(T), QT);
  if (const int fgrid = (int)plan.fused_decompress_grid) {  // small field of full blocks: count + dequantise + IDCT in ONE launch
    unsigned long long nb = nblk_full;
    const size_t ntiles = plan.ntiles;
    ScanBufs sb;
    TRY(scan_bufs(ctx, ntiles, &sb));
    TRY(grow(ctx, ctx->tile_off, ntiles * sizeof(unsigned)));
    CUtensorMap tmap;
    TRY(make_tile_map(ctx, &tmap, d_out, BLK * sizeof(T), nblk_full));
    T bw_ = bw, sf_ = sfT;
    QtConsts<T> qk_ = qk;
    unsigned *counts = sb.counts, *toff = (unsigned *)ctx->tile_off.p;
    unsigned long long *totals = ctx->d_cta_totals + (size_t)ctx->sm_count * 4, *bar = ctx->d_barrier + 1;
    unsigned long long base = ctx->barrier_base[1], lim = ac_limit;
    int dca = aligned16(d_dc) ? 1 : 0;
    unsigned long long *dbg = ctx->fused_stamps ? ctx->d_dbg + (size_t)ctx->sm_count * 4 * 8 : nullptr;
    ctx->dbg_grid[1] = ctx->fused_stamps ? fgrid : 0;
    void *args[] = {&d_bins, &d_dc, &d_ac, &d_qtable, &nb, &bw_, &sf_, &qk_, &tmap, &counts, &toff, &totals, &lim, &d_corrupt, &dca, &bar, &base, &dbg};
    CU(cudaLaunchCooperativeKernel((const void *)k_decompress_fused<T, QT>, dim3(fgrid), dim3(Cfg::THREADS), args, Cfg::SMEM, st));
    ctx->barrier_base[1] += (unsigned long long)fgrid;
    ctx->launches++;
    return DCTZ_GPU_OK;
  }
  if (nblk_full) {
    const size_t ntiles = plan.ntiles;
    if (ntiles > 0xFFFFF000ull) return fail(ctx, DCTZ_GPU_EINVAL, "slab too large: %zu tiles", ntiles);
    // No pre-pass (a count warpgroup publishes the tiles' outlier counts beside the decode warpgroup, count_units) where it
    // pays, DESIGN.md 4.3.  double: below one outlier per 128 elements (the caller states the number of outliers, so the
    // choice is made per call): 1.57 against 1.69 ms on the outlier-free 8 GiB slab, but 0.539 against 0.505 ms with 5 %
    // outliers (B200).  float: never -- the pre-pass kernel keeps 3 CTAs of decode warps per SM, the split kernel fits 2
    // (f32 slab 1.037 against 1.129 ms).
    const bool ahead = ctx->decomp_ahead > 0 || (ctx->decomp_ahead < 0 && sizeof(T) == 8 && ac_limit <= (unsigned long long)(N >> 7));
    if (ahead) {
      const int grid = (int)plan.ahead_grid;
      const unsigned batch = (unsigned)plan.ahead_batch;
      const size_t nunits = plan.ahead_units, ngroups = plan.ahead_groups, nsuper = plan.ahead_super;
      const size_t off_a = up128(ntiles * sizeof(unsigned)), off_s = off_a + up128(nunits * sizeof(unsigned)), off_t = off_s + up128(ngroups * 8),
                   total = off_t + up128(nsuper * 8);
      TRY(grow(ctx, ctx->ahead_buf, total));
      CU(cudaMemsetAsync(ctx->ahead_buf.p, 0, total, st));
      char *ab = (char *)ctx->ahead_buf.p;
      unsigned *tile_counts = (unsigned *)ab, *agg = (unsigned *)(ab + off_a);
      unsigned long long *S = (unsigned long long *)(ab + off_s), *Tt = (unsigned long long *)(ab + off_t);
      CUtensorMap tmap;
      TRY(make_tile_map(ctx, &tmap, d_out, BLK * sizeof(T), nblk_full));
      k_decompress<T, QT, true><<<grid, SplitCfg::THREADS, Cfg::SMEM, st>>>(d_bins, d_dc, d_ac, d_qtable, nblk_full, bw, sfT, qk, tmap, tile_counts, agg,
                                                                            S, Tt, ctx->d_nconsumed, ac_limit, &ctx->d_ctl[1], d_corrupt,
                                                                            aligned16(d_dc) ? 1 : 0, batch, ctx->l2_hints < 0 ? 3 : ctx->l2_hints);
      ctx->launches++;
      CU(cudaGetLastError());
    } else {
    ScanBufs sb;
    TRY(scan_bufs(ctx, ntiles, &sb));
    {
      const size_t want = (ntiles + 7) / 8;
      const int grid = (int)(want < (size_t)ctx->sm_count * 16 ? want : (size_t)ctx->sm_count * 16);
      FusedScan fused;
      fused.out = sb.out;
      fused.total = ctx->d_nconsumed;
      fused.n_entries = ((ntiles + 31) / 32 <= 1024) ? (unsigned)ntiles : 0u;  // small field: the last CTA scans
      k_count_bins<<<grid, 256, 0, st>>>(d_bins, nblk_full, sb.counts, ctx->d_done + 3, fused);
      ctx->launches++;
      if (!fused.n_entries) {
        k_scan_groups<<<sb.nchunks, 1024, 0, st>>>(sb.counts, (unsigned)ntiles, sb.out, ctx->d_nconsumed);
        ctx->launches++;
      }
    }
    const int grid = (int)plan.decompress_grid;
    CUtensorMap tmap;
    TRY(make_tile_map(ctx, &tmap, d_out, BLK * sizeof(T), nblk_full));
    k_decompress<T, QT, false><<<grid, Cfg::THREADS, Cfg::SMEM, st>>>(d_bins, d_dc, d_ac, d_qtable, nblk_full, bw, sfT, qk, tmap, sb.counts, nullptr,
                                                                      sb.out.group_prefix, sb.out.chunk_prefix, ctx->d_nconsumed, ac_limit,
                                                                      &ctx->d_ctl[1], d_corrupt, aligned16(d_dc) ? 1 : 0,
                                                                      (unsigned)plan.decompress_batch, ctx->l2_hints > 0 ? ctx->l2_hints : 0);
    ctx->launches++;
    CU(cudaGetLastError());
    }
  }
  if (rem) {
    k_tail_decompress<T, QT><<<1, 32, 0, st>>>(d_bins, d_dc, d_ac, d_qtable, rem, nblk_full, bw, sfT, qk, d_out,
                                               nblk_full ? ctx->d_nconsumed : nullptr, 0ull, ac_limit, d_corrupt);
    ctx->launches++;
    CU(cudaGetLastError());
  }
  return DCTZ_GPU_OK;
}

// sf comes from the stream header and may be any decade the reference writes (double 1e-307..1e308, float 1e-37..1e38).
// The decoders form c*sf BEFORE the inverse transform: near the top a scaled DC of up to 80 times sf overflows, near the
// bottom the coefficients become subnormal and lose bits.  Outside 2^-960..2^960 (float 2^-96..2^96) the kernels decode
// with sf*2^-E instead (E = the binary exponent of sf: an exact rescaling that commutes with every step of the decode) and
// k_scale multiplies the reconstruction by 2^E afterwards.  Returns E, or 0 inside the window (no extra pass).
static int decode_exponent(double sf, int datatype) {
  const bool dbl = datatype == DCTZ_GPU_DOUBLE;
  const int e = dbl ? ilogb(sf) : ilogbf((float)sf);
  const int w = dbl ? 960 : 96;
  return (e > w || e < -w) ? e : 0;
}
static double decode_sf(double sf, int datatype, int E) {
  return datatype == DCTZ_GPU_DOUBLE ? ldexp(sf, -E) : (double)ldexpf((float)sf, -E);
}
static int rescale_output(dctz_gpu_ctx *ctx, void *d_out, size_t N, int datatype, int E, cudaStream_t st) {
  const size_t want = (N + 255) / 256;
  const int grid = (int)(want < (size_t)ctx->sm_count * 16 ? want : (size_t)ctx->sm_count * 16);
  if (datatype == DCTZ_GPU_DOUBLE) k_scale<double><<<grid, 256, 0, st>>>((double *)d_out, N, ldexp(1.0, E), 1);
  else k_scale<float><<<grid, 256, 0, st>>>((float *)d_out, N, ldexpf(1.0f, E), 1);
  ctx->launches++;
  CU(cudaGetLastError());
  return DCTZ_GPU_OK;
}

extern "C" int dctz_gpu_decompress_dev(dctz_gpu_ctx *ctx, const uint8_t *d_bins, const float *d_dc, const float *d_ac,
                                       uint64_t n_outliers, const void *d_qtable, size_t N, int datatype, double eb, double sf, int mode_qt,
                                       void *d_out, uint32_t *d_corrupt, void *stream) {
  TRY(check_common(ctx, datatype, eb));
  if (!d_bins || !d_dc || !d_out || N == 0 || (n_outliers && !d_ac)) return fail(ctx, DCTZ_GPU_EINVAL, "decompress: NULL pointer or N == 0");
  if (mode_qt && !d_qtable) return fail(ctx, DCTZ_GPU_EINVAL, "decompress: QT mode needs the qtable");
  if (!aligned16(d_bins) || !aligned16(d_out)) return fail(ctx, DCTZ_GPU_EINVAL, "decompress: bin_index and output must be 16-byte aligned");
  if (((uintptr_t)d_dc & 3u) || ((uintptr_t)d_ac & 3u)) return fail(ctx, DCTZ_GPU_EINVAL, "decompress: DC / AC_exact must be float-aligned");
  if (!(sf > 0.0) || isinf(sf)) return fail(ctx, DCTZ_GPU_EINVAL, "decompress: scaling factor %g is not a positive finite number", sf);
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  unsigned *flag = d_corrupt ? (unsigned *)d_corrupt : &ctx->d_ctl[1].corrupt;  // the caller's flag, else a scratch word nobody reads
  const int E = decode_exponent(sf, datatype);
  const double sfk = decode_sf(sf, datatype, E);
  if (datatype == DCTZ_GPU_DOUBLE) {
    if (mode_qt) TRY((launch_decompress<double, true>(ctx, d_bins, d_dc, d_ac, n_outliers, (const double *)d_qtable, N, eb, sfk, (double *)d_out, flag, st)));
    else TRY((launch_decompress<double, false>(ctx, d_bins, d_dc, d_ac, n_outliers, (const double *)d_qtable, N, eb, sfk, (double *)d_out, flag, st)));
  } else {
    if (mode_qt) TRY((launch_decompress<float, true>(ctx, d_bins, d_dc, d_ac, n_outliers, (const float *)d_qtable, N, eb, sfk, (float *)d_out, flag, st)));
    else TRY((launch_decompress<float, false>(ctx, d_bins, d_dc, d_ac, n_outliers, (const float *)d_qtable, N, eb, sfk, (float *)d_out, flag, st)));
  }
  return E ? rescale_output(ctx, d_out, N, datatype, E, st) : DCTZ_GPU_OK;
}

// ------------------------------------------------------------------------------------------
// region decompression (ranges.cuh, DESIGN.md §4.4)
// ------------------------------------------------------------------------------------------
// Outlier index of an N-element slab: [RegionIndexHdr (128 B)][group_prefix][chunk_prefix][counts], the arrays laid out as
// scan_bufs lays them out in the context's scratch.
struct RegionLayout { size_t ntiles, nchunks, off_gp, off_cp, off_counts, bytes; };
static RegionLayout region_layout(size_t N) {
  RegionLayout L;
  L.ntiles = (N / BLK + WTILE - 1) / WTILE;
  const size_t ngroups = (L.ntiles + 31) / 32;
  L.nchunks = (ngroups + 1023) / 1024;
  L.off_gp = 128;
  L.off_cp = L.off_gp + up128(ngroups * 8);
  L.off_counts = L.off_cp + up128(L.nchunks * 8);
  L.bytes = L.off_counts + up128(L.ntiles * 4);
  return L;
}
static_assert(sizeof(RegionIndexHdr) <= 128, "index header");

extern "C" size_t dctz_gpu_outlier_index_bytes(size_t N) { return region_layout(N).bytes; }

static RegionIndex region_view(const void *d_index, size_t N) {
  const RegionLayout L = region_layout(N);
  const char *p = (const char *)d_index;
  RegionIndex v;
  v.hdr = (const RegionIndexHdr *)p;
  v.group_prefix = (const unsigned long long *)(p + L.off_gp);
  v.chunk_prefix = (const unsigned long long *)(p + L.off_cp);
  v.counts = (const unsigned *)(p + L.off_counts);
  return v;
}

extern "C" int dctz_gpu_outlier_index_dev(dctz_gpu_ctx *ctx, const uint8_t *d_bins, size_t N, void *d_index, uint64_t *d_n_outliers, void *stream) {
  if (!ctx) return fail(nullptr, DCTZ_GPU_EINVAL, "ctx is NULL");
  if (!d_bins || !d_index || N == 0) return fail(ctx, DCTZ_GPU_EINVAL, "outlier_index: NULL pointer or N == 0");
  if (!aligned16(d_bins) || !aligned16(d_index)) return fail(ctx, DCTZ_GPU_EINVAL, "outlier_index: bin_index and the index must be 16-byte aligned");
  if ((uintptr_t)d_n_outliers & 7u) return fail(ctx, DCTZ_GPU_EINVAL, "outlier_index: n_outliers must be 8-byte aligned");
  const RegionLayout L = region_layout(N);
  if (L.ntiles > 0xFFFFF000ull) return fail(ctx, DCTZ_GPU_EINVAL, "outlier_index: slab too large: %zu tiles", L.ntiles);
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  char *p = (char *)d_index;
  RegionIndexHdr *hdr = (RegionIndexHdr *)p;
  if (L.ntiles) {  // the decompress pre-pass, into the caller's buffer
    unsigned *counts = (unsigned *)(p + L.off_counts);
    FusedScan fused;
    fused.out.group_prefix = (unsigned long long *)(p + L.off_gp);
    fused.out.chunk_prefix = (unsigned long long *)(p + L.off_cp);
    fused.out.done = ctx->d_done + 1;
    fused.total = &hdr->n_full_outliers;
    fused.n_entries = ((L.ntiles + 31) / 32 <= 1024) ? (unsigned)L.ntiles : 0u;  // small slab: the last CTA scans
    const size_t want = (L.ntiles + 7) / 8;
    const int grid = (int)(want < (size_t)ctx->sm_count * 16 ? want : (size_t)ctx->sm_count * 16);
    k_count_bins<<<grid, 256, 0, st>>>(d_bins, N / BLK, counts, ctx->d_done + 3, fused);
    ctx->launches++;
    if (!fused.n_entries) {
      k_scan_groups<<<(unsigned)L.nchunks, 1024, 0, st>>>(counts, (unsigned)L.ntiles, fused.out, fused.total);
      ctx->launches++;
    }
  }
  k_index_finish<<<1, 32, 0, st>>>(d_bins, N, (unsigned)L.ntiles, hdr, (unsigned long long *)d_n_outliers);
  ctx->launches++;
  CU(cudaGetLastError());
  return DCTZ_GPU_OK;
}

// The range plan in ctx->region: [RangeCtl (128 B)][piece_at, out_at: per range][chunk_piece, chunk_out: per chunk of 1024]
static RangePlan range_plan_view(void *region, size_t nranges) {
  char *p = (char *)region;
  RangePlan plan;
  plan.ctl = (RangeCtl *)p;
  plan.piece_at = (unsigned long long *)(p + 128);
  plan.out_at = plan.piece_at + nranges;
  plan.chunk_piece = (unsigned long long *)(p + 128 + up128(nranges * 16));
  plan.chunk_out = plan.chunk_piece + (nranges + 1023) / 1024;
  return plan;
}

template <typename T, bool QT>
static int launch_ranges(dctz_gpu_ctx *ctx, const uint8_t *d_bins, const float *d_dc, const float *d_ac, unsigned long long n_outliers, const T *d_qtable,
                         size_t N, double eb, double sf, const void *d_index, const unsigned long long *d_ranges, size_t nranges, T *d_out,
                         unsigned *flag, cudaStream_t st) {
  typedef RangeCfg<T> Cfg;
  const size_t nchunks = (nranges + 1023) / 1024;
  TRY(grow(ctx, ctx->region, 128 + up128(nranges * 16) + up128(nchunks * 16), true));  // (a new allocation starts zeroed: RangeCtl::done)
  const RangePlan plan = range_plan_view(ctx->region.p, nranges);
  const RegionIndex idx = region_view(d_index, N);
  k_range_plan<<<(unsigned)nchunks, 1024, 0, st>>>(d_ranges, nranges, N, idx.hdr, plan, flag);
  ctx->launches++;
  // the grid: every resident CTA, or fewer when the ranges cannot have that many pieces
  const size_t ntiles = region_layout(N).ntiles;
  const size_t max_pieces = nranges > PIECE_LIMIT / (ntiles + 1) ? (size_t)PIECE_LIMIT : nranges * (ntiles + 1);
  const size_t resident = (size_t)ctx->sm_count * ctx->occ_ranges[sizeof(T) == 8][QT];
  const size_t ctas = (max_pieces + Cfg::WARPS - 1) / Cfg::WARPS;
  const int grid = (int)(ctas < resident ? ctas : resident);
  const QtConsts<T> qk = make_qt<T>(eb);
  const T bw = (sizeof(T) == 8) ? (T)(eb * 2 * 1.0) : (T)(float)((float)eb * 2 * 1.0);  // as launch_decompress
  k_decompress_ranges<T, QT><<<grid, Cfg::THREADS, Cfg::SMEM, st>>>(d_bins, d_dc, d_ac, d_qtable, N, bw, (T)sf, qk, idx, n_outliers, d_ranges, nranges,
                                                                    plan, d_out, flag);
  ctx->launches++;
  CU(cudaGetLastError());
  return DCTZ_GPU_OK;
}

extern "C" int dctz_gpu_decompress_ranges_dev(dctz_gpu_ctx *ctx, const uint8_t *d_bins, const float *d_dc, const float *d_ac, uint64_t n_outliers,
                                              const void *d_qtable, size_t N, int datatype, double eb, double sf, int mode_qt, const void *d_index,
                                              const uint64_t *d_ranges, size_t nranges, void *d_out, uint32_t *d_corrupt, void *stream) {
  TRY(check_common(ctx, datatype, eb));
  if (!d_bins || !d_dc || !d_index || !d_ranges || !d_out || N == 0 || nranges == 0 || (n_outliers && !d_ac))
    return fail(ctx, DCTZ_GPU_EINVAL, "decompress_ranges: NULL pointer, N == 0 or no ranges");
  if (mode_qt && !d_qtable) return fail(ctx, DCTZ_GPU_EINVAL, "decompress_ranges: QT mode needs the qtable");
  const size_t es = datatype == DCTZ_GPU_DOUBLE ? 8 : 4;
  if (!aligned16(d_bins) || !aligned16(d_index) || ((uintptr_t)d_ranges & 7u) || ((uintptr_t)d_out & (es - 1)))
    return fail(ctx, DCTZ_GPU_EINVAL, "decompress_ranges: bin_index and the index must be 16-byte aligned, the ranges 8-byte, the output element-aligned");
  if (((uintptr_t)d_dc & 3u) || ((uintptr_t)d_ac & 3u) || ((uintptr_t)d_qtable & (es - 1)))
    return fail(ctx, DCTZ_GPU_EINVAL, "decompress_ranges: DC / AC_exact must be float-aligned, the qtable element-aligned");
  if (!(sf > 0.0) || isinf(sf)) return fail(ctx, DCTZ_GPU_EINVAL, "decompress_ranges: scaling factor %g is not a positive finite number", sf);
  if (nranges > ((size_t)1 << 40)) return fail(ctx, DCTZ_GPU_EINVAL, "decompress_ranges: %zu ranges", nranges);
  if (region_layout(N).ntiles > 0xFFFFF000ull) return fail(ctx, DCTZ_GPU_EINVAL, "decompress_ranges: slab too large");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  unsigned *flag = d_corrupt ? (unsigned *)d_corrupt : &ctx->d_ctl[1].corrupt;  // the caller's flag, else a scratch word nobody reads
  const unsigned long long *rg = (const unsigned long long *)d_ranges;
  const int E = decode_exponent(sf, datatype);
  const double sfk = decode_sf(sf, datatype, E);
  if (datatype == DCTZ_GPU_DOUBLE) {
    if (mode_qt) TRY((launch_ranges<double, true>(ctx, d_bins, d_dc, d_ac, n_outliers, (const double *)d_qtable, N, eb, sfk, d_index, rg, nranges, (double *)d_out, flag, st)));
    else TRY((launch_ranges<double, false>(ctx, d_bins, d_dc, d_ac, n_outliers, (const double *)d_qtable, N, eb, sfk, d_index, rg, nranges, (double *)d_out, flag, st)));
  } else {
    if (mode_qt) TRY((launch_ranges<float, true>(ctx, d_bins, d_dc, d_ac, n_outliers, (const float *)d_qtable, N, eb, sfk, d_index, rg, nranges, (float *)d_out, flag, st)));
    else TRY((launch_ranges<float, false>(ctx, d_bins, d_dc, d_ac, n_outliers, (const float *)d_qtable, N, eb, sfk, d_index, rg, nranges, (float *)d_out, flag, st)));
  }
  if (!E) return DCTZ_GPU_OK;
  // the plan launch_ranges left in ctx->region: output offsets per range (the decode wrote the places of the valid ranges)
  const RangePlan plan = range_plan_view(ctx->region.p, nranges);
  const int grid = ctx->sm_count * 8;
  if (datatype == DCTZ_GPU_DOUBLE) k_scale_ranges<double><<<grid, 256, 0, st>>>((double *)d_out, rg, nranges, N, plan, ldexp(1.0, E));
  else k_scale_ranges<float><<<grid, 256, 0, st>>>((float *)d_out, rg, nranges, N, plan, ldexpf(1.0f, E));
  ctx->launches++;
  CU(cudaGetLastError());
  return DCTZ_GPU_OK;
}

extern "C" int dctz_gpu_scale_dev(dctz_gpu_ctx *ctx, void *d_x, size_t N, int datatype, double sf, int multiply, void *stream) {
  TRY(check_common(ctx, datatype, 1.0));
  if (!d_x || N == 0) return fail(ctx, DCTZ_GPU_EINVAL, "scale: NULL pointer or N == 0");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  size_t want = (N + 255) / 256;
  const int grid = (int)(want < (size_t)ctx->sm_count * 16 ? want : (size_t)ctx->sm_count * 16);
  if (datatype == DCTZ_GPU_DOUBLE) k_scale<double><<<grid, 256, 0, st>>>((double *)d_x, N, sf, multiply);
  else k_scale<float><<<grid, 256, 0, st>>>((float *)d_x, N, (float)sf, multiply);
  ctx->launches++;
  CU(cudaGetLastError());
  return DCTZ_GPU_OK;
}

// ------------------------------------------------------------------------------------------
// host-buffer API (the drop-in seam)
//
// The caller's buffers are ordinary host memory (dctz-test.c:130-174 reads its file into malloc'ed arrays).  A
// pageable pointer handed to cudaMemcpyAsync goes through the driver's own bounce buffers at a fraction of the link
// speed and serialises with everything else, so the library stages it itself: a ring of NSTAGE page-locked slots,
// filled (or drained) by the host worker threads while the previous slot is on the wire.  Page-locked buffers
// (dctz_gpu_host_alloc, cudaHostRegister) are detected and copied directly.  Uploads are chunked on a copy stream and
// the statistics kernel of chunk k runs on the compute stream while chunk k+1 is still arriving: the chunks play the
// part of ranks (k_finalize merges their {max,min,sum} in chunk order), so when the last byte has landed only the
// transform kernel is left to run.  The caller-visible x/sf (dctz-comp-lib.c:198,213 scale the input in place) is an
// IEEE division done by the host threads on the caller's own buffer: nothing travels back over PCIe for it.
// ------------------------------------------------------------------------------------------
static bool host_is_pinned(const void *p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

static int host_threads() {
  const char *e = getenv("DCTZ_HOST_THREADS");
  long n = e ? atol(e) : (long)std::thread::hardware_concurrency();
  if (n < 1) n = 1;
  if (n > 16) n = 16;
  return (int)n;
}

static int ensure_pool(dctz_gpu_ctx *ctx) {
  if (!ctx->pool) {
    ctx->pool = new (std::nothrow) HostPool(host_threads() - 1);  // the calling thread works too
    if (!ctx->pool) return fail(ctx, DCTZ_GPU_ENOMEM, "out of host memory");
  }
  return DCTZ_GPU_OK;
}

static int ensure_stage_events(dctz_gpu_ctx *ctx) {
  for (int i = 0; i < NSTAGE; i++)
    if (!ctx->stage_ev[i]) CU(cudaEventCreateWithFlags(&ctx->stage_ev[i], cudaEventDisableTiming));
  return DCTZ_GPU_OK;
}

static int ensure_stage(dctz_gpu_ctx *ctx) {
  TRY(ensure_pool(ctx));
  TRY(ensure_stage_events(ctx));
  for (int i = 0; i < NSTAGE; i++)
    if (!ctx->stage[i]) CU(cudaMallocHost(&ctx->stage[i], STAGE_BYTES));
  return DCTZ_GPU_OK;
}

static void pool_memcpy(HostPool *pool, void *dst, const void *src, size_t bytes) {
  const size_t piece = (size_t)1 << 20;
  const int parts = (int)((bytes + piece - 1) / piece);
  if (parts <= 1) { memcpy(dst, src, bytes); return; }
  pool->parallel_for(parts, [=](int i) {
    const size_t off = (size_t)i * piece, len = bytes - off < piece ? bytes - off : piece;
    memcpy((char *)dst + off, (const char *)src + off, len);
  });
}

// Host -> device on the copy stream.  after_chunk(index, byte offset, bytes) is called once a chunk's copy has been
// enqueued and the compute stream has been told to wait for it.  `dominant` marks the direction-dominant transfer of a
// call (it holds the link gate, see LinkGate); the other transfers from page-locked memory are submitted whole.
static int upload(dctz_gpu_ctx *ctx, void *d_dst, const void *h_src, size_t bytes, size_t chunk_align,
                  const std::function<int(size_t, size_t, size_t)> &after_chunk, bool dominant = false) {
  if (bytes == 0) return DCTZ_GPU_OK;
  const bool pinned = host_is_pinned(h_src);
  if (pinned) TRY(ensure_stage_events(ctx));
  else TRY(ensure_stage(ctx));
  size_t chunk = pinned ? PINNED_CHUNK : STAGE_BYTES;
  if (pinned && !after_chunk && !dominant) chunk = bytes + chunk_align;  // submitted whole
  chunk -= chunk % chunk_align;
  size_t c = 0;
  for (size_t off = 0; off < bytes; off += chunk, c++) {
    const size_t len = bytes - off < chunk ? bytes - off : chunk;
    const void *src = (const char *)h_src + off;
    const int s = (int)(c % NSTAGE);
    // staged: the slot's previous content (this upload's or an earlier one's) is on the device; page-locked: at most
    // NSTAGE chunks in flight -- one while another call wants the link
    CU(cudaEventSynchronize(ctx->stage_ev[s]));
    if (pinned && dominant && c > 0 && link_contended(ctx->device)) CU(cudaEventSynchronize(ctx->stage_ev[(c - 1) % NSTAGE]));
    if (!pinned) {
      pool_memcpy(ctx->pool, ctx->stage[s], src, len);
      src = ctx->stage[s];
    }
    CU(cudaMemcpyAsync((char *)d_dst + off, src, len, cudaMemcpyHostToDevice, ctx->copy_stream));
    CU(cudaEventRecord(ctx->stage_ev[s], ctx->copy_stream));
    CU(cudaEventRecord(ctx->ev_chain, ctx->copy_stream));
    CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_chain, 0));
    if (after_chunk) TRY(after_chunk(c, off, len));
  }
  ctx->h2d_bytes += bytes;
  return DCTZ_GPU_OK;
}

// Device -> host of data produced on the compute stream; synchronous.  on_ready(byte offset, bytes) reports every
// piece as soon as it is valid in the caller's buffer (the host library starts deflating it while the rest is still
// on its way).  `dominant`: as for upload().
static int download(dctz_gpu_ctx *ctx, void *h_dst, const void *d_src, size_t bytes, const std::function<void(size_t, size_t)> &on_ready,
                    bool dominant = false) {
  if (bytes == 0) return DCTZ_GPU_OK;
  CU(cudaEventRecord(ctx->ev_chain, ctx->stream));
  CU(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_chain, 0));
  const bool pinned = host_is_pinned(h_dst);
  ctx->d2h_bytes += bytes;
  if (pinned && !on_ready && !dominant) {  // submitted whole
    CU(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, ctx->copy_stream));
    CU(cudaStreamSynchronize(ctx->copy_stream));
    return DCTZ_GPU_OK;
  }
  if (pinned) TRY(ensure_stage_events(ctx));  // (the events are used in both modes)
  else TRY(ensure_stage(ctx));
  const size_t chunk = pinned ? PINNED_CHUNK : STAGE_BYTES;
  const size_t nchunks = (bytes + chunk - 1) / chunk;
  // chunks on the wire beside the one being handed over (none while another call wants the link, see LinkGate)
  const size_t depth = !pinned ? 1 : dominant && link_contended(ctx->device) ? 0 : NSTAGE - 1;
  auto span = [&](size_t c, size_t *off, size_t *len) { *off = c * chunk; *len = bytes - *off < chunk ? bytes - *off : chunk; };
  for (size_t c = 0; c < nchunks + depth; c++) {  // chunk c goes on the wire, chunk c-depth is handed over
    if (c < nchunks) {
      size_t off, len;
      span(c, &off, &len);
      const int s = (int)(c % NSTAGE);
      void *dst = pinned ? (void *)((char *)h_dst + off) : ctx->stage[s];
      CU(cudaMemcpyAsync(dst, (const char *)d_src + off, len, cudaMemcpyDeviceToHost, ctx->copy_stream));
      CU(cudaEventRecord(ctx->stage_ev[s], ctx->copy_stream));
    }
    if (c >= depth) {
      size_t off, len;
      span(c - depth, &off, &len);
      const int s = (int)((c - depth) % NSTAGE);
      CU(cudaEventSynchronize(ctx->stage_ev[s]));
      if (dominant && c == depth) ctx->times[6] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - ctx->t_call).count();
      if (!pinned) pool_memcpy(ctx->pool, (char *)h_dst + off, ctx->stage[s], len);
      if (on_ready) on_ready(off, len);
    }
  }
  return DCTZ_GPU_OK;
}

template <typename T> static void host_scale(HostPool *pool, T *dst, const T *src, size_t n, T sf) {
  const size_t piece = (size_t)1 << 18;
  const int parts = (int)((n + piece - 1) / piece);
  auto body = [=](int i) {
    const size_t a = (size_t)i * piece, b = a + piece < n ? a + piece : n;
    for (size_t k = a; k < b; k++) dst[k] = src[k] / sf;  // IEEE division, element type: dctz-comp-lib.c:198 / :213
  };
  if (parts <= 1 || !pool) { for (int i = 0; i < parts; i++) body(i); return; }
  pool->parallel_for(parts, body);
}

static float elapsed_ms(cudaEvent_t a, cudaEvent_t b) {
  float ms = 0.f;
  if (cudaEventElapsedTime(&ms, a, b) != cudaSuccess) { cudaGetLastError(); return 0.f; }
  return ms;
}

static int compress_core_impl(dctz_gpu_ctx *ctx, const void *in, size_t N, size_t N_total, const double *stats3, int first_piece,
                              int datatype, double eb, int mode_qt, void *scaled_out, uint8_t *bin_index, float *DC, float *AC_exact,
                              void *qtable, void *qtable_raw, dctz_gpu_info *info, dctz_gpu_section_cb cb, void *cb_user) {
  TRY(check_common(ctx, datatype, eb));
  if (!in || !bin_index || !DC || !AC_exact || !info || N == 0) return fail(ctx, DCTZ_GPU_EINVAL, "compress_core: NULL pointer or N == 0");
  if (mode_qt && !qtable) return fail(ctx, DCTZ_GPU_EINVAL, "compress_core: QT mode needs a qtable output");
  CU(cudaSetDevice(ctx->device));
  const size_t es = datatype == DCTZ_GPU_DOUBLE ? 8 : 4;
  const size_t nblk = (N + BLK - 1) / BLK;
  cudaStream_t st = ctx->stream;
  ctx->h2d_bytes = ctx->d2h_bytes = 0;
  for (double &t : ctx->times) t = 0.0;
  TRY(grow(ctx, ctx->in, N * es));
  TRY(grow(ctx, ctx->bins, N));
  TRY(grow(ctx, ctx->dc, nblk * 4));
  TRY(grow(ctx, ctx->ac, N * 4));
  TRY(grow(ctx, ctx->qt, BLK * 8));
  TRY(grow(ctx, ctx->qtraw, BLK * 8));
  dctz_gpu_info *d_info = (dctz_gpu_info *)ctx->d_info;
  const bool pinned_in = host_is_pinned(in);
  const size_t up_chunk = pinned_in ? PINNED_CHUNK : STAGE_BYTES;
  const size_t nchunks = (N * es + up_chunk - 1) / up_chunk;
  const auto t_begin = std::chrono::steady_clock::now();
  ctx->t_call = t_begin;
  BusyMark busy(ctx->device);
  if (ctx->timing) CU(cudaEventRecord(ctx->ev_time[0], st));
  // compress is the upload-heavy call: it holds the device's upload gate until its kernels have run (see LinkGate)
  std::unique_lock<std::mutex> up_gate;
  if (link_gates_enabled() && N * es >= GATE_BYTES && ctx->device < 64) up_gate = std::unique_lock<std::mutex>(g_gate[ctx->device].up);
  ctx->times[5] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();  // gate taken

  if (stats3) {  // the caller's global statistics decide the scaling factor
    CU(cudaMemcpyAsync(ctx->d_stats_host3, stats3, 3 * sizeof(double), cudaMemcpyHostToDevice, st));
    TRY(upload(ctx, ctx->in.p, in, N * es, 1024, nullptr, up_gate.owns_lock()));
    if (ctx->timing) { CU(cudaStreamSynchronize(st)); CU(cudaEventRecord(ctx->ev_time[1], st)); CU(cudaEventRecord(ctx->ev_time[2], st)); }
    TRY(dctz_gpu_compress_dev(ctx, ctx->in.p, N, N_total, datatype, eb, mode_qt, ctx->d_stats_host3, 1, first_piece, (uint8_t *)ctx->bins.p,
                              (float *)ctx->dc.p, (float *)ctx->ac.p, ctx->qtraw.p, d_info, st));
    if (mode_qt) TRY(dctz_gpu_qt_finish_dev(ctx, datatype, eb, ctx->qtraw.p, ctx->qt.p, (float *)ctx->ac.p, d_info, st));
  } else if (ctx->timing) {  // stage timers wanted (the reference's -DTIME_DEBUG lines): upload, statistics, transform one after the other
    TRY(upload(ctx, ctx->in.p, in, N * es, 1024, nullptr, up_gate.owns_lock()));
    CU(cudaStreamSynchronize(st));
    CU(cudaEventRecord(ctx->ev_time[1], st));
    TRY(dctz_gpu_stats_dev(ctx, ctx->in.p, N, datatype, ctx->d_stats3, st));
    CU(cudaEventRecord(ctx->ev_time[2], st));
    TRY(dctz_gpu_compress_dev(ctx, ctx->in.p, N, N, datatype, eb, mode_qt, ctx->d_stats3, 1, 1, (uint8_t *)ctx->bins.p, (float *)ctx->dc.p,
                              (float *)ctx->ac.p, ctx->qtraw.p, d_info, st));
    if (mode_qt) TRY(dctz_gpu_qt_finish_dev(ctx, datatype, eb, ctx->qtraw.p, ctx->qt.p, (float *)ctx->ac.p, d_info, st));
  } else if (nchunks == 1 || fused_grid(ctx, 0, N, es, mode_qt)) {  // one upload, then the single-field path (small fields: ONE launch)
    TRY(upload(ctx, ctx->in.p, in, N * es, 1024, nullptr, up_gate.owns_lock()));
    TRY(dctz_gpu_compress_field_dev(ctx, ctx->in.p, N, datatype, eb, mode_qt, (uint8_t *)ctx->bins.p, (float *)ctx->dc.p,
                                    (float *)ctx->ac.p, ctx->qt.p, ctx->qtraw.p, d_info, st));
  } else {  // statistics of chunk k while chunk k+1 is on the wire; the chunks are merged like ranks
    TRY(grow(ctx, ctx->chunk_stats, nchunks * 3 * sizeof(double)));
    double *d_cs = (double *)ctx->chunk_stats.p;
    TRY(upload(ctx, ctx->in.p, in, N * es, 1024, [&](size_t c, size_t off, size_t len) -> int {
      return dctz_gpu_stats_dev(ctx, (const char *)ctx->in.p + off, len / es, datatype, d_cs + 3 * c, st);
    }, up_gate.owns_lock()));
    TRY(dctz_gpu_compress_dev(ctx, ctx->in.p, N, N, datatype, eb, mode_qt, d_cs, (int)nchunks, 1, (uint8_t *)ctx->bins.p,
                              (float *)ctx->dc.p, (float *)ctx->ac.p, ctx->qtraw.p, d_info, st));
    if (mode_qt) TRY(dctz_gpu_qt_finish_dev(ctx, datatype, eb, ctx->qtraw.p, ctx->qt.p, (float *)ctx->ac.p, d_info, st));
  }
  if (ctx->timing) CU(cudaEventRecord(ctx->ev_time[3], st));
  CU(cudaMemcpyAsync(info, ctx->d_info, sizeof(Info), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  if (up_gate.owns_lock()) up_gate.unlock();
  ctx->d2h_bytes += sizeof(Info);
  if (info->status != 0)
    return fail(ctx, info->status, "compress_core: max|x| = %g gives no usable scaling factor (util.c:28 would yield 0/inf/NaN)", info->max_abs);
  const auto t_gpu = std::chrono::steady_clock::now();

  // the caller-visible scaled input: host threads, overlapping the downloads when those need no staging copies
  const bool scale = scaled_out && (info->sf != 1.0 || scaled_out != in);
  // (the staged downloads need the worker threads themselves: overlap only when none of them is staged)
  const bool overlap = scale && !cb && host_is_pinned(bin_index) && host_is_pinned(DC) && host_is_pinned(AC_exact);
  auto do_scale = [&](bool async) -> int {
    TRY(ensure_pool(ctx));
    if (info->sf == 1.0) { pool_memcpy(ctx->pool, scaled_out, in, N * es); return DCTZ_GPU_OK; }  // dctz-comp-lib.c:193/:208 skip the loop
    if (async) {
      const size_t piece = (size_t)1 << 18;
      const int parts = (int)((N + piece - 1) / piece);
      if (es == 8) {
        double *d = (double *)scaled_out; const double *s2 = (const double *)in; const double sf = info->sf;
        ctx->pool->start(parts, [=](int i) { const size_t a = (size_t)i * piece, b = a + piece < N ? a + piece : N; for (size_t k = a; k < b; k++) d[k] = s2[k] / sf; });
      } else {
        float *d = (float *)scaled_out; const float *s2 = (const float *)in; const float sf = (float)info->sf;
        ctx->pool->start(parts, [=](int i) { const size_t a = (size_t)i * piece, b = a + piece < N ? a + piece : N; for (size_t k = a; k < b; k++) d[k] = s2[k] / sf; });
      }
      return DCTZ_GPU_OK;
    }
    if (es == 8) host_scale<double>(ctx->pool, (double *)scaled_out, (const double *)in, N, info->sf);
    else host_scale<float>(ctx->pool, (float *)scaled_out, (const float *)in, N, (float)info->sf);
    return DCTZ_GPU_OK;
  };
  if (overlap) TRY(do_scale(info->sf != 1.0));

  auto section = [&](int id) -> std::function<void(size_t, size_t)> {
    if (!cb) return nullptr;
    return [=](size_t off, size_t len) { cb(cb_user, id, off, len); };
  };
  // the float sections first: they are small on the wire and slow to deflate, so the host library's workers start on them
  TRY(download(ctx, DC, ctx->dc.p, nblk * 4, section(1)));
  TRY(download(ctx, AC_exact, ctx->ac.p, (size_t)info->n_outliers * 4, section(2)));
  TRY(download(ctx, bin_index, ctx->bins.p, N, section(0)));
  if (cb && info->n_outliers == 0) cb(cb_user, 2, 0, 0);  // every section is reported at least once
  if (mode_qt) {
    CU(cudaMemcpyAsync(qtable, ctx->qt.p, BLK * es, cudaMemcpyDeviceToHost, st));
    if (qtable_raw) CU(cudaMemcpyAsync(qtable_raw, ctx->qtraw.p, BLK * es, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    ctx->d2h_bytes += (qtable_raw ? 2 : 1) * BLK * es;
  }
  if (overlap) { if (info->sf != 1.0) ctx->pool->wait(); }
  else if (scale) TRY(do_scale(false));
  if (ctx->timing) {
    ctx->times[0] = elapsed_ms(ctx->ev_time[0], ctx->ev_time[1]);  // upload
    ctx->times[1] = elapsed_ms(ctx->ev_time[1], ctx->ev_time[2]);  // statistics                          (the reference's sf_t)
    ctx->times[2] = elapsed_ms(ctx->ev_time[2], ctx->ev_time[3]);  // scale + DCT + quantise + outliers   (the reference's dct_t)
  }
  ctx->times[3] = std::chrono::duration<double, std::milli>(t_gpu - t_begin).count();                                   // upload + kernels (wall clock)
  ctx->times[4] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_gpu).count();          // downloads + host scaling
  return DCTZ_GPU_OK;
}

extern "C" int dctz_gpu_compress_core(dctz_gpu_ctx *ctx, const void *in, size_t N, int datatype, double eb, int mode_qt,
                                      void *scaled_out, uint8_t *bin_index, float *DC, float *AC_exact, void *qtable,
                                      void *qtable_raw, dctz_gpu_info *info) {
  return compress_core_impl(ctx, in, N, N, nullptr, 1, datatype, eb, mode_qt, scaled_out, bin_index, DC, AC_exact, qtable, qtable_raw, info,
                            nullptr, nullptr);
}

extern "C" int dctz_gpu_compress_core_cb(dctz_gpu_ctx *ctx, const void *in, size_t N, int datatype, double eb, int mode_qt,
                                         void *scaled_out, uint8_t *bin_index, float *DC, float *AC_exact, void *qtable,
                                         void *qtable_raw, dctz_gpu_info *info, dctz_gpu_section_cb on_ready, void *user) {
  return compress_core_impl(ctx, in, N, N, nullptr, 1, datatype, eb, mode_qt, scaled_out, bin_index, DC, AC_exact, qtable, qtable_raw, info,
                            on_ready, user);
}

extern "C" int dctz_gpu_compress_core_with_stats(dctz_gpu_ctx *ctx, const void *in, size_t N, size_t N_total, const double stats3[3],
                                                 int first_piece, int datatype, double eb, int mode_qt, void *scaled_out,
                                                 uint8_t *bin_index, float *DC, float *AC_exact, void *qtable, void *qtable_raw,
                                                 dctz_gpu_info *info) {
  if (!stats3 || N_total < N) return fail(ctx, DCTZ_GPU_EINVAL, "compress_core_with_stats: bad statistics arguments");
  return compress_core_impl(ctx, in, N, N_total, stats3, first_piece, datatype, eb, mode_qt, scaled_out, bin_index, DC, AC_exact, qtable,
                            qtable_raw, info, nullptr, nullptr);
}

// Phase boundaries of the last single-launch kernel (kernel 0 = compress, 1 = decompress), synchronous: for every stamp
// k (fused.cuh) the earliest and the latest CTA, in microseconds after the earliest CTA's start: out[2k], out[2k+1].
extern "C" int dctz_gpu_fused_phase_times(dctz_gpu_ctx *ctx, int kernel, double out_us[16]) {
  if (!ctx || kernel < 0 || kernel > 1 || !out_us) return fail(ctx, DCTZ_GPU_EINVAL, "fused_phase_times: bad arguments");
  const int grid = ctx->dbg_grid[kernel];
  if (grid <= 0) return fail(ctx, DCTZ_GPU_EINVAL, "fused_phase_times: no single-launch kernel has run with DCTZ_FUSED_STAMPS=1");
  CU(cudaSetDevice(ctx->device));
  CU(cudaDeviceSynchronize());
  std::vector<unsigned long long> h((size_t)grid * 8);
  CU(cudaMemcpy(h.data(), ctx->d_dbg + (size_t)kernel * ctx->sm_count * 4 * 8, h.size() * 8, cudaMemcpyDeviceToHost));
  unsigned long long t0 = ~0ull;
  for (int b = 0; b < grid; b++) t0 = h[8 * b] < t0 ? h[8 * b] : t0;
  const int nstamp = kernel == 0 ? 6 : 4;
  for (int k = 0; k < 8; k++) {
    unsigned long long lo = ~0ull, hi = 0;
    for (int b = 0; b < grid && k < nstamp; b++) { const unsigned long long v = h[8 * b + k]; lo = v < lo ? v : lo; hi = v > hi ? v : hi; }
    out_us[2 * k] = k < nstamp ? (double)(lo - t0) / 1e3 : 0.0;
    out_us[2 * k + 1] = k < nstamp ? (double)(hi - t0) / 1e3 : 0.0;
  }
  return DCTZ_GPU_OK;
}

extern "C" int dctz_gpu_set_timing(dctz_gpu_ctx *ctx, int on) {
  if (!ctx) return fail(nullptr, DCTZ_GPU_EINVAL, "ctx is NULL");
  const int prev = ctx->timing;
  ctx->timing = on ? 1 : 0;
  return prev;
}

extern "C" int dctz_gpu_last_call_stats(const dctz_gpu_ctx *ctx, double times_ms[8], uint64_t *h2d_bytes, uint64_t *d2h_bytes) {
  if (!ctx) return fail(nullptr, DCTZ_GPU_EINVAL, "ctx is NULL");
  if (times_ms) for (int i = 0; i < 8; i++) times_ms[i] = ctx->times[i];
  if (h2d_bytes) *h2d_bytes = ctx->h2d_bytes;
  if (d2h_bytes) *d2h_bytes = ctx->d2h_bytes;
  return DCTZ_GPU_OK;
}

template <typename T>
static int launch_quality(dctz_gpu_ctx *ctx, const T *a, const T *b, size_t N, double *d_out4, cudaStream_t st) {
  size_t want = (N + 255) / 256 / 8 + 1;
  const int grid = (int)(want < (size_t)ctx->stat_grid ? want : (size_t)ctx->stat_grid);
  k_quality<T><<<grid, 256, 0, st>>>(a, b, N, ctx->d_qpartials, ctx->d_done + 2, (QualityPartial *)d_out4);
  ctx->launches++;
  CU(cudaGetLastError());
  return DCTZ_GPU_OK;
}

extern "C" int dctz_gpu_quality_dev(dctz_gpu_ctx *ctx, const void *d_a, const void *d_b, size_t N, int datatype, double *d_out4, void *stream) {
  TRY(check_common(ctx, datatype, 1.0));
  if (!d_a || !d_b || !d_out4 || N == 0) return fail(ctx, DCTZ_GPU_EINVAL, "quality: NULL pointer or N == 0");
  CU(cudaSetDevice(ctx->device));
  if (datatype == DCTZ_GPU_DOUBLE) return launch_quality<double>(ctx, (const double *)d_a, (const double *)d_b, N, d_out4, (cudaStream_t)stream);
  return launch_quality<float>(ctx, (const float *)d_a, (const float *)d_b, N, d_out4, (cudaStream_t)stream);
}

extern "C" int dctz_gpu_quality(dctz_gpu_ctx *ctx, const void *a, const void *b, size_t N, int datatype, double out4[4]) {
  TRY(check_common(ctx, datatype, 1.0));
  if (!a || !b || !out4 || N == 0) return fail(ctx, DCTZ_GPU_EINVAL, "quality: NULL pointer or N == 0");
  CU(cudaSetDevice(ctx->device));
  const size_t es = datatype == DCTZ_GPU_DOUBLE ? 8 : 4;
  cudaStream_t st = ctx->stream;
  TRY(grow(ctx, ctx->in, N * es));
  TRY(grow(ctx, ctx->out, N * es));
  TRY(upload(ctx, ctx->in.p, a, N * es, 1024, nullptr));
  TRY(upload(ctx, ctx->out.p, b, N * es, 1024, nullptr));
  double *d_res = (double *)(ctx->d_qpartials + ctx->stat_grid);
  TRY(dctz_gpu_quality_dev(ctx, ctx->in.p, ctx->out.p, N, datatype, d_res, st));
  CU(cudaMemcpyAsync(out4, d_res, 4 * sizeof(double), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return DCTZ_GPU_OK;
}

extern "C" int dctz_gpu_stats(dctz_gpu_ctx *ctx, const void *in, size_t N, int datatype, dctz_gpu_info *info) {
  TRY(check_common(ctx, datatype, 1.0));
  if (!in || !info || N == 0) return fail(ctx, DCTZ_GPU_EINVAL, "stats: NULL pointer or N == 0");
  CU(cudaSetDevice(ctx->device));
  const size_t es = datatype == DCTZ_GPU_DOUBLE ? 8 : 4;
  cudaStream_t st = ctx->stream;
  TRY(grow(ctx, ctx->in, N * es));
  TRY(upload(ctx, ctx->in.p, in, N * es, 1024, nullptr));
  if (datatype == DCTZ_GPU_DOUBLE) TRY(launch_stats<double>(ctx, (const double *)ctx->in.p, N, ctx->d_stats3, 1, N, nullptr, ctx->d_info, st));
  else TRY(launch_stats<float>(ctx, (const float *)ctx->in.p, N, ctx->d_stats3, 1, N, nullptr, ctx->d_info, st));
  CU(cudaMemcpyAsync(info, ctx->d_info, sizeof(Info), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return DCTZ_GPU_OK;
}

extern "C" int dctz_gpu_decompress_core(dctz_gpu_ctx *ctx, const uint8_t *bin_index, const float *DC, const float *AC_exact,
                                        uint64_t n_outliers, const void *qtable, size_t N, int datatype, double eb, double sf,
                                        int mode_qt, void *out) {
  TRY(check_common(ctx, datatype, eb));
  if (!bin_index || !DC || !out || N == 0 || (n_outliers && !AC_exact)) return fail(ctx, DCTZ_GPU_EINVAL, "decompress_core: NULL pointer or N == 0");
  if (mode_qt && !qtable) return fail(ctx, DCTZ_GPU_EINVAL, "decompress_core: QT mode needs the qtable");
  CU(cudaSetDevice(ctx->device));
  const size_t es = datatype == DCTZ_GPU_DOUBLE ? 8 : 4;
  const size_t nblk = (N + BLK - 1) / BLK;
  cudaStream_t st = ctx->stream;
  TRY(grow(ctx, ctx->bins, N));
  TRY(grow(ctx, ctx->dc, nblk * 4));
  TRY(grow(ctx, ctx->ac, (n_outliers ? n_outliers : 1) * 4));
  TRY(grow(ctx, ctx->qt, BLK * 8));
  TRY(grow(ctx, ctx->out, N * es));
  ctx->h2d_bytes = ctx->d2h_bytes = 0;
  for (double &t : ctx->times) t = 0.0;
  const auto t_begin = std::chrono::steady_clock::now();
  ctx->t_call = t_begin;
  BusyMark busy(ctx->device);
  if (ctx->timing) CU(cudaEventRecord(ctx->ev_time[0], st));
  TRY(upload(ctx, ctx->bins.p, bin_index, N, 1024, nullptr));
  TRY(upload(ctx, ctx->dc.p, DC, nblk * 4, 4, nullptr));
  if (n_outliers) TRY(upload(ctx, ctx->ac.p, AC_exact, n_outliers * 4, 4, nullptr));
  if (mode_qt) { CU(cudaMemcpyAsync(ctx->qt.p, qtable, BLK * es, cudaMemcpyHostToDevice, st)); ctx->h2d_bytes += BLK * es; }
  if (ctx->timing) { CU(cudaStreamSynchronize(ctx->copy_stream)); CU(cudaEventRecord(ctx->ev_time[1], st)); }
  // The kernels never read past the n_outliers floats the caller handed over: a stream whose bin indices mark more
  // outliers than that is reported as corrupt (the reference would read whatever follows its buffer).
  CU(cudaMemsetAsync(&ctx->d_ctl[1].corrupt, 0, sizeof(unsigned), st));
  TRY(dctz_gpu_decompress_dev(ctx, (const uint8_t *)ctx->bins.p, (const float *)ctx->dc.p, (const float *)ctx->ac.p, n_outliers, ctx->qt.p, N,
                              datatype, eb, sf, mode_qt, ctx->out.p, &ctx->d_ctl[1].corrupt, st));
  if (ctx->timing) CU(cudaEventRecord(ctx->ev_time[2], st));
  unsigned corrupt = 0;
  CU(cudaMemcpyAsync(&corrupt, &ctx->d_ctl[1].corrupt, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
  const auto t_gpu = std::chrono::steady_clock::now();
  {  // decompress is the download-heavy call: it holds the device's download gate while the reconstruction travels
    std::unique_lock<std::mutex> down_gate;
    if (link_gates_enabled() && N * es >= GATE_BYTES && ctx->device < 64) down_gate = std::unique_lock<std::mutex>(g_gate[ctx->device].down);
    ctx->times[5] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - ctx->t_call).count();  // gate taken
    TRY(download(ctx, out, ctx->out.p, N * es, nullptr, down_gate.owns_lock()));
  }
  CU(cudaStreamSynchronize(st));
  if (ctx->timing) {
    ctx->times[0] = elapsed_ms(ctx->ev_time[0], ctx->ev_time[1]);  // upload
    ctx->times[2] = elapsed_ms(ctx->ev_time[1], ctx->ev_time[2]);  // outlier scan + dequantise + inverse DCT + de-scale (the reference's idct_t + sf_t)
  }
  ctx->times[3] = std::chrono::duration<double, std::milli>(t_gpu - t_begin).count();
  ctx->times[4] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_gpu).count();
  if (corrupt) return fail(ctx, DCTZ_GPU_ECORRUPT, "decompress_core: the bin indices mark more outliers than the %llu given", (unsigned long long)n_outliers);
  return DCTZ_GPU_OK;
}

// ------------------------------------------------------------------------------------------
// DCT-only entry point (dct.h:17-27 equivalents) and utilities
// ------------------------------------------------------------------------------------------
template <typename T>
static int dct_blocks_impl(dctz_gpu_ctx *ctx, const T *in, T *out, size_t nblocks, int dn, int inverse) {
  const size_t bytes = nblocks * (size_t)dn * sizeof(T);
  cudaStream_t st = ctx->stream;
  TRY(grow(ctx, ctx->in, bytes));
  TRY(grow(ctx, ctx->out, bytes));
  CU(cudaMemcpyAsync(ctx->in.p, in, bytes, cudaMemcpyHostToDevice, st));
  if (dn == BLK) {
    const unsigned grid = (unsigned)((nblocks + DCT_ONLY_THREADS - 1) / DCT_ONLY_THREADS);
    if (inverse) k_dct64_blocks<T, true><<<grid, DCT_ONLY_THREADS, 0, st>>>((const T *)ctx->in.p, (T *)ctx->out.p, nblocks);
    else k_dct64_blocks<T, false><<<grid, DCT_ONLY_THREADS, 0, st>>>((const T *)ctx->in.p, (T *)ctx->out.p, nblocks);
  } else {
    if (inverse) k_dct_generic_blocks<T, true><<<(unsigned)nblocks, 32, 0, st>>>((const T *)ctx->in.p, (T *)ctx->out.p, dn);
    else k_dct_generic_blocks<T, false><<<(unsigned)nblocks, 32, 0, st>>>((const T *)ctx->in.p, (T *)ctx->out.p, dn);
  }
  ctx->launches++;
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(out, ctx->out.p, bytes, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return DCTZ_GPU_OK;
}

extern "C" int dctz_gpu_dct_blocks(dctz_gpu_ctx *ctx, const void *in, void *out, size_t nblocks, int dn, int datatype, int inverse) {
  TRY(check_common(ctx, datatype, 1.0));
  if (!in || !out || nblocks == 0 || dn < 1 || dn > BLK) return fail(ctx, DCTZ_GPU_EINVAL, "dct_blocks: bad arguments (1 <= dn <= 64)");
  if (nblocks > 0x7FFFFFFFull) return fail(ctx, DCTZ_GPU_EINVAL, "dct_blocks: too many blocks");
  CU(cudaSetDevice(ctx->device));
  if (datatype == DCTZ_GPU_DOUBLE) return dct_blocks_impl<double>(ctx, (const double *)in, (double *)out, nblocks, dn, inverse);
  return dct_blocks_impl<float>(ctx, (const float *)in, (float *)out, nblocks, dn, inverse);
}

// Transform-only entry point on device buffers; variant 0 = register butterfly, 1 = FP64 DMMA matrix form.
static int ensure_dfrag(dctz_gpu_ctx *ctx, int inverse) {
  if (ctx->d_dfrag[inverse]) return DCTZ_GPU_OK;
  std::vector<double> f(BLK * BLK);
  const long double pi = 3.14159265358979323846264338327950288L;
  for (int i = 0; i < 8; i++)
    for (int s = 0; s < 16; s++)
      for (int lane = 0; lane < 32; lane++) {
        int row = 8 * i + lane / 4, col = 4 * s + lane % 4;  // entry M[row][col] of the matrix applied to a block
        int k = inverse ? col : row, n = inverse ? row : col;  // orthonormal DCT-II: C[k][n]; inverse = transpose
        long double v = sqrtl(2.0L / BLK) * cosl(pi * (long double)(((2 * n + 1) * k) % (4 * BLK)) / (2.0L * BLK));
        if (k == 0) v /= sqrtl(2.0L);
        f[(i * 16 + s) * 32 + lane] = (double)v;
      }
  CU(cudaMalloc(&ctx->d_dfrag[inverse], f.size() * sizeof(double)));
  CU(cudaMemcpy(ctx->d_dfrag[inverse], f.data(), f.size() * sizeof(double), cudaMemcpyHostToDevice));
  return DCTZ_GPU_OK;
}

static int ensure_dfrag_split(dctz_gpu_ctx *ctx, int inverse) {
  if (ctx->d_dfrag2[inverse]) return DCTZ_GPU_OK;
  std::vector<double> f(2 * 32 * 32);
  const long double pi = 3.14159265358979323846264338327950288L;
  for (int m = 0; m < 2; m++)
    for (int i = 0; i < 4; i++)
      for (int s = 0; s < 8; s++)
        for (int lane = 0; lane < 32; lane++) {
          const int row = 8 * i + lane / 4, col = 4 * s + lane % 4;
          const int kh = inverse ? col : row, n = inverse ? row : col;  // forward: M_m[kh][n] = C[2 kh + m][n]; inverse: transposed
          const int k = 2 * kh + m;
          long double v = sqrtl(2.0L / BLK) * cosl(pi * (long double)(((2 * n + 1) * k) % (4 * BLK)) / (2.0L * BLK));
          if (k == 0) v /= sqrtl(2.0L);
          f[(size_t)m * 1024 + (i * 8 + s) * 32 + lane] = (double)v;
        }
  CU(cudaMalloc(&ctx->d_dfrag2[inverse], f.size() * sizeof(double)));
  CU(cudaMemcpy(ctx->d_dfrag2[inverse], f.data(), f.size() * sizeof(double), cudaMemcpyHostToDevice));
  return DCTZ_GPU_OK;
}

// FP64 rate probes: kind 0 = DFMA (vector pipe), 1 = DMMA m8n8k4 (tensor pipe); *tflops = the measured rate.
extern "C" int dctz_gpu_fp64_rate(dctz_gpu_ctx *ctx, int kind, double *tflops) {
  if (!ctx || !tflops || kind < 0 || kind > 1) return fail(ctx, DCTZ_GPU_EINVAL, "fp64_rate: bad arguments");
  CU(cudaSetDevice(ctx->device));
  const int iters = 4096, grid = ctx->sm_count * 8;
  cudaEvent_t e0, e1;
  CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
  k_fp64_rate<<<grid, 256, 0, ctx->stream>>>(kind, 64, 1.0, ctx->d_stats3);  // warm-up
  CU(cudaEventRecord(e0, ctx->stream));
  k_fp64_rate<<<grid, 256, 0, ctx->stream>>>(kind, iters, 1.0, ctx->d_stats3);
  CU(cudaEventRecord(e1, ctx->stream));
  CU(cudaEventSynchronize(e1));
  float ms = 0.f;
  CU(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  ctx->launches += 2;
  // kind 0: 32 DFMA per thread and iteration = 64 flop; kind 1: 32 DMMA per WARP and iteration, 8*8*4*2 = 512 flop each
  const double flop = kind == 0 ? (double)grid * 256 * iters * 64.0 : (double)grid * 8 * iters * 32.0 * 512.0;
  *tflops = flop / (ms * 1e-3) / 1e12;
  return DCTZ_GPU_OK;
}

extern "C" int dctz_gpu_dct64_dev(dctz_gpu_ctx *ctx, const void *d_in, void *d_out, size_t nblocks, int datatype, int inverse, int variant,
                                  void *stream) {
  TRY(check_common(ctx, datatype, 1.0));
  if (!d_in || !d_out || nblocks == 0 || !aligned16(d_in) || !aligned16(d_out)) return fail(ctx, DCTZ_GPU_EINVAL, "dct64_dev: bad pointers");
  if (variant != 0 && !((variant == 1 || variant == 2) && datatype == DCTZ_GPU_DOUBLE)) return fail(ctx, DCTZ_GPU_EINVAL, "dct64_dev: variant %d not available for this type", variant);
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t es = datatype == DCTZ_GPU_DOUBLE ? 8 : 4;
  CUtensorMap tin, tout;
  TRY(make_tile_map(ctx, &tin, d_in, BLK * es, nblocks));
  TRY(make_tile_map(ctx, &tout, d_out, BLK * es, nblocks));
  const size_t ntiles = (nblocks + WTILE - 1) / WTILE, ctas = (ntiles + 3) / 4;
  const size_t resident = (size_t)ctx->sm_count * (datatype == DCTZ_GPU_DOUBLE ? 2 : 3);
  const int grid = (int)(ctas < resident ? ctas : resident);
  if (variant == 2) {
    TRY(ensure_dfrag_split(ctx, inverse ? 1 : 0));
    auto k = inverse ? k_dct64_dmma_split<true> : k_dct64_dmma_split<false>;
    CU(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, DctOnlyCfg<double>::SMEM));
    k<<<grid, DctOnlyCfg<double>::THREADS, DctOnlyCfg<double>::SMEM, st>>>(tin, tout, nblocks, ctx->d_dfrag2[inverse ? 1 : 0]);
  } else if (variant == 1) {
    TRY(ensure_dfrag(ctx, inverse ? 1 : 0));
    CU(cudaFuncSetAttribute(k_dct64_dmma, cudaFuncAttributeMaxDynamicSharedMemorySize, DctOnlyCfg<double>::SMEM));
    k_dct64_dmma<<<grid, DctOnlyCfg<double>::THREADS, DctOnlyCfg<double>::SMEM, st>>>(tin, tout, nblocks, ctx->d_dfrag[inverse ? 1 : 0]);
  } else if (datatype == DCTZ_GPU_DOUBLE) {
    auto k = inverse ? k_dct64_tile<double, true> : k_dct64_tile<double, false>;
    CU(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, DctOnlyCfg<double>::SMEM));
    k<<<grid, DctOnlyCfg<double>::THREADS, DctOnlyCfg<double>::SMEM, st>>>(tin, tout, nblocks);
  } else {
    auto k = inverse ? k_dct64_tile<float, true> : k_dct64_tile<float, false>;
    CU(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, DctOnlyCfg<float>::SMEM));
    k<<<grid, DctOnlyCfg<float>::THREADS, DctOnlyCfg<float>::SMEM, st>>>(tin, tout, nblocks);
  }
  ctx->launches++;
  CU(cudaGetLastError());
  return DCTZ_GPU_OK;
}

extern "C" int dctz_gpu_fill_hash_field(dctz_gpu_ctx *ctx, double *d_out, uint64_t start, uint64_t count, uint32_t dim, uint32_t seed,
                                        void *stream) {
  if (!ctx) return fail(nullptr, DCTZ_GPU_EINVAL, "ctx is NULL");
  if (!d_out || count == 0 || dim == 0 || (dim & (dim - 1))) return fail(ctx, DCTZ_GPU_EINVAL, "fill_hash_field: dim must be a power of two");
  CU(cudaSetDevice(ctx->device));
  k_fill_hash_field<<<ctx->sm_count * 16, 256, 0, (cudaStream_t)stream>>>(d_out, start, count, dim, seed);
  ctx->launches++;
  CU(cudaGetLastError());
  return DCTZ_GPU_OK;
}

extern "C" int dctz_gpu_selftest_division(dctz_gpu_ctx *ctx, int datatype, double b, uint64_t count, uint32_t seed,
                                          uint64_t *mismatches) {
  TRY(check_common(ctx, datatype, 1.0));
  if (!mismatches) return fail(ctx, DCTZ_GPU_EINVAL, "selftest: NULL pointer");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  CU(cudaMemsetAsync(ctx->d_mismatch, 0, 8, st));
  if (datatype == DCTZ_GPU_DOUBLE) k_selftest_division<double><<<ctx->sm_count * 8, 256, 0, st>>>(b, count, seed, ctx->d_mismatch);
  else k_selftest_division<float><<<ctx->sm_count * 8, 256, 0, st>>>((float)b, count, seed, ctx->d_mismatch);
  ctx->launches++;
  CU(cudaGetLastError());
  unsigned long long m = 0;
  CU(cudaMemcpyAsync(&m, ctx->d_mismatch, 8, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  *mismatches = m;
  return DCTZ_GPU_OK;
}
