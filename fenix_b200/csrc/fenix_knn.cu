// fenix_knn.cu — C ABI of libfenix_knn.so (declared in include/fenix_knn.h).
//
// Host side of the B200 exact k-NN path: device shard ownership, pinned staging, kernel
// dispatch and the certificate / refinement tiers. Kernels live in exact_scan.cuh (fp64 CUDA-core
// scan, merges, row norms), tc_filter.cuh (tcgen05/TMEM filter kernels, prepass, finish + rerank) and direct_scan.cuh
// (the single-launch latency path for a handful of queries over a small shard).
#include <cuda.h>
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>

#include <dlfcn.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../../include/fenix_knn.h"
#include "exact_scan.cuh"
#include "direct_scan.cuh"
#include "tc_filter.cuh"
#include "range_search.cuh"
#include "kmeans.cuh"

#include <cub/device/device_segmented_sort.cuh>

// ----------------------------------------------------------------------------------------
// error plumbing
// ----------------------------------------------------------------------------------------
static thread_local std::string g_last_error;

static int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

#define FX_CUDA(expr)                                                                      \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess)                                                                 \
      return fail(_e == cudaErrorMemoryAllocation ? FX_ENOMEM : FX_ECUDA, "%s failed: %s (%s:%d)", \
                  #expr, cudaGetErrorString(_e), __FILE__, __LINE__);                      \
  } while (0)

#define FX_TRY(expr)              \
  do {                            \
    int _r = (expr);              \
    if (_r != FX_OK) return _r;   \
  } while (0)

// NVTX ranges (header-only NVTX 3; no-ops unless a profiler is attached): upload, shadow build, search, exchange.
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

// ----------------------------------------------------------------------------------------
// objects
// ----------------------------------------------------------------------------------------
struct DevBuf {  // grow-only device scratch
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes) {
    if (bytes <= cap) return FX_OK;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 4;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(FX_ENOMEM, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e)); }
    cap = want;
    return FX_OK;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct HostBuf {  // grow-only pinned staging
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes) {
    if (bytes <= cap) return FX_OK;
    if (p) cudaFreeHost(p);
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 4;
    cudaError_t e = cudaMallocHost(&p, want);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(FX_ENOMEM, "cudaMallocHost(%zu) failed: %s", want, cudaGetErrorString(e)); }
    cap = want;
    return FX_OK;
  }
  void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

struct fx_ctx {
  int device = 0;
  int sm_count = 0;
  int cc_major = 0, cc_minor = 0;
  cudaStream_t stream = nullptr;   // compute
  cudaStream_t upload = nullptr;   // H2D of corpus chunks
  cudaEvent_t ev_start = nullptr, ev_stop = nullptr, ev_k0 = nullptr, ev_k1 = nullptr;
  std::mutex mu;                   // one search at a time per device context
  cudaEvent_t ev_x0 = nullptr, ev_x1 = nullptr;   // exchange (all-gather + merge) of a sharded search
  DevBuf d_q, d_rows, d_dist, d_mask, d_partial, d_qlist, d_tc, d_ref, d_maskn, d_floor, d_xchg, d_hdr, d_tickets;
  DevBuf d_hits, d_hits2, d_col, d_rmeta, d_rbatch, d_cub;   // range search: hit keys (+ sorted copy), distance columns,
                                                              // per-query and per-batch arrays, CUB scratch
  HostBuf h_q, h_rows, h_dist, h_flags;
  unsigned int* d_ticket = nullptr;   // direct scan: "last CTA merges" counter (zero between launches)
  unsigned long long* h_done = nullptr;   // pinned: direct scan completion word [0] = sequence number, [1] = kernel ns
  unsigned long long direct_seq = 0;
  int* h_word = nullptr;           // pinned: [0] flagged-query count of the last main pass, [1..] gathered per-rank counts
  int64_t launches = 0;
  fx::TcState tc;                  // driver entry points / kernel attributes / tuning knobs of the TC path
  bool capturing = false;          // the search being enqueued is captured into a CUDA graph (events become external nodes)
  uint64_t knob_epoch = 0;         // bumped by fx_set_option: captured graphs bake the plan in
};
constexpr int H_WORDS = 64;

constexpr size_t RING_BYTES = size_t(32) << 20;

struct fx_corpus {
  fx_ctx* ctx = nullptr;
  int64_t cap = 0, n = 0, row_base = 0;
  int dim = 0, pitch = 0;
  float* X = nullptr;
  void* Xb = nullptr;              // bf16 shadow of X (+ three -|x|^2/2 columns) for the bf16 filter, tiled (tc_filter.cuh)
  void* Xn = nullptr;              // bf16 shadow of the normalised rows (cosine), built by the first cosine search
  void* X8 = nullptr;              // int8 shadow of the normalised rows (exact cosine at small k), built by the first search that takes it
  float2* x8_tile = nullptr;       // (S_t, E_t) of every tile of X8 (tc_filter.cuh, i8_scale)
  bool xn_failed = false;          // no memory for Xn: cosine keeps the plain shadow + multiplicative epilogue
  bool x8_failed = false;          // no memory for X8: cosine keeps the bf16 shadows
  bool xb_failed = false;          // no memory for Xb: the TF32 filter over the fp32 rows serves L2 / inner product
  int shadow_mode = -1;            // FENIX_BF16_SHADOW at finalize: -1 lazy (default), 0 never, 1 plain shadow built at finalize
  int pitch_b = 0;                 // elements per row of the bf16 QUERY matrix that goes with the shadows (ShadowGeom::pitch_q)
  float* hx = nullptr;
  float* rx = nullptr;
  unsigned int* max_n2_bits = nullptr;   // device: [0] bits of max |x|^2, [2..3] double: sum of |x| (16 bytes)
  float max_norm = 0.f;            // max |x| over the shard (host copy, set by finalize)
  float mean_norm = 0.f;           // mean |x| over the shard: max / mean = how far the norms spread
  bool finalized = false;
  void* ring[2] = {nullptr, nullptr};
  cudaEvent_t ring_ev[2] = {nullptr, nullptr};
  int ring_next = 0;
  fx_stats stats{};
  fx::TcCorpus tc;                 // tensor map of the shard for the TC path
  struct GraphEntry {              // a small search captured as one CUDA graph (H2D, kernels, D2H), replayed from its second call on
    int64_t n_q = 0; int metric = 0, k = 0, precision = 0;
    int state = 0;                 // 0 new, 2 seen once (the next identical call captures), 1 ready, -1 capture failed (never again)
    cudaGraphExec_t exec = nullptr;
    void* ptrs[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // buffers baked into the graph
    uint64_t knob_epoch = 0;
    int path = 0, variant = 0, launches = 0, operand = 0;
  };
  std::vector<GraphEntry> graphs;
  // inverted index for batched IVF searches (fx_corpus_set_cells): local rows grouped by cell
  int* d_inv = nullptr; long long* d_cell_off = nullptr;
  std::vector<long long> h_cell_off;
  int64_t n_inv = 0, n_cells = 0;
};

// variant of fx::tc_search (bit 3: resident query tiles) -> fx_stats
static void set_variant(fx_corpus* c, int variant) {
  c->stats.last_variant = variant & 7;
  c->stats.last_resident_queries = (variant >> 3) & 1;
}

static int bind(fx_ctx* ctx) {
  FX_CUDA(cudaSetDevice(ctx->device));
  return FX_OK;
}

// ----------------------------------------------------------------------------------------
// live-handle registry: a corpus handle is checked (and leased) before it is dereferenced, so a call that races with
// fx_corpus_destroy of the same shard fails with FX_EINVAL - or finishes first - instead of running on freed memory.
// fx_corpus_destroy retires the handle, then waits for the leases already out.
// ----------------------------------------------------------------------------------------
struct HandleState { int users = 0; bool doomed = false; };
static std::mutex g_reg_mu;
static std::condition_variable g_reg_cv;
static std::unordered_map<const fx_corpus*, HandleState> g_live;

struct Lease {
  const fx_corpus* c;
  bool ok = false;
  explicit Lease(const fx_corpus* c_) : c(c_) {
    if (!c) return;
    std::lock_guard<std::mutex> lock(g_reg_mu);
    auto it = g_live.find(c);
    if (it == g_live.end() || it->second.doomed) return;
    it->second.users++;
    ok = true;
  }
  ~Lease() {
    if (!ok) return;
    std::lock_guard<std::mutex> lock(g_reg_mu);
    auto it = g_live.find(c);
    if (it != g_live.end() && --it->second.users == 0 && it->second.doomed) g_reg_cv.notify_all();
  }
  Lease(const Lease&) = delete;
  Lease& operator=(const Lease&) = delete;
};
#define FX_LEASE(c, who)                                                                             \
  Lease _lease(c);                                                                                   \
  if (!_lease.ok) return fail(FX_EINVAL, "%s: %s", who, (c) ? "not a live corpus handle (destroyed?)" : "corpus is NULL")

// ----------------------------------------------------------------------------------------
// lifetime
// ----------------------------------------------------------------------------------------
extern "C" int fx_abi_version(void) { return FX_ABI_VERSION; }
extern "C" const char* fx_last_error(void) { return g_last_error.c_str(); }

extern "C" int fx_init(int device, fx_ctx** out) {
  if (!out) return fail(FX_EINVAL, "fx_init: out is NULL");
  *out = nullptr;
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev == 0) {
    cudaGetLastError();
    return fail(FX_ECUDA, "fx_init: no CUDA device visible (%s); libfenix_knn has no CPU fallback",
                e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
  }
  if (device < 0 || device >= n_dev) return fail(FX_EINVAL, "fx_init: device %d out of range [0,%d)", device, n_dev);
  fx_ctx* ctx = new (std::nothrow) fx_ctx();
  if (!ctx) return fail(FX_ENOMEM, "fx_init: out of host memory");
  ctx->device = device;
  cudaDeviceProp prop;
  if (cudaSetDevice(device) != cudaSuccess || cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
    delete ctx;
    return fail(FX_ECUDA, "fx_init: cannot bind device %d: %s", device, cudaGetErrorString(cudaGetLastError()));
  }
  ctx->sm_count = prop.multiProcessorCount;
  ctx->cc_major = prop.major; ctx->cc_minor = prop.minor;
  if (prop.major != 10) {
    delete ctx;
    return fail(FX_EUNSUP, "fx_init: device %d is sm_%d%d; this library is built for sm_100a (B200) only",
                device, prop.major, prop.minor);
  }
  FX_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  FX_CUDA(cudaStreamCreateWithFlags(&ctx->upload, cudaStreamNonBlocking));
  FX_CUDA(cudaEventCreate(&ctx->ev_start));
  FX_CUDA(cudaEventCreate(&ctx->ev_stop));
  FX_CUDA(cudaEventCreate(&ctx->ev_k0));
  FX_CUDA(cudaEventCreate(&ctx->ev_k1));
  FX_CUDA(cudaEventCreate(&ctx->ev_x0));
  FX_CUDA(cudaEventCreate(&ctx->ev_x1));
  FX_CUDA(cudaMallocHost(reinterpret_cast<void**>(&ctx->h_word), H_WORDS * sizeof(int)));
  std::memset(ctx->h_word, 0, H_WORDS * sizeof(int));
  FX_CUDA(cudaMallocHost(reinterpret_cast<void**>(&ctx->h_done), 64));
  std::memset(ctx->h_done, 0, 64);
  FX_CUDA(cudaFuncSetAttribute(fx::exact_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  FX_CUDA(cudaFuncSetAttribute(fx::merge_keys_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024));
  FX_CUDA(cudaFuncSetAttribute(fx::merge_pairs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024));
  FX_CUDA(cudaMalloc(reinterpret_cast<void**>(&ctx->d_ticket), 256));
  FX_CUDA(cudaMemset(ctx->d_ticket, 0, 256));
  {
    std::string err;
    if (!fx::tc_init(&ctx->tc, ctx->sm_count, &err)) {
      delete ctx;
      return fail(FX_ECUDA, "fx_init: %s", err.c_str());
    }
  }
  *out = ctx;
  return FX_OK;
}

extern "C" int fx_shutdown(fx_ctx* ctx) {
  if (!ctx) return fail(FX_EINVAL, "fx_shutdown: ctx is NULL");
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  cudaStreamSynchronize(ctx->upload);
  ctx->d_q.release(); ctx->d_rows.release(); ctx->d_dist.release(); ctx->d_mask.release();
  ctx->d_partial.release(); ctx->d_qlist.release(); ctx->d_tc.release(); ctx->d_ref.release(); ctx->d_maskn.release();
  ctx->d_floor.release(); ctx->d_xchg.release(); ctx->d_hdr.release(); ctx->d_tickets.release();
  ctx->d_hits.release(); ctx->d_hits2.release(); ctx->d_col.release(); ctx->d_rmeta.release(); ctx->d_rbatch.release(); ctx->d_cub.release();
  ctx->h_q.release(); ctx->h_rows.release(); ctx->h_dist.release(); ctx->h_flags.release();
  if (ctx->h_word) cudaFreeHost(ctx->h_word);
  if (ctx->d_ticket) cudaFree(ctx->d_ticket);
  if (ctx->h_done) cudaFreeHost(ctx->h_done);
  cudaEventDestroy(ctx->ev_start); cudaEventDestroy(ctx->ev_stop);
  cudaEventDestroy(ctx->ev_k0); cudaEventDestroy(ctx->ev_k1);
  cudaEventDestroy(ctx->ev_x0); cudaEventDestroy(ctx->ev_x1);
  cudaStreamDestroy(ctx->stream); cudaStreamDestroy(ctx->upload);
  delete ctx;
  return FX_OK;
}

extern "C" int fx_corpus_create(fx_ctx* ctx, int64_t capacity_rows, int32_t dim, int32_t dtype,
                                int64_t row_base, fx_corpus** out) {
  if (!ctx || !out) return fail(FX_EINVAL, "fx_corpus_create: NULL argument");
  *out = nullptr;
  if (capacity_rows < 0) return fail(FX_EINVAL, "fx_corpus_create: negative capacity %lld", (long long)capacity_rows);
  if (dim < 1) return fail(FX_EINVAL, "fx_corpus_create: dim must be >= 1 (got %d)", dim);
  if (dtype != FX_DTYPE_F32) return fail(FX_EUNSUP, "fx_corpus_create: only float32 rows are supported (dtype=%d)", dtype);
  if (capacity_rows > int64_t(0xfffffff0ll)) return fail(FX_EUNSUP, "fx_corpus_create: a shard holds at most 2^32-16 rows; shard the corpus");
  if (dim > 16384) return fail(FX_EUNSUP, "fx_corpus_create: dim %d exceeds 16384", dim);
  std::lock_guard<std::mutex> lock(ctx->mu);
  FX_TRY(bind(ctx));
  fx_corpus* c = new (std::nothrow) fx_corpus();
  if (!c) return fail(FX_ENOMEM, "fx_corpus_create: out of host memory");
  c->ctx = ctx; c->cap = capacity_rows; c->dim = dim; c->pitch = (dim + 3) & ~3; c->row_base = row_base;
  size_t rows_alloc = size_t(std::max<int64_t>(capacity_rows, 1));
  // the tensor-core tiles read whole 256-row boxes; TMA clips to the tensor bounds, no padding needed
  cudaError_t e = cudaMalloc(&c->X, rows_alloc * c->pitch * sizeof(float));
  // norm terms are fetched in whole 256-entry tiles (1 KB bulk copies) by the tensor-core kernel
  const size_t norm_alloc = ((rows_alloc + 255) / 256) * 256;
  if (e == cudaSuccess) e = cudaMalloc(&c->hx, norm_alloc * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&c->rx, norm_alloc * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&c->max_n2_bits, 16);
  if (e != cudaSuccess) {
    cudaGetLastError();
    if (c->X) cudaFree(c->X);
    if (c->hx) cudaFree(c->hx);
    if (c->rx) cudaFree(c->rx);
    delete c;
    return fail(FX_ENOMEM, "fx_corpus_create: cannot allocate %zu rows x %d floats on device %d: %s",
                rows_alloc, c ? ((dim + 3) & ~3) : 0, ctx->device, cudaGetErrorString(e));
  }
  if (c->pitch != c->dim) FX_CUDA(cudaMemsetAsync(c->X, 0, rows_alloc * c->pitch * sizeof(float), ctx->upload));
  FX_CUDA(cudaMemsetAsync(c->hx, 0, norm_alloc * sizeof(float), ctx->upload));
  FX_CUDA(cudaMemsetAsync(c->rx, 0, norm_alloc * sizeof(float), ctx->upload));
  c->stats.dim = dim; c->stats.pitch = c->pitch;
  c->stats.device_bytes = int64_t(rows_alloc * (c->pitch + 2) * sizeof(float));
  {
    std::lock_guard<std::mutex> reg(g_reg_mu);
    g_live[c] = HandleState{};
  }
  *out = c;
  return FX_OK;
}

extern "C" int fx_set_option(fx_ctx* ctx, const char* name, const char* value) {
  if (!ctx || !name) return fail(FX_EINVAL, "fx_set_option: NULL argument");
  std::lock_guard<std::mutex> lock(ctx->mu);
  if (!fx::tc_set_knob(&ctx->tc.knobs, name, value)) return fail(FX_EINVAL, "fx_set_option: unknown option '%s'", name);
  ctx->knob_epoch++;
  return FX_OK;
}

static int ensure_ring(fx_corpus* c) {
  for (int i = 0; i < 2; ++i) {
    if (!c->ring[i]) {
      FX_CUDA(cudaMallocHost(&c->ring[i], RING_BYTES));
      FX_CUDA(cudaEventCreateWithFlags(&c->ring_ev[i], cudaEventDisableTiming));
    }
  }
  return FX_OK;
}

static int append_impl(fx_corpus* c, const void* rows, int64_t n_rows, bool on_device) {
  FX_LEASE(c, "fx_corpus_append");
  NvtxRange nvtx("fenix:corpus_append");
  if (n_rows < 0) return fail(FX_EINVAL, "fx_corpus_append: negative row count");
  if (n_rows == 0) return FX_OK;
  if (!rows) return fail(FX_EINVAL, "fx_corpus_append: rows is NULL");
  fx_ctx* ctx = c->ctx;
  std::lock_guard<std::mutex> lock(ctx->mu);
  if (c->finalized) return fail(FX_ESTATE, "fx_corpus_append: shard is already finalized");
  if (c->n + n_rows > c->cap)
    return fail(FX_EINVAL, "fx_corpus_append: %lld rows would exceed capacity %lld (have %lld)",
                (long long)n_rows, (long long)c->cap, (long long)c->n);
  FX_TRY(bind(ctx));
  const size_t src_pitch = size_t(c->dim) * sizeof(float), dst_pitch = size_t(c->pitch) * sizeof(float);
  float* dst = c->X + size_t(c->n) * c->pitch;
  if (on_device) {
    FX_CUDA(cudaMemcpy2DAsync(dst, dst_pitch, rows, src_pitch, src_pitch, size_t(n_rows), cudaMemcpyDeviceToDevice, ctx->upload));
    FX_CUDA(cudaStreamSynchronize(ctx->upload));  // caller may free its buffer on return
  } else {
    // pageable Arrow buffer -> pinned ring (CPU copy) -> async H2D, double buffered
    FX_TRY(ensure_ring(c));
    const int64_t rows_per_slot = std::max<int64_t>(1, int64_t(RING_BYTES / src_pitch));
    const char* src = static_cast<const char*>(rows);
    for (int64_t done = 0; done < n_rows;) {
      int64_t take = std::min(rows_per_slot, n_rows - done);
      int slot = c->ring_next;
      c->ring_next ^= 1;
      FX_CUDA(cudaEventSynchronize(c->ring_ev[slot]));
      std::memcpy(c->ring[slot], src + size_t(done) * src_pitch, size_t(take) * src_pitch);
      FX_CUDA(cudaMemcpy2DAsync(dst + size_t(done) * c->pitch, dst_pitch, c->ring[slot], src_pitch, src_pitch,
                                size_t(take), cudaMemcpyHostToDevice, ctx->upload));
      FX_CUDA(cudaEventRecord(c->ring_ev[slot], ctx->upload));
      done += take;
    }
  }
  c->n += n_rows;
  return FX_OK;
}

extern "C" int fx_corpus_append(fx_corpus* c, const void* host_rows, int64_t n_rows) {
  return append_impl(c, host_rows, n_rows, false);
}
extern "C" int fx_corpus_append_device(fx_corpus* c, const void* device_rows, int64_t n_rows) {
  return append_impl(c, device_rows, n_rows, true);
}

static bool ensure_plain_shadow(fx_corpus* c);

extern "C" int fx_corpus_finalize(fx_corpus* c) {
  FX_LEASE(c, "fx_corpus_finalize");
  NvtxRange nvtx("fenix:corpus_finalize");
  fx_ctx* ctx = c->ctx;
  std::lock_guard<std::mutex> lock(ctx->mu);
  if (c->finalized) return FX_OK;
  FX_TRY(bind(ctx));
  FX_CUDA(cudaStreamSynchronize(ctx->upload));
  FX_CUDA(cudaMemsetAsync(c->max_n2_bits, 0, 16, ctx->stream));
  if (c->n > 0) {
    int blocks = int(std::min<int64_t>((c->n + 7) / 8, int64_t(ctx->sm_count) * 8));
    fx::row_norms_kernel<<<blocks, 256, 0, ctx->stream>>>(c->X, c->n, c->pitch, c->hx, c->rx, c->max_n2_bits,
                                                          reinterpret_cast<double*>(c->max_n2_bits + 2));
    FX_CUDA(cudaGetLastError());
    ctx->launches++; c->stats.kernel_launches++;
  }
  unsigned int words[4] = {0, 0, 0, 0};
  FX_CUDA(cudaMemcpyAsync(words, c->max_n2_bits, sizeof words, cudaMemcpyDeviceToHost, ctx->stream));
  FX_CUDA(cudaStreamSynchronize(ctx->stream));
  float n2; std::memcpy(&n2, &words[0], sizeof n2);
  double nsum; std::memcpy(&nsum, &words[2], sizeof nsum);
  c->max_norm = std::sqrt(n2) * (1.0f + 1e-6f);
  c->mean_norm = c->n > 0 ? float(nsum / double(c->n)) : 0.f;
  for (int i = 0; i < 2; ++i) {
    if (c->ring[i]) { cudaFreeHost(c->ring[i]); c->ring[i] = nullptr; cudaEventDestroy(c->ring_ev[i]); c->ring_ev[i] = nullptr; }
  }
  // bf16 shadows (tiled for streaming, see tc_filter.cuh): the exact (fp32) mode filters with 2x-rate bf16 MMAs and half
  // the operand bytes - measured gains: C3 (D=768) 95 -> 49 ms, one C4 shard (D=96) 49 -> 39 ms. Each of the two shadows
  // costs +50 % HBM per shard and only ONE is read by any given metric (plain + augmented columns: L2 / inner product;
  // normalised rows: cosine), so each is built by the first search that streams it (ensure_plain_shadow /
  // ensure_norm_shadow) - a table searched with one metric holds fp32 rows + one shadow. FENIX_BF16_SHADOW=0: never
  // build one (TF32 filter over the fp32 rows); =1: build the plain shadow here, at finalize.
  {
    const fx::ShadowGeom g = fx::shadow_geom(c->dim);
    c->pitch_b = g.pitch_q;
    const char* e = std::getenv("FENIX_BF16_SHADOW");
    c->shadow_mode = e ? (std::atoi(e) != 0 ? 1 : 0) : -1;
  }
  {
    std::string err;
    const fx::ShadowGeom g = fx::shadow_geom(c->dim);
    if (!fx::tc_bind_corpus(&ctx->tc, &c->tc, c->X, c->n, c->dim, c->pitch, nullptr, g.n_kb_data + (g.aug_separate ? 1 : 0), &err))
      return fail(FX_ECUDA, "fx_corpus_finalize: %s", err.c_str());
  }
  c->stats.n_rows = c->n;
  c->finalized = true;
  if (c->shadow_mode == 1) ensure_plain_shadow(c);
  return FX_OK;
}

extern "C" int fx_corpus_destroy(fx_corpus* c) {
  if (!c) return fail(FX_EINVAL, "fx_corpus_destroy: corpus is NULL");
  {
    // retire the handle (new calls on it fail), then wait for the calls already inside the library
    std::unique_lock<std::mutex> reg(g_reg_mu);
    auto it = g_live.find(c);
    if (it == g_live.end() || it->second.doomed) return fail(FX_EINVAL, "fx_corpus_destroy: not a live corpus handle (destroyed twice?)");
    it->second.doomed = true;
    g_reg_cv.wait(reg, [&] { return g_live[c].users == 0; });
    g_live.erase(c);
  }
  fx_ctx* ctx = c->ctx;
  std::lock_guard<std::mutex> lock(ctx->mu);
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->upload);
  cudaStreamSynchronize(ctx->stream);
  for (int i = 0; i < 2; ++i) {
    if (c->ring[i]) { cudaFreeHost(c->ring[i]); cudaEventDestroy(c->ring_ev[i]); }
  }
  for (auto& g : c->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
  if (c->X) cudaFree(c->X);
  if (c->Xb) cudaFree(c->Xb);
  if (c->Xn) cudaFree(c->Xn);
  if (c->X8) cudaFree(c->X8);
  if (c->x8_tile) cudaFree(c->x8_tile);
  if (c->hx) cudaFree(c->hx);
  if (c->rx) cudaFree(c->rx);
  if (c->max_n2_bits) cudaFree(c->max_n2_bits);
  if (c->d_inv) cudaFree(c->d_inv);
  if (c->d_cell_off) cudaFree(c->d_cell_off);
  delete c;
  return FX_OK;
}

extern "C" int fx_get_stats(fx_corpus* c, fx_stats* out) {
  if (!out) return fail(FX_EINVAL, "fx_get_stats: NULL argument");
  FX_LEASE(c, "fx_get_stats");
  std::lock_guard<std::mutex> lock(c->ctx->mu);
  c->stats.n_rows = c->n;
  *out = c->stats;
  return FX_OK;
}

// ----------------------------------------------------------------------------------------
// exact scan dispatch
// ----------------------------------------------------------------------------------------
static int next_pow2(int v) { int p = 1; while (p < v) p <<= 1; return p; }
constexpr int SCAN_K_PASS = 2048;   // neighbours one pass of the scan selects (shared-memory candidate buffers)

// One pass of the fp64 scan for `n_list` queries (all of them when d_qlist == null): the k smallest (distance, row)
// keys ABOVE each query's floor key (d_floor, optional) land in columns [out_off, out_off + k) of the listed
// queries' output rows (out_stride entries per query); the last key becomes the next floor (floor_out, optional).
static int run_scan_pass(fx_corpus* c, const float* d_q, int n_q, const int* d_qlist, int n_list, int metric, int k,
                         const uint8_t* d_mask, int64_t* d_out_rows, float* d_out_dist, int out_stride, int out_off,
                         uint64_t* d_floor) {
  fx_ctx* ctx = c->ctx;
  if (n_list == 0) return FX_OK;
  const int buf = next_pow2(k + fx::SCAN_THREADS);
  const size_t per_q = size_t(c->pitch) * 8 + 8 + 8 + 8 + size_t(buf) * 8 + 4;
  const size_t smem_limit = 200 * 1024;
  int qb = int(std::min<size_t>(fx::SCAN_MAX_QB, smem_limit / per_q));
  if (qb < 1) return fail(FX_EUNSUP, "exact scan: dim %d with k %d needs %zu B of shared memory per query", c->dim, k, per_q);
  qb = std::min(qb, n_list);
  const int groups = (n_list + qb - 1) / qb;
  const int64_t tiles = std::max<int64_t>(1, (c->n + fx::SCAN_THREADS - 1) / fx::SCAN_THREADS);
  int W = int(std::min<int64_t>(tiles, std::max<int64_t>(1, (2 * int64_t(ctx->sm_count) + groups - 1) / groups)));
  W = std::max(1, std::min(W, 8192 / std::max(k, 1)));
  if (groups > 65535) {
    // grid.y limit: process in slabs of 65535 groups
    int done = 0;
    while (done < n_list) {
      int take = std::min(n_list - done, 65535 * qb);
      if (d_qlist) {
        FX_TRY(run_scan_pass(c, d_q, n_q, d_qlist + done, take, metric, k, d_mask, d_out_rows, d_out_dist, out_stride, out_off,
                             d_floor ? d_floor + done : nullptr));
      } else {
        // build an explicit list for the slab
        std::vector<int> idx(take);
        for (int i = 0; i < take; ++i) idx[i] = done + i;
        DevBuf tmp;
        FX_TRY(tmp.ensure(size_t(take) * sizeof(int)));
        FX_CUDA(cudaMemcpyAsync(tmp.p, idx.data(), size_t(take) * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        int r = run_scan_pass(c, d_q, n_q, static_cast<int*>(tmp.p), take, metric, k, d_mask, d_out_rows, d_out_dist, out_stride,
                              out_off, d_floor ? d_floor + done : nullptr);
        cudaStreamSynchronize(ctx->stream);
        tmp.release();
        FX_TRY(r);
      }
      done += take;
    }
    return FX_OK;
  }
  FX_TRY(ctx->d_partial.ensure(size_t(n_list) * W * k * sizeof(uint64_t)));
  fx::ScanParams p{};
  p.X = c->X; p.n_rows = c->n; p.pitch = c->pitch; p.dim = c->dim; p.Q = d_q; p.n_q = n_q;
  p.metric = metric; p.mask = d_mask; p.q_list = d_qlist; p.n_list = n_list; p.k = k; p.buf = buf; p.qb = qb;
  p.floor = d_floor;
  p.partial = static_cast<uint64_t*>(ctx->d_partial.p); p.dist_out = nullptr;
  const size_t smem = per_q * qb + 16;
  fx::exact_scan_kernel<<<dim3(W, groups), fx::SCAN_THREADS, smem, ctx->stream>>>(p);
  FX_CUDA(cudaGetLastError());
  const int n_sort = next_pow2(std::max(W * k, 2));
  fx::merge_keys_kernel<<<n_list, 256, size_t(n_sort) * 8, ctx->stream>>>(
      p.partial, W, k, n_sort, d_qlist, c->row_base, d_out_rows, d_out_dist, out_stride, out_off, d_floor);
  FX_CUDA(cudaGetLastError());
  ctx->launches += 2; c->stats.kernel_launches += 2;
  return FX_OK;
}

// The fp64 scan for any k: passes of at most SCAN_K_PASS neighbours, each admitting only keys above the last
// (distance, row) key of the one before ((distance, row) keys are unique, so the passes partition the order).
static int run_exact_scan(fx_corpus* c, const float* d_q, int n_q, const int* d_qlist, int n_list,
                          int metric, int k, const uint8_t* d_mask, int64_t* d_out_rows, float* d_out_dist) {
  fx_ctx* ctx = c->ctx;
  if (k <= SCAN_K_PASS) return run_scan_pass(c, d_q, n_q, d_qlist, n_list, metric, k, d_mask, d_out_rows, d_out_dist, k, 0, nullptr);
  FX_TRY(ctx->d_floor.ensure(size_t(n_list) * sizeof(uint64_t)));
  FX_CUDA(cudaMemsetAsync(ctx->d_floor.p, 0, size_t(n_list) * sizeof(uint64_t), ctx->stream));
  for (int done = 0; done < k; done += SCAN_K_PASS) {
    const int kp = std::min(SCAN_K_PASS, k - done);
    FX_TRY(run_scan_pass(c, d_q, n_q, d_qlist, n_list, metric, kp, d_mask, d_out_rows, d_out_dist, k, done,
                         static_cast<uint64_t*>(ctx->d_floor.p)));
  }
  return FX_OK;
}

// ----------------------------------------------------------------------------------------
// search
// ----------------------------------------------------------------------------------------
// The normalised bf16 shadow (cosine scores straight out of the MMA) is built by the first cosine search that
// can use it; when HBM is short the search keeps the plain shadow and the multiplicative epilogue.
static bool shadow_allowed(const fx_corpus* c) { return c->shadow_mode != 0 && c->dim >= 16 && c->n >= 4096 && c->tc.ok; }

// The plain bf16 shadow (+ four augmented columns per row): operand of the L2 / inner-product filter, and of cosine
// when there is no room for the normalised shadow.
static bool ensure_plain_shadow(fx_corpus* c) {
  fx_ctx* ctx = c->ctx;
  if (c->tc.ok_b) return true;
  NvtxRange nvtx("fenix:build_plain_shadow");
  if (c->xb_failed || !shadow_allowed(c)) return false;
  const fx::ShadowGeom g = fx::shadow_geom(c->dim);
  const int n_kb = g.n_kb_data, aug_blocks = g.aug_separate ? 1 : 0;
  const int64_t n_tiles = (c->n + fx::TC_BN - 1) / fx::TC_BN;
  const size_t shadow_bytes = size_t(n_tiles) * (n_kb + aug_blocks) * fx::TC_BN * 64 * 2;
  size_t free_b = 0, total_b = 0;
  const bool forced = c->shadow_mode == 1;
  if ((!forced && (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess || free_b < shadow_bytes + (size_t(4) << 30))) ||
      cudaMalloc(&c->Xb, shadow_bytes) != cudaSuccess) {
    cudaGetLastError(); c->Xb = nullptr; c->xb_failed = true;   // not fatal: the TF32 filter needs no shadow
    return false;
  }
  const int64_t total = int64_t(shadow_bytes / 4);
  int blocks = int(std::min<int64_t>((total + 255) / 256, int64_t(ctx->sm_count) * 16));
  // -|x|^2/2 is stored shrunk by the accumulation-rounding allowance (10 % margin for the rounding of the product itself)
  const float h_scale = float(1.0 - 1.1 * fx::tc_c_add(c->dim, true));
  fx::to_bf16_tiled_kernel<<<blocks, 256, 0, ctx->stream>>>(c->X, c->n, c->pitch, c->dim, c->hx, c->rx, 0,
                                                            static_cast<__nv_bfloat16*>(c->Xb), n_kb, n_tiles, g.aug_col, aug_blocks, h_scale);
  std::string err;
  if (cudaGetLastError() != cudaSuccess || cudaStreamSynchronize(ctx->stream) != cudaSuccess ||
      !fx::tc_bind_shadow(&ctx->tc, &c->tc.map_xb, &c->tc.map_xb_h, c->Xb, c->n, n_kb + aug_blocks, &err)) {
    cudaGetLastError(); cudaFree(c->Xb); c->Xb = nullptr; c->xb_failed = true;
    return false;
  }
  ctx->launches++; c->stats.kernel_launches++;
  c->stats.device_bytes += int64_t(shadow_bytes);
  c->tc.ok_b = true;
  return true;
}

static bool ensure_norm_shadow(fx_corpus* c) {
  fx_ctx* ctx = c->ctx;
  if (c->tc.ok_n) return true;
  if (c->xn_failed || !shadow_allowed(c) || ctx->tc.knobs.no_norm_shadow) return false;
  const int n_kb = fx::shadow_geom(c->dim).n_kb_data;
  const int64_t n_tiles = (c->n + fx::TC_BN - 1) / fx::TC_BN;
  const size_t shadow_bytes = size_t(n_tiles) * n_kb * fx::TC_BN * 64 * 2;
  size_t free_b = 0, total_b = 0;
  if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess || free_b < shadow_bytes + (size_t(4) << 30) ||
      cudaMalloc(&c->Xn, shadow_bytes) != cudaSuccess) {
    cudaGetLastError(); c->Xn = nullptr; c->xn_failed = true;
    return false;
  }
  const int64_t total = int64_t(shadow_bytes / 4);
  int blocks = int(std::min<int64_t>((total + 255) / 256, int64_t(ctx->sm_count) * 16));
  fx::to_bf16_tiled_kernel<<<blocks, 256, 0, ctx->stream>>>(c->X, c->n, c->pitch, c->dim, c->hx, c->rx, 1,
                                                            static_cast<__nv_bfloat16*>(c->Xn), n_kb, n_tiles, 0, 0, 1.f);
  std::string err;
  if (cudaGetLastError() != cudaSuccess || cudaStreamSynchronize(ctx->stream) != cudaSuccess ||
      !fx::tc_bind_shadow(&ctx->tc, &c->tc.map_xn, &c->tc.map_xn_h, c->Xn, c->n, n_kb, &err)) {
    cudaGetLastError(); cudaFree(c->Xn); c->Xn = nullptr; c->xn_failed = true;
    return false;
  }
  ctx->launches++; c->stats.kernel_launches++;
  c->stats.device_bytes += int64_t(shadow_bytes);
  c->tc.ok_n = true;
  return true;
}

// The int8 normalised shadow (kind 2: 128 int8 columns per k-block, a (S_t, E_t) pair per tile): operand of exact cosine
// searches at small k over rows wider than the resident-query kernel's (int8_wanted). Half the bytes of the bf16
// normalised shadow and twice its tensor rate; its scores are certified upper bounds with a looser error than bf16's,
// so K' grows (TC_KP_I8) and large k keeps the bf16 shadow. FENIX_BF16_SHADOW=0 and FENIX_NO_NORM_SHADOW stop it too.
static bool ensure_i8_shadow(fx_corpus* c) {
  fx_ctx* ctx = c->ctx;
  if (c->tc.ok_8) return true;
  if (c->x8_failed || !shadow_allowed(c) || ctx->tc.knobs.no_norm_shadow) return false;
  NvtxRange nvtx("fenix:build_int8_shadow");
  const int n_kb = fx::i8_n_kb(c->dim);
  const int64_t n_tiles = (c->n + fx::TC_BN - 1) / fx::TC_BN;
  const size_t shadow_bytes = size_t(n_tiles) * n_kb * fx::TC_BN * fx::I8_KB, tile_bytes = size_t(n_tiles) * sizeof(float2);
  size_t free_b = 0, total_b = 0;
  if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess || free_b < shadow_bytes + tile_bytes + (size_t(4) << 30) ||
      cudaMalloc(&c->X8, shadow_bytes) != cudaSuccess || cudaMalloc(&c->x8_tile, tile_bytes) != cudaSuccess) {
    cudaGetLastError();
    if (c->X8) cudaFree(c->X8);
    c->X8 = nullptr; c->x8_tile = nullptr; c->x8_failed = true;
    return false;
  }
  const int blocks = int(std::min<int64_t>(n_tiles, int64_t(ctx->sm_count) * 8));
  fx::to_i8_tiled_kernel<<<blocks, 256, 0, ctx->stream>>>(c->X, c->n, c->pitch, c->dim, n_kb, n_tiles,
                                                          static_cast<int8_t*>(c->X8), c->x8_tile);
  std::string err;
  if (cudaGetLastError() != cudaSuccess || cudaStreamSynchronize(ctx->stream) != cudaSuccess ||
      !fx::tc_bind_shadow(&ctx->tc, &c->tc.map_x8, &c->tc.map_x8_h, c->X8, c->n, n_kb, &err, 1)) {
    cudaGetLastError(); cudaFree(c->X8); cudaFree(c->x8_tile); c->X8 = nullptr; c->x8_tile = nullptr; c->x8_failed = true;
    return false;
  }
  ctx->launches++; c->stats.kernel_launches++;
  c->stats.device_bytes += int64_t(shadow_bytes + tile_bytes);
  c->tc.ok_8 = true;
  return true;
}

// Exact cosine searches the int8 filter takes (FENIX_INT8 -1): rows wider than 192 columns - narrower ones take the
// resident-query kernel, which its epilogue binds - and k <= 16, where K' = TC_KP_I8 covers the rows the int8 bound lets
// past the k-th neighbour (k = 32 would need ~700).
static bool int8_wanted(const fx_corpus* c, int metric, int k, int precision) {
  const int knob = c->ctx->tc.knobs.int8;
  if (metric != 1 || precision != FX_PREC_FP32 || knob == 0 || c->ctx->tc.knobs.fp32_filter_tf32) return false;
  return knob > 0 || (c->dim > 192 && k <= 16);
}

// Operand kind, shadow and epilogue form of one filter launch (see TcSearch). With a row mask the per-row
// epilogue term carries the mask: masked rows get -inf (additive forms) or NaN (multiplicative form), which can
// never pass the threshold test.
static int configure_filter(fx_corpus* c, int metric, int kind, const uint8_t* d_mask, fx::TcSearch* s) {
  fx_ctx* ctx = c->ctx;
  s->kind = kind; s->pitch_b = c->pitch_b; s->shadow = 0; s->aug = 0; s->epi = metric;
  s->hx = c->hx; s->rx = c->rx; s->i8_tile = c->x8_tile;
  if (kind == 2) {   // cosine over the int8 normalised shadow: upper bounds straight out of the MMA and the tile constants
    s->epi = 2; s->pitch_b = fx::I8_KB * fx::i8_n_kb(c->dim);
  } else if (kind == 1) {
    if (metric == 0) { s->aug = 1; s->epi = 2; }                       // -|x|^2/2 and the row's error weight ride in the shadow's extra columns
    else if (metric == 1) { if (ensure_norm_shadow(c)) { s->shadow = 1; s->epi = 2; } else ensure_plain_shadow(c); }
    else if (c->max_norm > 2.0f * c->mean_norm) s->aug = 2;           // inner product over rows whose norms spread:
                                                                       // per-row error weights instead of c |q| max|x| for every row
    s->c_pair = s->aug != 0 ? fx::tc_c_pair(c->dim, s->aug) : 0.0;
  }
  if (d_mask) {
    const int64_t n_alloc = ((c->n + 255) / 256) * 256;
    FX_TRY(ctx->d_maskn.ensure(size_t(n_alloc) * sizeof(float)));
    float* mn = static_cast<float*>(ctx->d_maskn.p);
    // mode 0: hx or -inf (added), 1: rx or NaN (multiplied), 2: 0 or -inf (added), 3: int8 filter's integer term
    const int mode = kind == 2 ? 3 : (s->epi == 2 ? 2 : s->epi);
    fx::masked_norms_kernel<<<int(std::min<int64_t>((n_alloc + 255) / 256, int64_t(ctx->sm_count) * 8)), 256, 0, ctx->stream>>>(
        d_mask, mode == 1 ? c->rx : c->hx, c->n, n_alloc, mode, mn);
    FX_CUDA(cudaGetLastError());
    ctx->launches++; c->stats.kernel_launches++;
    s->hx = mn; s->rx = mn;
    if (s->epi == 2) s->epi = 0;
  }
  return FX_OK;
}

static int check_search_args(fx_corpus* c, const void* q, int64_t n_q, int metric, int k, int precision,
                             const void* out_rows, const void* out_dist, bool outs_required = true) {
  if (!c->finalized) return fail(FX_ESTATE, "fx_search: corpus is not finalized");
  if (n_q < 0) return fail(FX_EINVAL, "fx_search: negative query count");
  if (n_q > 0 && (!q || (outs_required && (!out_rows || !out_dist)))) return fail(FX_EINVAL, "fx_search: NULL buffer");
  if ((out_rows == nullptr) != (out_dist == nullptr)) return fail(FX_EINVAL, "fx_search: out_rows and out_dist must both be given, or neither");
  if (n_q > int64_t(1) << 24) return fail(FX_EUNSUP, "fx_search: at most 2^24 queries per call");
  if (metric < 0 || metric > 2) return fail(FX_EINVAL, "fx_search: unknown metric %d", metric);
  if (k < 1) return fail(FX_EINVAL, "fx_search: k must be >= 1 (got %d)", k);
  if (n_q * int64_t(k) > (int64_t(1) << 33)) return fail(FX_EUNSUP, "fx_search: n_q * k = %lld results exceed 2^33", (long long)(n_q * int64_t(k)));
  if (precision != FX_PREC_FP32 && precision != FX_PREC_TF32 && precision != FX_PREC_BF16 && precision != FX_PREC_EXACT_SCAN)
    return fail(FX_EINVAL, "fx_search: unknown precision mode %d", precision);
  return FX_OK;
}

// A search runs in two phases so that callers can queue whatever follows (result copies, the all-gather and merge of
// a sharded search) behind the kernels WITHOUT a host synchronisation in between:
//   search_enqueue  launches prep / prepass / filter / finish (or the scan) on the context's stream and queues the copy
//                   of the "flagged queries" counter into pinned memory;
//   search_settle   after the caller's ONE synchronisation: nothing to do when no certificate failed (the common
//                   case); otherwise the re-run / refinement / scan tiers repair the flagged queries' results in place
//                   and the caller repeats its copies.
// The single-launch direct scan (direct_scan.cuh) takes exact searches of a handful of queries over a shard small enough
// that reading its fp32 rows once beats the fixed cost of the tensor-core pipeline (FENIX_DIRECT, FENIX_DIRECT_MAX_MB).
static fx::DirectPlan direct_plan_for(const fx_corpus* c, int64_t n_q, int k, int precision) {
  const fx::TcKnobs& kn = c->ctx->tc.knobs;
  if (kn.direct == 0 || precision != FX_PREC_FP32) return fx::DirectPlan{};
  if (double(c->n) * c->pitch * 4.0 > double(kn.direct_mb) * 1048576.0) return fx::DirectPlan{};
  return fx::direct_plan(c->n, c->pitch, n_q, k, c->ctx->sm_count);
}

struct SearchRun {
  bool tc = false;            // the tensor-core path ran (flags are meaningful)
  int path = 0;               // 0 exact scan, 1 tensor-core TF32 filter, 2 tensor-core shadow filter (bf16 or int8), 3 direct scan (one launch)
  int operand = 0;            // operand kind of the filter: 0 fp32 / TF32, 1 bf16, 2 int8
  fx::TcSearch s{};
  fx::TcLaunch L{};
  const float* d_q = nullptr; int64_t n_q = 0; int metric = 0, k = 0;
  const uint8_t* d_mask = nullptr; int64_t* d_out_rows = nullptr; float* d_out_dist = nullptr;
  const float* inline_q = nullptr;   // set by the caller: HOST queries small enough to ride in the direct scan's kernel parameters
  bool spin = false;                 // set by the caller: results go to mapped host memory and the host spins on the kernel's completion word
                                     // (no events are recorded around the launch)
};

static int search_enqueue(fx_corpus* c, const float* d_q, int64_t n_q, int metric, int k, int precision,
                          const uint8_t* d_mask, int64_t* d_out_rows, float* d_out_dist, SearchRun* run) {
  fx_ctx* ctx = c->ctx;
  run->tc = false; run->path = 0; run->operand = 0; run->d_q = d_q; run->n_q = n_q; run->metric = metric; run->k = k;
  run->d_mask = d_mask; run->d_out_rows = d_out_rows; run->d_out_dist = d_out_dist;
  ctx->h_word[0] = 0;
  const unsigned ev_flags = ctx->capturing ? cudaEventRecordExternal : cudaEventRecordDefault;
  const fx::DirectPlan dpl = direct_plan_for(c, n_q, k, precision);
  const bool spin = run->spin && dpl.ok && c->n > 0;
  if (!spin) FX_CUDA(cudaEventRecordWithFlags(ctx->ev_start, ctx->stream, ev_flags));
  const bool want_tc = !dpl.ok && precision != FX_PREC_EXACT_SCAN &&
                       fx::tc_supported(&ctx->tc, &c->tc, c->n, c->dim, k, int(n_q));
  if (c->n == 0) {
    // empty shard: all pads
    fx::fill_pad_kernel<<<int(std::min<int64_t>((n_q * k + 255) / 256, 65535)), 256, 0, ctx->stream>>>(d_out_rows, d_out_dist, n_q * k);
    FX_CUDA(cudaGetLastError());
    ctx->launches++; c->stats.kernel_launches++;
    FX_CUDA(cudaEventRecordWithFlags(ctx->ev_k0, ctx->stream, ev_flags));
    FX_CUDA(cudaEventRecordWithFlags(ctx->ev_k1, ctx->stream, ev_flags));
  } else if (dpl.ok) {
    // one kernel per four queries: fp64 distances of every (live) row, per-CTA top-k, join by the last CTA. d_out_* may be
    // mapped pinned host memory (fx_search passes its staging buffers and, for small query blocks, the queries by value:
    // no copies)
    FX_TRY(ctx->d_partial.ensure(dpl.partial_bytes));
    if (ctx->tc.knobs.debug_direct) {
      FX_TRY(ctx->h_flags.ensure(size_t(512) * 8));
      std::memset(ctx->h_flags.p, 0, 512 * 8);
    }
    for (int64_t q0 = 0; q0 < n_q; q0 += fx::DS_LAUNCH_Q) {
      const int64_t nq_l = std::min<int64_t>(fx::DS_LAUNCH_Q, n_q - q0);
      const fx::DirectPlan pl = fx::direct_plan(c->n, c->pitch, nq_l, k, ctx->sm_count);
      fx::DirectParams p{};
      p.X = c->X; p.n_rows = c->n; p.pitch = c->pitch; p.dim = c->dim; p.row_base = c->row_base;
      p.Q = d_q + q0 * c->dim; p.n_q = int(nq_l); p.metric = metric; p.k = k; p.mask = d_mask;
      if (run->inline_q != nullptr) { p.Q = nullptr; std::memcpy(p.q_inline, run->inline_q + q0 * c->dim, size_t(nq_l) * c->dim * sizeof(float)); }
      p.partial = static_cast<uint64_t*>(ctx->d_partial.p); p.ticket = ctx->d_ticket; p.cap_steps = pl.cap_steps;
      p.out_rows = d_out_rows + q0 * k; p.out_dist = d_out_dist + q0 * k;
      const bool last = q0 + fx::DS_LAUNCH_Q >= n_q;
      // (launches of one stream complete in order: the host waits for the last one's word; the first one leaves its time in [3])
      if (spin) {
        if (q0 == 0) ctx->h_done[3] = 0;
        p.done = last ? ctx->h_done : ctx->h_done + 2;
        p.seq = last ? ++ctx->direct_seq : 0;
      }
      if (ctx->tc.knobs.debug_direct && last) p.dbg = static_cast<unsigned long long*>(ctx->h_flags.p);
      FX_CUDA(fx::direct_launch(pl, p, ctx->stream));
      ctx->launches++; c->stats.kernel_launches++;
    }
    run->path = 3;
  } else if (want_tc) {
    fx::TcSearch& s = run->s;
    s = fx::TcSearch{};
    s.X = c->X; s.hx = c->hx; s.rx = c->rx; s.n_rows = c->n; s.dim = c->dim; s.pitch = c->pitch;
    s.row_base = c->row_base; s.max_norm = c->max_norm; s.Q = d_q; s.n_q = int(n_q); s.metric = metric; s.k = k;
    s.certify = precision == FX_PREC_FP32; s.out_rows = d_out_rows; s.out_dist = d_out_dist;
    s.stream = ctx->stream; s.ev_k0 = ctx->ev_k0; s.ev_k1 = ctx->ev_k1; s.ev_flags = ev_flags; s.dbg = nullptr; s.tau_fixed = nullptr;
    // operand kind of the filter: exact mode takes the int8 normalised shadow for cosine at small k (int8_wanted), else the
    // bf16 shadow when the shard has one (the shadow a search streams is built here, by its first search: normalised rows
    // for cosine, else the plain one)
    const bool have_i8 = int8_wanted(c, metric, k, precision) && ensure_i8_shadow(c);
    const bool want_bf16 = precision == FX_PREC_BF16 || (precision == FX_PREC_FP32 && !ctx->tc.knobs.fp32_filter_tf32);
    const bool have_shadow = !have_i8 && want_bf16 && ((metric == 1 && ensure_norm_shadow(c)) || ensure_plain_shadow(c));
    const int kind = have_i8 ? 2 : (have_shadow ? 1 : 0);
    if (precision == FX_PREC_BF16 && !have_shadow)
      return fail(FX_ESTATE, "fx_search: FX_PREC_BF16 needs a bf16 shadow (none could be built: FENIX_BF16_SHADOW=0, a tiny shard, or no HBM left)");
    FX_TRY(configure_filter(c, metric, kind, d_mask, &s));
    run->L = fx::tc_prepare(&ctx->tc, s);
    FX_TRY(ctx->d_tc.ensure(run->L.scratch_bytes));
    std::string err;
    int launched = 0, variant = 0;
    if (!fx::tc_search(&ctx->tc, &c->tc, s, run->L, ctx->d_tc.p, &launched, &err, &variant)) return fail(FX_ECUDA, "fx_search: %s", err.c_str());
    run->tc = true; run->path = kind == 0 ? 1 : 2; run->operand = kind;
    set_variant(c, variant);
    ctx->launches += launched; c->stats.kernel_launches += launched;
    if (s.certify) FX_CUDA(cudaMemcpyAsync(ctx->h_word, fx::tc_flag_count(ctx->d_tc.p), sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  } else {
    FX_CUDA(cudaEventRecordWithFlags(ctx->ev_k0, ctx->stream, ev_flags));
    FX_TRY(run_exact_scan(c, d_q, int(n_q), nullptr, int(n_q), metric, k, d_mask, d_out_rows, d_out_dist));
    FX_CUDA(cudaEventRecordWithFlags(ctx->ev_k1, ctx->stream, ev_flags));
  }
  if (!spin) FX_CUDA(cudaEventRecordWithFlags(ctx->ev_stop, ctx->stream, ev_flags));
  return FX_OK;
}

// Precondition: the stream has been synchronised since search_enqueue. *changed: results were rewritten.
static int search_settle(fx_corpus* c, SearchRun* run, bool* changed) {
  fx_ctx* ctx = c->ctx;
  *changed = false;
  if (!run->tc || !run->s.certify || ctx->h_word[0] == 0) return FX_OK;
  *changed = true;
  const fx::TcSearch& s = run->s;
  const int64_t n_q = run->n_q;
  const int k = run->k, metric = run->metric;
  const float* d_q = run->d_q;
  int64_t* d_out_rows = run->d_out_rows; float* d_out_dist = run->d_out_dist;
  std::string err;
  // queries whose certificate failed: flag 1; fewer than k candidates survived (a sample threshold that came out too tight): flag 2
  FX_TRY(ctx->h_flags.ensure(size_t(n_q) * sizeof(int)));
  int* h_flags = static_cast<int*>(ctx->h_flags.p);
  const int* d_flags = fx::tc_flags(run->L, ctx->d_tc.p);
  FX_CUDA(cudaMemcpyAsync(h_flags, d_flags, size_t(n_q) * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  FX_CUDA(cudaStreamSynchronize(ctx->stream));
  std::vector<int> bad, starved;
  for (int64_t i = 0; i < n_q; ++i) { if (h_flags[i] == 2) starved.push_back(int(i)); else if (h_flags[i]) bad.push_back(int(i)); }
  // Flagged queries are settled by further filter passes over their own (small) batch:
  //  tier 0 (queries left with fewer than k candidates - there is no k-th distance to refine from): the search again with
  //         FULL candidate lists (K' entries each). Stage a keeps the sample prepass: the small batch draws its own sample
  //         (other tiles, other rank), which settles what starves on clustered rows - the sample statistic assumes rows
  //         exchangeable across tiles, and the reference tests' batches of 1000 rows around a common offset are not: 8 % of
  //         the queries of a C2-scale batch starve in the main pass, none after stage a (1.0 ms for ~800 queries; 1.1 ms
  //         through the adaptive search). What stage a leaves starved runs adaptively, without prepass (stage b);
  //  tier 1: preset-threshold refinement: the admission threshold is the query's k-th distance minus the error
  //         bound and every survivor is reranked, so the result is exact.
  std::vector<int> to_refine;
  to_refine.swap(bad);                 // certificate failures of the main pass: tier 1
  bool adaptive_done = false;
  for (int stage = starved.empty() ? 2 : 0; stage <= 2; ++stage) {
    if (stage == 1 && adaptive_done) continue;
    std::vector<int>& in = stage == 2 ? to_refine : starved;
    if (in.empty()) continue;
    const int n_f = int(in.size());
    FX_TRY(ctx->d_qlist.ensure(size_t(n_f) * sizeof(int)));
    FX_CUDA(cudaMemcpyAsync(ctx->d_qlist.p, in.data(), size_t(n_f) * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~size_t(255); return o; };
    const size_t o_q = take(size_t(n_f) * c->dim * 4), o_tau = take(size_t(n_f) * 4);
    const size_t o_rows = take(size_t(n_f) * k * 8), o_dist = take(size_t(n_f) * k * 4);
    FX_TRY(ctx->d_ref.ensure(off));
    char* rb = static_cast<char*>(ctx->d_ref.p);
    float* q_r = reinterpret_cast<float*>(rb + o_q);
    uint32_t* tau_fixed = reinterpret_cast<uint32_t*>(rb + o_tau);
    int64_t* rows2 = reinterpret_cast<int64_t*>(rb + o_rows);
    float* dist2 = reinterpret_cast<float*>(rb + o_dist);
    // gathers the flagged queries (and derives the preset thresholds tier 1 uses)
    double c_err = 0.0, c_add = 0.0, c_abs = 0.0;
    fx::tc_cert_consts(s, &c_err, &c_add, &c_abs);
    fx::refine_prep_kernel<<<n_f, 128, 0, ctx->stream>>>(d_q, static_cast<const int*>(ctx->d_qlist.p), c->dim, metric, k,
                                                        d_out_dist, c->max_norm, c_err, c_add, c_abs, q_r, tau_fixed,
                                                        s.kind == 2 ? 1 : 0);
    FX_CUDA(cudaGetLastError());
    fx::TcSearch s2 = s;
    s2.Q = q_r; s2.n_q = n_f; s2.out_rows = rows2; s2.out_dist = dist2; s2.certify = true;
    s2.tau_fixed = stage == 2 ? tau_fixed : nullptr; s2.no_prepass = stage == 0 ? 0 : 1; s2.full_lists = stage < 2 ? 1 : 0;
    s2.ev_k0 = nullptr; s2.ev_k1 = nullptr;   // keep the timing of the main pass
    const fx::TcLaunch L2 = fx::tc_prepare(&ctx->tc, s2);
    if (stage == 0 && !L2.with_pre) adaptive_done = true;   // (no sample for this small batch: stage a already ran adaptively)
    FX_TRY(ctx->d_tc.ensure(L2.scratch_bytes));
    int launched2 = 0;
    if (!fx::tc_search(&ctx->tc, &c->tc, s2, L2, ctx->d_tc.p, &launched2, &err)) return fail(FX_ECUDA, "fx_search (refine): %s", err.c_str());
    const int* d_flags2 = fx::tc_flags(L2, ctx->d_tc.p);
    // tier 0 results replace the first pass's in any case (they hold k real neighbours for tier 1 to refine from);
    // tier 1 results only where their certificate holds
    fx::refine_scatter_kernel<<<std::min((n_f * k + 255) / 256, 1024), 256, 0, ctx->stream>>>(
        static_cast<const int*>(ctx->d_qlist.p), stage == 2 ? d_flags2 : nullptr, n_f, k, rows2, dist2, d_out_rows, d_out_dist);
    FX_CUDA(cudaGetLastError());
    ctx->launches += launched2 + 2; c->stats.kernel_launches += launched2 + 2;
    FX_CUDA(cudaMemcpyAsync(h_flags, d_flags2, size_t(n_f) * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    FX_CUDA(cudaStreamSynchronize(ctx->stream));
    // stage a: still starved -> stage b, certificate failures -> tier 1; stage b: whatever is flagged -> tier 1;
    // tier 1: whatever is flagged -> the fp64 scan
    std::vector<int> still_starved, still;
    for (int i = 0; i < n_f; ++i) {
      if (h_flags[i] == 0) continue;
      if (stage == 0 && h_flags[i] == 2 && !adaptive_done) still_starved.push_back(in[i]);
      else still.push_back(in[i]);
    }
    c->stats.refined_queries += int64_t(n_f - int(still.size()) - int(still_starved.size()));
    if (stage < 2) { starved.swap(still_starved); to_refine.insert(to_refine.end(), still.begin(), still.end()); }
    else bad.swap(still);
  }
  if (!bad.empty()) {
    // tier 2: the certificate-free fp64 scan
    FX_TRY(ctx->d_qlist.ensure(bad.size() * sizeof(int)));
    FX_CUDA(cudaMemcpyAsync(ctx->d_qlist.p, bad.data(), bad.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    FX_TRY(run_exact_scan(c, d_q, int(n_q), static_cast<int*>(ctx->d_qlist.p), int(bad.size()), metric, k,
                          run->d_mask, d_out_rows, d_out_dist));
    FX_CUDA(cudaStreamSynchronize(ctx->stream));  // `bad` must outlive the H2D copy
    c->stats.fallback_queries += int64_t(bad.size());
  }
  FX_CUDA(cudaEventRecord(ctx->ev_stop, ctx->stream));   // the search now ends here
  return FX_OK;
}

// After the final synchronisation of a search: device times from the events, counters.
static void search_account(fx_corpus* c, const SearchRun& run) {
  fx_ctx* ctx = c->ctx;
  float ms = 0.f, kms = 0.f;
  if (run.spin && run.path == 3) ms = float(double(ctx->h_done[1] + ctx->h_done[3]) * 1e-6);   // the kernels' own globaltimer stamps
  else cudaEventElapsedTime(&ms, ctx->ev_start, ctx->ev_stop);
  if (run.path == 3) kms = ms;   // the direct scan is its one kernel (no inner events: they cost host time on the latency path)
  else cudaEventElapsedTime(&kms, ctx->ev_k0, ctx->ev_k1);
  c->stats.last_search_ms = ms; c->stats.last_main_kernel_ms = kms; c->stats.last_path = run.path; c->stats.last_operand = run.operand;
  c->stats.searches++; c->stats.queries += run.n_q;
}

extern "C" int fx_search_device(fx_corpus* c, const float* d_queries, int64_t n_q, int32_t metric, int32_t k,
                                int32_t precision, const uint8_t* d_row_mask, int64_t* d_out_rows, float* d_out_dist) {
  FX_LEASE(c, "fx_search_device");
  NvtxRange nvtx("fenix:search_device");
  FX_TRY(check_search_args(c, d_queries, n_q, metric, k, precision, d_out_rows, d_out_dist));
  if (n_q == 0) return FX_OK;
  fx_ctx* ctx = c->ctx;
  std::lock_guard<std::mutex> lock(ctx->mu);
  FX_TRY(bind(ctx));
  SearchRun run;
  FX_TRY(search_enqueue(c, d_queries, n_q, metric, k, precision, d_row_mask, d_out_rows, d_out_dist, &run));
  FX_CUDA(cudaStreamSynchronize(ctx->stream));
  bool changed = false;
  FX_TRY(search_settle(c, &run, &changed));
  if (changed) FX_CUDA(cudaStreamSynchronize(ctx->stream));
  search_account(c, run);
  return FX_OK;
}

static bool is_pinned(const void* p) {
  cudaPointerAttributes attr{};
  const bool pinned = cudaPointerGetAttributes(&attr, p) == cudaSuccess && attr.type == cudaMemoryTypeHost;
  cudaGetLastError();
  return pinned;
}

// Small searches are launch-bound: six kernels, three copies and their host calls around a few microseconds of device
// work each. From its second identical call on (same shard, batch size, metric, k, precision; no row mask) such a
// search is ONE cudaGraphLaunch: queries are staged in the context's pinned buffer, the graph copies them in, runs
// prep / filter / finish and copies results and the flagged-query counter back to pinned memory. A flagged query (rare)
// sends the call down the ordinary path.
constexpr int64_t GRAPH_MAX_Q = 64;

static fx_corpus::GraphEntry* graph_entry(fx_corpus* c, int64_t n_q, int metric, int k, int precision) {
  for (auto& g : c->graphs)
    if (g.n_q == n_q && g.metric == metric && g.k == k && g.precision == precision) return &g;
  if (c->graphs.size() >= 16) {          // bounded: drop the oldest
    if (c->graphs.front().exec) cudaGraphExecDestroy(c->graphs.front().exec);
    c->graphs.erase(c->graphs.begin());
  }
  c->graphs.emplace_back();
  auto& g = c->graphs.back();
  g.n_q = n_q; g.metric = metric; g.k = k; g.precision = precision;
  return &g;
}

static bool graph_buffers_match(const fx_ctx* ctx, const fx_corpus::GraphEntry& g) {
  const void* now[7] = {ctx->d_q.p, ctx->d_rows.p, ctx->d_dist.p, ctx->d_tc.p, ctx->h_q.p, ctx->h_rows.p, ctx->h_dist.p};
  for (int i = 0; i < 7; ++i) if (now[i] != g.ptrs[i]) return false;
  return g.knob_epoch == ctx->knob_epoch;
}

// Captures H2D + search + D2H of this call into an executable graph (the caller launches it). false: not captured - the
// entry is marked and the caller takes the ordinary path.
static bool graph_capture(fx_corpus* c, fx_corpus::GraphEntry* g, int64_t n_q, int metric, int k, int precision,
                                     size_t q_bytes, size_t r_bytes, size_t d_bytes, SearchRun* run) {
  fx_ctx* ctx = c->ctx;
  if (cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); g->state = -1; return false; }
  ctx->capturing = true;
  bool ok = cudaMemcpyAsync(ctx->d_q.p, ctx->h_q.p, q_bytes, cudaMemcpyHostToDevice, ctx->stream) == cudaSuccess;
  const int64_t launches0 = c->stats.kernel_launches;
  ok = ok && search_enqueue(c, static_cast<const float*>(ctx->d_q.p), n_q, metric, k, precision, nullptr,
                            static_cast<int64_t*>(ctx->d_rows.p), static_cast<float*>(ctx->d_dist.p), run) == FX_OK;
  ok = ok && cudaMemcpyAsync(ctx->h_rows.p, ctx->d_rows.p, r_bytes, cudaMemcpyDeviceToHost, ctx->stream) == cudaSuccess;
  ok = ok && cudaMemcpyAsync(ctx->h_dist.p, ctx->d_dist.p, d_bytes, cudaMemcpyDeviceToHost, ctx->stream) == cudaSuccess;
  ctx->capturing = false;
  cudaGraph_t graph = nullptr;
  const cudaError_t ee = cudaStreamEndCapture(ctx->stream, &graph);
  if (!ok || ee != cudaSuccess || !graph || !run->tc) {      // only the tensor-core path is worth a graph
    cudaGetLastError();
    if (graph) cudaGraphDestroy(graph);
    g->state = -1;
    return false;
  }
  cudaGraphExec_t exec = nullptr;
  if (cudaGraphInstantiate(&exec, graph, 0) != cudaSuccess) { cudaGetLastError(); cudaGraphDestroy(graph); g->state = -1; return false; }
  cudaGraphDestroy(graph);
  g->exec = exec; g->state = 1; g->knob_epoch = ctx->knob_epoch;
  const void* now[7] = {ctx->d_q.p, ctx->d_rows.p, ctx->d_dist.p, ctx->d_tc.p, ctx->h_q.p, ctx->h_rows.p, ctx->h_dist.p};
  for (int i = 0; i < 7; ++i) g->ptrs[i] = const_cast<void*>(now[i]);
  g->path = run->path; g->operand = run->operand; g->variant = c->stats.last_variant | (c->stats.last_resident_queries << 3); g->launches = int(c->stats.kernel_launches - launches0);
  c->stats.kernel_launches = launches0;   // counted when the graph runs
  return true;
}

extern "C" int fx_search(fx_corpus* c, const float* queries, int64_t n_q, int32_t metric, int32_t k,
                         int32_t precision, const uint8_t* row_mask, int64_t* out_rows, float* out_dist) {
  FX_LEASE(c, "fx_search");
  NvtxRange nvtx("fenix:search");
  FX_TRY(check_search_args(c, queries, n_q, metric, k, precision, out_rows, out_dist));
  if (n_q == 0) return FX_OK;
  fx_ctx* ctx = c->ctx;
  std::lock_guard<std::mutex> lock(ctx->mu);
  FX_TRY(bind(ctx));
  const size_t q_bytes = size_t(n_q) * c->dim * sizeof(float);
  const size_t r_bytes = size_t(n_q) * k * sizeof(int64_t), d_bytes = size_t(n_q) * k * sizeof(float);
  FX_TRY(ctx->d_q.ensure(q_bytes));
  FX_TRY(ctx->d_rows.ensure(r_bytes));
  FX_TRY(ctx->d_dist.ensure(d_bytes));
  // ---- a handful of queries over a small shard: one launch. Small query blocks ride in the kernel parameters, the
  // results are written straight to mapped pinned staging (cudaMallocHost memory is device-addressable under unified
  // addressing): no H2D / D2H copies on the common single-query call ----
  if (c->n > 0 && direct_plan_for(c, n_q, k, precision).ok) {
    FX_TRY(ctx->h_rows.ensure(r_bytes));
    FX_TRY(ctx->h_dist.ensure(d_bytes));
    SearchRun run;
    run.spin = !ctx->tc.knobs.debug_direct;   // (the timeline's stamps land after the completion word)
    if (n_q * int64_t(c->dim) <= fx::DS_INLINE_FLOATS) {
      run.inline_q = queries;
    } else {
      FX_TRY(ctx->h_q.ensure(q_bytes));
      std::memcpy(ctx->h_q.p, queries, q_bytes);
      FX_CUDA(cudaMemcpyAsync(ctx->d_q.p, ctx->h_q.p, q_bytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    const uint8_t* d_mask = nullptr;
    if (row_mask) {
      FX_TRY(ctx->d_mask.ensure(size_t(c->n)));
      FX_CUDA(cudaMemcpyAsync(ctx->d_mask.p, row_mask, size_t(c->n), cudaMemcpyHostToDevice, ctx->stream));
      d_mask = static_cast<const uint8_t*>(ctx->d_mask.p);
    }
    FX_TRY(search_enqueue(c, static_cast<const float*>(ctx->d_q.p), n_q, metric, k, precision, d_mask,
                          static_cast<int64_t*>(ctx->h_rows.p), static_cast<float*>(ctx->h_dist.p), &run));
    if (run.spin) {
      // the last CTA writes the results, then the sequence number, into mapped host memory: spinning on that word skips the
      // driver's stream-completion latency. A kernel that does not report within 2 ms (a fault) falls back to the stream wait.
      volatile unsigned long long* done = ctx->h_done;
      const auto t0 = std::chrono::steady_clock::now();
      for (unsigned it = 1; done[0] != ctx->direct_seq; ++it) {
        if ((it & 0x3ff) == 0 && std::chrono::steady_clock::now() - t0 > std::chrono::milliseconds(2)) {
          FX_CUDA(cudaStreamSynchronize(ctx->stream));
          break;
        }
      }
      std::atomic_thread_fence(std::memory_order_acquire);
    } else {
      FX_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    std::memcpy(out_rows, ctx->h_rows.p, r_bytes);
    std::memcpy(out_dist, ctx->h_dist.p, d_bytes);
    search_account(c, run);
    if (ctx->tc.knobs.debug_direct && ctx->h_flags.p) {
      static_cast<volatile unsigned long long*>(ctx->h_flags.p)[500] = 1;
      const int grid = direct_plan_for(c, n_q, k, precision).grid;
      const unsigned long long* t = static_cast<const unsigned long long*>(ctx->h_flags.p);
      unsigned long long lo = ~0ull, hi = 0;
      for (int i = 0; i < grid; ++i) { lo = std::min(lo, t[8 + i]); hi = std::max(hi, t[8 + i]); }
      fprintf(stderr, "[fenix direct] last CTA: start 0, staged %llu, scanned %llu, published %llu, ticket %llu, joined %llu, end %llu ns; "
                      "scan ends over all %d CTAs: first %lld, last %lld ns after that start; event time %.1f us\n",
              t[1] - t[0], t[2] - t[0], t[3] - t[0], t[4] - t[0], t[5] - t[0], t[6] - t[0], grid,
              (long long)(lo - t[0]), (long long)(hi - t[0]), c->stats.last_search_ms * 1e3);
    }
    return FX_OK;
  }
  // ---- small searches: replay (or capture) the whole call as one CUDA graph ----
  if (n_q <= GRAPH_MAX_Q && !row_mask && c->n > 0 && ctx->tc.knobs.graph != 0 && precision != FX_PREC_EXACT_SCAN &&
      fx::tc_supported(&ctx->tc, &c->tc, c->n, c->dim, k, int(n_q))) {
    fx_corpus::GraphEntry* g = graph_entry(c, n_q, metric, k, precision);
    if (g->state == 1 && !graph_buffers_match(ctx, *g)) {     // a buffer grew or a knob changed since the capture
      cudaGraphExecDestroy(g->exec); g->exec = nullptr; g->state = 0;
    }
    bool launched = false;
    SearchRun run;
    if (g->state >= 0) {
      FX_TRY(ctx->h_q.ensure(q_bytes));
      FX_TRY(ctx->h_rows.ensure(r_bytes));
      FX_TRY(ctx->h_dist.ensure(d_bytes));
    }
    if (g->state == 1) {
      std::memcpy(ctx->h_q.p, queries, q_bytes);
      ctx->h_word[0] = 0;
      FX_CUDA(cudaGraphLaunch(g->exec, ctx->stream));
      run.tc = true; run.path = g->path; run.operand = g->operand; run.n_q = n_q;
      set_variant(c, g->variant);
      ctx->launches += g->launches; c->stats.kernel_launches += g->launches;
      launched = true;
    } else if (g->state == 2) {
      // second identical call: everything it needs (shadows, scratch) exists and is big enough - capture it
      std::memcpy(ctx->h_q.p, queries, q_bytes);
      if (graph_capture(c, g, n_q, metric, k, precision, q_bytes, r_bytes, d_bytes, &run)) {
        ctx->h_word[0] = 0;
        FX_CUDA(cudaGraphLaunch(g->exec, ctx->stream));
        ctx->launches += g->launches; c->stats.kernel_launches += g->launches;
        launched = true;
      }
    } else if (g->state == 0) {
      g->state = 2;   // seen once: the next identical call captures
    }
    if (launched) {
      FX_CUDA(cudaStreamSynchronize(ctx->stream));
      if (ctx->h_word[0] == 0) {
        std::memcpy(out_rows, ctx->h_rows.p, r_bytes);
        std::memcpy(out_dist, ctx->h_dist.p, d_bytes);
        search_account(c, run);
        return FX_OK;
      }
      // a certificate failed: the ordinary path below recomputes the call, with its repair tiers
    }
  }
  // queries: direct DMA when the caller's buffer is pinned, otherwise through pinned staging
  const void* q_src = queries;
  if (!is_pinned(queries)) {
    FX_TRY(ctx->h_q.ensure(q_bytes));
    std::memcpy(ctx->h_q.p, queries, q_bytes);
    q_src = ctx->h_q.p;
  }
  FX_CUDA(cudaMemcpyAsync(ctx->d_q.p, q_src, q_bytes, cudaMemcpyHostToDevice, ctx->stream));
  const uint8_t* d_mask = nullptr;
  if (row_mask && c->n > 0) {
    FX_TRY(ctx->d_mask.ensure(size_t(c->n)));
    FX_CUDA(cudaMemcpyAsync(ctx->d_mask.p, row_mask, size_t(c->n), cudaMemcpyHostToDevice, ctx->stream));
    d_mask = static_cast<const uint8_t*>(ctx->d_mask.p);
  }
  SearchRun run;
  FX_TRY(search_enqueue(c, static_cast<const float*>(ctx->d_q.p), n_q, metric, k, precision, d_mask,
                        static_cast<int64_t*>(ctx->d_rows.p), static_cast<float*>(ctx->d_dist.p), &run));
  // results: straight into the caller's buffers when pinned, else via pinned staging. The copies are queued behind the
  // kernels; the one synchronisation below covers the flagged-query counter too.
  const bool direct = is_pinned(out_rows) && is_pinned(out_dist);
  void* dst_rows = out_rows; void* dst_dist = out_dist;
  if (!direct) {
    FX_TRY(ctx->h_rows.ensure(r_bytes));
    FX_TRY(ctx->h_dist.ensure(d_bytes));
    dst_rows = ctx->h_rows.p; dst_dist = ctx->h_dist.p;
  }
  for (int attempt = 0; attempt < 2; ++attempt) {
    FX_CUDA(cudaMemcpyAsync(dst_rows, ctx->d_rows.p, r_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    FX_CUDA(cudaMemcpyAsync(dst_dist, ctx->d_dist.p, d_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    FX_CUDA(cudaStreamSynchronize(ctx->stream));
    if (attempt == 1) break;
    bool changed = false;
    FX_TRY(search_settle(c, &run, &changed));
    if (!changed) break;
  }
  if (!direct) {
    std::memcpy(out_rows, ctx->h_rows.p, r_bytes);
    std::memcpy(out_dist, ctx->h_dist.p, d_bytes);
  }
  search_account(c, run);
  return FX_OK;
}

// ----------------------------------------------------------------------------------------
// batched IVF: an inverted index per shard, one launch per query batch (direct_scan.cuh, LISTS mode)
// ----------------------------------------------------------------------------------------
extern "C" int fx_corpus_set_cells(fx_corpus* c, const int32_t* inv_rows, int64_t n_inv, const int64_t* cell_off, int64_t n_cells) {
  FX_LEASE(c, "fx_corpus_set_cells");
  if (!c->finalized) return fail(FX_ESTATE, "fx_corpus_set_cells: corpus is not finalized");
  if (n_inv < 0 || n_cells < 0 || (n_inv > 0 && !inv_rows) || !cell_off) return fail(FX_EINVAL, "fx_corpus_set_cells: bad arguments");
  if (cell_off[0] != 0 || cell_off[n_cells] != n_inv) return fail(FX_EINVAL, "fx_corpus_set_cells: cell_off must run from 0 to n_inv");
  for (int64_t i = 0; i < n_cells; ++i) if (cell_off[i + 1] < cell_off[i]) return fail(FX_EINVAL, "fx_corpus_set_cells: cell_off must not decrease");
  for (int64_t i = 0; i < n_inv; ++i) if (inv_rows[i] < 0 || inv_rows[i] >= c->n) return fail(FX_EINVAL, "fx_corpus_set_cells: row %d out of range", inv_rows[i]);
  fx_ctx* ctx = c->ctx;
  std::lock_guard<std::mutex> lock(ctx->mu);
  FX_TRY(bind(ctx));
  FX_CUDA(cudaStreamSynchronize(ctx->stream));
  if (c->d_inv) { cudaFree(c->d_inv); c->d_inv = nullptr; }
  if (c->d_cell_off) { cudaFree(c->d_cell_off); c->d_cell_off = nullptr; }
  c->n_inv = 0; c->n_cells = 0; c->h_cell_off.clear();
  if (cudaMalloc(reinterpret_cast<void**>(&c->d_inv), size_t(std::max<int64_t>(n_inv, 1)) * sizeof(int)) != cudaSuccess ||
      cudaMalloc(reinterpret_cast<void**>(&c->d_cell_off), size_t(n_cells + 1) * sizeof(long long)) != cudaSuccess) {
    cudaGetLastError();
    if (c->d_inv) { cudaFree(c->d_inv); c->d_inv = nullptr; }
    return fail(FX_ENOMEM, "fx_corpus_set_cells: no device memory for %lld rows in %lld cells", (long long)n_inv, (long long)n_cells);
  }
  FX_CUDA(cudaMemcpy(c->d_inv, inv_rows, size_t(n_inv) * sizeof(int), cudaMemcpyHostToDevice));
  FX_CUDA(cudaMemcpy(c->d_cell_off, cell_off, size_t(n_cells + 1) * sizeof(long long), cudaMemcpyHostToDevice));
  c->h_cell_off.assign(cell_off, cell_off + n_cells + 1);
  c->n_inv = n_inv; c->n_cells = n_cells;
  return FX_OK;
}

extern "C" int fx_search_cells(fx_corpus* c, const float* queries, int64_t n_q, int32_t metric, int32_t k, const int32_t* probes,
                               int32_t n_probe, const uint8_t* row_mask, int64_t* out_rows, float* out_dist) {
  FX_LEASE(c, "fx_search_cells");
  NvtxRange nvtx("fenix:search_cells");
  FX_TRY(check_search_args(c, queries, n_q, metric, k, FX_PREC_FP32, out_rows, out_dist));
  if (n_q == 0) return FX_OK;
  if (!probes || n_probe < 1) return fail(FX_EINVAL, "fx_search_cells: no probes");
  fx_ctx* ctx = c->ctx;
  std::lock_guard<std::mutex> lock(ctx->mu);   // (also against a concurrent fx_corpus_set_cells on this shard)
  if (!c->d_cell_off) return fail(FX_ESTATE, "fx_search_cells: the shard has no cells (fx_corpus_set_cells)");
  // the longest candidate list of the batch sizes the grid; cell numbers are validated on the way
  int64_t max_items = 0;
  for (int64_t q = 0; q < n_q; ++q) {
    int64_t items = 0;
    for (int t = 0; t < n_probe; ++t) {
      const int cell = probes[q * n_probe + t];
      if (cell >= c->n_cells) return fail(FX_EINVAL, "fx_search_cells: cell %d out of range [0, %lld)", cell, (long long)c->n_cells);
      if (cell >= 0) items += c->h_cell_off[cell + 1] - c->h_cell_off[cell];
    }
    if (items > (int64_t(1) << 31) - 1) return fail(FX_EUNSUP, "fx_search_cells: a query probes more than 2^31 rows");
    max_items = std::max(max_items, items);
  }
  const fx::CellsPlan pl = fx::cells_plan(c->pitch, n_q, k, n_probe, max_items, ctx->sm_count);
  if (!pl.ok) return fail(FX_EUNSUP, "fx_search_cells: shape not supported by the one-launch path (k %d <= 128, probes %d <= 512, queries %lld <= 65535, dim %d)",
                          k, n_probe, (long long)n_q, c->dim);
  FX_TRY(bind(ctx));
  const size_t q_bytes = size_t(n_q) * c->dim * sizeof(float), p_bytes = size_t(n_q) * n_probe * sizeof(int);
  const size_t r_bytes = size_t(n_q) * k * sizeof(int64_t), d_bytes = size_t(n_q) * k * sizeof(float);
  FX_TRY(ctx->d_q.ensure(q_bytes));
  FX_TRY(ctx->d_rows.ensure(r_bytes));
  FX_TRY(ctx->d_dist.ensure(d_bytes));
  FX_TRY(ctx->d_qlist.ensure(p_bytes));
  FX_TRY(ctx->d_tickets.ensure(size_t(n_q) * sizeof(unsigned int)));
  FX_TRY(ctx->d_partial.ensure(pl.partial_bytes));
  FX_TRY(ctx->h_q.ensure(q_bytes + p_bytes));
  FX_TRY(ctx->h_rows.ensure(r_bytes));
  FX_TRY(ctx->h_dist.ensure(d_bytes));
  std::memcpy(ctx->h_q.p, queries, q_bytes);
  std::memcpy(static_cast<char*>(ctx->h_q.p) + q_bytes, probes, p_bytes);
  FX_CUDA(cudaEventRecord(ctx->ev_start, ctx->stream));
  FX_CUDA(cudaMemcpyAsync(ctx->d_q.p, ctx->h_q.p, q_bytes, cudaMemcpyHostToDevice, ctx->stream));
  FX_CUDA(cudaMemcpyAsync(ctx->d_qlist.p, static_cast<char*>(ctx->h_q.p) + q_bytes, p_bytes, cudaMemcpyHostToDevice, ctx->stream));
  FX_CUDA(cudaMemsetAsync(ctx->d_tickets.p, 0, size_t(n_q) * sizeof(unsigned int), ctx->stream));
  const uint8_t* d_mask = nullptr;
  if (row_mask) {
    FX_TRY(ctx->d_mask.ensure(size_t(c->n)));
    FX_CUDA(cudaMemcpyAsync(ctx->d_mask.p, row_mask, size_t(c->n), cudaMemcpyHostToDevice, ctx->stream));
    d_mask = static_cast<const uint8_t*>(ctx->d_mask.p);
  }
  fx::DirectParams p{};
  p.X = c->X; p.n_rows = c->n; p.pitch = c->pitch; p.dim = c->dim; p.row_base = c->row_base;
  p.Q = static_cast<const float*>(ctx->d_q.p); p.n_q = int(n_q); p.metric = metric; p.k = k; p.mask = d_mask;
  p.partial = static_cast<uint64_t*>(ctx->d_partial.p); p.ticket = static_cast<unsigned int*>(ctx->d_tickets.p); p.cap_steps = pl.cap_steps;
  p.out_rows = static_cast<int64_t*>(ctx->d_rows.p); p.out_dist = static_cast<float*>(ctx->d_dist.p);
  p.inv_rows = c->d_inv; p.cell_off = c->d_cell_off; p.probes = static_cast<const int*>(ctx->d_qlist.p); p.n_probe = n_probe;
  FX_CUDA(fx::cells_launch(pl, p, int(n_q), ctx->stream));
  ctx->launches++; c->stats.kernel_launches++;
  FX_CUDA(cudaEventRecord(ctx->ev_stop, ctx->stream));
  FX_CUDA(cudaMemcpyAsync(ctx->h_rows.p, ctx->d_rows.p, r_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  FX_CUDA(cudaMemcpyAsync(ctx->h_dist.p, ctx->d_dist.p, d_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  FX_CUDA(cudaStreamSynchronize(ctx->stream));
  std::memcpy(out_rows, ctx->h_rows.p, r_bytes);
  std::memcpy(out_dist, ctx->h_dist.p, d_bytes);
  SearchRun run; run.path = 3; run.n_q = n_q;
  search_account(c, run);
  return FX_OK;
}

extern "C" int fx_distances(fx_corpus* c, const float* query, int32_t metric, float* out_dist) {
  FX_LEASE(c, "fx_distances");
  if (!c->finalized) return fail(FX_ESTATE, "fx_distances: corpus is not finalized");
  if (metric < 0 || metric > 2) return fail(FX_EINVAL, "fx_distances: unknown metric %d", metric);
  if (c->n == 0) return FX_OK;
  if (!query || !out_dist) return fail(FX_EINVAL, "fx_distances: NULL buffer");
  fx_ctx* ctx = c->ctx;
  std::lock_guard<std::mutex> lock(ctx->mu);
  FX_TRY(bind(ctx));
  const size_t q_bytes = size_t(c->dim) * sizeof(float), d_bytes = size_t(c->n) * sizeof(float);
  FX_TRY(ctx->d_q.ensure(q_bytes));
  FX_TRY(ctx->d_dist.ensure(d_bytes));
  FX_CUDA(cudaMemcpyAsync(ctx->d_q.p, query, q_bytes, cudaMemcpyHostToDevice, ctx->stream));
  const size_t per_q = size_t(c->pitch) * 8 + 8 + 8 + 8 + 2 * 8 + 4;
  if (per_q > 200 * 1024) return fail(FX_EUNSUP, "fx_distances: dim %d too large", c->dim);
  fx::ScanParams p{};
  p.X = c->X; p.n_rows = c->n; p.pitch = c->pitch; p.dim = c->dim; p.Q = static_cast<const float*>(ctx->d_q.p);
  p.n_q = 1; p.metric = metric; p.mask = nullptr; p.q_list = nullptr; p.n_list = 1; p.k = 0; p.buf = 2; p.qb = 1;
  p.floor = nullptr;
  p.partial = nullptr; p.dist_out = static_cast<float*>(ctx->d_dist.p);
  const int64_t tiles = (c->n + fx::SCAN_THREADS - 1) / fx::SCAN_THREADS;
  int W = int(std::min<int64_t>(tiles, int64_t(ctx->sm_count) * 8));
  fx::exact_scan_kernel<<<dim3(W, 1), fx::SCAN_THREADS, per_q + 16, ctx->stream>>>(p);
  FX_CUDA(cudaGetLastError());
  ctx->launches++; c->stats.kernel_launches++;
  FX_TRY(ctx->h_dist.ensure(d_bytes));
  FX_CUDA(cudaMemcpyAsync(ctx->h_dist.p, ctx->d_dist.p, d_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  FX_CUDA(cudaStreamSynchronize(ctx->stream));
  std::memcpy(out_dist, ctx->h_dist.p, d_bytes);
  return FX_OK;
}

// ----------------------------------------------------------------------------------------
// range search: every row within a radius (DESIGN.md, "Range search")
// ----------------------------------------------------------------------------------------
// Grows `b` to `need` bytes keeping its first `used` bytes (the hit buffer fills in several steps).
static int grow_keep(fx_ctx* ctx, DevBuf& b, size_t used, size_t need) {
  if (need <= b.cap) return FX_OK;
  DevBuf nb;
  FX_TRY(nb.ensure(need));
  if (used) FX_CUDA(cudaMemcpyAsync(nb.p, b.p, used, cudaMemcpyDeviceToDevice, ctx->stream));
  FX_CUDA(cudaStreamSynchronize(ctx->stream));
  b.release();
  b = nb;
  return FX_OK;
}

// Distance columns of a range-search batch: at most this much scratch (or one column), whatever n_q x N is.
constexpr size_t RANGE_COL_BYTES = size_t(256) << 20;

// Hits of the listed queries by the exact scan: the distance columns of a batch of queries at a time, then the unmasked
// rows within the radius become keys in each query's segment of ctx->d_hits, appended at *used. seg / hits: host
// arrays over every query of the search.
static int range_scan(fx_corpus* c, const float* d_q, int64_t n_q, const std::vector<int>& list, int metric, float radius,
                      const uint8_t* d_mask, std::vector<int64_t>& seg, std::vector<int64_t>& hits, size_t* used) {
  fx_ctx* ctx = c->ctx;
  const size_t per_q = size_t(c->pitch) * 8 + 8 + 8 + 8 + 2 * 8 + 4;   // exact_scan_kernel's shared memory, column mode
  const int qb = int(std::min<size_t>(fx::SCAN_MAX_QB, (200 * 1024) / per_q));
  if (qb < 1) return fail(FX_EUNSUP, "fx_search_range: dim %d too large for the exact scan", c->dim);
  const int batch = int(std::max<int64_t>(1, std::min<int64_t>(4096, int64_t(RANGE_COL_BYTES / (size_t(c->n) * 4)))));
  const int nb_max = int(std::min<size_t>(size_t(batch), list.size()));
  FX_TRY(ctx->d_col.ensure(size_t(nb_max) * c->n * 4));
  FX_TRY(ctx->d_rbatch.ensure(size_t(nb_max) * 24));   // per slot: list entry, count, fill (int) and segment (int64)
  FX_TRY(ctx->h_flags.ensure(size_t(nb_max) * sizeof(int)));
  float* col = static_cast<float*>(ctx->d_col.p);
  int64_t* d_seg = static_cast<int64_t*>(ctx->d_rbatch.p);
  int* d_list = reinterpret_cast<int*>(d_seg + nb_max);
  int* d_cnt = d_list + nb_max;
  int* d_fill = d_cnt + nb_max;
  int* h_cnt = static_cast<int*>(ctx->h_flags.p);
  std::vector<int64_t> seg_b(nb_max);
  const int64_t tiles = (c->n + fx::SCAN_THREADS - 1) / fx::SCAN_THREADS;
  const int cblocks = int(std::min<int64_t>((c->n + 255) / 256, 256));
  for (size_t b0 = 0; b0 < list.size(); b0 += size_t(batch)) {
    const int nb = int(std::min<size_t>(size_t(batch), list.size() - b0));
    FX_CUDA(cudaMemcpyAsync(d_list, list.data() + b0, size_t(nb) * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    FX_CUDA(cudaMemsetAsync(d_cnt, 0, size_t(2 * nb_max) * sizeof(int), ctx->stream));   // counts and fills
    fx::ScanParams p{};
    p.X = c->X; p.n_rows = c->n; p.pitch = c->pitch; p.dim = c->dim; p.Q = d_q; p.n_q = int(n_q); p.metric = metric;
    p.mask = nullptr; p.q_list = d_list; p.n_list = nb; p.k = 0; p.buf = 2; p.qb = std::min(qb, nb); p.floor = nullptr;
    p.partial = nullptr; p.dist_out = col;
    const int groups = (nb + p.qb - 1) / p.qb;
    const int W = int(std::min<int64_t>(tiles, std::max<int64_t>(1, (8 * int64_t(ctx->sm_count) + groups - 1) / groups)));
    fx::exact_scan_kernel<<<dim3(W, groups), fx::SCAN_THREADS, per_q * p.qb + 16, ctx->stream>>>(p);
    FX_CUDA(cudaGetLastError());
    fx::range_col_count_kernel<<<dim3(cblocks, nb), 256, 0, ctx->stream>>>(col, c->n, d_mask, radius, d_cnt);
    FX_CUDA(cudaGetLastError());
    FX_CUDA(cudaMemcpyAsync(h_cnt, d_cnt, size_t(nb) * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    FX_CUDA(cudaStreamSynchronize(ctx->stream));
    const size_t before = *used;
    for (int i = 0; i < nb; ++i) {
      const int q = list[b0 + i];
      seg[q] = seg_b[i] = int64_t(*used);
      hits[q] = h_cnt[i];
      *used += size_t(h_cnt[i]);
    }
    FX_TRY(grow_keep(ctx, ctx->d_hits, before * 8, std::max<size_t>(*used, 1) * 8));
    FX_CUDA(cudaMemcpyAsync(d_seg, seg_b.data(), size_t(nb) * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
    fx::range_col_compact_kernel<<<dim3(cblocks, nb), 256, 0, ctx->stream>>>(col, c->n, d_mask, radius, d_seg, d_fill,
                                                                             static_cast<uint64_t*>(ctx->d_hits.p));
    FX_CUDA(cudaGetLastError());
    ctx->launches += 3; c->stats.kernel_launches += 3;
  }
  return FX_OK;
}

extern "C" int fx_search_range(fx_corpus* c, const float* queries, int64_t n_q, int32_t metric, float radius,
                               int32_t precision, const uint8_t* row_mask, int64_t capacity, int64_t* out_offsets,
                               int64_t* out_rows, float* out_dist) {
  FX_LEASE(c, "fx_search_range");
  NvtxRange nvtx("fenix:search_range");
  if (!c->finalized) return fail(FX_ESTATE, "fx_search_range: corpus is not finalized");
  if (n_q < 0 || capacity < 0) return fail(FX_EINVAL, "fx_search_range: negative query count or capacity");
  if (!out_offsets || (n_q > 0 && !queries) || (capacity > 0 && (!out_rows || !out_dist)))
    return fail(FX_EINVAL, "fx_search_range: NULL buffer");
  if (n_q > int64_t(1) << 24) return fail(FX_EUNSUP, "fx_search_range: at most 2^24 queries per call");
  if (metric < 0 || metric > 2) return fail(FX_EINVAL, "fx_search_range: unknown metric %d", metric);
  if (radius != radius) return fail(FX_EINVAL, "fx_search_range: radius is NaN");
  if (precision == FX_PREC_TF32 || precision == FX_PREC_BF16)
    return fail(FX_EUNSUP, "fx_search_range: range search is exact only (FX_PREC_FP32 or FX_PREC_EXACT_SCAN)");
  if (precision != FX_PREC_FP32 && precision != FX_PREC_EXACT_SCAN)
    return fail(FX_EINVAL, "fx_search_range: unknown precision mode %d", precision);
  std::fill(out_offsets, out_offsets + n_q + 1, int64_t(0));
  if (n_q == 0 || c->n == 0) return FX_OK;
  fx_ctx* ctx = c->ctx;
  std::lock_guard<std::mutex> lock(ctx->mu);
  FX_TRY(bind(ctx));
  const size_t q_bytes = size_t(n_q) * c->dim * sizeof(float);
  FX_TRY(ctx->d_q.ensure(q_bytes));
  FX_TRY(ctx->h_q.ensure(q_bytes));
  std::memcpy(ctx->h_q.p, queries, q_bytes);
  FX_CUDA(cudaEventRecord(ctx->ev_start, ctx->stream));
  FX_CUDA(cudaMemcpyAsync(ctx->d_q.p, ctx->h_q.p, q_bytes, cudaMemcpyHostToDevice, ctx->stream));
  const float* d_q = static_cast<const float*>(ctx->d_q.p);
  const uint8_t* d_mask = nullptr;
  if (row_mask) {
    FX_TRY(ctx->d_mask.ensure(size_t(c->n)));
    FX_CUDA(cudaMemcpyAsync(ctx->d_mask.p, row_mask, size_t(c->n), cudaMemcpyHostToDevice, ctx->stream));
    d_mask = static_cast<const uint8_t*>(ctx->d_mask.p);
  }
  // per-query device arrays: segment start, candidate count, segment end (int64), output offsets [n_q + 1],
  // preset threshold, hit count
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~size_t(255); return o; };
  const size_t o_seg = take(size_t(n_q) * 8), o_cand = take(size_t(n_q) * 8), o_end = take(size_t(n_q) * 8);
  const size_t o_off = take(size_t(n_q + 1) * 8), o_tau = take(size_t(n_q) * 4), o_hits = take(size_t(n_q) * 4);
  FX_TRY(ctx->d_rmeta.ensure(off));
  char* rm = static_cast<char*>(ctx->d_rmeta.p);
  int64_t* d_seg = reinterpret_cast<int64_t*>(rm + o_seg);
  int64_t* d_cand = reinterpret_cast<int64_t*>(rm + o_cand);
  int64_t* d_end = reinterpret_cast<int64_t*>(rm + o_end);
  int64_t* d_off = reinterpret_cast<int64_t*>(rm + o_off);
  uint32_t* d_tau = reinterpret_cast<uint32_t*>(rm + o_tau);
  int* d_hitcnt = reinterpret_cast<int*>(rm + o_hits);
  FX_TRY(ctx->h_rows.ensure(size_t(n_q + 1) * 8));
  int64_t* h_i64 = static_cast<int64_t*>(ctx->h_rows.p);

  std::vector<int64_t> seg(n_q, 0), hits(n_q, 0);
  std::vector<int> scan_list;
  size_t used = 0;
  SearchRun run;
  run.n_q = n_q;
  // tensor-core path: the operand an exact k = 1 search would filter with, thresholds from the radius, no selection
  const bool want_tc = precision == FX_PREC_FP32 && fx::tc_supported(&ctx->tc, &c->tc, c->n, c->dim, 1, int(n_q));
  if (want_tc) {
    fx::TcSearch s{};
    s.X = c->X; s.hx = c->hx; s.rx = c->rx; s.n_rows = c->n; s.dim = c->dim; s.pitch = c->pitch;
    s.row_base = c->row_base; s.max_norm = c->max_norm; s.Q = d_q; s.n_q = int(n_q); s.metric = metric; s.k = 1;
    s.certify = true; s.out_rows = nullptr; s.out_dist = nullptr;
    s.stream = ctx->stream; s.ev_k0 = ctx->ev_k0; s.ev_k1 = ctx->ev_k1; s.ev_flags = cudaEventRecordDefault; s.dbg = nullptr;
    s.tau_fixed = d_tau; s.no_prepass = 1; s.full_lists = 1; s.no_finish = 1;
    const bool have_i8 = int8_wanted(c, metric, 1, FX_PREC_FP32) && ensure_i8_shadow(c);
    const bool have_shadow = !have_i8 && !ctx->tc.knobs.fp32_filter_tf32 &&
                             ((metric == 1 && ensure_norm_shadow(c)) || ensure_plain_shadow(c));
    const int kind = have_i8 ? 2 : (have_shadow ? 1 : 0);
    FX_TRY(configure_filter(c, metric, kind, d_mask, &s));
    double c_err = 0.0, c_add = 0.0, c_abs = 0.0;
    fx::tc_cert_consts(s, &c_err, &c_add, &c_abs);
    fx::range_prep_kernel<<<int((n_q + 3) / 4), 128, 0, ctx->stream>>>(d_q, int(n_q), c->dim, metric, radius, c->max_norm,
                                                                       c_err, c_add, c_abs, kind == 2 ? 1 : 0, d_tau);
    FX_CUDA(cudaGetLastError());
    const fx::TcLaunch L = fx::tc_prepare(&ctx->tc, s);
    FX_TRY(ctx->d_tc.ensure(L.scratch_bytes));
    std::string err;
    int launched = 0, variant = 0;
    if (!fx::tc_search(&ctx->tc, &c->tc, s, L, ctx->d_tc.p, &launched, &err, &variant)) return fail(FX_ECUDA, "fx_search_range: %s", err.c_str());
    const fx::FinishParams f = fx::tc_finish_params(s, L.pl, ctx->d_tc.p);
    fx::range_count_kernel<<<int((n_q + 7) / 8), 256, 0, ctx->stream>>>(f, d_cand);
    FX_CUDA(cudaGetLastError());
    FX_CUDA(cudaMemcpyAsync(h_i64, d_cand, size_t(n_q) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    FX_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int64_t q = 0; q < n_q; ++q) {
      if (h_i64[q] < 0) { scan_list.push_back(int(q)); continue; }   // a candidate list overflowed
      seg[q] = int64_t(used);
      used += size_t(h_i64[q]);
    }
    FX_TRY(ctx->d_hits.ensure(std::max<size_t>(used, 1) * 8));
    FX_CUDA(cudaMemcpyAsync(d_seg, seg.data(), size_t(n_q) * 8, cudaMemcpyHostToDevice, ctx->stream));
    fx::range_finish_kernel<<<int(n_q), 256, size_t(c->pitch) * 4 + 16, ctx->stream>>>(f, radius, d_seg,
                                                                                      static_cast<uint64_t*>(ctx->d_hits.p), d_hitcnt);
    FX_CUDA(cudaGetLastError());
    ctx->launches += launched + 3; c->stats.kernel_launches += launched + 3;   // (+ prep, count, finish)
    run.tc = true; run.path = kind == 0 ? 1 : 2; run.operand = kind;
    set_variant(c, variant);
    c->stats.fallback_queries += int64_t(scan_list.size());
  } else {
    scan_list.resize(size_t(n_q));
    for (int64_t q = 0; q < n_q; ++q) scan_list[size_t(q)] = int(q);
    FX_CUDA(cudaEventRecord(ctx->ev_k0, ctx->stream));
  }
  if (want_tc) {
    // hit counts of the tensor-core queries (the scan's own are counted on the host)
    FX_CUDA(cudaMemcpyAsync(h_i64, d_hitcnt, size_t(n_q) * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    FX_CUDA(cudaStreamSynchronize(ctx->stream));
    const int* h_hits = reinterpret_cast<const int*>(h_i64);
    for (int64_t q = 0; q < n_q; ++q) hits[q] = h_hits[q];
  }
  if (!scan_list.empty()) FX_TRY(range_scan(c, d_q, n_q, scan_list, metric, radius, d_mask, seg, hits, &used));
  if (!want_tc) FX_CUDA(cudaEventRecord(ctx->ev_k1, ctx->stream));
  for (int64_t q = 0; q < n_q; ++q) out_offsets[q + 1] = out_offsets[q] + hits[q];
  const int64_t total = out_offsets[n_q];
  if (total > capacity || total == 0) {
    FX_CUDA(cudaEventRecord(ctx->ev_stop, ctx->stream));
    FX_CUDA(cudaStreamSynchronize(ctx->stream));
    search_account(c, run);
    if (total > capacity)
      return fail(FX_ETRUNC, "fx_search_range: %lld hits exceed the capacity of %lld (out_offsets holds the sizes needed)",
                  (long long)total, (long long)capacity);
    return FX_OK;
  }
  if (used > size_t(INT32_MAX)) return fail(FX_EUNSUP, "fx_search_range: %zu candidates exceed 2^31 - 1 (split the query batch)", used);
  // sort every query's segment by (distance, row), then write rows and distances at its output offset
  {
    std::vector<int64_t> end(n_q);
    for (int64_t q = 0; q < n_q; ++q) end[q] = seg[q] + hits[q];
    FX_CUDA(cudaMemcpyAsync(d_seg, seg.data(), size_t(n_q) * 8, cudaMemcpyHostToDevice, ctx->stream));
    FX_CUDA(cudaMemcpyAsync(d_end, end.data(), size_t(n_q) * 8, cudaMemcpyHostToDevice, ctx->stream));
    FX_CUDA(cudaMemcpyAsync(d_off, out_offsets, size_t(n_q + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    FX_TRY(ctx->d_hits2.ensure(used * 8));
    const uint64_t* keys = static_cast<const uint64_t*>(ctx->d_hits.p);
    uint64_t* sorted = static_cast<uint64_t*>(ctx->d_hits2.p);
    size_t tmp_bytes = 0;
    FX_CUDA(cub::DeviceSegmentedSort::SortKeys(nullptr, tmp_bytes, keys, sorted, int(used), int(n_q), d_seg, d_end, ctx->stream));
    FX_TRY(ctx->d_cub.ensure(std::max<size_t>(tmp_bytes, 1)));
    FX_CUDA(cub::DeviceSegmentedSort::SortKeys(ctx->d_cub.p, tmp_bytes, keys, sorted, int(used), int(n_q), d_seg, d_end, ctx->stream));
    FX_TRY(ctx->d_rows.ensure(size_t(total) * 8));
    FX_TRY(ctx->d_dist.ensure(size_t(total) * 4));
    fx::range_gather_kernel<<<int(n_q), 256, 0, ctx->stream>>>(sorted, d_seg, d_off, c->row_base,
                                                              static_cast<int64_t*>(ctx->d_rows.p), static_cast<float*>(ctx->d_dist.p));
    FX_CUDA(cudaGetLastError());
    ctx->launches += 2; c->stats.kernel_launches += 2;   // (the sort: counted as one)
  }
  FX_CUDA(cudaEventRecord(ctx->ev_stop, ctx->stream));
  FX_TRY(ctx->h_rows.ensure(size_t(total) * 8));
  FX_TRY(ctx->h_dist.ensure(size_t(total) * 4));
  FX_CUDA(cudaMemcpyAsync(ctx->h_rows.p, ctx->d_rows.p, size_t(total) * 8, cudaMemcpyDeviceToHost, ctx->stream));
  FX_CUDA(cudaMemcpyAsync(ctx->h_dist.p, ctx->d_dist.p, size_t(total) * 4, cudaMemcpyDeviceToHost, ctx->stream));
  FX_CUDA(cudaStreamSynchronize(ctx->stream));
  std::memcpy(out_rows, ctx->h_rows.p, size_t(total) * 8);
  std::memcpy(out_dist, ctx->h_dist.p, size_t(total) * 4);
  search_account(c, run);
  return FX_OK;
}

// ----------------------------------------------------------------------------------------
// codebook training: one epoch of mini-batch k-means per call (DESIGN.md §4.11; csrc/kmeans.cuh)
// ----------------------------------------------------------------------------------------
// Staging buffer on the training device when the rows span several devices (two of them, filled alternately).
constexpr size_t TRAIN_STAGE_BYTES = size_t(256) << 20;

namespace {
// Per-call device memory and events of fx_train_codebooks, released on every return path after the streams drain.
struct TrainScratch {
  struct Alloc { int device; void* p; };
  struct Event { int device; cudaEvent_t e; };
  std::vector<Alloc> allocs;
  std::vector<Event> events;
  std::vector<std::pair<int, cudaStream_t>> streams;
  ~TrainScratch() {
    for (auto& s : streams) { cudaSetDevice(s.first); cudaStreamSynchronize(s.second); }
    for (auto& a : allocs) { cudaSetDevice(a.device); cudaFree(a.p); }
    for (auto& e : events) { cudaSetDevice(e.device); cudaEventDestroy(e.e); }
    cudaGetLastError();
  }
  template <typename T>
  int alloc(int device, size_t count, T** out) {
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T));
    if (e != cudaSuccess) {
      cudaGetLastError();
      return fail(FX_ENOMEM, "fx_train_codebooks: cudaMalloc(%zu) on device %d failed: %s", count * sizeof(T), device,
                  cudaGetErrorString(e));
    }
    allocs.push_back({device, p});
    *out = static_cast<T*>(p);
    return FX_OK;
  }
  int event(int device, cudaEvent_t* out) {
    FX_CUDA(cudaEventCreateWithFlags(out, cudaEventDisableTiming));
    events.push_back({device, *out});
    return FX_OK;
  }
};
}  // namespace

extern "C" int fx_train_codebooks(fx_corpus* const* shards, int32_t n_shards, int32_t metric, int32_t n_books, int32_t k,
                                  int32_t batch, const int64_t* positions, int64_t n_steps, float* books) {
  if (!shards || !books || (n_steps > 0 && !positions)) return fail(FX_EINVAL, "fx_train_codebooks: NULL argument");
  if (n_shards < 1 || n_books < 1 || k < 1 || batch < 1 || n_steps < 0)
    return fail(FX_EINVAL, "fx_train_codebooks: n_shards, n_books, k and batch must be >= 1 and n_steps >= 0");
  if (metric < 0 || metric > 2) return fail(FX_EINVAL, "fx_train_codebooks: unknown metric %d", metric);
  if (n_books > 65535) return fail(FX_EUNSUP, "fx_train_codebooks: at most 65535 codebooks");
  std::vector<std::unique_ptr<Lease>> leases;
  for (int i = 0; i < n_shards; ++i) {
    leases.emplace_back(new Lease(shards[i]));
    if (!leases.back()->ok) return fail(FX_EINVAL, "fx_train_codebooks: shard %d is not a live corpus handle", i);
    if (!shards[i]->finalized) return fail(FX_ESTATE, "fx_train_codebooks: shard %d is not finalized", i);
    if (shards[i]->dim != shards[0]->dim)
      return fail(FX_EINVAL, "fx_train_codebooks: shard %d has dim %d, shard 0 has %d", i, shards[i]->dim, shards[0]->dim);
    if (i > 0 && shards[i]->row_base != shards[i - 1]->row_base + shards[i - 1]->n)
      return fail(FX_EINVAL, "fx_train_codebooks: shards must hold contiguous row ranges in order (shard %d starts at %lld, expected %lld)",
                  i, (long long)shards[i]->row_base, (long long)(shards[i - 1]->row_base + shards[i - 1]->n));
  }
  const int dim = shards[0]->dim;
  const int64_t pitch = shards[0]->pitch;
  const int64_t lo = shards[0]->row_base, hi = shards[n_shards - 1]->row_base + shards[n_shards - 1]->n;
  const int64_t per_step = int64_t(n_books) * batch;
  if (per_step > (int64_t(1) << 30) || int64_t(k) * dim > (int64_t(1) << 40))
    return fail(FX_EUNSUP, "fx_train_codebooks: n_books * batch or k * dim too large");
  for (int64_t s = 0; s < n_steps; ++s) {
    const int64_t* ps = positions + s * per_step;
    for (int64_t t = 0; t < per_step; ++t) {
      if (ps[t] < lo || ps[t] >= hi)
        return fail(FX_EINVAL, "fx_train_codebooks: position %lld of step %lld is outside the shards' rows [%lld, %lld)",
                    (long long)ps[t], (long long)s, (long long)lo, (long long)hi);
      if (t > 0 && ps[t] < ps[t - 1])
        return fail(FX_EINVAL, "fx_train_codebooks: positions of step %lld are not ascending", (long long)s);
    }
  }
  if (n_steps == 0) return FX_OK;

  // every distinct context locked once, in address order (two shards may share a context)
  std::vector<fx_ctx*> ctxs;
  for (int i = 0; i < n_shards; ++i) ctxs.push_back(shards[i]->ctx);
  std::sort(ctxs.begin(), ctxs.end());
  ctxs.erase(std::unique(ctxs.begin(), ctxs.end()), ctxs.end());
  std::vector<std::unique_lock<std::mutex>> locks;
  for (fx_ctx* x : ctxs) locks.emplace_back(x->mu);

  fx_corpus* c0 = shards[0];
  fx_ctx* ctx = c0->ctx;
  TrainScratch scratch;
  int64_t launches = 0;
  const size_t book_floats = size_t(n_books) * k * dim;
  FX_TRY(bind(ctx));
  scratch.streams.push_back({ctx->device, ctx->stream});
  fx::KmParams p{};
  FX_TRY(scratch.alloc(ctx->device, book_floats, &p.books));
  FX_TRY(scratch.alloc(ctx->device, size_t(per_step), &p.keys));
  FX_TRY(scratch.alloc(ctx->device, size_t(per_step), &p.xx));
  FX_TRY(scratch.alloc(ctx->device, size_t(n_books) * (k + 1), &p.off));
  FX_TRY(scratch.alloc(ctx->device, size_t(n_books) * k, &p.cur));
  FX_TRY(scratch.alloc(ctx->device, size_t(per_step), &p.order));
  int64_t* d_idx = nullptr;
  FX_TRY(scratch.alloc(ctx->device, size_t(n_steps * per_step), &d_idx));
  const size_t upd_smem = size_t(dim) * sizeof(double);
  FX_CUDA(cudaFuncSetAttribute(fx::km_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(upd_smem)));
  FX_CUDA(cudaMemcpyAsync(p.books, books, book_floats * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  FX_CUDA(cudaMemsetAsync(p.keys, 0xff, size_t(per_step) * sizeof(unsigned long long), ctx->stream));
  p.pitch = pitch; p.dim = dim; p.k = k; p.batch = batch; p.metric = metric;

  // assignment grid: row tiles x codeword ranges x codebooks, codeword ranges split until the grid fills the device
  const int row_tiles = (batch + fx::KM_TR - 1) / fx::KM_TR, cw_tiles = (k + fx::KM_TC - 1) / fx::KM_TC;
  const int64_t rows_blocks = int64_t(row_tiles) * n_books;
  const int splits = int(std::min<int64_t>(cw_tiles, std::max<int64_t>(1, (2 * int64_t(ctx->sm_count) + rows_blocks - 1) / rows_blocks)));
  p.cw_per_block = ((cw_tiles + splits - 1) / splits) * fx::KM_TC;
  const dim3 assign_grid(row_tiles, (k + p.cw_per_block - 1) / p.cw_per_block, n_books);
  auto run_steps = [&](int64_t s0, int64_t s1, const float* X) -> int {
    p.X = X;
    for (int64_t s = s0; s < s1; ++s) {
      p.idx = d_idx + s * per_step;
      fx::km_assign_kernel<<<assign_grid, fx::KM_THREADS, 0, ctx->stream>>>(p);
      fx::km_bucket_kernel<<<n_books, fx::KM_BUCKET_THREADS, 0, ctx->stream>>>(p);
      fx::km_update_kernel<<<dim3(k, n_books), fx::KM_UPDATE_THREADS, upd_smem, ctx->stream>>>(p);
      FX_CUDA(cudaGetLastError());
      launches += 3;
    }
    return FX_OK;
  };

  std::vector<int64_t> idx(size_t(n_steps * per_step));
  if (n_shards == 1) {
    // one shard: the steps read the sample rows straight from its rows
    for (size_t t = 0; t < idx.size(); ++t) idx[t] = positions[t] - lo;
    FX_CUDA(cudaMemcpyAsync(d_idx, idx.data(), idx.size() * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
    FX_TRY(run_steps(0, n_steps, c0->X));
  } else {
    // several shards: per chunk of steps, every shard gathers its part of the chunk's sample rows (in position order)
    // and copies it into one of two staging buffers on shard 0's device; the steps read the rows from there
    const int64_t chunk = std::max<int64_t>(1, int64_t(TRAIN_STAGE_BYTES / (size_t(per_step) * pitch * sizeof(float))));
    const int64_t n_chunks = (n_steps + chunk - 1) / chunk;
    std::vector<std::vector<int64_t>> rows(n_shards);          // local rows each shard gathers, chunk after chunk
    std::vector<int64_t> cnt(size_t(n_chunks) * n_shards, 0);  // rows of shard i in chunk q
    std::vector<int64_t> at(n_shards);
    auto shard_of = [&](int64_t pos) {
      int i = 0;
      while (i + 1 < n_shards && pos >= shards[i + 1]->row_base) ++i;
      return i;
    };
    for (int64_t q = 0; q < n_chunks; ++q) {
      const int64_t t0 = q * chunk * per_step, t1 = std::min(n_steps, (q + 1) * chunk) * per_step;
      int64_t* cq = cnt.data() + q * n_shards;
      for (int64_t t = t0; t < t1; ++t) cq[shard_of(positions[t])]++;
      for (int i = 0, o = 0; i < n_shards; o += int(cq[i]), ++i) at[i] = o;
      for (int64_t t = t0; t < t1; ++t) {   // idx: the row's slot in the chunk's staging buffer, shard after shard
        const int i = shard_of(positions[t]);
        idx[size_t(t)] = at[i]++;
        rows[i].push_back(positions[t] - shards[i]->row_base);
      }
    }
    float* stage[2] = {nullptr, nullptr};
    const size_t stage_rows = size_t(std::min(chunk, n_steps) * per_step);
    FX_TRY(scratch.alloc(ctx->device, stage_rows * pitch, &stage[0]));
    FX_TRY(scratch.alloc(ctx->device, n_chunks > 1 ? stage_rows * pitch : 0, &stage[1]));
    cudaEvent_t consumed[2];
    FX_TRY(scratch.event(ctx->device, &consumed[0]));
    FX_TRY(scratch.event(ctx->device, &consumed[1]));
    std::vector<int64_t*> d_rows(n_shards, nullptr);
    std::vector<float*> gbuf(n_shards, nullptr);
    std::vector<cudaEvent_t> copied(n_shards, nullptr);
    for (int i = 0; i < n_shards; ++i) {
      fx_ctx* xi = shards[i]->ctx;
      int64_t most = 0;
      for (int64_t q = 0; q < n_chunks; ++q) most = std::max(most, cnt[size_t(q * n_shards + i)]);
      FX_TRY(bind(xi));
      scratch.streams.push_back({xi->device, xi->stream});
      FX_TRY(scratch.alloc(xi->device, rows[i].size(), &d_rows[i]));
      FX_CUDA(cudaMemcpyAsync(d_rows[i], rows[i].data(), rows[i].size() * sizeof(int64_t), cudaMemcpyHostToDevice, xi->stream));
      if (i > 0) {
        FX_TRY(scratch.alloc(xi->device, size_t(most) * pitch, &gbuf[i]));
        FX_TRY(scratch.event(xi->device, &copied[i]));
      }
    }
    FX_TRY(bind(ctx));
    FX_CUDA(cudaMemcpyAsync(d_idx, idx.data(), idx.size() * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
    std::vector<int64_t> done(n_shards, 0);   // rows of shard i gathered so far
    for (int64_t q = 0; q < n_chunks; ++q) {
      const int b = int(q & 1);
      int64_t slot = 0;
      for (int i = 0; i < n_shards; ++i) {
        const int64_t m = cnt[size_t(q * n_shards + i)];
        if (m == 0) continue;
        fx_ctx* xi = shards[i]->ctx;
        FX_TRY(bind(xi));
        const int blocks = int(std::min<int64_t>(m, 4 * int64_t(xi->sm_count)));
        if (i == 0) {
          fx::km_gather_kernel<<<blocks, 256, 0, xi->stream>>>(shards[i]->X, pitch, d_rows[i] + done[i], m,
                                                               stage[b] + slot * pitch);
          FX_CUDA(cudaGetLastError());
        } else {
          if (q >= 2) FX_CUDA(cudaStreamWaitEvent(xi->stream, consumed[b], 0));
          fx::km_gather_kernel<<<blocks, 256, 0, xi->stream>>>(shards[i]->X, pitch, d_rows[i] + done[i], m, gbuf[i]);
          FX_CUDA(cudaGetLastError());
          FX_CUDA(cudaMemcpyPeerAsync(stage[b] + slot * pitch, ctx->device, gbuf[i], xi->device,
                                      size_t(m) * pitch * sizeof(float), xi->stream));
          FX_CUDA(cudaEventRecord(copied[i], xi->stream));
          FX_TRY(bind(ctx));
          FX_CUDA(cudaStreamWaitEvent(ctx->stream, copied[i], 0));
        }
        launches++;
        done[i] += m;
        slot += m;
      }
      FX_TRY(bind(ctx));
      FX_TRY(run_steps(q * chunk, std::min(n_steps, (q + 1) * chunk), stage[b]));
      FX_CUDA(cudaEventRecord(consumed[b], ctx->stream));
    }
  }
  FX_CUDA(cudaMemcpyAsync(books, p.books, book_floats * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  FX_CUDA(cudaStreamSynchronize(ctx->stream));
  ctx->launches += launches;
  c0->stats.kernel_launches += launches;
  return FX_OK;
}

extern "C" int fx_debug_scores(fx_corpus* c, const float* queries, int64_t n_q, int32_t metric, float* out_scores) {
  if (!queries || !out_scores) return fail(FX_EINVAL, "fx_debug_scores: NULL argument");
  FX_LEASE(c, "fx_debug_scores");
  if (!c->finalized) return fail(FX_ESTATE, "fx_debug_scores: corpus is not finalized");
  if (n_q < 1 || metric < 0 || metric > 2) return fail(FX_EINVAL, "fx_debug_scores: bad arguments");
  fx_ctx* ctx = c->ctx;
  std::lock_guard<std::mutex> lock(ctx->mu);
  FX_TRY(bind(ctx));
  if (!fx::tc_supported(&ctx->tc, &c->tc, c->n, c->dim, 10, int(n_q)))
    return fail(FX_EUNSUP, "fx_debug_scores: the tensor-core path does not cover this shard");
  const size_t q_bytes = size_t(n_q) * c->dim * sizeof(float);
  FX_TRY(ctx->d_q.ensure(q_bytes));
  FX_TRY(ctx->d_rows.ensure(size_t(n_q) * 10 * sizeof(int64_t)));
  FX_TRY(ctx->d_dist.ensure(size_t(n_q) * 10 * sizeof(float) + 128 * 256 * sizeof(float) + 256));
  FX_CUDA(cudaMemcpyAsync(ctx->d_q.p, queries, q_bytes, cudaMemcpyHostToDevice, ctx->stream));
  float* d_dbg = reinterpret_cast<float*>(static_cast<char*>(ctx->d_dist.p) + ((size_t(n_q) * 10 * sizeof(float) + 255) & ~size_t(255)));
  FX_CUDA(cudaMemsetAsync(d_dbg, 0, 128 * 256 * sizeof(float), ctx->stream));
  fx::TcSearch s{};
  s.X = c->X; s.hx = c->hx; s.rx = c->rx; s.n_rows = c->n; s.dim = c->dim; s.pitch = c->pitch;
  s.row_base = c->row_base; s.max_norm = c->max_norm; s.Q = static_cast<const float*>(ctx->d_q.p); s.n_q = int(n_q);
  s.metric = metric; s.k = 10; s.certify = false; s.out_rows = static_cast<int64_t*>(ctx->d_rows.p);
  s.out_dist = static_cast<float*>(ctx->d_dist.p); s.stream = ctx->stream; s.ev_k0 = ctx->ev_k0; s.ev_k1 = ctx->ev_k1;
  s.dbg = d_dbg; s.tau_fixed = nullptr;
  // operand: FENIX_INT8=1 and cosine - the int8 filter's upper bounds; FENIX_DEBUG_BF16 - the bf16 filter; else TF32
  const bool i8 = metric == 1 && ctx->tc.knobs.int8 > 0 && ensure_i8_shadow(c);
  const bool b16 = !i8 && ctx->tc.knobs.debug_bf16 && ((metric == 1 && ensure_norm_shadow(c)) || ensure_plain_shadow(c));
  FX_TRY(configure_filter(c, metric, i8 ? 2 : (b16 ? 1 : 0), nullptr, &s));
  const fx::TcLaunch L = fx::tc_prepare(&ctx->tc, s);
  FX_TRY(ctx->d_tc.ensure(L.scratch_bytes));
  std::string err; int launched = 0;
  if (!fx::tc_search(&ctx->tc, &c->tc, s, L, ctx->d_tc.p, &launched, &err)) return fail(FX_ECUDA, "fx_debug_scores: %s", err.c_str());
  FX_CUDA(cudaMemcpyAsync(out_scores, d_dbg, 128 * 256 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  FX_CUDA(cudaStreamSynchronize(ctx->stream));
  return FX_OK;
}

// ----------------------------------------------------------------------------------------
// merge of per-shard lists
// ----------------------------------------------------------------------------------------
// Lists are [n_q][k] each (rows int64, distances f32), sorted by (distance, row), pads last; list l sits
// l * rows_stride / l * dist_stride bytes into the two arrays.
static int enqueue_merge(fx_ctx* ctx, const int64_t* d_rows, const float* d_dist, int n_lists, int64_t n_q, int k,
                         int64_t rows_stride, int64_t dist_stride, int64_t* d_out_rows, float* d_out_dist) {
  const int64_t total = int64_t(n_lists) * k;
  // the lists arrive sorted: ranking every entry by binary searches over the other lists beats re-sorting them in shared
  // memory from ~128 candidates per query on (C4's exchange, 8 x 100 per query: 0.59 -> 0.35 ms)
  if (total < 128) {
    const int n_sort = next_pow2(std::max(int(total), 2));
    fx::merge_pairs_kernel<<<unsigned(n_q), 256, size_t(n_sort) * 12, ctx->stream>>>(
        d_rows, d_dist, n_lists, n_q, k, n_sort, rows_stride, dist_stride, d_out_rows, d_out_dist);
  } else {
    fx::merge_rank_kernel<<<unsigned(n_q), 256, 0, ctx->stream>>>(d_rows, d_dist, n_lists, n_q, k, rows_stride, dist_stride,
                                                                 d_out_rows, d_out_dist);
  }
  FX_CUDA(cudaGetLastError());
  ctx->launches++;
  return FX_OK;
}

extern "C" int fx_merge_topk(fx_ctx* ctx, const int64_t* d_rows, const float* d_dist, int32_t n_lists,
                             int64_t n_q, int32_t k, int64_t* d_out_rows, float* d_out_dist) {
  if (!ctx) return fail(FX_EINVAL, "fx_merge_topk: ctx is NULL");
  if (n_lists < 1 || n_q < 0 || k < 1) return fail(FX_EINVAL, "fx_merge_topk: bad sizes (lists=%d, n_q=%lld, k=%d)", n_lists, (long long)n_q, k);
  if (n_q == 0) return FX_OK;
  if (!d_rows || !d_dist || !d_out_rows || !d_out_dist) return fail(FX_EINVAL, "fx_merge_topk: NULL buffer");
  std::lock_guard<std::mutex> lock(ctx->mu);
  FX_TRY(bind(ctx));
  // list-major inputs: list l starts l * n_q * k entries into each array
  FX_TRY(enqueue_merge(ctx, d_rows, d_dist, n_lists, n_q, k, n_q * int64_t(k) * 8, n_q * int64_t(k) * 4, d_out_rows, d_out_dist));
  FX_CUDA(cudaStreamSynchronize(ctx->stream));
  return FX_OK;
}

// ----------------------------------------------------------------------------------------
// multi-GPU: NCCL communicator owned by the library, sharded search with one host synchronisation
// ----------------------------------------------------------------------------------------
// NCCL comes from the process (torch ships libnccl.so.2; the Python binding pre-loads it for a bare server): nothing
// links against it and the header is not needed - the few entry points used here have had a stable ABI since NCCL 2.0.
namespace {
typedef struct ncclComm* ncclComm_t;
struct ncclUniqueId { char internal[128]; };
static_assert(sizeof(ncclUniqueId) == FX_COMM_ID_BYTES, "ncclUniqueId is 128 bytes");
constexpr int kNcclInt8 = 0;   // ncclInt8 / ncclChar

struct NcclApi {
  void* handle = nullptr;
  int (*GetUniqueId)(ncclUniqueId*) = nullptr;
  int (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  int (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  int (*CommDestroy)(ncclComm_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  std::string error;
};

NcclApi* nccl_api() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    const char* name = std::getenv("FENIX_NCCL_LIB");
    api.handle = dlopen(name && *name ? name : "libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!api.handle) {
      const char* why = dlerror();
      api.error = std::string("cannot load NCCL (") + (why ? why : "?") + "); set FENIX_NCCL_LIB to the path of libnccl.so.2";
      return;
    }
    auto sym = [&](const char* s) { void* p = dlsym(api.handle, s); if (!p && api.error.empty()) api.error = std::string("NCCL symbol missing: ") + s; return p; };
    api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
    api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
    api.CommInitAll = reinterpret_cast<decltype(api.CommInitAll)>(sym("ncclCommInitAll"));
    api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
    api.AllGather = reinterpret_cast<decltype(api.AllGather)>(sym("ncclAllGather"));
    api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
  });
  return &api;
}
}  // namespace

#define FX_NCCL(expr)                                                                             \
  do {                                                                                            \
    int _r = (expr);                                                                              \
    if (_r != 0) return fail(FX_ECUDA, "%s failed: %s", #expr, nccl_api()->GetErrorString ? nccl_api()->GetErrorString(_r) : "?"); \
  } while (0)

struct fx_comm {
  fx_ctx* ctx = nullptr;
  ncclComm_t comm = nullptr;
  int world = 1, rank = 0;
};

static int nccl_ready() {
  NcclApi* api = nccl_api();
  if (!api->error.empty() || !api->handle) return fail(FX_EUNSUP, "multi-GPU search: %s", api->error.c_str());
  return FX_OK;
}

extern "C" int fx_comm_unique_id(void* out_id) {
  if (!out_id) return fail(FX_EINVAL, "fx_comm_unique_id: NULL argument");
  FX_TRY(nccl_ready());
  ncclUniqueId id;
  FX_NCCL(nccl_api()->GetUniqueId(&id));
  std::memcpy(out_id, &id, sizeof id);
  return FX_OK;
}

extern "C" int fx_comm_init_rank(fx_ctx* ctx, const void* id, int32_t world, int32_t rank, fx_comm** out) {
  if (!ctx || !id || !out) return fail(FX_EINVAL, "fx_comm_init_rank: NULL argument");
  *out = nullptr;
  if (world < 1 || rank < 0 || rank >= world) return fail(FX_EINVAL, "fx_comm_init_rank: bad rank %d of %d", rank, world);
  if (world + 1 > H_WORDS) return fail(FX_EUNSUP, "fx_comm_init_rank: at most %d ranks", H_WORDS - 1);
  FX_TRY(nccl_ready());
  std::lock_guard<std::mutex> lock(ctx->mu);
  FX_TRY(bind(ctx));
  ncclUniqueId uid;
  std::memcpy(&uid, id, sizeof uid);
  fx_comm* cm = new (std::nothrow) fx_comm();
  if (!cm) return fail(FX_ENOMEM, "fx_comm_init_rank: out of host memory");
  cm->ctx = ctx; cm->world = world; cm->rank = rank;
  int r = nccl_api()->CommInitRank(&cm->comm, world, uid, rank);
  if (r != 0) { delete cm; return fail(FX_ECUDA, "ncclCommInitRank failed: %s", nccl_api()->GetErrorString(r)); }
  *out = cm;
  return FX_OK;
}

extern "C" int fx_comm_destroy(fx_comm* cm) {
  if (!cm) return fail(FX_EINVAL, "fx_comm_destroy: comm is NULL");
  {
    std::lock_guard<std::mutex> lock(cm->ctx->mu);
    cudaSetDevice(cm->ctx->device);
    cudaStreamSynchronize(cm->ctx->stream);
    if (cm->comm && nccl_api()->CommDestroy) nccl_api()->CommDestroy(cm->comm);
  }
  delete cm;
  return FX_OK;
}

// Per-rank body of a sharded search (ctx->mu held, device bound). Collective: every rank of the communicator runs it
// with the same (n_q, metric, k, precision). `queries`: host (whole batch; this rank uploads its slice) or device
// (whole batch). Outputs host, device or null.
static int sharded_search_locked(fx_corpus* c, fx_comm* cm, const float* queries, bool q_on_device, int64_t n_q, int metric,
                                 int k, int precision, const uint8_t* row_mask, bool mask_on_device, int64_t* out_rows,
                                 float* out_dist, bool out_on_device) {
  fx_ctx* ctx = c->ctx;
  NcclApi* api = nccl_api();
  NvtxRange nvtx("fenix:search_sharded");
  const int W = cm->world, rank = cm->rank;
  const int64_t per = (n_q + W - 1) / W;                    // queries per rank slice (the last slices may be short / empty)
  const size_t row_bytes = size_t(c->dim) * sizeof(float);
  // ---- queries: upload 1/W of the batch, all-gather the slices over NVLink ----
  const float* d_q = queries;
  if (!q_on_device) {
    FX_TRY(ctx->d_q.ensure(size_t(per) * W * row_bytes));
    char* qall = static_cast<char*>(ctx->d_q.p);
    const int64_t lo = std::min<int64_t>(n_q, rank * per), hi = std::min<int64_t>(n_q, lo + per);
    if (hi > lo) {
      const char* src = reinterpret_cast<const char*>(queries) + size_t(lo) * row_bytes;
      const size_t bytes = size_t(hi - lo) * row_bytes;
      if (!is_pinned(queries)) {
        FX_TRY(ctx->h_q.ensure(bytes));
        std::memcpy(ctx->h_q.p, src, bytes);
        src = static_cast<const char*>(ctx->h_q.p);
      }
      FX_CUDA(cudaMemcpyAsync(qall + size_t(lo) * row_bytes, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    if (W > 1) FX_NCCL(api->AllGather(qall + size_t(rank) * per * row_bytes, qall, size_t(per) * row_bytes, kNcclInt8, cm->comm, ctx->stream));
    d_q = reinterpret_cast<const float*>(qall);
  }
  const uint8_t* d_mask = nullptr;
  if (row_mask && c->n > 0) {
    if (mask_on_device) d_mask = row_mask;
    else {
      FX_TRY(ctx->d_mask.ensure(size_t(c->n)));
      FX_CUDA(cudaMemcpyAsync(ctx->d_mask.p, row_mask, size_t(c->n), cudaMemcpyHostToDevice, ctx->stream));
      d_mask = static_cast<const uint8_t*>(ctx->d_mask.p);
    }
  }
  // ---- exchange buffer: W slots of [rows n_q*k int64][distances n_q*k f32][header 16 B]; the shard search writes
  // this rank's slot in place and the all-gather is in place too ----
  const size_t nk = size_t(n_q) * k;
  const size_t hdr_off = (nk * 12 + 15) & ~size_t(15), slot = hdr_off + 16;
  FX_TRY(ctx->d_xchg.ensure(slot * W));
  char* xb = static_cast<char*>(ctx->d_xchg.p);
  char* mine = xb + slot * rank;
  int64_t* my_rows = reinterpret_cast<int64_t*>(mine);
  float* my_dist = reinterpret_cast<float*>(mine + nk * 8);
  const bool want_out = out_rows != nullptr;
  int64_t* d_res_rows = nullptr; float* d_res_dist = nullptr;
  if (want_out) {
    if (out_on_device) { d_res_rows = out_rows; d_res_dist = out_dist; }
    else {
      FX_TRY(ctx->d_rows.ensure(nk * 8));
      FX_TRY(ctx->d_dist.ensure(nk * 4));
      d_res_rows = static_cast<int64_t*>(ctx->d_rows.p); d_res_dist = static_cast<float*>(ctx->d_dist.p);
    }
  }
  const bool direct = want_out && !out_on_device && is_pinned(out_rows) && is_pinned(out_dist);
  void* h_rows = out_rows; void* h_dist = out_dist;
  if (want_out && !out_on_device && !direct) {
    FX_TRY(ctx->h_rows.ensure(nk * 8));
    FX_TRY(ctx->h_dist.ensure(nk * 4));
    h_rows = ctx->h_rows.p; h_dist = ctx->h_dist.p;
  }

  SearchRun run;
  FX_TRY(search_enqueue(c, d_q, n_q, metric, k, precision, d_mask, my_rows, my_dist, &run));
  for (int attempt = 0; attempt < 2; ++attempt) {
    // header word 0: queries of this shard whose result is not final yet (first exchange only)
    if (attempt == 0 && run.tc && run.s.certify)
      FX_CUDA(cudaMemcpyAsync(mine + hdr_off, fx::tc_flag_count(ctx->d_tc.p), sizeof(int), cudaMemcpyDeviceToDevice, ctx->stream));
    else
      FX_CUDA(cudaMemsetAsync(mine + hdr_off, 0, 16, ctx->stream));
    NvtxRange nvtx_x("fenix:exchange (all-gather + merge)");
    FX_CUDA(cudaEventRecord(ctx->ev_x0, ctx->stream));
    if (W > 1) FX_NCCL(api->AllGather(mine, xb, slot, kNcclInt8, cm->comm, ctx->stream));
    if (want_out) {
      FX_TRY(enqueue_merge(ctx, reinterpret_cast<const int64_t*>(xb), reinterpret_cast<const float*>(xb + nk * 8), W, n_q, k,
                           int64_t(slot), int64_t(slot), d_res_rows, d_res_dist));
    }
    FX_CUDA(cudaEventRecord(ctx->ev_x1, ctx->stream));
    if (want_out && !out_on_device) {
      FX_CUDA(cudaMemcpyAsync(h_rows, d_res_rows, nk * 8, cudaMemcpyDeviceToHost, ctx->stream));
      FX_CUDA(cudaMemcpyAsync(h_dist, d_res_dist, nk * 4, cudaMemcpyDeviceToHost, ctx->stream));
    }
    // every rank's header word, strided out of the gathered slots -> pinned h_word[1 .. W]
    FX_CUDA(cudaMemcpy2DAsync(ctx->h_word + 1, sizeof(int), xb + hdr_off, slot, sizeof(int), size_t(W), cudaMemcpyDeviceToHost, ctx->stream));
    FX_CUDA(cudaStreamSynchronize(ctx->stream));   // the ONE synchronisation of the common path
    if (attempt == 1) break;
    bool any = false;
    for (int r = 0; r < W; ++r) any = any || ctx->h_word[1 + r] != 0;
    if (!any) break;
    // some shard's certificate failed for some query: those ranks repair their lists, then EVERY rank repeats the exchange
    bool changed = false;
    FX_TRY(search_settle(c, &run, &changed));
  }
  if (want_out && !out_on_device && !direct) {
    std::memcpy(out_rows, ctx->h_rows.p, nk * 8);
    std::memcpy(out_dist, ctx->h_dist.p, nk * 4);
  }
  search_account(c, run);
  float xms = 0.f;
  cudaEventElapsedTime(&xms, ctx->ev_x0, ctx->ev_x1);
  c->stats.last_exchange_ms = xms;
  return FX_OK;
}

extern "C" int fx_search_sharded(fx_corpus* c, fx_comm* cm, const float* queries, int64_t n_q, int32_t metric, int32_t k,
                                 int32_t precision, const uint8_t* row_mask, int64_t* out_rows, float* out_dist) {
  if (!cm) return fail(FX_EINVAL, "fx_search_sharded: comm is NULL");
  FX_LEASE(c, "fx_search_sharded");
  FX_TRY(check_search_args(c, queries, n_q, metric, k, precision, out_rows, out_dist, false));
  if (cm->ctx != c->ctx) return fail(FX_EINVAL, "fx_search_sharded: corpus and communicator live on different contexts");
  if (n_q == 0) return FX_OK;
  fx_ctx* ctx = c->ctx;
  std::lock_guard<std::mutex> lock(ctx->mu);
  FX_TRY(bind(ctx));
  return sharded_search_locked(c, cm, queries, false, n_q, metric, k, precision, row_mask, false, out_rows, out_dist, false);
}

extern "C" int fx_search_sharded_device(fx_corpus* c, fx_comm* cm, const float* d_queries, int64_t n_q, int32_t metric,
                                        int32_t k, int32_t precision, const uint8_t* d_row_mask, int64_t* d_out_rows,
                                        float* d_out_dist) {
  if (!cm) return fail(FX_EINVAL, "fx_search_sharded_device: comm is NULL");
  FX_LEASE(c, "fx_search_sharded_device");
  FX_TRY(check_search_args(c, d_queries, n_q, metric, k, precision, d_out_rows, d_out_dist, false));
  if (cm->ctx != c->ctx) return fail(FX_EINVAL, "fx_search_sharded_device: corpus and communicator live on different contexts");
  if (n_q == 0) return FX_OK;
  fx_ctx* ctx = c->ctx;
  std::lock_guard<std::mutex> lock(ctx->mu);
  FX_TRY(bind(ctx));
  return sharded_search_locked(c, cm, d_queries, true, n_q, metric, k, precision, d_row_mask, true, d_out_rows, d_out_dist, true);
}

// ----------------------------------------------------------------------------------------
// one process, several devices: a context, a communicator and a worker thread per device
// ----------------------------------------------------------------------------------------
struct GroupJob {
  fx_corpus* const* shards = nullptr;
  const float* queries = nullptr; int64_t n_q = 0; int metric = 0, k = 0, precision = 0;
  const uint8_t* row_mask = nullptr; int64_t* out_rows = nullptr; float* out_dist = nullptr;
};

struct fx_group {
  int n = 0;
  std::vector<fx_ctx*> ctxs;
  std::vector<fx_comm*> comms;
  std::vector<std::thread> workers;
  std::mutex search_mu;            // collective searches on a group serialise
  std::mutex mu;                   // job hand-off
  std::condition_variable cv_go, cv_done;
  uint64_t generation = 0;
  int pending = 0;
  bool quit = false;
  GroupJob job;
  std::vector<int> rc;
  std::vector<std::string> err;
};

static void group_worker(fx_group* g, int i) {
  uint64_t seen = 0;
  cudaSetDevice(g->ctxs[i]->device);
  for (;;) {
    GroupJob job;
    {
      std::unique_lock<std::mutex> lock(g->mu);
      g->cv_go.wait(lock, [&] { return g->quit || g->generation != seen; });
      if (g->quit) return;
      seen = g->generation;
      job = g->job;
    }
    fx_corpus* c = job.shards[i];
    const uint8_t* mask = job.row_mask ? job.row_mask + (c->row_base - job.shards[0]->row_base) : nullptr;
    int rc = fx_search_sharded(c, g->comms[i], job.queries, job.n_q, job.metric, job.k, job.precision, mask,
                               i == 0 ? job.out_rows : nullptr, i == 0 ? job.out_dist : nullptr);
    {
      std::lock_guard<std::mutex> lock(g->mu);
      g->rc[i] = rc;
      if (rc != FX_OK) g->err[i] = g_last_error;   // thread-local of the worker: hand it to the caller
      if (--g->pending == 0) g->cv_done.notify_all();
    }
  }
}

extern "C" int fx_group_create(const int32_t* devices, int32_t n_devices, fx_group** out) {
  if (!devices || !out) return fail(FX_EINVAL, "fx_group_create: NULL argument");
  *out = nullptr;
  if (n_devices < 1 || n_devices + 1 > H_WORDS) return fail(FX_EINVAL, "fx_group_create: bad device count %d", n_devices);
  for (int i = 0; i < n_devices; ++i)
    for (int j = 0; j < i; ++j)
      if (devices[i] == devices[j]) return fail(FX_EINVAL, "fx_group_create: device %d listed twice", devices[i]);
  fx_group* g = new (std::nothrow) fx_group();
  if (!g) return fail(FX_ENOMEM, "fx_group_create: out of host memory");
  g->n = n_devices;
  auto cleanup = [&]() {
    for (fx_comm* cm : g->comms) if (cm) { if (cm->comm && nccl_api()->CommDestroy) nccl_api()->CommDestroy(cm->comm); delete cm; }
    for (fx_ctx* c : g->ctxs) if (c) fx_shutdown(c);
    delete g;
  };
  for (int i = 0; i < n_devices; ++i) {
    fx_ctx* ctx = nullptr;
    int r = fx_init(devices[i], &ctx);
    if (r != FX_OK) { cleanup(); return r; }
    g->ctxs.push_back(ctx);
  }
  if (n_devices > 1) {
    int r = nccl_ready();
    if (r != FX_OK) { cleanup(); return r; }
    std::vector<ncclComm_t> comms(n_devices, nullptr);
    std::vector<int> devs(devices, devices + n_devices);
    int nr = nccl_api()->CommInitAll(comms.data(), n_devices, devs.data());
    if (nr != 0) { cleanup(); return fail(FX_ECUDA, "ncclCommInitAll failed: %s", nccl_api()->GetErrorString(nr)); }
    for (int i = 0; i < n_devices; ++i) {
      fx_comm* cm = new fx_comm();
      cm->ctx = g->ctxs[i]; cm->comm = comms[i]; cm->world = n_devices; cm->rank = i;
      g->comms.push_back(cm);
    }
    g->rc.assign(n_devices, FX_OK);
    g->err.assign(n_devices, std::string());
    for (int i = 0; i < n_devices; ++i) g->workers.emplace_back(group_worker, g, i);
  }
  *out = g;
  return FX_OK;
}

extern "C" int fx_group_size(fx_group* g) { return g ? g->n : fail(FX_EINVAL, "fx_group_size: group is NULL"); }
extern "C" fx_ctx* fx_group_ctx(fx_group* g, int32_t i) {
  if (!g || i < 0 || i >= g->n) { fail(FX_EINVAL, "fx_group_ctx: bad argument"); return nullptr; }
  return g->ctxs[i];
}

extern "C" int fx_group_search(fx_group* g, fx_corpus* const* shards, const float* queries, int64_t n_q, int32_t metric,
                               int32_t k, int32_t precision, const uint8_t* row_mask, int64_t* out_rows, float* out_dist) {
  if (!g || !shards) return fail(FX_EINVAL, "fx_group_search: NULL argument");
  if (n_q > 0 && (!queries || !out_rows || !out_dist)) return fail(FX_EINVAL, "fx_group_search: NULL buffer");
  if (n_q == 0) return FX_OK;
  std::vector<std::unique_ptr<Lease>> leases;
  for (int i = 0; i < g->n; ++i) {
    leases.emplace_back(new Lease(shards[i]));
    if (!leases.back()->ok) return fail(FX_EINVAL, "fx_group_search: shard %d is not a live corpus handle", i);
    if (shards[i]->ctx != g->ctxs[i]) return fail(FX_EINVAL, "fx_group_search: shard %d does not live on fx_group_ctx(g, %d)", i, i);
    if (i > 0 && shards[i]->row_base != shards[i - 1]->row_base + shards[i - 1]->n)
      return fail(FX_EINVAL, "fx_group_search: shards must hold contiguous row ranges in order (shard %d starts at %lld, expected %lld)",
                  i, (long long)shards[i]->row_base, (long long)(shards[i - 1]->row_base + shards[i - 1]->n));
  }
  if (g->n == 1) return fx_search(shards[0], queries, n_q, metric, k, precision, row_mask, out_rows, out_dist);
  std::lock_guard<std::mutex> serial(g->search_mu);
  {
    std::lock_guard<std::mutex> lock(g->mu);
    g->job = GroupJob{shards, queries, n_q, metric, k, precision, row_mask, out_rows, out_dist};
    g->pending = g->n;
    g->generation++;
  }
  g->cv_go.notify_all();
  {
    std::unique_lock<std::mutex> lock(g->mu);
    g->cv_done.wait(lock, [&] { return g->pending == 0; });
  }
  for (int i = 0; i < g->n; ++i)
    if (g->rc[i] != FX_OK) return fail(g->rc[i], "fx_group_search (device %d): %s", g->ctxs[i]->device, g->err[i].c_str());
  return FX_OK;
}

extern "C" int fx_group_destroy(fx_group* g) {
  if (!g) return fail(FX_EINVAL, "fx_group_destroy: group is NULL");
  {
    std::lock_guard<std::mutex> serial(g->search_mu);
    {
      std::lock_guard<std::mutex> lock(g->mu);
      g->quit = true;
    }
    g->cv_go.notify_all();
    for (std::thread& t : g->workers) t.join();
  }
  for (fx_comm* cm : g->comms) fx_comm_destroy(cm);
  for (fx_ctx* c : g->ctxs) fx_shutdown(c);
  delete g;
  return FX_OK;
}
