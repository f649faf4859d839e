// bbq_api.cu — host side of libbbq_b200.so: the C ABI declared in include/bbq_b200.h.
// Owns device memory, the stream and the launch sequence; no torch, no CPU fallback.
#include <cuda_runtime.h>
#include <atomic>
#include <dlfcn.h>
#include <nccl.h>  // types and prototypes only: the library is dlopen'ed on first use (bbq_comm_*), never linked

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/bbq_b200.h"
#include "bbq_kernels.cuh"
#include "bbq_mma.cuh"

using namespace bbqk;

// ------------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static thread_local int64_t g_err_vec = -1, g_err_pos = -1;

static int fail(int status, const std::string& msg, int64_t vec = -1, int64_t pos = -1) {
  g_err = msg;
  g_err_vec = vec;
  g_err_pos = pos;
  return status;
}

#define CU(expr)                                                                                   \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess) {                                                                       \
      const int _st = (_e == cudaErrorMemoryAllocation) ? BBQ_ERR_OOM : BBQ_ERR_CUDA;              \
      return fail(_st, std::string(#expr) + ": " + cudaGetErrorString(_e));                        \
    }                                                                                              \
  } while (0)

#define TRY(expr)                 \
  do {                            \
    const int _s = (expr);        \
    if (_s != BBQ_OK) return _s;  \
  } while (0)

static std::atomic<uint64_t> g_scratch_gen{0};  // bumped whenever any scratch buffer moves: a captured launch sequence holds its address
struct DevBuf {  // grow-only device scratch, freed with its owner (on the owner's device)
  void* p = nullptr;
  size_t cap = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() {
    if (p) cudaFree(p);
  }
  int reserve(size_t bytes) {
    if (bytes <= cap) return BBQ_OK;
    g_scratch_gen++;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    CU(cudaMalloc(&p, bytes));
    cap = bytes;
    return BBQ_OK;
  }
  template <class T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

struct bbq_ctx {
  int refs = 1;           // the handle itself + one per live index (destroy order must not matter to callers)
  bool destroyed = false;
  bbq_config cfg;
  int device = 0;
  cudaStream_t stream = nullptr;
  int sm_count = 148;
  uint64_t launches = 0;
  bbq_stats stats{};
  int force_path = -1;  // BBQ_FORCE_PATH: 1 sampled+filtered, 2 exact chunked (tests)
  // build scratch
  DevBuf T, stage, cacc, chain, norms;  // chain: the centroid's running sum, dim words + one status word
  // query scratch
  DevBuf qrows, qT, qcodes, qcorr, planes, qterms, tau, dump, cand, cand_cnt, lists_a, lists_b,
      out_idx, out_score, dots, images, qscreen, tau_bits, rr_true, rr_idx, rr_q, rr_t, cenv, qoff, qenv;
  int popc_form = 0;        // BBQ_POPC_FORM=tile forces the shared-memory tile form of the popcount scan (tests)
  bool dynamic_tau = true;  // BBQ_DYNTAU=0 keeps the sampled threshold fixed during the tensor-core scan (tests)
  int query_quantizer = 0;  // BBQ_QQUANT: thread / warp / cta force one form of K4 (tests, A/B); default by batch size
  // query screening armed by an entry point for the batch that starts at validate_base: the next K4 launches do it
  const float* validate_base = nullptr;
  // bbq_search keeps ONE host synchronisation per call: the filtered search leaves its overflow flag in h_flag and the
  // entry point looks at it after the synchronisation it needs anyway for the results (pending_overflow_nq >= 0)
  bool defer_overflow = false;
  int pending_overflow_nq = -1;
  // A narrow batch is launch-latency bound (a single query: ~10 stream operations around 60-90 us of kernels), and
  // its whole device sequence — screening, K4, planes / B images, threshold sample, scan, selection, status read-back —
  // depends only on (index, batch size, k): bbq_search captures it into a CUDA graph the second time the same key
  // arrives and replays it from then on (batches of up to GRAPH_MAX_NQ queries).
  struct SearchGraphKey {
    uint64_t ix = 0, n = 0, base = 0; const void* codes = nullptr; const void* rscreen = nullptr;
    uint32_t nq = 0, k = 0; uint64_t scratch_gen = 0;
    bool operator==(const SearchGraphKey& o) const {
      return ix == o.ix && n == o.n && base == o.base && codes == o.codes && rscreen == o.rscreen && nq == o.nq && k == o.k &&
             scratch_gen == o.scratch_gen;
    }
  };
  struct SearchGraph {
    cudaGraphExec_t exec = nullptr;
    SearchGraphKey key, seen;   // key: what exec was captured for; seen: the key of the previous eligible call
    uint64_t launches = 0;      // this library's kernel launches inside the captured sequence
    int pending_nq = -1;
    uint32_t last_path = 0, last_engine = 0;
    uint64_t replays = 0;
  } sgraph;
  int scan_engine = 0;  // BBQ_SCAN: 0 auto, 1 popcount kernel only, 2 tensor-core kernel whenever it can run
  uint32_t* h_flag = nullptr;  // pinned: [0..nq) candidate counts, [nq] overflow flag, then 2 words: first invalid query
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;  // ordering between the context's stream and a caller's stream (StreamBridge)
  // sharded search (bbq_comm_init): one NCCL communicator per context = per GPU = per process
  // atomic: a device group's caller thread clears it (then aborts the communicator) while the workers may read it
  std::atomic<ncclComm_t> comm{nullptr};
  int rank = 0, world = 1;
  DevBuf keys_local, keys_all, loc_idx, loc_score, bad, nglob;
  const bbq_group* group = nullptr;  // the device group that owns this context: its collectives run on that group's worker
  // profiling (bbq_set_profiling): event pairs per kernel group, drained by bbq_get_stats
  bool profiling = false;
  struct EvPair { cudaEvent_t a, b; int kind; };
  std::vector<EvPair> ev_pending;
  std::vector<cudaEvent_t> ev_pool;
};

// The worker thread of a device group runs the collective entries of its own context; anyone else calling them on a
// group's context would wait forever for peers that are not coming.
static thread_local const bbq_ctx* t_group_worker = nullptr;
static int group_guard(const bbq_ctx* c) {
  if (c->group && t_group_worker != c)
    return fail(BBQ_ERR_INVALID_ARG, "this context belongs to a device group: its collective entries run through the "
                                     "bbq_group_* entries");
  return BBQ_OK;
}

enum { PROF_SCAN = 0, PROF_QUANT = 1, PROF_SELECT = 2, PROF_SAMPLE = 3 };
struct ProfScope {  // records an event pair around a group of launches when profiling is on
  bbq_ctx* c;
  cudaStream_t st;
  cudaEvent_t a = nullptr, b = nullptr;
  int kind;
  ProfScope(bbq_ctx* c_, cudaStream_t st_, int kind_) : c(c_), st(st_), kind(kind_) {
    if (!c->profiling) return;
    auto get = [&]() {
      cudaEvent_t e = nullptr;
      if (!c->ev_pool.empty()) {
        e = c->ev_pool.back();
        c->ev_pool.pop_back();
      } else {
        cudaEventCreate(&e);
      }
      return e;
    };
    a = get();
    b = get();
    cudaEventRecord(a, st);
  }
  ~ProfScope() {
    if (!a) return;
    cudaEventRecord(b, st);
    c->ev_pending.push_back({a, b, kind});
  }
};

// All searches of a context share its scratch buffers.  When a caller hands in a stream of its own, the work it gets
// there is ordered AFTER everything already queued on the context's stream and BEFORE anything queued on it later, so
// that a host-pointer call (context stream) and a device-pointer call (caller stream) can follow each other without
// an explicit synchronisation.  Two caller streams used concurrently on one context remain the caller's business.
struct StreamBridge {
  bbq_ctx* c;
  cudaStream_t st;
  StreamBridge(bbq_ctx* c_, cudaStream_t st_) : c(c_), st(st_) {
    if (st == c->stream) return;
    cudaEventRecord(c->ev_in, c->stream);
    cudaStreamWaitEvent(st, c->ev_in, 0);
  }
  ~StreamBridge() {
    if (st == c->stream) return;
    cudaEventRecord(c->ev_out, st);
    cudaStreamWaitEvent(c->stream, c->ev_out, 0);
  }
};

static std::atomic<uint64_t> g_index_serial{0};
struct bbq_index {
  bbq_ctx* ctx = nullptr;
  uint64_t serial = ++g_index_serial;  // never reused (an address can be): part of the key of a captured launch sequence
  uint64_t n = 0;
  uint32_t dim = 0;
  int ib = 1;             // index bits (planes per 128-dim chunk of a row)
  int row_bytes = 0;
  uint8_t* codes = nullptr;
  double *lower = nullptr, *upper = nullptr, *addc = nullptr;
  uint32_t* compsum = nullptr;
  float* centroid = nullptr;  // device
  std::vector<float> centroid_h;
  double cdp = 0.0;
  uint64_t base = 0;
  IndexBounds* bounds = nullptr;  // device; valid for bounds_n rows (tensor-core screen margins)
  float* rows = nullptr;          // device [rows_n][dim]: original rows for the exact re-rank (bbq_index_attach_rows)
  uint64_t rows_n = 0;            // rows attached: the re-rank refuses an index that has grown (appended) since
  float4* rscreen = nullptr;      // device [capacity]: per-row screen constants, same validity
  uint64_t bounds_n = 0;
  uint64_t capacity = 0;  // rows allocated (== n except while a streaming build is in progress)
  uint64_t n_global = 0, n_global_for = ~0ull;  // sharded search: rows over all ranks, valid while n == n_global_for
};

static constexpr int64_t BUILD_CHUNK = 32768;   // rows per build chunk (transposed scratch = dim*chunk*4 B)
static constexpr uint32_t QUERY_BATCH = 4096;   // queries per internal pass (12-bit query field of a parked hit)
static constexpr uint32_t GRAPH_MAX_NQ = 16;    // widest batch whose device sequence bbq_search captures (bbq_ctx::sgraph)
static constexpr int64_t SAMPLE_TILES = 128;    // threshold sample = 128 tiles = 16384 rows ...
static constexpr int64_t SAMPLE_TILES_MAX = 2048;  // ... grown with k*n up to 262144 rows (see search_filtered)
static constexpr uint32_t CAND_CAP = SELECT_MAX;
static constexpr uint32_t K_MAX = 4096;

// device row: 16-byte chunks, index_bits planes per 128-dim chunk (k_osq_index); index_bits == 1: the packed row padded to 16 B
static inline int row_bytes_for(uint32_t dim, uint32_t index_bits = 1) { return (int)(((dim + 127) / 128) * 16 * index_bits); }
static constexpr uint32_t INDEX_BITS_MAX = 2;  // 1 = the reference's searchable layout, 2 = this build's extension

// ------------------------------------------------------------------------------------------------
// lifecycle
// ------------------------------------------------------------------------------------------------
extern "C" int bbq_abi_version(void) { return BBQ_B200_ABI_VERSION; }
extern "C" const char* bbq_last_error(void) { return g_err.c_str(); }
extern "C" void bbq_last_error_pos(int64_t* vector, int64_t* position) {
  if (vector) *vector = g_err_vec;
  if (position) *position = g_err_pos;
}

// src/binaryQuantizationFormat.ts:143-148
static int check_config(const bbq_config* config) {
  if (config->query_bits < 1 || config->query_bits > 8) return fail(BBQ_ERR_QUERY_BITS, "queryBits must be in 1..8");
  if (config->index_bits < 1 || config->index_bits > 8) return fail(BBQ_ERR_INDEX_BITS, "indexBits must be in 1..8");
  if (config->similarity > 2) return fail(BBQ_ERR_INVALID_ARG, "unknown similarity function");
  return BBQ_OK;
}
static int device_count(int* ndev) {
  *ndev = 0;
  if (cudaGetDeviceCount(ndev) != cudaSuccess || *ndev == 0) {
    cudaGetLastError();
    *ndev = 0;
    return fail(BBQ_ERR_NO_DEVICE, "no CUDA device: libbbq_b200 has no CPU fallback");
  }
  return BBQ_OK;
}

extern "C" int bbq_create(const bbq_config* config, bbq_ctx** out_ctx) {
  if (!config || !out_ctx) return fail(BBQ_ERR_NULL, "config/out_ctx is null");
  *out_ctx = nullptr;
  TRY(check_config(config));
  int ndev = 0;
  TRY(device_count(&ndev));
  int dev = config->device;
  if (dev < 0) CU(cudaGetDevice(&dev));
  if (dev >= ndev) return fail(BBQ_ERR_NO_DEVICE, "device ordinal out of range");
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10)
    return fail(BBQ_ERR_NO_DEVICE, std::string("device is sm_") + std::to_string(prop.major * 10 + prop.minor) +
                                       "; this library is built for sm_100a (B200) only");
  CU(cudaSetDevice(dev));
  bbq_ctx* c = new bbq_ctx();
  c->cfg = *config;
  c->device = dev;
  c->sm_count = prop.multiProcessorCount;
  CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  CU(cudaMallocHost(&c->h_flag, (QUERY_BATCH + 4) * sizeof(uint32_t)));
  CU(cudaEventCreateWithFlags(&c->ev_in, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&c->ev_out, cudaEventDisableTiming));
  if (const char* e = getenv("BBQ_FORCE_PATH")) c->force_path = atoi(e);
  if (const char* e = getenv("BBQ_POPC_FORM")) c->popc_form = !strcmp(e, "tile") ? 1 : 0;
  if (const char* e = getenv("BBQ_DYNTAU")) c->dynamic_tau = atoi(e) != 0;
  if (const char* e = getenv("BBQ_QQUANT")) c->query_quantizer = !strcmp(e, "thread") ? 1 : !strcmp(e, "warp") ? 2 : !strcmp(e, "cta") ? 3 : 0;
  if (const char* e = getenv("BBQ_SCAN")) c->scan_engine = !strcmp(e, "popc") ? 1 : !strcmp(e, "mma") ? 2 : 0;
  *out_ctx = c;
  return BBQ_OK;
}

static void comm_release(bbq_ctx* c);
static void ctx_release(bbq_ctx* c) {
  if (--c->refs > 0) return;
  cudaSetDevice(c->device);  // also for the scratch buffers, which `delete c` frees
  cudaStreamSynchronize(c->stream);
  comm_release(c);
  if (c->h_flag) cudaFreeHost(c->h_flag);
  if (c->sgraph.exec) cudaGraphExecDestroy(c->sgraph.exec);
  if (c->ev_in) cudaEventDestroy(c->ev_in);
  if (c->ev_out) cudaEventDestroy(c->ev_out);
  for (auto& p : c->ev_pending) {
    cudaEventDestroy(p.a);
    cudaEventDestroy(p.b);
  }
  for (auto e : c->ev_pool) cudaEventDestroy(e);
  cudaStreamDestroy(c->stream);
  delete c;
}

extern "C" void bbq_destroy(bbq_ctx* c) {
  if (!c || c->destroyed) return;
  c->destroyed = true;  // indexes that are still alive keep the context (its stream and scratch) until they go
  ctx_release(c);
}

extern "C" int bbq_get_stats(bbq_ctx* c, bbq_stats* out) {
  if (!c || !out) return fail(BBQ_ERR_NULL, "null");
  for (auto& p : c->ev_pending) {
    float ms = 0.f;
    CU(cudaEventSynchronize(p.b));
    CU(cudaEventElapsedTime(&ms, p.a, p.b));
    if (p.kind == PROF_SCAN) {
      c->stats.scan_ms += ms;
    } else if (p.kind == PROF_QUANT) {
      c->stats.quantize_ms += ms;
    } else if (p.kind == PROF_SAMPLE) {
      c->stats.sample_ms += ms;
    } else {
      c->stats.select_ms += ms;
    }
    c->ev_pool.push_back(p.a);
    c->ev_pool.push_back(p.b);
  }
  c->ev_pending.clear();
  *out = c->stats;
  out->kernel_launches = c->launches;
  return BBQ_OK;
}
extern "C" int bbq_set_profiling(bbq_ctx* c, int enabled) {
  if (!c) return fail(BBQ_ERR_NULL, "null");
  c->profiling = enabled != 0;
  return BBQ_OK;
}
extern "C" int bbq_reset_profiling(bbq_ctx* c) {
  if (!c) return fail(BBQ_ERR_NULL, "null");
  bbq_stats tmp;
  TRY(bbq_get_stats(c, &tmp));
  c->stats.scan_launches = 0;
  c->stats.scan_ms = c->stats.quantize_ms = c->stats.select_ms = c->stats.sample_ms = 0.0;
  return BBQ_OK;
}

#define LAUNCH(ctx, kernel, grid, block, smem, st, ...)       \
  do {                                                        \
    kernel<<<grid, block, smem, st>>>(__VA_ARGS__);           \
    (ctx)->launches++;                                        \
    CU(cudaGetLastError());                                   \
  } while (0)

// ------------------------------------------------------------------------------------------------
// index build
// ------------------------------------------------------------------------------------------------
static int index_alloc(bbq_ctx* c, uint64_t n, uint32_t dim, bbq_index** out) {
  bbq_index* ix = new bbq_index();
  ix->ctx = c;
  c->refs++;
  ix->n = n;
  ix->dim = dim;
  ix->ib = (int)c->cfg.index_bits;
  ix->row_bytes = row_bytes_for(dim, c->cfg.index_bits);
  ix->capacity = n;
  *out = ix;
  CU(cudaMalloc(&ix->codes, (size_t)n * ix->row_bytes));
  CU(cudaMalloc(&ix->lower, n * sizeof(double)));
  CU(cudaMalloc(&ix->upper, n * sizeof(double)));
  CU(cudaMalloc(&ix->addc, n * sizeof(double)));
  CU(cudaMalloc(&ix->compsum, n * sizeof(uint32_t)));
  CU(cudaMalloc(&ix->centroid, dim * sizeof(float)));
  ix->centroid_h.resize(dim);
  return BBQ_OK;
}

extern "C" void bbq_index_destroy(bbq_index* ix) {
  if (!ix) return;
  cudaSetDevice(ix->ctx->device);
  cudaStreamSynchronize(ix->ctx->stream);
  cudaFree(ix->codes);
  cudaFree(ix->lower);
  cudaFree(ix->upper);
  cudaFree(ix->addc);
  cudaFree(ix->compsum);
  cudaFree(ix->centroid);
  if (ix->bounds) cudaFree(ix->bounds);
  if (ix->rscreen) cudaFree(ix->rscreen);
  if (ix->rows) cudaFree(ix->rows);
  bbq_ctx* c = ix->ctx;
  delete ix;
  ctx_release(c);
}

// an index under construction: destroyed on every early return unless released to the caller
struct IndexGuard {
  bbq_index* ix = nullptr;
  IndexGuard() = default;
  IndexGuard(const IndexGuard&) = delete;
  IndexGuard& operator=(const IndexGuard&) = delete;
  ~IndexGuard() { bbq_index_destroy(ix); }
  bbq_index* release() {
    bbq_index* r = ix;
    ix = nullptr;
    return r;
  }
};

static int finish_centroid(bbq_index* ix) {
  bbq_ctx* c = ix->ctx;
  TRY(c->cacc.reserve(sizeof(double)));
  LAUNCH(c, k_centroid_dp, 1, 32, 0, c->stream, ix->centroid, (int)ix->dim, c->cacc.as<double>());
  CU(cudaMemcpyAsync(&ix->cdp, c->cacc.p, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(ix->centroid_h.data(), ix->centroid, ix->dim * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return BBQ_OK;
}

// Rows [off, off + rows_here) of `rows` (host when is_host, else device; row-major) into the transposed scratch T
// (leading dimension R), normalised for COSINE.  A host chunk goes through `stage`: the context's stream orders the
// next chunk's copy behind this chunk's kernels.
static int stage_chunk(bbq_ctx* c, const float* rows, bool is_host, uint32_t dim, int64_t R, int64_t off,
                       int64_t rows_here) {
  TRY(c->T.reserve((size_t)R * dim * sizeof(float)));
  const float* src = rows + off * (int64_t)dim;
  if (is_host) {
    TRY(c->stage.reserve((size_t)R * dim * sizeof(float)));
    CU(cudaMemcpyAsync(c->stage.p, src, (size_t)rows_here * dim * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    src = c->stage.as<float>();
  }
  dim3 grid((unsigned)((rows_here + 31) / 32), (dim + 31) / 32), block(32, 8);
  LAUNCH(c, k_transpose, grid, block, 0, c->stream, src, rows_here, (int)dim, c->T.as<float>(), R);
  if (c->cfg.similarity == BBQ_SIM_COSINE)
    LAUNCH(c, k_normalize_T, (unsigned)((rows_here + 127) / 128), 128, 0, c->stream, c->T.as<float>(), R, rows_here,
           (int)dim, 1);
  return BBQ_OK;
}

// quantise rows [0, n) of `rows` into index rows [ix->n, ix->n + n) with the index's centroid
static int append_impl(bbq_index* ix, const float* rows, bool is_host, uint64_t n) {
  if (!ix) return fail(BBQ_ERR_NULL, "null index");
  if (!rows) return fail(BBQ_ERR_NULL, "rows is null");
  if (ix->n + n > ix->capacity) return fail(BBQ_ERR_INVALID_ARG, "append exceeds the reserved capacity");
  bbq_ctx* c = ix->ctx;
  CU(cudaSetDevice(c->device));
  const int64_t R = (int64_t)std::min<uint64_t>(std::max<uint64_t>(n, 1), BUILD_CHUNK);
  for (int64_t off = 0; off < (int64_t)n; off += R) {
    const int64_t rows_here = std::min<int64_t>(R, (int64_t)n - off);
    TRY(stage_chunk(c, rows, is_host, ix->dim, R, off, rows_here));
    const unsigned grid = (unsigned)((rows_here + 127) / 128);
    if (ix->ib == 1)
      LAUNCH(c, k_osq_index<1>, grid, 128, 0, c->stream, c->T.as<float>(), R, rows_here, (int)ix->dim, ix->centroid,
             (int)c->cfg.similarity, c->cfg.lambda, (int)c->cfg.iters, ix->codes, ix->row_bytes, (int64_t)ix->n + off,
             ix->lower, ix->upper, ix->addc, ix->compsum);
    else
      LAUNCH(c, k_osq_index<2>, grid, 128, 0, c->stream, c->T.as<float>(), R, rows_here, (int)ix->dim, ix->centroid,
             (int)c->cfg.similarity, c->cfg.lambda, (int)c->cfg.iters, ix->codes, ix->row_bytes, (int64_t)ix->n + off,
             ix->lower, ix->upper, ix->addc, ix->compsum);
  }
  CU(cudaStreamSynchronize(c->stream));
  ix->n += n;
  return BBQ_OK;
}

// COSINE: the f64 norms of device rows [0, n) into c->norms, ahead of a chain over them (they do not depend on the sum)
static int row_norms(bbq_ctx* c, const float* d_rows, int64_t n, uint32_t dim) {
  if (c->cfg.similarity != BBQ_SIM_COSINE || n == 0) return BBQ_OK;
  TRY(c->norms.reserve((size_t)n * sizeof(double)));
  LAUNCH(c, k_row_norms, (unsigned)((n + 127) / 128), 128, 0, c->stream, d_rows, n, (int)dim, c->norms.as<double>());
  return BBQ_OK;
}

// The reference's running sum (device, d_acc[0, dim)) continued over rows [0, n) (host when is_host, else device), in
// stream order.  starts_corpus: rows[0] is the corpus's row 0.  norms_ready: c->norms already holds the COSINE norms
// of all n device rows (row_norms); otherwise they are computed chunk by chunk here.  COSINE chunks are normalised into
// the scratch T (row-major here) by a parallel pass, so that the chain itself only adds.
static int chain_rows(bbq_ctx* c, const float* rows, bool is_host, uint64_t n, uint32_t dim, bool starts_corpus,
                      float* d_acc, bool norms_ready = false) {
  const bool cosine = c->cfg.similarity == BBQ_SIM_COSINE;
  const unsigned grid = (dim + 31) / 32;
  if (!is_host && !cosine) {  // one pass over the caller's rows
    LAUNCH(c, k_centroid_chain, grid, 32, 0, c->stream, rows, (int64_t)n, (int)dim, d_acc, starts_corpus ? 1 : 0);
    return BBQ_OK;
  }
  const int64_t R = (int64_t)std::min<uint64_t>(std::max<uint64_t>(n, 1), BUILD_CHUNK);
  for (int64_t off = 0; off < (int64_t)n; off += R) {
    const int64_t rows_here = std::min<int64_t>(R, (int64_t)n - off);
    const float* src = rows + off * (int64_t)dim;
    if (is_host) {  // the stream orders this copy behind the previous chunk's kernels
      TRY(c->stage.reserve((size_t)R * dim * sizeof(float)));
      CU(cudaMemcpyAsync(c->stage.p, src, (size_t)rows_here * dim * sizeof(float), cudaMemcpyHostToDevice, c->stream));
      src = c->stage.as<float>();
    }
    if (cosine) {
      const double* norms = c->norms.as<double>() + off;
      if (is_host || !norms_ready) {
        TRY(row_norms(c, src, rows_here, dim));
        norms = c->norms.as<double>();
      }
      TRY(c->T.reserve((size_t)R * dim * sizeof(float)));
      const int64_t elems = rows_here * (int64_t)dim;
      LAUNCH(c, k_normalize_rows, (unsigned)std::min<int64_t>((elems + 255) / 256, 8 * (int64_t)c->sm_count * 8), 256, 0,
             c->stream, src, rows_here, (int)dim, norms, c->T.as<float>());
      src = c->T.as<float>();
    }
    LAUNCH(c, k_centroid_chain, grid, 32, 0, c->stream, src, rows_here, (int)dim, d_acc, starts_corpus && off == 0 ? 1 : 0);
  }
  return BBQ_OK;
}

// rows: host (is_host) or device pointer.  The centroid (unless given) from one pass over the rows, then the rows are
// appended to an index reserved for all of them.
static int build_impl(bbq_ctx* c, const float* rows, bool is_host, uint64_t n, uint32_t dim, const float* centroid,
                      bbq_index** out_index) {
  if (!c || !out_index) return fail(BBQ_ERR_NULL, "null ctx/out_index");
  *out_index = nullptr;
  if (!rows) return fail(BBQ_ERR_NULL, "rows is null");
  if (n == 0) return fail(BBQ_ERR_EMPTY, "vector set must not be empty");
  if (dim == 0) return fail(BBQ_ERR_INVALID_ARG, "dim must be > 0");
  if (n > 0x7FFFFFF0ull) return fail(BBQ_ERR_UNSUPPORTED, "more than 2^31 rows per shard (result ids are int32)");
  if (c->cfg.index_bits > INDEX_BITS_MAX)
    return fail(BBQ_ERR_UNSUPPORTED,
                "indexBits > 2: the reference's search cannot run any indexBits != 1 (createDirectPackedBuffer throws); "
                "this build searches 1-bit indexes (reference behaviour) and 2-bit ones (extension)");
  CU(cudaSetDevice(c->device));
  IndexGuard g;
  TRY(index_alloc(c, n, dim, &g.ix));
  bbq_index* ix = g.ix;
  ix->n = 0;
  if (centroid) {
    CU(cudaMemcpyAsync(ix->centroid, centroid, dim * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  } else {
    TRY(chain_rows(c, rows, is_host, n, dim, /*starts_corpus=*/true, ix->centroid));
    LAUNCH(c, k_centroid_finish, (dim + 127) / 128, 128, 0, c->stream, ix->centroid, (int)dim, (double)n);
  }
  TRY(finish_centroid(ix));
  TRY(append_impl(ix, rows, is_host, n));
  *out_index = g.release();
  return BBQ_OK;
}

// Reference validation order: COSINE rows are normalised first (binaryQuantizationFormat.ts:174-176), so a
// row holding NaN becomes all-NaN (first offender: position 0) and a row holding +-Inf (norm = Inf) turns
// the Inf components into NaN; otherwise the first non-finite component is reported as NaN or Infinity
// (:196-211).  Returns BBQ_OK or the status with (vector, position) set.
static int validate_rows(const float* rows, uint64_t n, uint32_t dim, bool cosine) {
  for (uint64_t i = 0; i < n; i++) {
    const float* r = rows + i * (uint64_t)dim;
    bool bad = false;
    for (uint32_t j = 0; j < dim; j++) bad |= !std::isfinite(r[j]);
    if (!bad) continue;
    if (cosine) {
      for (uint32_t j = 0; j < dim; j++)
        if (std::isnan(r[j])) return fail(BBQ_ERR_NAN, "vector contains NaN", (int64_t)i, 0);
      double n2 = 0;
      for (uint32_t j = 0; j < dim; j++) n2 += (double)r[j] * (double)r[j];
      (void)n2;  // norm is +Inf here: finite/Inf -> 0, Inf/Inf -> NaN
      for (uint32_t j = 0; j < dim; j++)
        if (std::isinf(r[j])) return fail(BBQ_ERR_NAN, "vector contains NaN", (int64_t)i, (int64_t)j);
    } else {
      for (uint32_t j = 0; j < dim; j++) {
        if (std::isnan(r[j])) return fail(BBQ_ERR_NAN, "vector contains NaN", (int64_t)i, (int64_t)j);
        if (std::isinf(r[j])) return fail(BBQ_ERR_INF, "vector contains Infinity", (int64_t)i, (int64_t)j);
      }
    }
  }
  return BBQ_OK;
}

extern "C" int bbq_index_build(bbq_ctx* c, const float* rows, uint64_t n, uint32_t dim, const float* centroid,
                               bbq_index** out_index) {
  if (!c || !out_index) return fail(BBQ_ERR_NULL, "null ctx/out_index");
  *out_index = nullptr;
  if (n == 0) return fail(BBQ_ERR_EMPTY, "vector set must not be empty");
  if (!rows) return fail(BBQ_ERR_NULL, "rows is null");
  TRY(validate_rows(rows, n, dim, c->cfg.similarity == BBQ_SIM_COSINE));
  return build_impl(c, rows, true, n, dim, centroid, out_index);
}

extern "C" int bbq_index_build_device(bbq_ctx* c, const float* d_rows, uint64_t n, uint32_t dim,
                                      const float* centroid, bbq_index** out_index) {
  return build_impl(c, d_rows, false, n, dim, centroid, out_index);
}

extern "C" int bbq_index_reserve(bbq_ctx* c, uint64_t capacity, uint32_t dim, const float* centroid,
                                 bbq_index** out_index) {
  if (!c || !out_index) return fail(BBQ_ERR_NULL, "null ctx/out_index");
  *out_index = nullptr;
  if (!centroid) return fail(BBQ_ERR_NULL, "a streaming build needs an explicit centroid");
  if (capacity == 0) return fail(BBQ_ERR_EMPTY, "vector set must not be empty");
  if (dim == 0) return fail(BBQ_ERR_INVALID_ARG, "dim must be > 0");
  if (capacity > 0x7FFFFFF0ull) return fail(BBQ_ERR_UNSUPPORTED, "more than 2^31 rows per shard");
  if (c->cfg.index_bits > INDEX_BITS_MAX) return fail(BBQ_ERR_UNSUPPORTED, "indexBits > 2 is not built on device");
  CU(cudaSetDevice(c->device));
  IndexGuard g;
  TRY(index_alloc(c, capacity, dim, &g.ix));
  g.ix->n = 0;
  CU(cudaMemcpy(g.ix->centroid, centroid, dim * sizeof(float), cudaMemcpyHostToDevice));
  TRY(finish_centroid(g.ix));
  *out_index = g.release();
  return BBQ_OK;
}
extern "C" int bbq_index_append(bbq_index* ix, const float* rows, uint64_t n) {
  if (!ix) return fail(BBQ_ERR_NULL, "null index");
  if (n == 0) return BBQ_OK;
  if (!rows) return fail(BBQ_ERR_NULL, "rows is null");
  TRY(validate_rows(rows, n, ix->dim, ix->ctx->cfg.similarity == BBQ_SIM_COSINE));
  return append_impl(ix, rows, true, n);
}
extern "C" int bbq_index_append_device(bbq_index* ix, const float* d_rows, uint64_t n) {
  if (n == 0) return BBQ_OK;
  return append_impl(ix, d_rows, false, n);
}

// The reference centroid's running sum over a slice of the corpus: host running[0, dim) in and out
static int accumulate_impl(bbq_ctx* c, const float* rows, bool is_host, uint64_t n, uint32_t dim, uint64_t rows_before,
                           float* running) {
  if (!c || !running) return fail(BBQ_ERR_NULL, "null ctx/running");
  if (dim == 0) return fail(BBQ_ERR_INVALID_ARG, "dim must be > 0");
  if (n == 0) return BBQ_OK;
  if (!rows) return fail(BBQ_ERR_NULL, "rows is null");
  if (is_host) {
    const int st = validate_rows(rows, n, dim, c->cfg.similarity == BBQ_SIM_COSINE);
    if (st != BBQ_OK) return fail(st, g_err, (int64_t)rows_before + g_err_vec, g_err_pos);  // the corpus's vector index
  }
  CU(cudaSetDevice(c->device));
  TRY(c->chain.reserve((size_t)dim * sizeof(float)));
  float* acc = c->chain.as<float>();
  if (rows_before > 0) CU(cudaMemcpyAsync(acc, running, dim * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  TRY(chain_rows(c, rows, is_host, n, dim, rows_before == 0, acc));
  CU(cudaMemcpyAsync(running, acc, dim * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return BBQ_OK;
}
extern "C" int bbq_centroid_accumulate(bbq_ctx* c, const float* rows, uint64_t n, uint32_t dim, uint64_t rows_before,
                                       float* running) {
  return accumulate_impl(c, rows, true, n, dim, rows_before, running);
}
extern "C" int bbq_centroid_accumulate_device(bbq_ctx* c, const float* d_rows, uint64_t n, uint32_t dim,
                                              uint64_t rows_before, float* running) {
  return accumulate_impl(c, d_rows, false, n, dim, rows_before, running);
}
// k_centroid_finish on the host: f32(f64 sum / f64 N).  Dividing by float(N) instead rounds N once N > 2^24.
extern "C" int bbq_centroid_finish(const float* running, uint32_t dim, uint64_t n_total, float* centroid) {
  if (!running || !centroid) return fail(BBQ_ERR_NULL, "null running/centroid");
  if (n_total == 0) return fail(BBQ_ERR_EMPTY, "vector set must not be empty");
  for (uint32_t i = 0; i < dim; i++) centroid[i] = (float)((double)running[i] / (double)n_total);
  return BBQ_OK;
}

// Host-side conversion between the caller's row form and the device row (cold paths: adopt / export).
// index_bits == 1: the caller's row is the packed MSB-first row (ceil(dim/8) bytes) and the device row is that row
// zero-padded.  index_bits >= 2: the caller's row is what BinarizedByteVectorValuesImpl holds for such an index —
// dim UNPACKED codes (src/binaryQuantizationFormat.ts:221-249) — and the device row is plane-interleaved.
static void row_to_device(const uint8_t* src, uint32_t dim, int ib, uint8_t* dst, int row_bytes) {
  memset(dst, 0, (size_t)row_bytes);
  if (ib == 1) {
    const int P = (int)((dim + 7) / 8);
    memcpy(dst, src, P);
    if (dim & 7) dst[P - 1] &= (uint8_t)(0xFF << (8 - (dim & 7)));  // tail bits are zero by contract
    return;
  }
  for (uint32_t i = 0; i < dim; i++) {
    const uint32_t rc = i >> 7, j = (i & 127) >> 3, t = i & 7;
    for (int p = 0; p < ib; p++)
      if ((src[i] >> p) & 1) dst[(rc * ib + p) * 16 + j] |= (uint8_t)(1u << (7 - t));
  }
}
static void row_from_device(const uint8_t* src, uint32_t dim, int ib, uint8_t* dst) {
  if (ib == 1) {
    memcpy(dst, src, (dim + 7) / 8);
    return;
  }
  for (uint32_t i = 0; i < dim; i++) {
    const uint32_t rc = i >> 7, j = (i & 127) >> 3, t = i & 7;
    uint8_t v = 0;
    for (int p = 0; p < ib; p++) v |= (uint8_t)(((src[(rc * ib + p) * 16 + j] >> (7 - t)) & 1) << p);
    dst[i] = v;
  }
}
static inline size_t caller_row_bytes(uint32_t dim, int ib) { return ib == 1 ? (dim + 7) / 8 : dim; }

extern "C" int bbq_index_from_quantized(bbq_ctx* c, const uint8_t* packed, const double* corr4, const float* centroid,
                                        uint64_t n, uint32_t dim, bbq_index** out_index) {
  if (!c || !out_index) return fail(BBQ_ERR_NULL, "null ctx/out_index");
  *out_index = nullptr;
  if (!packed || !corr4 || !centroid) return fail(BBQ_ERR_NULL, "null input");
  if (n == 0) return fail(BBQ_ERR_EMPTY, "vector set must not be empty");
  if (dim == 0) return fail(BBQ_ERR_INVALID_ARG, "dim must be > 0");
  if (c->cfg.index_bits > INDEX_BITS_MAX) return fail(BBQ_ERR_UNSUPPORTED, "only 1- and 2-bit indexes can be adopted");
  CU(cudaSetDevice(c->device));
  IndexGuard g;
  TRY(index_alloc(c, n, dim, &g.ix));
  bbq_index* ix = g.ix;
  const size_t P = caller_row_bytes(dim, ix->ib);
  const int RB = ix->row_bytes;
  std::vector<uint8_t> codes((size_t)n * RB, 0);
  std::vector<double> lo(n), up(n), ad(n);
  std::vector<uint32_t> cs(n);
  for (uint64_t i = 0; i < n; i++) {
    row_to_device(packed + i * P, dim, ix->ib, codes.data() + i * RB, RB);
    lo[i] = corr4[4 * i];
    up[i] = corr4[4 * i + 1];
    ad[i] = corr4[4 * i + 2];
    cs[i] = (uint32_t)corr4[4 * i + 3];
  }
  CU(cudaMemcpy(ix->codes, codes.data(), codes.size(), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(ix->lower, lo.data(), n * sizeof(double), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(ix->upper, up.data(), n * sizeof(double), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(ix->addc, ad.data(), n * sizeof(double), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(ix->compsum, cs.data(), n * sizeof(uint32_t), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(ix->centroid, centroid, dim * sizeof(float), cudaMemcpyHostToDevice));
  TRY(finish_centroid(ix));
  *out_index = g.release();
  return BBQ_OK;
}

extern "C" uint64_t bbq_index_size(const bbq_index* ix) { return ix ? ix->n : 0; }
extern "C" uint32_t bbq_index_dim(const bbq_index* ix) { return ix ? ix->dim : 0; }
extern "C" int bbq_index_centroid(const bbq_index* ix, float* out_centroid, double* out_cdp) {
  if (!ix) return fail(BBQ_ERR_NULL, "null index");
  if (out_centroid) memcpy(out_centroid, ix->centroid_h.data(), ix->dim * sizeof(float));
  if (out_cdp) *out_cdp = ix->cdp;
  return BBQ_OK;
}
extern "C" int bbq_index_set_base(bbq_index* ix, uint64_t base) {
  if (!ix) return fail(BBQ_ERR_NULL, "null index");
  if (base + ix->n > 0x7FFFFFFFull) return fail(BBQ_ERR_UNSUPPORTED, "global row ids must fit in int32");
  ix->base = base;
  return BBQ_OK;
}

extern "C" int bbq_index_export(const bbq_index* ix, uint64_t first, uint64_t count, uint8_t* packed, double* corr4) {
  if (!ix) return fail(BBQ_ERR_NULL, "null index");
  if (first + count > ix->n) return fail(BBQ_ERR_INVALID_ARG, "row range out of bounds");
  if (count == 0) return BBQ_OK;
  CU(cudaSetDevice(ix->ctx->device));
  CU(cudaStreamSynchronize(ix->ctx->stream));
  const size_t P = caller_row_bytes(ix->dim, ix->ib);
  const int RB = ix->row_bytes;
  if (packed) {
    std::vector<uint8_t> tmp((size_t)count * RB);
    CU(cudaMemcpy(tmp.data(), ix->codes + first * RB, tmp.size(), cudaMemcpyDeviceToHost));
    for (uint64_t i = 0; i < count; i++) row_from_device(tmp.data() + i * RB, ix->dim, ix->ib, packed + i * P);
  }
  if (corr4) {
    std::vector<double> lo(count), up(count), ad(count);
    std::vector<uint32_t> cs(count);
    CU(cudaMemcpy(lo.data(), ix->lower + first, count * sizeof(double), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(up.data(), ix->upper + first, count * sizeof(double), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(ad.data(), ix->addc + first, count * sizeof(double), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(cs.data(), ix->compsum + first, count * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    for (uint64_t i = 0; i < count; i++) {
      corr4[4 * i] = lo[i];
      corr4[4 * i + 1] = up[i];
      corr4[4 * i + 2] = ad[i];
      corr4[4 * i + 3] = (double)cs[i];
    }
  }
  return BBQ_OK;
}

// ------------------------------------------------------------------------------------------------
// search
// ------------------------------------------------------------------------------------------------
static constexpr unsigned K1S_CTAS_PER_SM = 4;  // persistent CTAs per SM of the streaming scan (its __launch_bounds__)
template <int MODE>
static int launch_scan_nb(bbq_ctx* c, int nb, bool stream_form, dim3 grid, size_t smem, cudaStream_t st,
                          const ScanParams& p) {
#define BBQ_SCAN_CASE(NB)                                                                                          \
  case NB:                                                                                                         \
    if (stream_form) {                                                                                             \
      const unsigned sgrid = std::min<unsigned>(grid.x, (unsigned)c->sm_count * K1S_CTAS_PER_SM);                  \
      switch (p.row_bytes >> 4) {                                                                                  \
        case 1: LAUNCH(c, (k_scan_stream<NB, MODE, 1>), dim3(sgrid), TILE_ROWS, 0, st, p); break;                  \
        case 2: LAUNCH(c, (k_scan_stream<NB, MODE, 2>), dim3(sgrid), TILE_ROWS, 0, st, p); break;                  \
        case 3: LAUNCH(c, (k_scan_stream<NB, MODE, 3>), dim3(sgrid), TILE_ROWS, 0, st, p); break;                  \
        case 4: LAUNCH(c, (k_scan_stream<NB, MODE, 4>), dim3(sgrid), TILE_ROWS, 0, st, p); break;                  \
        case 6: LAUNCH(c, (k_scan_stream<NB, MODE, 6>), dim3(sgrid), TILE_ROWS, 0, st, p); break;                  \
        case 8: LAUNCH(c, (k_scan_stream<NB, MODE, 8>), dim3(sgrid), TILE_ROWS, 0, st, p); break;                  \
        case 12: LAUNCH(c, (k_scan_stream<NB, MODE, 12>), dim3(sgrid), TILE_ROWS, 0, st, p); break;                \
        default: return fail(BBQ_ERR_UNSUPPORTED, "no streaming scan for this row size");                          \
      }                                                                                                            \
    } else {                                                                                                       \
      if (smem > 48 * 1024)                                                                                        \
        CU(cudaFuncSetAttribute(k_scan<NB, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));        \
      LAUNCH(c, (k_scan<NB, MODE>), grid, TILE_ROWS, smem, st, p);                                                 \
    }                                                                                                              \
    break;
  switch (nb) {
    BBQ_SCAN_CASE(1)
    BBQ_SCAN_CASE(2)
    BBQ_SCAN_CASE(3)
    BBQ_SCAN_CASE(4)
    BBQ_SCAN_CASE(5)
    BBQ_SCAN_CASE(6)
    BBQ_SCAN_CASE(7)
    BBQ_SCAN_CASE(8)
    case 9:  // 8-bit queries on a 2-bit index: 9 virtual planes, shared-memory tile form only
      if (stream_form) return fail(BBQ_ERR_UNSUPPORTED, "no streaming scan for 9 planes");
      if (smem > 48 * 1024) CU(cudaFuncSetAttribute(k_scan<9, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      LAUNCH(c, (k_scan<9, MODE>), grid, TILE_ROWS, smem, st, p);
      break;
    default:
      return fail(BBQ_ERR_QUERY_BITS, "queryBits must be in 1..8");
  }
#undef BBQ_SCAN_CASE
  return BBQ_OK;
}

// tiles [tile_first, tile_first + ntiles*tile_stride) step tile_stride, queries [0, nq)
static int launch_scan(bbq_index* ix, int mode, ScanParams p, int64_t ntiles, cudaStream_t st) {
  bbq_ctx* c = ix->ctx;
  const int nb = (int)c->cfg.query_bits + ix->ib - 1;  // (virtual) query bit-planes, k_query_planes
  const int w4 = ix->row_bytes / 16, s4 = w4 | 1;
  int qb = std::min(p.nq, 32);
  auto smem_for = [&](int q) {
    return (size_t)TILE_ROWS * s4 * 16 + (size_t)q * nb * w4 * 16 + (size_t)q * sizeof(bbqn::QueryTerms) +
           (size_t)q * sizeof(float) + 16;
  };
  while (qb > 1 && smem_for(qb) > 160 * 1024) qb /= 2;
  if (smem_for(qb) > 227 * 1024) return fail(BBQ_ERR_UNSUPPORTED, "dimension too large for the scan tile");
  p.q_block = qb;
  const bool is_sample = mode == SCAN_DUMP && p.tile_stride > 1;
  ProfScope prof(c, st, is_sample ? PROF_SAMPLE : PROF_SCAN);
  if (!is_sample) c->stats.scan_launches++;
  dim3 grid((unsigned)ntiles, (unsigned)((p.nq + qb - 1) / qb));
  p.ntiles = ntiles;
  // one or a few queries: the streaming (register/shuffle, HBM-bound) form; it needs >= 2 rows per 512-byte load
  const bool stream_ok = w4 == 1 || w4 == 2 || w4 == 3 || w4 == 4 || w4 == 6 || w4 == 8 || w4 == 12;  // dims 128..1536
  const bool stream_form = c->popc_form != 1 && p.nq <= 4 && stream_ok && nb <= 8;
  if (mode == SCAN_DUMP) return launch_scan_nb<SCAN_DUMP>(c, nb, stream_form, grid, smem_for(qb), st, p);
  return launch_scan_nb<SCAN_FILTER>(c, nb, stream_form, grid, smem_for(qb), st, p);
}

template <int MODE>
static int launch_select(bbq_ctx* c, const SelectParams& p, uint32_t m_max, cudaStream_t st) {
  uint32_t m2 = 2;
  while (m2 < m_max || m2 < p.k) m2 <<= 1;
  if (m2 > (uint32_t)SELECT_MAX) return fail(BBQ_ERR_UNSUPPORTED, "selection exceeds SELECT_MAX keys");
  const size_t smem = (size_t)m2 * sizeof(uint64_t);
  ProfScope prof(c, st, PROF_SELECT);
  if (smem > 48 * 1024)
    CU(cudaFuncSetAttribute(k_select<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  LAUNCH(c, (k_select<MODE>), p.nq, SELECT_THREADS, smem, st, p, m2);
  return BBQ_OK;
}

// K4 for nq queries already in device memory (row-major f32): fills ctx->planes / qterms (/qcodes,qcorr).
// ntimes = how often a COSINE query is normalised: 2 on the search path (src/binaryQuantizationFormat.ts:337 and
// :279), 1 for a direct quantizeQueryVector call (:271-299).
static int quantize_rows(bbq_ctx* c, const float* d_queries, int nq, int dim, int row_bytes, const float* d_centroid,
                         int ntimes, cudaStream_t st) {
  // row_bytes: the DEVICE row of the index the queries are for (planes included); codes are stored per real dim
  const int ib = (int)c->cfg.index_bits <= (int)INDEX_BITS_MAX ? (int)c->cfg.index_bits : 1;
  const int nb = (int)c->cfg.query_bits, nbv = nb + ib - 1, words = row_bytes / 4, code_ld = row_bytes * 8 / ib;
  TRY(c->qT.reserve((size_t)nq * dim * sizeof(float)));
  TRY(c->qcodes.reserve((size_t)nq * code_ld));
  TRY(c->qcorr.reserve((size_t)nq * 4 * sizeof(double)));
  TRY(c->planes.reserve((size_t)nq * nbv * words * sizeof(uint32_t)));
  TRY(c->qterms.reserve((size_t)nq * sizeof(bbqn::QueryTerms)));
  ProfScope prof(c, st, PROF_QUANT);
  const size_t per_warp = (size_t)((dim + 3) & ~3) * sizeof(float) + 14 * 33 * sizeof(double);
  const size_t smem = per_warp * OSQW_WARPS;
  const size_t smem_cta = (size_t)OSQC_TERM_ROWS * 33 * sizeof(double) + (2 * (OSQC_PRODUCERS + 1) + 8) * sizeof(double) +
                          (size_t)((dim + 3) & ~3) * sizeof(float);
  // 0 = by batch size: one CTA per query for a narrow batch (K4 is the longest kernel of a single-query search and
  // the CTA form runs each pass at the latency of the add chain), one warp per query otherwise
  const int form = c->query_quantizer != 0 ? c->query_quantizer : (nq <= 2 * c->sm_count ? 3 : 2);
  // query screening (NaN / Infinity): armed by the entry point, done by K4 itself while it stages the query
  unsigned long long* bad = nullptr;
  int q_base = 0;
  if (c->validate_base != nullptr) {
    bad = c->bad.as<unsigned long long>();
    q_base = (int)((d_queries - c->validate_base) / dim);
  }
  float* d_q = const_cast<float*>(d_queries);  // (an offending query is zeroed in place; the entry points own the buffer)
  if (form == 3 && smem_cta <= 200 * 1024) {
    if (smem_cta > 48 * 1024)
      CU(cudaFuncSetAttribute(k_osq_query_cta, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cta));
    LAUNCH(c, k_osq_query_cta, nq, OSQC_THREADS, smem_cta, st, d_q, nq, dim, d_centroid, (int)c->cfg.similarity, nb,
           c->cfg.lambda, (int)c->cfg.iters, ntimes, c->qcodes.as<uint8_t>(), code_ld, c->qcorr.as<double>(), bad, q_base);
  } else if (form != 1 && smem <= 200 * 1024) {
    // one warp per query
    if (smem > 48 * 1024)
      CU(cudaFuncSetAttribute(k_osq_query_warp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    LAUNCH(c, k_osq_query_warp, (nq + OSQW_WARPS - 1) / OSQW_WARPS, OSQW_WARPS * 32, smem, st, d_q, nq, dim,
           d_centroid, (int)c->cfg.similarity, nb, c->cfg.lambda, (int)c->cfg.iters, ntimes, c->qcodes.as<uint8_t>(),
           code_ld, c->qcorr.as<double>(), bad, q_base);
  } else {
    // throughput form: one thread per query over the transposed scratch (same code as the index build)
    if (bad != nullptr)
      LAUNCH(c, k_validate_queries, (nq + 3) / 4, 128, 0, st, d_q, nq, dim, c->cfg.similarity == BBQ_SIM_COSINE ? 1 : 0, ntimes,
             bad, q_base);
    float* T = c->qT.as<float>();
    dim3 grid((nq + 31) / 32, (dim + 31) / 32), block(32, 8);
    LAUNCH(c, k_transpose, grid, block, 0, st, d_queries, (int64_t)nq, dim, T, (int64_t)nq);
    if (ntimes) LAUNCH(c, k_normalize_T, (nq + 63) / 64, 64, 0, st, T, (int64_t)nq, (int64_t)nq, dim, ntimes);
    LAUNCH(c, k_osq_query, (nq + 63) / 64, 64, 0, st, T, (int64_t)nq, nq, dim, d_centroid, (int)c->cfg.similarity, nb,
           c->cfg.lambda, (int)c->cfg.iters, c->qcodes.as<uint8_t>(), code_ld, c->qcorr.as<double>());
  }
  const int64_t total = std::max<int64_t>((int64_t)nq * nbv * words, nq);
  LAUNCH(c, k_query_planes, (unsigned)((total + 127) / 128), 128, 0, st, c->qcodes.as<uint8_t>(), code_ld,
         c->qcorr.as<double>(), nq, nb, ib, words, c->planes.as<uint32_t>(), c->qterms.as<bbqn::QueryTerms>());
  return BBQ_OK;
}
static int quantize_queries(bbq_index* ix, const float* d_queries, int nq, cudaStream_t st) {
  bbq_ctx* c = ix->ctx;
  return quantize_rows(c, d_queries, nq, (int)ix->dim, ix->row_bytes, ix->centroid,
                       c->cfg.similarity == BBQ_SIM_COSINE ? 2 : 0, st);
}

// ---- tensor-core scan (K2) -------------------------------------------------------------------------
struct MmaPlan {
  int n_tile = 0, passes = 0, nstage = 0, kbytes = 0;
  int cpq = 1;  // accumulator columns per query: 2 when the code is split into nibbles (k_query_tiles)
  int nissuers = 2;  // MMA issuing threads
  int layout = 0;  // MmaLayout: 0 = 8 epilogue warps + 1 expansion group, 1 = 4 + 2 (few resident queries: feed-bound)
  size_t smem = 0;
};
static bool mma_plan(const bbq_index* ix, int nq, MmaPlan* out) {
  const bbq_ctx* c = ix->ctx;
  if (c->scan_engine == 1) return false;
  const int qb_ = (int)c->cfg.query_bits;
  // B elements are code << plane << (0..3): they fit a byte while (2^qb - 1) * 2^(ib-1) <= 31; wider codes are split
  // into two nibble columns per query
  MmaPlan pl;
  pl.cpq = (((1 << qb_) - 1) << (ix->ib - 1)) <= 31 ? 1 : 2;
  const int64_t max_dot = (int64_t)((1 << qb_) - 1) * ((1 << ix->ib) - 1) * ix->dim;
  if (max_dot >= (1ll << HIT_DOT_BITS) || nq > 4096) return false;  // parked-hit word: 21-bit dot, 12-bit query
  if (ix->row_bytes * 8 > 4096) return false;                        // K bytes per row the resident B block is planned for
  pl.kbytes = ix->row_bytes * 8;
  const size_t budget = 227 * 1024 - 1024 - (HIT_RING * sizeof(uint64_t) + 64);
  int n_cap = (int)(budget / ((size_t)pl.kbytes + 64)) / 16 * 16;
  n_cap = std::min(n_cap, MMA_N_MAX);
  if (n_cap < 16) return false;
  // 1-4 queries: the streaming popcount scan (HBM/latency bound, ~43 us per query and 1M rows).  From 5 queries on the
  // tensor-core scan wins: one pass over 1M x 1024 costs 0.145 ms whatever the block size (operand-feed bound), the
  // popcount tile scan 0.03 ms per query (tools/crossover.sh: 8 queries 0.145 vs 0.257 ms, 48 queries 0.154 vs 1.43 ms)
  if (c->scan_engine != 2 && nq < 5) return false;
  const int ncols = nq * pl.cpq;
  pl.passes = (ncols + n_cap - 1) / n_cap;
  pl.n_tile = (((ncols + pl.passes - 1) / pl.passes) + 15) / 16 * 16;
  pl.nstage = std::min(8, (512 - 2 * pl.n_tile) / 32);
  // Role layout by the width of the resident block (profiles/r02_k2_narrow_layout.txt, 1 M x 1024, ms per pass, wide -> narrow:
  // 16 columns 0.136 -> 0.109, 64: 0.146 -> 0.127, 96: 0.151 -> 0.137, 128: 0.157 -> 0.155 (EUCLIDEAN: 0.175 -> 0.185), 208: 0.213 ->
  // 0.218).  A narrow batch is bound by the ISSUE of its tcgen05 operations (32 MMAs + 12 commits per 128-row tile whatever
  // the width, ~100-150 cycles each for the issuing thread), so the narrow layout also runs three issuing threads.
  constexpr int MMA_NARROW_MAX = 96;  // widest resident block (accumulator columns) that takes the narrow layout
  pl.layout = pl.n_tile <= MMA_NARROW_MAX ? 1 : 0;
  pl.nissuers = pl.layout == 1 ? 3 : 2;
  pl.smem = (size_t)pl.n_tile * pl.kbytes + (size_t)pl.n_tile * (sizeof(QScreen) + sizeof(bbqn::QueryTerms)) + 26 * 8 + sizeof(HitCtx) + HIT_RING * sizeof(uint64_t) + 16 + 16;
  *out = pl;
  return true;
}

static int ensure_bounds(bbq_index* ix, cudaStream_t st) {
  bbq_ctx* c = ix->ctx;
  if (ix->bounds && ix->bounds_n == ix->n) return BBQ_OK;
  if (!ix->bounds) CU(cudaMalloc(&ix->bounds, sizeof(IndexBounds)));
  if (!ix->rscreen) CU(cudaMalloc(&ix->rscreen, (size_t)ix->capacity * sizeof(float4)));
  CU(cudaMemsetAsync(ix->bounds, 0, sizeof(IndexBounds), st));
  LAUNCH(c, k_index_bounds, 592, 256, 0, st, ix->lower, ix->upper, ix->addc, ix->compsum, (int64_t)ix->n,
         (int)c->cfg.similarity, bbqn::index_lx_div(ix->ib), reinterpret_cast<uint32_t*>(ix->bounds), ix->rscreen);
  ix->bounds_n = ix->n;
  return BBQ_OK;
}

// B images for the whole query batch (after quantize_queries)
static int prepare_mma_operands(bbq_index* ix, int nq, const MmaPlan& pl, cudaStream_t st) {
  bbq_ctx* c = ix->ctx;
  const size_t bytes = (size_t)pl.passes * pl.n_tile * pl.kbytes;
  TRY(c->images.reserve(bytes));
  // per-query tables are indexed by query SLOT: pass * (n_tile / cpq) + position in the pass
  TRY(c->qscreen.reserve((size_t)pl.passes * pl.n_tile * sizeof(QScreen)));
  TRY(c->tau_bits.reserve((size_t)pl.passes * pl.n_tile * sizeof(uint32_t)));
  TRY(c->qoff.reserve((size_t)pl.passes * pl.n_tile * sizeof(int32_t)));
  TRY(c->qenv.reserve((size_t)pl.passes * sizeof(QEnv)));
  ProfScope prof(c, st, PROF_QUANT);
  const int64_t threads = (int64_t)pl.passes * pl.n_tile * (pl.kbytes / 16);
  LAUNCH(c, k_query_tiles, (unsigned)((threads + 255) / 256), 256, 0, st, c->qcodes.as<uint8_t>(),
         ix->row_bytes * 8 / ix->ib, nq, pl.n_tile, pl.kbytes, ix->ib, pl.cpq, c->images.as<uint8_t>());
  return BBQ_OK;
}

template <int MODE, int LAYOUT>
static int launch_mma_sim(bbq_ctx* c, int sim, int cpq, unsigned grid, size_t smem, cudaStream_t st, const MmaParams& p) {
#define BBQ_MMA_CASE(S)                                                                                                  \
  case S:                                                                                                                \
    if (cpq == 1) {                                                                                                      \
      CU(cudaFuncSetAttribute(k_scan_mma<MODE, S, 1, LAYOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
      LAUNCH(c, (k_scan_mma<MODE, S, 1, LAYOUT>), grid, MmaLayout<LAYOUT>::THREADS, smem, st, p);                       \
    } else {                                                                                                             \
      CU(cudaFuncSetAttribute(k_scan_mma<MODE, S, 2, LAYOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
      LAUNCH(c, (k_scan_mma<MODE, S, 2, LAYOUT>), grid, MmaLayout<LAYOUT>::THREADS, smem, st, p);                       \
    }                                                                                                                    \
    break;
  switch (sim) {
    BBQ_MMA_CASE(0)
    BBQ_MMA_CASE(1)
    BBQ_MMA_CASE(2)
    default:
      return fail(BBQ_ERR_INVALID_ARG, "unknown similarity");
  }
#undef BBQ_MMA_CASE
  return BBQ_OK;
}

static int launch_scan_mma(bbq_index* ix, int mode, int nq, uint32_t k, const MmaPlan& pl, int64_t tile_first, int64_t tile_stride,
                           int64_t ntiles, float* dump, int64_t dump_ld, uint64_t* cand, uint32_t* cand_cnt,
                           uint32_t cap, uint32_t* overflow, cudaStream_t st, int32_t* dots = nullptr) {
  bbq_ctx* c = ix->ctx;
  MmaParams p{};
  p.codes = ix->codes;
  p.lower = ix->lower;
  p.upper = ix->upper;
  p.addc = ix->addc;
  p.compsum = ix->compsum;
  p.n = (int64_t)ix->n;
  p.row_bytes = ix->row_bytes;
  p.kbytes = pl.kbytes;
  p.images = c->images.as<uint8_t>();
  p.qscreen = c->qscreen.as<QScreen>();
  p.rscreen = ix->rscreen;
  p.qoff = mode == SCAN_FILTER ? c->qoff.as<int32_t>() : nullptr;  // the dump (sample, taps) reads plain accumulators
  p.qenv = mode == SCAN_FILTER ? c->qenv.as<QEnv>() : nullptr;
  p.tau_bits = c->tau_bits.as<uint32_t>();
  p.bounds = ix->bounds;
  p.k = c->dynamic_tau ? k : 0xFFFFFFFFu;
  p.qterms = c->qterms.as<bbqn::QueryTerms>();
  p.nq = nq;
  p.n_tile = pl.n_tile;
  p.passes = pl.passes;
  p.nstage = pl.nstage;
  p.nissuers = pl.nissuers;
  p.dim = (double)ix->dim;
  p.cdp = ix->cdp;
  p.sim = (int)c->cfg.similarity;
  p.one_bit_query = bbqn::score_mode((int)c->cfg.query_bits, ix->ib);
  p.lx_div = bbqn::index_lx_div(ix->ib);
  p.base = (uint32_t)ix->base;
  p.tile_first = tile_first;
  p.tile_stride = tile_stride;
  p.ntiles = ntiles;
  p.dump = dump;
  p.dump_ld = dump_ld;
  p.dots = dots;
  p.cand = cand;
  p.cand_cnt = cand_cnt;
  p.cap = cap;
  p.overflow = overflow;
  ProfScope prof(c, st, mode == SCAN_DUMP ? PROF_SAMPLE : PROF_SCAN);
  if (mode != SCAN_DUMP) c->stats.scan_launches++;
  c->stats.mma_n_tile = (uint32_t)pl.n_tile;
  if (mode != SCAN_DUMP) c->stats.mma_layout = (uint32_t)pl.layout;
  c->stats.mma_passes = (uint32_t)pl.passes;
  const unsigned grid = (unsigned)std::min<int64_t>(ntiles, c->sm_count);
  // (the dump — threshold sample, parity taps — always runs the wide-batch roles: it is a few hundred tiles)
  if (mode == SCAN_DUMP) return launch_mma_sim<SCAN_DUMP, 0>(c, p.sim, pl.cpq, grid, pl.smem, st, p);
  if (pl.layout == 1) return launch_mma_sim<SCAN_FILTER, 1>(c, p.sim, pl.cpq, grid, pl.smem, st, p);
  return launch_mma_sim<SCAN_FILTER, 0>(c, p.sim, pl.cpq, grid, pl.smem, st, p);
}

static ScanParams base_scan_params(bbq_index* ix, int nq) {
  bbq_ctx* c = ix->ctx;
  ScanParams p{};
  p.codes = ix->codes;
  p.lower = ix->lower;
  p.upper = ix->upper;
  p.addc = ix->addc;
  p.compsum = ix->compsum;
  p.n = (int64_t)ix->n;
  p.row_bytes = ix->row_bytes;
  p.planes = c->planes.as<uint32_t>();
  p.qterms = c->qterms.as<bbqn::QueryTerms>();
  p.nq = nq;
  p.dim = (double)ix->dim;
  p.cdp = ix->cdp;
  p.sim = (int)c->cfg.similarity;
  p.one_bit_query = bbqn::score_mode((int)c->cfg.query_bits, ix->ib);
  p.lx_div = bbqn::index_lx_div(ix->ib);
  p.base = (uint32_t)ix->base;
  p.tile_first = 0;
  p.tile_stride = 1;
  return p;
}

// Deterministic merge of `lists` per-query lists [lists][nq][k] into out_idx / out_score [nq][k], in groups of
// max(2, SELECT_MAX / k) lists per selection.  The input is read in place: idx/score pairs, or 64-bit keys when in_keys
// is set.  The levels in between are keys, alternating between lists_a and lists_b (the first in the one that does not
// hold the input).  A key carries exactly what its pair carries, so the result does not depend on the form.
static int merge_topk(bbq_ctx* c, const int32_t* in_idx, const float* in_score, const uint64_t* in_keys, uint32_t lists,
                      int nq, uint32_t k, int32_t* out_idx, float* out_score, cudaStream_t st) {
  const uint32_t group = std::max<uint32_t>(2u, (uint32_t)SELECT_MAX / k);
  const size_t cnt = (size_t)nq * k;
  const void* in = in_keys ? (const void*)in_keys : (const void*)in_idx;
  DevBuf* dst = in == c->lists_a.p ? &c->lists_b : &c->lists_a;
  while (true) {
    const uint32_t ngroups = (lists + group - 1) / group;
    if (ngroups > 1) TRY(dst->reserve((size_t)ngroups * cnt * sizeof(uint64_t)));
    for (uint32_t g = 0; g < ngroups; g++) {
      SelectParams s{};
      s.nq = nq;
      s.k = k;
      s.lists = std::min(group, lists - g * group);
      s.k_in = k;
      const size_t off = (size_t)g * group * cnt;
      if (ngroups == 1) {
        s.out_idx = out_idx;
        s.out_score = out_score;
      } else {
        s.out_keys = dst->as<uint64_t>() + (size_t)g * cnt;
      }
      if (in_keys) {
        s.keys = in_keys + off;
        TRY(launch_select<SEL_KLISTS>(c, s, s.lists * k, st));
      } else {
        s.in_idx = in_idx + off;
        s.in_score = in_score + off;
        TRY(launch_select<SEL_PAIRS>(c, s, s.lists * k, st));
      }
    }
    if (ngroups == 1) return BBQ_OK;
    in_keys = dst->as<uint64_t>();
    dst = dst == &c->lists_a ? &c->lists_b : &c->lists_a;
    lists = ngroups;
  }
}

// Exact chunked path: every chunk of <= SELECT_MAX rows is scored densely and selected; partial lists
// are merged.  One chunk == the direct path for small indexes.
static int search_exact_chunked(bbq_index* ix, int nq, uint32_t k, int32_t* d_out_idx, float* d_out_score,
                                cudaStream_t st) {
  bbq_ctx* c = ix->ctx;
  const int64_t n = (int64_t)ix->n;
  const int64_t chunk_rows = SELECT_MAX, chunk_tiles = chunk_rows / TILE_ROWS;
  const int64_t ntiles = (n + TILE_ROWS - 1) / TILE_ROWS;
  const uint32_t nchunks = (uint32_t)((n + chunk_rows - 1) / chunk_rows);
  TRY(c->dump.reserve((size_t)nq * chunk_rows * sizeof(float)));
  if (nchunks > 1) TRY(c->lists_a.reserve((size_t)nchunks * nq * k * (sizeof(int32_t) + sizeof(float))));
  int32_t* la_idx = c->lists_a.as<int32_t>();
  float* la_score = reinterpret_cast<float*>(la_idx + (size_t)nchunks * nq * k);
  for (uint32_t ch = 0; ch < nchunks; ch++) {
    const int64_t t0 = (int64_t)ch * chunk_tiles, tn = std::min(chunk_tiles, ntiles - t0);
    const int64_t rows_here = std::min(chunk_rows, n - t0 * TILE_ROWS);
    ScanParams p = base_scan_params(ix, nq);
    p.tile_first = t0;
    p.dump = c->dump.as<float>();
    p.dump_ld = chunk_rows;
    TRY(launch_scan(ix, SCAN_DUMP, p, tn, st));
    SelectParams s{};
    s.nq = nq;
    s.k = k;
    s.scores = c->dump.as<float>();
    s.ld = chunk_rows;
    s.m = (uint32_t)rows_here;
    s.tile_first = t0;
    s.tile_stride = 1;
    s.base = (uint32_t)ix->base;
    if (nchunks == 1) {
      s.out_idx = d_out_idx;
      s.out_score = d_out_score;
    } else {
      s.out_idx = la_idx + (size_t)ch * nq * k;
      s.out_score = la_score + (size_t)ch * nq * k;
    }
    TRY(launch_select<SEL_DENSE>(c, s, (uint32_t)rows_here, st));
  }
  if (nchunks > 1) TRY(merge_topk(c, la_idx, la_score, nullptr, nchunks, nq, k, d_out_idx, d_out_score, st));
  return BBQ_OK;
}

// after the stream has been synchronised: must the last filtered search be redone on the exact chunked path?  Yes when a
// candidate list overflowed, and when a query has fewer than want = min(k, n) candidates.  tau is a lower bound of the
// k-th best finite score and the scans never admit a NaN score, so a short list means that fewer than k rows score
// finitely and rows that score NaN belong at the tail of the answer.
static bool resolve_filtered(bbq_ctx* c, int nq, uint32_t want) {
  uint64_t tot = 0;
  bool short_list = false;
  for (int q = 0; q < nq; q++) {
    tot += c->h_flag[q];
    short_list |= c->h_flag[q] < want;
  }
  c->stats.last_candidates = tot;
  return c->h_flag[nq] != 0 || short_list;
}

// Sampled-threshold path: tau[q] = k-th best score over a strided sample of full tiles (a valid lower
// bound of the final k-th best), then one filtered scan appends every row with score >= tau[q], then
// the final selection.  *overflowed is set (after a sync) when a candidate list overflowed.
static int search_filtered(bbq_index* ix, int nq, uint32_t k, int32_t* d_out_idx, float* d_out_score, cudaStream_t st,
                           bool* overflowed) {
  bbq_ctx* c = ix->ctx;
  const int64_t n = (int64_t)ix->n;
  const int64_t ntiles = (n + TILE_ROWS - 1) / TILE_ROWS, full_tiles = n / TILE_ROWS;
  MmaPlan pl;
  const bool use_mma = mma_plan(ix, nq, &pl);
  // Sample size.  With the running threshold of the tensor-core scan (k <= RETIGHTEN_KMAX) the sample only has to
  // give the scan something to start from.  With a FIXED threshold about k * n / sample_rows rows pass it, so the
  // sample grows with k * n until that expectation is a quarter of a candidate list (otherwise a large k or a large
  // shard would overflow the lists on perfectly ordinary data and fall back to the exact chunked path every time).
  const bool running = use_mma && c->dynamic_tau && k <= RETIGHTEN_KMAX;
  int64_t want_tiles = SAMPLE_TILES;
  if (!running) {
    const int64_t need_rows = (int64_t)std::min<double>(4.0 * (double)k * (double)n / (double)CAND_CAP, 1e12);
    want_tiles = std::max(want_tiles, std::min<int64_t>(SAMPLE_TILES_MAX, (need_rows + TILE_ROWS - 1) / TILE_ROWS));
    // the sample's scores are dumped densely: keep that scratch below ~1 GiB whatever the batch size
    want_tiles = std::max<int64_t>(SAMPLE_TILES, std::min<int64_t>(want_tiles, (int64_t)(1ll << 28) / ((int64_t)nq * TILE_ROWS)));
  }
  const int64_t stiles = std::min<int64_t>(want_tiles, full_tiles);
  const int64_t stride = std::max<int64_t>(1, full_tiles / stiles);
  const int64_t sample_ld = stiles * TILE_ROWS;
  TRY(c->dump.reserve((size_t)nq * sample_ld * sizeof(float)));
  TRY(c->tau.reserve((size_t)nq * sizeof(float)));
  TRY(c->cand.reserve((size_t)nq * CAND_CAP * sizeof(uint64_t)));
  TRY(c->cand_cnt.reserve((size_t)(nq + 1) * sizeof(uint32_t)));
  c->stats.last_engine = use_mma ? 2 : 1;
  if (use_mma) {
    TRY(prepare_mma_operands(ix, nq, pl, st));
    TRY(ensure_bounds(ix, st));
  }
  {
    ScanParams p = base_scan_params(ix, nq);
    p.tile_stride = stride;
    p.dump = c->dump.as<float>();
    p.dump_ld = sample_ld;
    if (use_mma)
      TRY(launch_scan_mma(ix, SCAN_DUMP, nq, k, pl, 0, stride, stiles, c->dump.as<float>(), sample_ld, nullptr, nullptr, 0,
                          nullptr, st));
    else
      TRY(launch_scan(ix, SCAN_DUMP, p, stiles, st));
    ProfScope prof(c, st, PROF_SELECT);
    if (k <= (uint32_t)TAU_THREADS) {
      LAUNCH(c, k_tau_from_sample<TAU_THREADS>, nq, TAU_THREADS, 0, st, c->dump.as<float>(),
             sample_ld, (uint32_t)sample_ld, k, c->tau.as<float>());
    } else {
      const size_t smem = TAU_BINS_MAX * sizeof(uint32_t);
      CU(cudaFuncSetAttribute(k_tau_from_sample<TAU_BINS_MAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      LAUNCH(c, k_tau_from_sample<TAU_BINS_MAX>, nq, TAU_THREADS, smem, st, c->dump.as<float>(), sample_ld,
             (uint32_t)sample_ld, k, c->tau.as<float>());
    }
  }
  uint32_t* cnt = c->cand_cnt.as<uint32_t>();
  CU(cudaMemsetAsync(cnt, 0, (size_t)(nq + 1) * sizeof(uint32_t), st));
  {
    ScanParams p = base_scan_params(ix, nq);
    p.tau = c->tau.as<float>();
    p.cand = c->cand.as<uint64_t>();
    p.cand_cnt = cnt;
    p.cap = CAND_CAP;
    p.overflow = cnt + nq;
    if (use_mma) {
      {
        ProfScope prof(c, st, PROF_QUANT);
        LAUNCH(c, k_query_screen, pl.passes, 256, 0, st, c->qterms.as<bbqn::QueryTerms>(), c->tau.as<float>(), nq,
               pl.n_tile / pl.cpq, (double)ix->dim, ix->cdp, (int)c->cfg.similarity,
               bbqn::score_mode((int)c->cfg.query_bits, ix->ib), ix->bounds,
               c->qscreen.as<QScreen>(), c->tau_bits.as<uint32_t>(), c->qoff.as<int32_t>(), c->qenv.as<QEnv>());
      }
      // the running threshold reads candidate slots that may be reserved but not yet written: they must read as 0
      CU(cudaMemset2DAsync(p.cand, (size_t)CAND_CAP * sizeof(uint64_t), 0, (size_t)RETIGHTEN_ZCAP * sizeof(uint64_t), nq, st));
      TRY(launch_scan_mma(ix, SCAN_FILTER, nq, k, pl, 0, 1, ntiles, nullptr, 0, p.cand, cnt, CAND_CAP, cnt + nq, st));
    } else {
      TRY(launch_scan(ix, SCAN_FILTER, p, ntiles, st));
    }
  }
  {
    SelectParams s{};
    s.nq = nq;
    s.k = k;
    s.keys = c->cand.as<uint64_t>();
    s.cnt = cnt;
    s.cap = CAND_CAP;
    s.out_idx = d_out_idx;
    s.out_score = d_out_score;
    TRY(launch_select<SEL_KEYS>(c, s, CAND_CAP, st));
  }
  CU(cudaMemcpyAsync(c->h_flag, cnt, (size_t)(nq + 1) * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  if (c->defer_overflow) {  // the caller synchronises once, then calls resolve_filtered
    c->pending_overflow_nq = nq;
    *overflowed = false;
    return BBQ_OK;
  }
  CU(cudaStreamSynchronize(st));
  *overflowed = resolve_filtered(c, nq, (uint32_t)std::min<int64_t>(k, n));
  return BBQ_OK;
}

static int search_batch(bbq_index* ix, const float* d_queries, int nq, uint32_t k, int32_t* d_out_idx,
                        float* d_out_score, cudaStream_t st) {
  bbq_ctx* c = ix->ctx;
  TRY(quantize_queries(ix, d_queries, nq, st));
  int path = ((int64_t)ix->n <= SELECT_MAX) ? 0 : 1;
  if (c->force_path == 2) path = 2;
  if (c->force_path == 1 && (int64_t)ix->n >= TILE_ROWS) path = 1;
  c->stats.last_overflow = 0;
  if (path == 1) {
    bool over = false;
    TRY(search_filtered(ix, nq, k, d_out_idx, d_out_score, st, &over));
    if (over) {
      c->stats.last_overflow = 1;
      path = 2;
    }
  }
  if (path != 1) TRY(search_exact_chunked(ix, nq, k, d_out_idx, d_out_score, st));
  c->stats.last_path = (uint32_t)path;
  return BBQ_OK;
}

extern "C" int bbq_search_device(bbq_index* ix, const float* d_queries, uint32_t nq, uint32_t k, int32_t* d_out_idx,
                                 float* d_out_score, void* stream) {
  if (!ix) return fail(BBQ_ERR_NULL, "target vector set must not be null");
  if (!d_queries || !d_out_idx || !d_out_score) return fail(BBQ_ERR_NULL, "query vector must not be null");
  if (nq == 0 || k == 0) return BBQ_OK;
  if (k > K_MAX) return fail(BBQ_ERR_UNSUPPORTED, "k > 4096 is not supported by the device top-k");
  bbq_ctx* c = ix->ctx;
  CU(cudaSetDevice(c->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : c->stream;
  StreamBridge bridge(c, st);
  for (uint32_t q0 = 0; q0 < nq; q0 += QUERY_BATCH) {
    const int nb = (int)std::min<uint32_t>(QUERY_BATCH, nq - q0);
    TRY(search_batch(ix, d_queries + (size_t)q0 * ix->dim, nb, k, d_out_idx + (size_t)q0 * k,
                     d_out_score + (size_t)q0 * k, st));
  }
  return BBQ_OK;
}

// Query screening on the device (NaN / Infinity): while a QueryScreen is alive, the K4 launches that follow screen the
// batch that starts at d_queries while they stage it (see osq_query_team) and zero an offending query in place.
// read_back enqueues the copy of the verdict into the pinned flag block; verdict() reads it after the caller's
// synchronisation.  Leaving the scope disarms: an entry point that fails half-way leaves nothing armed for the next.
struct QueryScreen {
  bbq_ctx* c;
  int armed;  // status of arming: returned by the caller before any device work
  QueryScreen(bbq_ctx* c_, const float* d_queries, cudaStream_t st) : c(c_), armed(arm(d_queries, st)) {}
  ~QueryScreen() { c->validate_base = nullptr; }
  int read_back(cudaStream_t st) {
    c->validate_base = nullptr;
    CU(cudaMemcpyAsync(c->h_flag + QUERY_BATCH + 2, c->bad.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    return BBQ_OK;
  }
  static int verdict(bbq_ctx* c) {
    unsigned long long v;
    memcpy(&v, c->h_flag + QUERY_BATCH + 2, sizeof v);
    if (v == ~0ull) return BBQ_OK;
    const int64_t q = (int64_t)(v >> 34), pos = (int64_t)(v & 0xFFFFFFFFull);
    if (((v >> 32) & 3ull) == 2ull) return fail(BBQ_ERR_INF, "vector contains Infinity", q, pos);
    return fail(BBQ_ERR_NAN, "vector contains NaN", q, pos);
  }

 private:
  int arm(const float* d_queries, cudaStream_t st) {
    TRY(c->bad.reserve(sizeof(unsigned long long)));
    CU(cudaMemsetAsync(c->bad.p, 0xFF, sizeof(unsigned long long), st));
    c->validate_base = d_queries;
    return BBQ_OK;
  }
};

// the nq host queries of a host-pointer call into qrows, on the context's stream
static int stage_queries(bbq_ctx* c, const float* queries, uint64_t nq, uint32_t dim) {
  TRY(c->qrows.reserve((size_t)nq * dim * sizeof(float)));
  CU(cudaMemcpyAsync(c->qrows.p, queries, (size_t)nq * dim * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  return BBQ_OK;
}

// nq device rows of kk elements (stride kk) into the caller's host rows of stride k
static int copy_rows_out(void* dst, size_t k, const DevBuf& src, uint32_t kk, uint32_t nq, size_t elem, cudaStream_t st) {
  if (kk == k)
    CU(cudaMemcpyAsync(dst, src.p, (size_t)nq * kk * elem, cudaMemcpyDeviceToHost, st));
  else
    CU(cudaMemcpy2DAsync(dst, k * elem, src.p, (size_t)kk * elem, (size_t)kk * elem, nq, cudaMemcpyDeviceToHost, st));
  return BBQ_OK;
}

// the lists of a host-pointer search (out_idx / out_score) into the caller's rows, then the call's synchronisation
static int copy_results(bbq_ctx* c, uint32_t nq, size_t k, uint32_t kk, int32_t* out_idx, float* out_score) {
  TRY(copy_rows_out(out_idx, k, c->out_idx, kk, nq, sizeof(int32_t), c->stream));
  TRY(copy_rows_out(out_score, k, c->out_score, kk, nq, sizeof(float), c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return BBQ_OK;
}

extern "C" int bbq_search(bbq_index* ix, const float* queries, uint32_t nq, int64_t k, int32_t* out_idx,
                          float* out_score, uint32_t* out_count) {
  if (out_count) *out_count = 0;
  // src/binaryQuantizationFormat.ts:318-334
  if (!queries) return fail(BBQ_ERR_NULL, "query vector must not be null");
  if (!ix) return fail(BBQ_ERR_NULL, "target vector set must not be null");
  if (k < 0) return fail(BBQ_ERR_NEGATIVE_K, "k must not be negative");
  if (k == 0 || nq == 0) return BBQ_OK;
  if (!out_idx || !out_score) return fail(BBQ_ERR_NULL, "output buffers must not be null");
  bbq_ctx* c = ix->ctx;
  const uint32_t kk = (uint32_t)std::min<int64_t>(k, (int64_t)ix->n);  // :385 k2 = min(k, vectorCount)
  if (kk > K_MAX) return fail(BBQ_ERR_UNSUPPORTED, "k > 4096 is not supported by the device top-k");
  CU(cudaSetDevice(c->device));
  TRY(c->out_idx.reserve((size_t)nq * kk * sizeof(int32_t)));
  TRY(c->out_score.reserve((size_t)nq * kk * sizeof(float)));
  TRY(stage_queries(c, queries, nq, ix->dim));
  // scalarQuantize validates the (normalised) query, optimizedScalarQuantizer.ts:138-148: done on the device, ahead
  // of the search in the same stream (an offending query is zeroed), and read back at the one synchronisation below.
  // One host synchronisation per call (a single-batch call; larger ones keep the per-batch check): the overflow flag of
  // the filtered search travels with the results and is looked at after the synchronisation below.
  c->pending_overflow_nq = -1;
  auto enqueue_device_sequence = [&]() -> int {  // everything between the H2D of the queries and the D2H of the results
    QueryScreen screen(c, c->qrows.as<float>(), c->stream);
    TRY(screen.armed);
    c->defer_overflow = nq <= QUERY_BATCH;
    const int st_search = bbq_search_device(ix, c->qrows.as<float>(), nq, kk, c->out_idx.as<int32_t>(), c->out_score.as<float>(), c->stream);
    c->defer_overflow = false;
    TRY(st_search);
    return screen.read_back(c->stream);
  };
  const bool graph_ok = nq <= GRAPH_MAX_NQ && !c->profiling;
  bbq_ctx::SearchGraphKey key;
  key.ix = ix->serial; key.n = ix->n; key.base = ix->base; key.codes = ix->codes; key.rscreen = ix->rscreen;
  key.nq = nq; key.k = kk; key.scratch_gen = g_scratch_gen;
  bbq_ctx::SearchGraph& sg = c->sgraph;
  if (graph_ok && sg.exec != nullptr && sg.key == key) {
    CU(cudaGraphLaunch(sg.exec, c->stream));
    c->launches += sg.launches;
    c->pending_overflow_nq = sg.pending_nq;
    c->stats.last_path = sg.last_path;
    c->stats.last_engine = sg.last_engine;
    c->stats.last_overflow = 0;
    sg.replays++;
    c->stats.graph_replays = sg.replays;
  } else if (graph_ok && sg.seen == key) {
    // second call in a row with this key: every scratch buffer has its final size (no allocation can happen inside the
    // capture) — record the sequence, then run it
    if (sg.exec) {
      cudaGraphExecDestroy(sg.exec);
      sg.exec = nullptr;
    }
    const uint64_t l0 = c->launches;
    CU(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeRelaxed));
    const int st_seq = enqueue_device_sequence();
    cudaGraph_t graph = nullptr;
    const cudaError_t ec = cudaStreamEndCapture(c->stream, &graph);
    if (st_seq != BBQ_OK || ec != cudaSuccess || graph == nullptr || g_scratch_gen != key.scratch_gen) {
      if (graph) cudaGraphDestroy(graph);
      cudaGetLastError();
      sg.seen = bbq_ctx::SearchGraphKey{};  // do not try again until the key has been seen twice more
      if (st_seq != BBQ_OK) return st_seq;
      c->pending_overflow_nq = -1;
      TRY(enqueue_device_sequence());       // nothing ran during the failed capture: run the sequence directly
    } else {
      const cudaError_t ei = cudaGraphInstantiate(&sg.exec, graph, 0);
      cudaGraphDestroy(graph);
      if (ei != cudaSuccess) {
        sg.exec = nullptr;
        cudaGetLastError();
        return fail(BBQ_ERR_CUDA, "cudaGraphInstantiate failed");
      }
      sg.key = key;
      sg.launches = c->launches - l0;
      sg.pending_nq = c->pending_overflow_nq;
      sg.last_path = c->stats.last_path;
      sg.last_engine = c->stats.last_engine;
      CU(cudaGraphLaunch(sg.exec, c->stream));
    }
  } else {
    if (graph_ok) sg.seen = key;  // (if scratch grows during this call the next call's key differs and re-arms)
    TRY(enqueue_device_sequence());
  }
  TRY(copy_results(c, nq, (size_t)k, kk, out_idx, out_score));
  if (c->pending_overflow_nq >= 0) {
    const bool over = resolve_filtered(c, c->pending_overflow_nq, kk);
    c->pending_overflow_nq = -1;
    if (over) {  // a candidate list overflowed (adversarial input) or came up short: the exact chunked path redoes the batch
      c->stats.last_overflow = 1;
      c->stats.last_path = 2;
      TRY(search_exact_chunked(ix, (int)nq, kk, c->out_idx.as<int32_t>(), c->out_score.as<float>(), c->stream));
      TRY(copy_results(c, nq, (size_t)k, kk, out_idx, out_score));
    }
  }
  TRY(QueryScreen::verdict(c));
  if (out_count) *out_count = kk;
  return BBQ_OK;
}

static int attach_rows(bbq_index* ix, const float* rows, cudaMemcpyKind kind) {
  if (!ix || !rows) return fail(BBQ_ERR_NULL, "null");
  bbq_ctx* c = ix->ctx;
  CU(cudaSetDevice(c->device));
  const size_t bytes = (size_t)ix->n * ix->dim * sizeof(float);
  if (ix->rows) CU(cudaFree(ix->rows));
  ix->rows = nullptr;
  ix->rows_n = 0;
  CU(cudaMalloc(&ix->rows, bytes));
  CU(cudaMemcpyAsync(ix->rows, rows, bytes, kind, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  ix->rows_n = ix->n;
  return BBQ_OK;
}

// the rows the exact re-rank reads must cover the whole index (not an index appended to after bbq_index_attach_rows)
static int check_attached_rows(const bbq_index* ix) {
  if (!ix->rows) return fail(BBQ_ERR_INVALID_ARG, "no original rows attached (bbq_index_attach_rows)");
  if (ix->rows_n != ix->n)
    return fail(BBQ_ERR_INVALID_ARG, "rows attached for " + std::to_string(ix->rows_n) + " rows, index has " +
                                         std::to_string(ix->n));
  return BBQ_OK;
}

static int launch_rerank_scores(bbq_index* ix, bool owned_only, const float* d_queries, uint32_t nq, uint32_t m,
                                const int32_t* d_cand_idx, double* d_true, cudaStream_t st) {
  bbq_ctx* c = ix->ctx;
  const int64_t pairs = (int64_t)nq * m;
  const unsigned grid = (unsigned)((pairs + RERANK_WARPS - 1) / RERANK_WARPS);
  if (owned_only) {
    LAUNCH(c, k_rerank_scores<true>, grid, RERANK_WARPS * 32, 0, st, ix->rows, (int)ix->dim, d_queries, (int)nq, (int)m,
           d_cand_idx, (uint32_t)ix->base, (uint32_t)ix->rows_n, d_true);
  } else {
    LAUNCH(c, k_rerank_scores<false>, grid, RERANK_WARPS * 32, 0, st, ix->rows, (int)ix->dim, d_queries, (int)nq, (int)m,
           d_cand_idx, (uint32_t)ix->base, (uint32_t)ix->rows_n, d_true);
  }
  return BBQ_OK;
}
extern "C" int bbq_index_attach_rows(bbq_index* ix, const float* rows) { return attach_rows(ix, rows, cudaMemcpyHostToDevice); }
extern "C" int bbq_index_attach_rows_device(bbq_index* ix, const float* d_rows) {
  return attach_rows(ix, d_rows, cudaMemcpyDeviceToDevice);
}

// scratch of a re-rank call: m candidates and kk results per query
static int reserve_rerank(bbq_ctx* c, uint32_t dim, uint32_t nq, uint32_t m, uint32_t kk) {
  TRY(c->qrows.reserve((size_t)nq * dim * sizeof(float)));
  TRY(c->out_idx.reserve((size_t)nq * m * sizeof(int32_t)));
  TRY(c->out_score.reserve((size_t)nq * m * sizeof(float)));
  TRY(c->rr_true.reserve((size_t)nq * m * sizeof(double)));
  TRY(c->rr_idx.reserve((size_t)nq * kk * sizeof(int32_t)));
  TRY(c->rr_q.reserve((size_t)nq * kk * sizeof(float)));
  TRY(c->rr_t.reserve((size_t)nq * kk * sizeof(double)));
  return BBQ_OK;
}

// the tail of a re-rank call, once rr_true holds the exact score of every candidate in out_idx / out_score: the kk
// best per query into the caller's rows of stride k, one synchronisation, then the verdict of the query screening
static int rerank_select_and_copy(bbq_ctx* c, cudaStream_t st, uint32_t nq, uint32_t m, uint32_t k, uint32_t kk,
                                  int32_t* out_idx, float* out_qscore, double* out_true) {
  {
    ProfScope prof(c, st, PROF_SELECT);
    LAUNCH(c, k_rerank_select, nq, 256, 0, st, c->rr_true.as<double>(), c->out_idx.as<int32_t>(), c->out_score.as<float>(),
           (int)m, kk, c->rr_idx.as<int32_t>(), c->rr_q.as<float>(), c->rr_t.as<double>());
  }
  TRY(copy_rows_out(out_idx, k, c->rr_idx, kk, nq, sizeof(int32_t), st));
  TRY(copy_rows_out(out_qscore, k, c->rr_q, kk, nq, sizeof(float), st));
  TRY(copy_rows_out(out_true, k, c->rr_t, kk, nq, sizeof(double), st));
  CU(cudaStreamSynchronize(st));
  return QueryScreen::verdict(c);
}

extern "C" int bbq_search_rerank(bbq_index* ix, const float* queries, uint32_t nq, uint32_t k, uint32_t factor,
                                 int32_t* out_idx, float* out_qscore, double* out_true, uint32_t* out_count) {
  if (out_count) *out_count = 0;
  if (!ix) return fail(BBQ_ERR_NULL, "target vector set must not be null");
  if (!queries) return fail(BBQ_ERR_NULL, "query vector must not be null");
  TRY(check_attached_rows(ix));
  if (nq == 0 || k == 0) return BBQ_OK;
  if (!out_idx || !out_qscore || !out_true) return fail(BBQ_ERR_NULL, "output buffers must not be null");
  if (factor == 0 || (uint64_t)k * factor > K_MAX) return fail(BBQ_ERR_UNSUPPORTED, "k * oversampleFactor must be in 1..4096");
  bbq_ctx* c = ix->ctx;
  const uint32_t m = (uint32_t)std::min<uint64_t>((uint64_t)k * factor, ix->n);  // candidates per query
  const uint32_t kk = std::min(k, m);
  CU(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  TRY(reserve_rerank(c, ix->dim, nq, m, kk));
  TRY(stage_queries(c, queries, nq, ix->dim));
  {
    QueryScreen screen(c, c->qrows.as<float>(), st);
    TRY(screen.armed);
    TRY(bbq_search_device(ix, c->qrows.as<float>(), nq, m, c->out_idx.as<int32_t>(), c->out_score.as<float>(), st));
    TRY(screen.read_back(st));
  }
  {
    ProfScope prof(c, st, PROF_SELECT);
    TRY(launch_rerank_scores(ix, /*owned_only=*/false, c->qrows.as<float>(), nq, m, c->out_idx.as<int32_t>(),
                             c->rr_true.as<double>(), st));
  }
  TRY(rerank_select_and_copy(c, st, nq, m, k, kk, out_idx, out_qscore, out_true));
  if (out_count) *out_count = kk;
  return BBQ_OK;
}

extern "C" int bbq_merge_topk_device(bbq_ctx* c, const int32_t* d_idx, const float* d_score, uint32_t lists,
                                     uint32_t nq, uint32_t k, int32_t* d_out_idx, float* d_out_score, void* stream) {
  if (!c || !d_idx || !d_score || !d_out_idx || !d_out_score) return fail(BBQ_ERR_NULL, "null");
  if (lists == 0 || nq == 0 || k == 0) return BBQ_OK;
  if (k > K_MAX) return fail(BBQ_ERR_UNSUPPORTED, "k > 4096");
  CU(cudaSetDevice(c->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : c->stream;
  return merge_topk(c, d_idx, d_score, nullptr, lists, (int)nq, k, d_out_idx, d_out_score, st);
}


// ------------------------------------------------------------------------------------------------
// sharded search (SURVEY §8e): row shards on the GPUs of one box, one process / context / communicator per GPU;
// per-shard top-k lists travel as 64-bit keys in ONE ncclAllGather over NVLink and are merged by k_select.
// NCCL is dlopen'ed on first use so that a single-GPU host needs no NCCL installation.
// ------------------------------------------------------------------------------------------------
struct NcclApi {
  decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
  decltype(&ncclCommInitRank) CommInitRank = nullptr;
  decltype(&ncclCommDestroy) CommDestroy = nullptr;
  decltype(&ncclCommAbort) CommAbort = nullptr;
  decltype(&ncclAllGather) AllGather = nullptr;
  decltype(&ncclAllReduce) AllReduce = nullptr;
  decltype(&ncclGetErrorString) GetErrorString = nullptr;
  decltype(&ncclGetVersion) GetVersion = nullptr;
  std::string error;
  bool ok = false;
};
static void nccl_load(NcclApi& api) {
    void* h = nullptr;
    const char* names[] = {getenv("BBQ_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
      if (nm && !h) h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
    }
    if (!h) {
      api.error = std::string("cannot load NCCL (libnccl.so.2): ") + (dlerror() ? dlerror() : "not found");
      return;
    }
#define BBQ_NCCL_SYM(field, name)                                            \
  api.field = reinterpret_cast<decltype(api.field)>(dlsym(h, name));        \
  if (!api.field) {                                                          \
    api.error = std::string("NCCL symbol missing: ") + name;                 \
    return;                                                                  \
  }
    BBQ_NCCL_SYM(GetUniqueId, "ncclGetUniqueId")
    BBQ_NCCL_SYM(CommInitRank, "ncclCommInitRank")
    BBQ_NCCL_SYM(CommDestroy, "ncclCommDestroy")
    BBQ_NCCL_SYM(CommAbort, "ncclCommAbort")
    BBQ_NCCL_SYM(AllGather, "ncclAllGather")
    BBQ_NCCL_SYM(AllReduce, "ncclAllReduce")
    BBQ_NCCL_SYM(GetErrorString, "ncclGetErrorString")
    BBQ_NCCL_SYM(GetVersion, "ncclGetVersion")
#undef BBQ_NCCL_SYM
    api.ok = true;
}
// the workers of a device group reach this at the same time
static NcclApi* nccl_api() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, nccl_load, std::ref(api));
  return &api;
}
#define NC(expr)                                                                                        \
  do {                                                                                                  \
    ncclResult_t _r = (expr);                                                                           \
    if (_r != ncclSuccess) return fail(BBQ_ERR_COMM, std::string(#expr) + ": " + nccl_api()->GetErrorString(_r)); \
  } while (0)

// Implicit release (bbq_destroy, a garbage collector's finalizer): ncclCommAbort — LOCAL, never waits for a peer.
// ncclCommDestroy synchronises with the other ranks and deadlocks when one rank's context is finalised while its
// peers are elsewhere (seen: rank 0 in a destructor, rank 1 in a barrier).  bbq_comm_destroy is the orderly,
// collective way out.
static void comm_release(bbq_ctx* c) {
  if (c->comm) {
    NcclApi* a = nccl_api();
    if (a->ok) a->CommAbort(c->comm);
    c->comm = nullptr;
  }
}

extern "C" int bbq_comm_unique_id(uint8_t* out_id) {
  if (!out_id) return fail(BBQ_ERR_NULL, "null");
  static_assert(sizeof(ncclUniqueId) == BBQ_COMM_ID_BYTES, "BBQ_COMM_ID_BYTES must equal sizeof(ncclUniqueId)");
  NcclApi* a = nccl_api();
  if (!a->ok) return fail(BBQ_ERR_COMM, a->error);
  ncclUniqueId id;
  NC(a->GetUniqueId(&id));
  memcpy(out_id, &id, sizeof id);
  return BBQ_OK;
}

extern "C" int bbq_comm_init(bbq_ctx* c, const uint8_t* id_bytes, int rank, int world) {
  if (!c || !id_bytes) return fail(BBQ_ERR_NULL, "null");
  TRY(group_guard(c));
  if (world < 1 || rank < 0 || rank >= world) return fail(BBQ_ERR_INVALID_ARG, "rank/world out of range");
  if (c->comm) return fail(BBQ_ERR_INVALID_ARG, "this context already has a communicator");
  NcclApi* a = nccl_api();
  if (!a->ok) return fail(BBQ_ERR_COMM, a->error);
  CU(cudaSetDevice(c->device));
  ncclUniqueId id;
  memcpy(&id, id_bytes, sizeof id);
  ncclComm_t comm = nullptr;
  NC(a->CommInitRank(&comm, world, id, rank));
  c->comm = comm;
  c->rank = rank;
  c->world = world;
  return BBQ_OK;
}

extern "C" int bbq_comm_destroy(bbq_ctx* c) {
  if (!c) return fail(BBQ_ERR_NULL, "null");
  TRY(group_guard(c));
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));
  if (c->comm) {
    NcclApi* a = nccl_api();
    if (a->ok) NC(a->CommDestroy(c->comm));
    c->comm = nullptr;
  }
  c->rank = 0;
  c->world = 1;
  return BBQ_OK;
}

extern "C" int bbq_comm_info(bbq_ctx* c, int* rank, int* world, int* nccl_version) {
  if (!c) return fail(BBQ_ERR_NULL, "null");
  if (rank) *rank = c->rank;
  if (world) *world = c->comm ? c->world : 1;
  if (nccl_version) {
    *nccl_version = 0;
    NcclApi* a = nccl_api();
    if (c->comm && a->ok) a->GetVersion(nccl_version);
  }
  return BBQ_OK;
}

// rows over all shards (cached per index; one 8-byte all-reduce when the shard has grown)
static int global_rows(bbq_index* ix, cudaStream_t st, uint64_t* out) {
  bbq_ctx* c = ix->ctx;
  if (!c->comm || c->world == 1) {
    *out = ix->n;
    return BBQ_OK;
  }
  if (ix->n_global_for != ix->n) {
    TRY(c->nglob.reserve(2 * sizeof(unsigned long long)));
    unsigned long long mine = ix->n, all = 0;
    CU(cudaMemcpyAsync(c->nglob.p, &mine, sizeof mine, cudaMemcpyHostToDevice, st));
    NC(nccl_api()->AllReduce(c->nglob.p, c->nglob.as<unsigned long long>() + 1, 1, ncclUint64, ncclSum, c->comm, st));
    CU(cudaMemcpyAsync(&all, c->nglob.as<unsigned long long>() + 1, sizeof all, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    ix->n_global = all;
    ix->n_global_for = ix->n;
  }
  *out = ix->n_global;
  return BBQ_OK;
}

extern "C" int bbq_search_sharded_device(bbq_index* ix, const float* d_queries, uint32_t nq, uint32_t k,
                                         int32_t* d_out_idx, float* d_out_score, void* stream) {
  if (!ix) return fail(BBQ_ERR_NULL, "target vector set must not be null");
  if (!d_queries || !d_out_idx || !d_out_score) return fail(BBQ_ERR_NULL, "query vector must not be null");
  if (nq == 0 || k == 0) return BBQ_OK;
  if (k > K_MAX) return fail(BBQ_ERR_UNSUPPORTED, "k > 4096 is not supported by the device top-k");
  bbq_ctx* c = ix->ctx;
  TRY(group_guard(c));
  if (!c->comm || c->world == 1) return bbq_search_device(ix, d_queries, nq, k, d_out_idx, d_out_score, stream);
  CU(cudaSetDevice(c->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : c->stream;
  StreamBridge bridge(c, st);  // (the local search inside builds its own, nested: harmless)
  const size_t cnt = (size_t)nq * k;
  TRY(c->loc_idx.reserve(cnt * sizeof(int32_t)));
  TRY(c->loc_score.reserve(cnt * sizeof(float)));
  TRY(c->keys_local.reserve(cnt * sizeof(uint64_t)));
  TRY(c->keys_all.reserve(cnt * sizeof(uint64_t) * (size_t)c->world));
  TRY(bbq_search_device(ix, d_queries, nq, k, c->loc_idx.as<int32_t>(), c->loc_score.as<float>(), st));
  {
    ProfScope prof(c, st, PROF_SELECT);
    LAUNCH(c, k_pack_keys, (unsigned)((cnt + 255) / 256), 256, 0, st, c->loc_idx.as<int32_t>(), c->loc_score.as<float>(),
           (int64_t)cnt, c->keys_local.as<uint64_t>());
  }
  NC(nccl_api()->AllGather(c->keys_local.p, c->keys_all.p, cnt, ncclUint64, c->comm, st));
  // merge: every rank selects the k best of world * k keys per query (identical result on every rank)
  return merge_topk(c, nullptr, nullptr, c->keys_all.as<uint64_t>(), (uint32_t)c->world, (int)nq, k, d_out_idx,
                    d_out_score, st);
}

extern "C" int bbq_search_sharded(bbq_index* ix, const float* queries, uint32_t nq, int64_t k, int32_t* out_idx,
                                  float* out_score, uint32_t* out_count) {
  if (out_count) *out_count = 0;
  if (!queries) return fail(BBQ_ERR_NULL, "query vector must not be null");
  if (!ix) return fail(BBQ_ERR_NULL, "target vector set must not be null");
  if (k < 0) return fail(BBQ_ERR_NEGATIVE_K, "k must not be negative");
  if (k == 0 || nq == 0) return BBQ_OK;
  if (!out_idx || !out_score) return fail(BBQ_ERR_NULL, "output buffers must not be null");
  bbq_ctx* c = ix->ctx;
  TRY(group_guard(c));
  if (!c->comm || c->world == 1) return bbq_search(ix, queries, nq, k, out_idx, out_score, out_count);  // one shard: the plain entry
  CU(cudaSetDevice(c->device));
  uint64_t n_all = 0;
  TRY(global_rows(ix, c->stream, &n_all));
  const uint32_t kk = (uint32_t)std::min<int64_t>(k, (int64_t)std::min<uint64_t>(n_all, 0x7FFFFFFFull));
  if (kk > K_MAX) return fail(BBQ_ERR_UNSUPPORTED, "k > 4096 is not supported by the device top-k");
  TRY(c->out_idx.reserve((size_t)nq * kk * sizeof(int32_t)));
  TRY(c->out_score.reserve((size_t)nq * kk * sizeof(float)));
  TRY(stage_queries(c, queries, nq, ix->dim));
  {
    QueryScreen screen(c, c->qrows.as<float>(), c->stream);
    TRY(screen.armed);
    TRY(bbq_search_sharded_device(ix, c->qrows.as<float>(), nq, kk, c->out_idx.as<int32_t>(), c->out_score.as<float>(),
                                  c->stream));
    TRY(screen.read_back(c->stream));
  }
  TRY(copy_results(c, nq, (size_t)k, kk, out_idx, out_score));
  TRY(QueryScreen::verdict(c));
  if (out_count) *out_count = kk;
  return BBQ_OK;
}

// ------------------------------------------------------------------------------------------------
// oversampled search + exact re-rank across row shards: the sharded search's global top-m candidates on every rank,
// each candidate scored exactly by the one rank that holds its row (bbq_rerank_owned_device), the f64 bits summed as
// integers in one ncclAllReduce (every other rank contributes 0), and the same k_rerank_select on every rank.
// ------------------------------------------------------------------------------------------------
extern "C" int bbq_rerank_owned_device(bbq_index* ix, const float* d_queries, uint32_t nq, const int32_t* d_cand_idx,
                                       uint32_t m, uint64_t* d_true_bits, void* stream) {
  if (!ix) return fail(BBQ_ERR_NULL, "target vector set must not be null");
  if (!d_queries || !d_cand_idx || !d_true_bits) return fail(BBQ_ERR_NULL, "null");
  TRY(check_attached_rows(ix));
  if (nq == 0 || m == 0) return BBQ_OK;
  bbq_ctx* c = ix->ctx;
  CU(cudaSetDevice(c->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : c->stream;
  StreamBridge bridge(c, st);
  return launch_rerank_scores(ix, /*owned_only=*/true, d_queries, nq, m, d_cand_idx, reinterpret_cast<double*>(d_true_bits), st);
}

// One all-gather of every rank's {base, rows, rows attached, status of its local preparation}, before any collective
// that depends on per-rank state: every rank derives the same verdict from the same words, so either all ranks go on
// or all return the same status and message.  Attached rows must cover each shard (an empty shard needs none), and
// the shards' id ranges must be disjoint: two owners of one id would add their bits together.
static int agree_on_shards(bbq_index* ix, int local_status, cudaStream_t st, uint64_t* n_global) {
  bbq_ctx* c = ix->ctx;
  const int world = c->world;
  TRY(c->nglob.reserve((size_t)(4 + 4 * world) * sizeof(unsigned long long)));
  unsigned long long* d = c->nglob.as<unsigned long long>();
  const unsigned long long mine[4] = {ix->base, ix->n, ix->rows_n, (unsigned long long)local_status};
  std::vector<unsigned long long> all((size_t)4 * world);
  CU(cudaMemcpyAsync(d, mine, sizeof mine, cudaMemcpyHostToDevice, st));
  NC(nccl_api()->AllGather(d, d + 4, 4, ncclUint64, c->comm, st));
  CU(cudaMemcpyAsync(all.data(), d + 4, all.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  auto word = [&](int r, int f) { return all[(size_t)4 * r + f]; };
  for (int r = 0; r < world; r++)
    if (word(r, 3) != BBQ_OK)
      return fail((int)word(r, 3), "sharded re-rank: rank " + std::to_string(r) + " could not reserve its scratch (status " +
                                       std::to_string(word(r, 3)) + ")");
  uint64_t total = 0;
  std::vector<int> order;
  for (int r = 0; r < world; r++) {
    const uint64_t n = word(r, 1), rows_n = word(r, 2);
    if (n > 0 && rows_n == 0)
      return fail(BBQ_ERR_INVALID_ARG, "sharded re-rank: rank " + std::to_string(r) +
                                           " has no original rows attached (bbq_index_attach_rows)");
    if (n > 0 && rows_n != n)
      return fail(BBQ_ERR_INVALID_ARG, "sharded re-rank: rank " + std::to_string(r) + " has rows attached for " +
                                           std::to_string(rows_n) + " rows, index has " + std::to_string(n));
    if (n > 0) order.push_back(r);
    total += n;
  }
  std::sort(order.begin(), order.end(), [&](int a, int b) { return word(a, 0) < word(b, 0) || (word(a, 0) == word(b, 0) && a < b); });
  for (size_t i = 1; i < order.size(); i++) {
    const int a = order[i - 1], b = order[i];
    if (word(a, 0) + word(a, 1) > word(b, 0))
      return fail(BBQ_ERR_INVALID_ARG, "sharded re-rank: the row ids of rank " + std::to_string(a) + " [" +
                                           std::to_string(word(a, 0)) + ", " + std::to_string(word(a, 0) + word(a, 1)) +
                                           ") overlap those of rank " + std::to_string(b) + " [" + std::to_string(word(b, 0)) +
                                           ", " + std::to_string(word(b, 0) + word(b, 1)) + ")");
  }
  *n_global = total;
  return BBQ_OK;
}

extern "C" int bbq_search_rerank_sharded(bbq_index* ix, const float* queries, uint32_t nq, uint32_t k, uint32_t factor,
                                         int32_t* out_idx, float* out_qscore, double* out_true, uint32_t* out_count) {
  if (out_count) *out_count = 0;
  if (!ix) return fail(BBQ_ERR_NULL, "target vector set must not be null");
  if (!queries) return fail(BBQ_ERR_NULL, "query vector must not be null");
  bbq_ctx* c = ix->ctx;
  TRY(group_guard(c));
  if (!c->comm || c->world == 1)  // one shard: the plain entry
    return bbq_search_rerank(ix, queries, nq, k, factor, out_idx, out_qscore, out_true, out_count);
  // the replicated arguments: every rank reaches the same verdict on them without communicating
  const bool work = nq != 0 && k != 0;
  if (work && (!out_idx || !out_qscore || !out_true)) return fail(BBQ_ERR_NULL, "output buffers must not be null");
  if (work && (factor == 0 || (uint64_t)k * factor > K_MAX))
    return fail(BBQ_ERR_UNSUPPORTED, "k * oversampleFactor must be in 1..4096");
  CU(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  const uint32_t mk = work ? k * factor : 0;  // candidates per query before the clamp to the rows of all shards
  const int prep = work ? reserve_rerank(c, ix->dim, nq, mk, k) : BBQ_OK;
  uint64_t n_global = 0;
  TRY(agree_on_shards(ix, prep, st, &n_global));
  const uint32_t m = (uint32_t)std::min<uint64_t>(mk, n_global);
  const uint32_t kk = std::min(k, m);
  if (m == 0) return BBQ_OK;
  TRY(stage_queries(c, queries, nq, ix->dim));
  {
    QueryScreen screen(c, c->qrows.as<float>(), st);
    TRY(screen.armed);
    TRY(bbq_search_sharded_device(ix, c->qrows.as<float>(), nq, m, c->out_idx.as<int32_t>(), c->out_score.as<float>(), st));
    TRY(screen.read_back(st));
  }
  {
    ProfScope prof(c, st, PROF_SELECT);
    TRY(launch_rerank_scores(ix, /*owned_only=*/true, c->qrows.as<float>(), nq, m, c->out_idx.as<int32_t>(),
                             c->rr_true.as<double>(), st));
    // integer sum, never a floating-point one: exactly one rank owns each filled slot, so the owner's bits arrive
    // unchanged (-0.0 and NaN payloads included)
    NC(nccl_api()->AllReduce(c->rr_true.p, c->rr_true.p, (size_t)nq * m, ncclUint64, ncclSum, c->comm, st));
  }
  TRY(rerank_select_and_copy(c, st, nq, m, k, kk, out_idx, out_qscore, out_true));
  if (out_count) *out_count = kk;
  return BBQ_OK;
}

#include "bbq_io.cuh"  // index image on disk, whole and across row shards (uses the NCCL plumbing above)

// ------------------------------------------------------------------------------------------------
// the index build across row shards (collective).  Ranks hold consecutive row ranges in rank order.  The reference
// centroid is one f32 sum in row order, which shards cannot split, so it is CHAINED: rank r continues the running sum
// of ranks 0 .. r-1 over its rows (k_centroid_chain), and one integer-sum ncclAllReduce, to which every other rank
// contributes 0, hands the owner's bits to every rank.  Everything else (validation, norms, quantisation) runs on all
// ranks at once.  Every phase ends in an exchange of each rank's status, as in the sharded save and load.
// ------------------------------------------------------------------------------------------------
// the verdict on an exchange whose words 0 and 1 carry the failing rank's (vector, position) in the whole corpus
static int first_failure_at(const std::vector<RankWord>& all, const char* what) {
  for (size_t r = 0; r < all.size(); r++)
    if (all[r].status != BBQ_OK)
      return fail((int)all[r].status, std::string(what) + ": rank " + std::to_string(r) + ": " + all[r].msg,
                  (int64_t)all[r].w[0], (int64_t)all[r].w[1]);
  return BBQ_OK;
}

// this rank's shard once the centroid is known: the chained sum over N rows (d_sum) or the caller's centroid, its
// centroidDP, then its rows quantised, and its base
static int finish_shard(bbq_index* ix, const float* d_sum, const float* centroid, uint64_t total, const float* rows,
                        bool is_host, uint64_t n, uint64_t base) {
  bbq_ctx* c = ix->ctx;
  if (centroid) {
    CU(cudaMemcpyAsync(ix->centroid, centroid, ix->dim * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  } else {
    CU(cudaMemcpyAsync(ix->centroid, d_sum, ix->dim * sizeof(float), cudaMemcpyDeviceToDevice, c->stream));
    LAUNCH(c, k_centroid_finish, (ix->dim + 127) / 128, 128, 0, c->stream, ix->centroid, (int)ix->dim, (double)total);
  }
  TRY(finish_centroid(ix));
  if (n > 0) TRY(append_impl(ix, rows, is_host, n));
  return bbq_index_set_base(ix, base);
}

// rows_validated: the caller has validated the host rows already (a device group does it before any collective)
static int build_sharded(bbq_ctx* c, const float* rows, bool is_host, uint64_t n, uint32_t dim, const float* centroid,
                         bbq_index** out_index, bool rows_validated = false) {
  if (!c) return fail(BBQ_ERR_NULL, "null ctx/out_index");
  TRY(group_guard(c));
  if (!c->comm || c->world == 1) {  // one shard: the plain entry
    if (is_host && rows_validated) return build_impl(c, rows, true, n, dim, centroid, out_index);
    return is_host ? bbq_index_build(c, rows, n, dim, centroid, out_index)
                   : bbq_index_build_device(c, rows, n, dim, centroid, out_index);
  }
  if (out_index) *out_index = nullptr;
  CU(cudaSetDevice(c->device));
  const char* what = "sharded build";
  const int world = c->world;
  std::vector<RankWord> all;
  // 1. every rank's {rows, dim, similarity, indexBits, centroid given, centroid fingerprint} and argument status
  int st = BBQ_OK;
  if (!out_index) st = fail(BBQ_ERR_NULL, "null ctx/out_index");
  else if (n > 0 && !rows) st = fail(BBQ_ERR_NULL, "rows is null");
  else if (n > 0 && dim == 0) st = fail(BBQ_ERR_INVALID_ARG, "dim must be > 0");
  RankWord mine = rank_word(st);
  const uint64_t shape[6] = {n, dim, (uint64_t)c->cfg.similarity, (uint64_t)c->cfg.index_bits, centroid ? 1u : 0u,
                             centroid ? bbqio::fingerprint(centroid, (size_t)dim * sizeof(float)) : 0};
  memcpy(mine.w, shape, sizeof shape);
  TRY(gather_ranks(c, mine, all));
  TRY(first_failure(all, what));
  std::vector<uint64_t> rows_of((size_t)world);
  uint64_t total = 0, base = 0;
  uint32_t D = 0;
  int first_full = -1;
  for (int r = 0; r < world; r++) {
    rows_of[r] = all[r].w[0];
    if (rows_of[r] > 0x7FFFFFF0ull)
      return fail(BBQ_ERR_UNSUPPORTED, std::string(what) + ": rank " + std::to_string(r) +
                                           " holds more than 2^31 rows (result ids are int32)");
    if (r < c->rank) base += rows_of[r];
    total += rows_of[r];
    if (rows_of[r] > 0 && first_full < 0) {
      first_full = r;
      D = (uint32_t)all[r].w[1];
    }
  }
  if (total == 0) return fail(BBQ_ERR_EMPTY, "vector set must not be empty");
  if (total > 0x7FFFFFFFull)
    return fail(BBQ_ERR_UNSUPPORTED, std::string(what) + ": " + std::to_string(total) +
                                         " rows over all ranks (global row ids are int32)");
  for (int r = 0; r < world; r++) {
    const uint64_t d = all[r].w[1];
    if (d != D && (rows_of[r] > 0 || d != 0))
      return fail(BBQ_ERR_INVALID_ARG, std::string(what) + ": rank " + std::to_string(r) + " has dimension " +
                                           std::to_string(d) + ", the rows of rank " + std::to_string(first_full) +
                                           " have " + std::to_string(D));
    if (all[r].w[2] != all[0].w[2] || all[r].w[3] != all[0].w[3])
      return fail(BBQ_ERR_INVALID_ARG, std::string(what) + ": rank " + std::to_string(r) + " has similarity " +
                                           std::to_string(all[r].w[2]) + " and indexBits " + std::to_string(all[r].w[3]) +
                                           ", rank 0 has " + std::to_string(all[0].w[2]) + " and " +
                                           std::to_string(all[0].w[3]));
    if (all[r].w[4] != all[0].w[4] || all[r].w[5] != all[0].w[5])
      return fail(BBQ_ERR_INVALID_ARG, std::string(what) + ": the centroid of rank " + std::to_string(r) +
                                           " differs from rank 0's (every rank passes NULL, or the same centroid)");
  }
  if (c->cfg.index_bits > INDEX_BITS_MAX)
    return fail(BBQ_ERR_UNSUPPORTED, "indexBits > 2 is not built on device");
  // 2. host rows validated (positions in the whole corpus), this rank's index reserved and, for device rows, the
  //    COSINE norms computed ahead of its turn in the chain
  const bool cosine = c->cfg.similarity == BBQ_SIM_COSINE;
  int64_t bad_vec = -1, bad_pos = -1;
  st = is_host && n > 0 && !rows_validated ? validate_rows(rows, n, D, cosine) : BBQ_OK;
  if (st != BBQ_OK) {
    bad_vec = (int64_t)base + g_err_vec;
    bad_pos = g_err_pos;
  }
  IndexGuard g;
  if (st == BBQ_OK && (st = index_alloc(c, std::max<uint64_t>(n, 1), D, &g.ix)) == BBQ_OK) g.ix->n = 0;
  if (st == BBQ_OK && !centroid) st = c->chain.reserve(((size_t)D + 1) * sizeof(uint32_t));
  if (st == BBQ_OK && !centroid && !is_host) st = row_norms(c, rows, (int64_t)n, D);
  mine = rank_word(st);
  mine.w[0] = (uint64_t)bad_vec;
  mine.w[1] = (uint64_t)bad_pos;
  TRY(gather_ranks(c, mine, all));
  TRY(first_failure_at(all, what));
  // 3. the chain, rank by rank (ranks without rows are skipped: every rank knows the row counts)
  float* sum = c->chain.as<float>();
  if (!centroid) {
    uint32_t* status_word = c->chain.as<uint32_t>() + D;
    for (int r = 0; r < world; r++) {
      if (rows_of[r] == 0) continue;
      int mine_st = BBQ_OK;
      if (r == c->rank) {
        mine_st = chain_rows(c, rows, is_host, n, D, base == 0, sum, /*norms_ready=*/!is_host);
        const uint32_t s = (uint32_t)mine_st;
        CU(cudaMemcpyAsync(status_word, &s, sizeof s, cudaMemcpyHostToDevice, c->stream));
      } else {
        CU(cudaMemsetAsync(sum, 0, ((size_t)D + 1) * sizeof(uint32_t), c->stream));
      }
      // integer sum: the owner's bits arrive unchanged (-0.0, subnormals and NaN payloads included)
      NC(nccl_api()->AllReduce(sum, sum, (size_t)D + 1, ncclUint32, ncclSum, c->comm, c->stream));
      uint32_t verdict = 0;
      CU(cudaMemcpyAsync(&verdict, status_word, sizeof verdict, cudaMemcpyDeviceToHost, c->stream));
      CU(cudaStreamSynchronize(c->stream));
      if (verdict != BBQ_OK) {  // the owner's message reaches every rank
        TRY(gather_ranks(c, rank_word(mine_st), all));
        return first_failure(all, what);
      }
    }
  }
  // 4. every rank quantises its rows; a failure on any rank fails all, and none keeps a half-built shard
  TRY(gather_ranks(c, rank_word(finish_shard(g.ix, sum, centroid, total, rows, is_host, n, base)), all));
  TRY(first_failure(all, what));
  *out_index = g.release();
  return BBQ_OK;
}

extern "C" int bbq_index_build_sharded(bbq_ctx* c, const float* rows, uint64_t n, uint32_t dim, const float* centroid,
                                       bbq_index** out_index) {
  return build_sharded(c, rows, true, n, dim, centroid, out_index);
}
extern "C" int bbq_index_build_sharded_device(bbq_ctx* c, const float* d_rows, uint64_t n, uint32_t dim,
                                              const float* centroid, bbq_index** out_index) {
  return build_sharded(c, d_rows, false, n, dim, centroid, out_index);
}

// Page-locked host buffers for hosts that want the H2D / D2H copies of bbq_search* to run at full PCIe speed
// (a Node host wraps them in external ArrayBuffers; any host pointer works, pageable memory is merely slower).
extern "C" void* bbq_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) {
    cudaGetLastError();
    fail(BBQ_ERR_OOM, "cudaMallocHost failed");
    return nullptr;
  }
  return p;
}
extern "C" void bbq_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

// ------------------------------------------------------------------------------------------------
// quantizeQueryVector / computeQuantizationAccuracy (the class members beside the search path)
// ------------------------------------------------------------------------------------------------
extern "C" int bbq_quantize_query(bbq_ctx* c, const float* query, const float* centroid, uint32_t dim, uint8_t* codes,
                                  double* corr4) {
  if (!c || !query || !centroid) return fail(BBQ_ERR_NULL, "null");
  if (dim == 0) return fail(BBQ_ERR_INVALID_ARG, "dim must be > 0");
  CU(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  const int row_bytes = row_bytes_for(dim, std::min<uint32_t>(c->cfg.index_bits, INDEX_BITS_MAX));
  TRY(c->cenv.reserve((size_t)dim * sizeof(float)));
  TRY(stage_queries(c, query, 1, dim));
  CU(cudaMemcpyAsync(c->cenv.p, centroid, (size_t)dim * sizeof(float), cudaMemcpyHostToDevice, st));
  const bool cosine = c->cfg.similarity == BBQ_SIM_COSINE;
  QueryScreen screen(c, c->qrows.as<float>(), st);
  TRY(screen.armed);
  TRY(quantize_rows(c, c->qrows.as<float>(), 1, (int)dim, row_bytes, c->cenv.as<float>(), cosine ? 1 : 0, st));
  if (codes) CU(cudaMemcpyAsync(codes, c->qcodes.p, dim, cudaMemcpyDeviceToHost, st));
  if (corr4) CU(cudaMemcpyAsync(corr4, c->qcorr.p, 4 * sizeof(double), cudaMemcpyDeviceToHost, st));
  TRY(screen.read_back(st));
  CU(cudaStreamSynchronize(st));
  return QueryScreen::verdict(c);
}

extern "C" int bbq_quantization_accuracy(bbq_ctx* c, const float* rows, const float* queries, uint64_t n, uint32_t dim,
                                         uint64_t target_ord, double* out5) {
  if (!c || !out5) return fail(BBQ_ERR_NULL, "null");
  if (n == 0 || !rows || !queries) return fail(BBQ_ERR_EMPTY, "vector sets must not be empty");
  if (target_ord >= n) return fail(BBQ_ERR_INVALID_ARG, "target row out of range");
  const uint32_t qb = c->cfg.query_bits;
  // computeQuantizedScore, src/binaryQuantizedScorer.ts:78-97: only 1-bit and 4-bit queries
  if (qb != 1 && qb != 4) return fail(BBQ_ERR_UNSUPPORTED, "unsupported query bits: only 1 and 4 (computeQuantizedScore)");
  if (c->cfg.index_bits != 1) return fail(BBQ_ERR_UNSUPPORTED, "computeQuantizationAccuracy scores through the single-vector scorer, which knows 1-bit indexes only");
  if (n > 0x7FFFFFF0ull) return fail(BBQ_ERR_UNSUPPORTED, "too many vectors");
  IndexGuard g;
  TRY(bbq_index_build(c, rows, n, dim, nullptr, &g.ix));  // 1. quantizeVectors(originalVectors), reference-order centroid
  bbq_index* ix = g.ix;
  cudaStream_t st = c->stream;
  const bool cosine = c->cfg.similarity == BBQ_SIM_COSINE;
  TRY(c->rr_q.reserve((size_t)dim * sizeof(float)));
  TRY(c->rr_true.reserve((size_t)n * sizeof(double)));
  TRY(c->rr_t.reserve((size_t)n * sizeof(double)));
  TRY(c->cacc.reserve(5 * sizeof(double)));
  TRY(stage_queries(c, queries, n, dim));
  CU(cudaMemcpyAsync(c->rr_q.p, rows + target_ord * dim, (size_t)dim * sizeof(float), cudaMemcpyHostToDevice, st));
  QueryScreen screen(c, c->qrows.as<float>(), st);
  TRY(screen.armed);
  // 2. quantizeQueryVector(query, centroid): ONE normalisation for COSINE (:271-299)
  TRY(quantize_rows(c, c->qrows.as<float>(), (int)n, (int)dim, ix->row_bytes, ix->centroid, cosine ? 1 : 0, st));
  LAUNCH(c, k_accuracy_scores, (unsigned)((n + RERANK_WARPS - 1) / RERANK_WARPS), RERANK_WARPS * 32, 0, st,
         c->qcodes.as<uint8_t>(), ix->row_bytes * 8, c->qcorr.as<double>(), (int)n, qb == 1 ? 1 : 0,
         ix->codes + target_ord * ix->row_bytes, ix->lower + target_ord, ix->upper + target_ord, ix->addc + target_ord,
         ix->compsum + target_ord, c->qrows.as<float>(), c->rr_q.as<float>(), (int)dim, (int)c->cfg.similarity,
         qb == 1 ? ix->cdp : 0.0, c->rr_true.as<double>(), c->rr_t.as<double>());
  // 3. statistics (sequential sums, one thread: the reference's order)
  LAUNCH(c, k_accuracy_stats, 1, 32, 0, st, c->rr_true.as<double>(), c->rr_t.as<double>(), (int64_t)n, c->cacc.as<double>());
  CU(cudaMemcpyAsync(out5, c->cacc.p, 5 * sizeof(double), cudaMemcpyDeviceToHost, st));
  TRY(screen.read_back(st));
  CU(cudaStreamSynchronize(st));
  return QueryScreen::verdict(c);
}

// ------------------------------------------------------------------------------------------------
// parity / debug taps
// ------------------------------------------------------------------------------------------------
static int debug_prepare_query(bbq_index* ix, const float* query) {
  if (!ix || !query) return fail(BBQ_ERR_NULL, "null");
  bbq_ctx* c = ix->ctx;
  CU(cudaSetDevice(c->device));
  TRY(c->qrows.reserve((size_t)ix->dim * sizeof(float)));
  CU(cudaMemcpyAsync(c->qrows.p, query, (size_t)ix->dim * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  return quantize_queries(ix, c->qrows.as<float>(), 1, c->stream);
}

extern "C" int bbq_debug_quantize_query(bbq_index* ix, const float* query, uint8_t* codes, double* corr4) {
  TRY(debug_prepare_query(ix, query));
  bbq_ctx* c = ix->ctx;
  if (codes) CU(cudaMemcpyAsync(codes, c->qcodes.p, ix->dim, cudaMemcpyDeviceToHost, c->stream));
  if (corr4) CU(cudaMemcpyAsync(corr4, c->qcorr.p, 4 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return BBQ_OK;
}

static int debug_dense(bbq_index* ix, const float* query, int32_t* out_dots, float* out_scores) {
  TRY(debug_prepare_query(ix, query));
  bbq_ctx* c = ix->ctx;
  const int64_t n = (int64_t)ix->n, ntiles = (n + TILE_ROWS - 1) / TILE_ROWS;
  TRY(c->dump.reserve((size_t)ntiles * TILE_ROWS * sizeof(float)));
  TRY(c->dots.reserve((size_t)n * sizeof(int32_t)));
  ScanParams p = base_scan_params(ix, 1);
  p.dump = c->dump.as<float>();
  p.dump_ld = ntiles * TILE_ROWS;
  p.dots = c->dots.as<int32_t>();
  TRY(launch_scan(ix, SCAN_DUMP, p, ntiles, c->stream));
  if (out_dots) CU(cudaMemcpyAsync(out_dots, c->dots.p, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  if (out_scores) CU(cudaMemcpyAsync(out_scores, c->dump.p, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return BBQ_OK;
}

extern "C" int bbq_debug_qcdist(bbq_index* ix, const float* query, int32_t* out_dots) {
  return debug_dense(ix, query, out_dots, nullptr);
}
extern "C" int bbq_debug_scores(bbq_index* ix, const float* query, float* out_scores) {
  return debug_dense(ix, query, nullptr, out_scores);
}

// The tensor-core scan's integers: accumulator >> 3 of every (query, row) pair, through k_scan_mma<SCAN_DUMP>
// (the popcount kernel is NOT involved) — the tap bbq_debug_qcdist lacks.  out_dots: [nq][n] int32, HOST.
extern "C" int bbq_debug_qcdist_batch(bbq_index* ix, const float* queries, uint32_t nq, int32_t* out_dots) {
  if (!ix || !queries || !out_dots) return fail(BBQ_ERR_NULL, "null");
  if (nq == 0) return BBQ_OK;
  bbq_ctx* c = ix->ctx;
  CU(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  const int saved_engine = c->scan_engine;
  c->scan_engine = 2;  // whatever the batch size: this tap exists to exercise tcgen05
  MmaPlan pl;
  const bool ok = mma_plan(ix, (int)nq, &pl);
  c->scan_engine = saved_engine;
  if (!ok) return fail(BBQ_ERR_UNSUPPORTED, "the tensor-core scan cannot run this configuration (queryBits > 5, dim > 4096 or > 4096 queries)");
  TRY(c->qrows.reserve((size_t)nq * ix->dim * sizeof(float)));
  CU(cudaMemcpyAsync(c->qrows.p, queries, (size_t)nq * ix->dim * sizeof(float), cudaMemcpyHostToDevice, st));
  TRY(quantize_queries(ix, c->qrows.as<float>(), (int)nq, st));
  TRY(prepare_mma_operands(ix, (int)nq, pl, st));
  TRY(ensure_bounds(ix, st));
  const int64_t n = (int64_t)ix->n, ntiles = (n + TILE_ROWS - 1) / TILE_ROWS;
  // a bounded scratch: tiles are dumped in groups and copied out row-range by row-range
  const int64_t group_tiles = std::max<int64_t>(1, std::min<int64_t>(ntiles, (int64_t)(1ll << 28) / ((int64_t)nq * TILE_ROWS)));
  const int64_t ld = group_tiles * TILE_ROWS;
  TRY(c->dots.reserve((size_t)nq * ld * sizeof(int32_t)));
  for (int64_t t0 = 0; t0 < ntiles; t0 += group_tiles) {
    const int64_t tn = std::min(group_tiles, ntiles - t0);
    const int64_t rows_here = std::min<int64_t>(tn * TILE_ROWS, n - t0 * TILE_ROWS);
    TRY(launch_scan_mma(ix, SCAN_DUMP, (int)nq, 1, pl, t0, 1, tn, nullptr, ld, nullptr, nullptr, 0, nullptr, st,
                        c->dots.as<int32_t>()));
    CU(cudaMemcpy2DAsync(out_dots + t0 * TILE_ROWS, (size_t)n * sizeof(int32_t), c->dots.p, (size_t)ld * sizeof(int32_t),
                         (size_t)rows_here * sizeof(int32_t), nq, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
  }
  return BBQ_OK;
}

#include "bbq_group.cuh"  // device groups: one process, one caller thread, the collectives above on every GPU
