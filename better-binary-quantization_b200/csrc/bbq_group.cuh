// bbq_group.cuh — device groups (included by bbq_api.cu after the collective entries it drives).
//
// One process drives every GPU of a box: a group owns one context, one NCCL communicator and one persistent host
// worker thread per GPU.  Each group entry checks its arguments on the caller's thread, hands the EXISTING collective
// entry of every rank to that rank's worker, waits for all of them, and returns what the lowest failing rank returned
// (or rank 0's results).  Rank r holds rows [r*per, min(N, (r+1)*per)), per = ceil(N / n) (host/sharded.py
// shard_bounds, what bbq_index_load_sharded does), with its base set, so every result id is global.
#include <chrono>
#include <condition_variable>
#include <functional>
#include <thread>

struct GroupResult {
  int status = BBQ_OK;
  std::string msg;
  int64_t vec = -1, pos = -1;
};

struct bbq_group {
  std::vector<int> devices;
  std::vector<bbq_ctx*> ctx;
  std::vector<std::thread> workers;
  std::mutex mu;
  std::condition_variable cv_job, cv_done;
  std::function<int(uint32_t)> job;  // what every worker runs for the current generation, given its rank
  uint64_t gen = 0;
  uint32_t done = 0;
  bool stop = false;
  std::vector<GroupResult> res;
  std::vector<char> finished;
  int live = 0;  // group indexes alive
  bool comms = false;  // the communicators are being created or exist: only then can a rank strand its peers
  bool failed = false;
  std::string failed_msg;
  // only rank 0 writes into the caller's buffers; rank r >= 1 writes its (identical) lists here
  std::vector<std::vector<int32_t>> h_idx;
  std::vector<std::vector<float>> h_score;
  std::vector<std::vector<double>> h_true;
  uint32_t size() const { return (uint32_t)devices.size(); }
};

struct bbq_group_index {
  bbq_group* g = nullptr;
  std::vector<bbq_index*> shards;
  std::vector<uint64_t> lo;  // first row of each shard, lo[n_devices] = n
  uint64_t n = 0;
  uint32_t dim = 0;
  int ib = 1;
  std::vector<float> centroid;
  double cdp = 0.0;
  bool rows_attached = false;
};

// After a runtime failure of one rank, how long the others get to return on their own: the collective entries
// exchange most failures, so their peers return the same status right after.
static constexpr auto GROUP_ABORT_GRACE = std::chrono::seconds(5);

static void group_worker(bbq_group* g, uint32_t rank) {
  uint64_t seen = 0;
  std::unique_lock<std::mutex> lk(g->mu);
  for (;;) {
    g->cv_job.wait(lk, [&] { return g->stop || g->gen != seen; });
    if (g->stop) return;
    seen = g->gen;
    const std::function<int(uint32_t)>& job = g->job;
    lk.unlock();
    g_err.clear();
    g_err_vec = g_err_pos = -1;
    const int st = job(rank);
    GroupResult r{st, g_err, g_err_vec, g_err_pos};
    t_group_worker = g->ctx[rank];  // set once its context exists (the first job creates it)
    lk.lock();
    g->res[rank] = std::move(r);
    g->finished[rank] = 1;
    g->done++;
    g->cv_done.notify_all();
  }
}

static void group_join(bbq_group* g) {
  {
    std::lock_guard<std::mutex> lk(g->mu);
    g->stop = true;
  }
  g->cv_job.notify_all();
  for (auto& t : g->workers) t.join();
  g->workers.clear();
}

// Every communicator aborted (ncclCommAbort is local and makes the NCCL kernels of a collective that waits for a
// peer return), the way torch's NCCL watchdog unblocks its process group.  The workers are still running, so:
// - the pointer is swapped out atomically before the abort: a worker that reads it afterwards passes NCCL a null
//   communicator and gets an error back, or, at the top of a sharded entry, takes the one-GPU path; its results are
//   discarded either way, because the group is marked failed;
// - a worker that loaded the pointer before the swap and enters NCCL only after the abort has freed the communicator
//   hands NCCL a dangling pointer.  The window is the few instructions between that load and the call; the workers
//   this path exists for are already blocked inside a collective.  Closing it would need a lock the blocked worker
//   holds, which the abort could then never take.
static void group_abort_comms(bbq_group* g) {
  NcclApi* a = nccl_api();
  for (bbq_ctx* c : g->ctx) {
    if (!c) continue;
    ncclComm_t cm = c->comm.exchange(nullptr);
    if (cm && a->ok) a->CommAbort(cm);
  }
}

// Runs job(rank) on every worker and waits for all of them.  Returns the lowest failing rank's status, with its message
// and (vector, position) copied into the caller's thread.  A runtime failure (status >= 100) on one rank while others
// are still running after GROUP_ABORT_GRACE means those wait in a collective the failed rank never joins: every
// communicator is aborted, the workers are joined and the group is marked failed.
static int group_run(bbq_group* g, std::function<int(uint32_t)> job) {
  const uint32_t n = g->size();
  int aborted_after = -1;
  {
    std::unique_lock<std::mutex> lk(g->mu);
    g->job = std::move(job);
    g->done = 0;
    std::fill(g->finished.begin(), g->finished.end(), 0);
    g->gen++;
    g->cv_job.notify_all();
    while (g->done < n) {
      int r_fail = -1;
      for (uint32_t r = 0; r < n && r_fail < 0; r++)
        if (g->finished[r] && g->res[r].status >= BBQ_ERR_NO_DEVICE) r_fail = (int)r;
      if (r_fail < 0 || !g->comms) {  // without communicators no rank can wait for another
        g->cv_done.wait(lk);
        continue;
      }
      if (g->cv_done.wait_for(lk, GROUP_ABORT_GRACE, [&] { return g->done == n; })) break;
      aborted_after = r_fail;
      lk.unlock();
      group_abort_comms(g);
      lk.lock();
      g->cv_done.wait(lk, [&] { return g->done == n; });
    }
  }
  if (aborted_after >= 0) {  // the other ranks' errors come from the abort: report the rank that caused it
    group_join(g);
    const GroupResult& x = g->res[(size_t)aborted_after];
    g->failed = true;
    g->failed_msg = "device group aborted after rank " + std::to_string(aborted_after) + " failed: " + x.msg;
    return fail(x.status, g->failed_msg, x.vec, x.pos);
  }
  for (uint32_t r = 0; r < n; r++) {
    const GroupResult& x = g->res[r];
    if (x.status != BBQ_OK) return fail(x.status, x.msg, x.vec, x.pos);
  }
  return BBQ_OK;
}

static int group_usable(const bbq_group* g) {
  if (g->failed) return fail(BBQ_ERR_COMM, g->failed_msg);
  return BBQ_OK;
}

// Releases what a group holds once its workers are joined (contexts that still hold a communicator abort it locally).
static void group_free(bbq_group* g) {
  group_join(g);
  for (bbq_ctx* c : g->ctx) {
    if (!c) continue;
    c->group = nullptr;
    bbq_destroy(c);
  }
  delete g;
}

extern "C" int bbq_group_create(const bbq_config* config, const int32_t* devices, uint32_t n_devices, bbq_group** out) {
  if (!config || !out) return fail(BBQ_ERR_NULL, "config/out is null");
  *out = nullptr;
  if (!devices || n_devices == 0) return fail(BBQ_ERR_INVALID_ARG, "the device list is empty");
  for (uint32_t i = 0; i < n_devices; i++) {
    if (devices[i] < 0)
      return fail(BBQ_ERR_INVALID_ARG, "device list entry " + std::to_string(i) + " is negative (" +
                                           std::to_string(devices[i]) + ")");
    for (uint32_t j = 0; j < i; j++)
      if (devices[j] == devices[i])
        return fail(BBQ_ERR_INVALID_ARG, "device " + std::to_string(devices[i]) + " appears twice in the device list");
  }
  TRY(check_config(config));
  int ndev = 0;
  TRY(device_count(&ndev));  // no device: no worker is ever started
  for (uint32_t i = 0; i < n_devices; i++)
    if (devices[i] >= ndev) return fail(BBQ_ERR_NO_DEVICE, "device ordinal out of range");
  bbq_group* g = new bbq_group();
  g->devices.assign(devices, devices + n_devices);
  g->ctx.assign(n_devices, nullptr);
  g->res.resize(n_devices);
  g->finished.assign(n_devices, 0);
  g->h_idx.resize(n_devices);
  g->h_score.resize(n_devices);
  g->h_true.resize(n_devices);
  for (uint32_t r = 0; r < n_devices; r++) g->workers.emplace_back(group_worker, g, r);
  // 1. a context on every device; only when all exist, 2. the communicators, all at once
  const bbq_config cfg = *config;
  int st = group_run(g, [g, cfg](uint32_t r) {
    bbq_config c = cfg;
    c.device = g->devices[r];
    const int s = bbq_create(&c, &g->ctx[r]);
    if (s == BBQ_OK) g->ctx[r]->group = g;
    return s;
  });
  if (st == BBQ_OK && n_devices > 1) {
    uint8_t id[BBQ_COMM_ID_BYTES];
    st = bbq_comm_unique_id(id);
    g->comms = true;
    if (st == BBQ_OK)
      st = group_run(g, [g, &id, n_devices](uint32_t r) { return bbq_comm_init(g->ctx[r], id, (int)r, (int)n_devices); });
  }
  if (st != BBQ_OK) {
    const std::string msg = g_err;
    const int64_t v = g_err_vec, p = g_err_pos;
    group_free(g);
    return fail(st, msg, v, p);
  }
  *out = g;
  return BBQ_OK;
}

extern "C" int bbq_group_destroy(bbq_group* g) {
  if (!g) return fail(BBQ_ERR_NULL, "null group");
  if (g->live > 0)
    return fail(BBQ_ERR_INVALID_ARG, std::to_string(g->live) + " group index(es) of this group are still alive");
  int st = BBQ_OK;
  if (!g->failed && g->size() > 1)  // the orderly way out: ncclCommDestroy on every GPU at once
    st = group_run(g, [g](uint32_t r) { return bbq_comm_destroy(g->ctx[r]); });
  const std::string msg = g_err;
  group_free(g);
  return st == BBQ_OK ? BBQ_OK : fail(st, msg);
}

extern "C" int bbq_group_info(const bbq_group* g, uint32_t* n_devices, int32_t* devices) {
  if (!g) return fail(BBQ_ERR_NULL, "null group");
  if (n_devices) *n_devices = g->size();
  if (devices)
    for (uint32_t r = 0; r < g->size(); r++) devices[r] = g->devices[r];
  return BBQ_OK;
}

extern "C" bbq_ctx* bbq_group_context(bbq_group* g, uint32_t rank) {
  if (!g || rank >= g->size()) {
    fail(BBQ_ERR_INVALID_ARG, "no such rank in the device group");
    return nullptr;
  }
  return g->ctx[rank];
}

// ---- group indexes -------------------------------------------------------------------------------------------------
static bbq_group_index* gindex_new(bbq_group* g, uint64_t n) {
  bbq_group_index* gi = new bbq_group_index();
  gi->g = g;
  const uint32_t w = g->size();
  gi->shards.assign(w, nullptr);
  gi->lo.resize(w + 1);
  const uint64_t per = n / w + (n % w != 0);
  for (uint32_t r = 0; r < w; r++) gi->lo[r] = std::min<uint64_t>(n, (uint64_t)r * per);
  gi->lo[w] = n;
  gi->n = n;
  return gi;
}

static void gindex_free(bbq_group_index* gi) {
  for (bbq_index* s : gi->shards) bbq_index_destroy(s);
  delete gi;
}

// after every shard exists: the metadata the read-only members answer from (rank 0 always holds rows)
static int gindex_publish(bbq_group_index* gi, bbq_group_index** out) {
  bbq_index* s0 = gi->shards[0];
  gi->dim = s0->dim;
  gi->ib = s0->ib;
  gi->centroid = s0->centroid_h;
  gi->cdp = s0->cdp;
  gi->g->live++;
  *out = gi;
  return BBQ_OK;
}

// runs a job that creates gi's shards; on failure nothing is kept
static int gindex_make(bbq_group_index* gi, std::function<int(uint32_t)> job, bbq_group_index** out) {
  const int st = group_run(gi->g, std::move(job));
  if (st != BBQ_OK) {
    const std::string msg = g_err;
    const int64_t v = g_err_vec, p = g_err_pos;
    gindex_free(gi);
    return fail(st, msg, v, p);
  }
  return gindex_publish(gi, out);
}

extern "C" int bbq_group_index_build(bbq_group* g, const float* rows, uint64_t n, uint32_t dim, const float* centroid,
                                     bbq_group_index** out) {
  // the checks of bbq_index_build, in its order
  if (!g || !out) return fail(BBQ_ERR_NULL, "null ctx/out_index");
  *out = nullptr;
  TRY(group_usable(g));
  if (n == 0) return fail(BBQ_ERR_EMPTY, "vector set must not be empty");
  if (!rows) return fail(BBQ_ERR_NULL, "rows is null");
  bbq_group_index* gi = gindex_new(g, n);
  // 1. every worker validates its slice; a NaN / Infinity is reported at its vector index in the whole corpus
  const bool cosine = g->ctx[0]->cfg.similarity == BBQ_SIM_COSINE;
  int st = group_run(g, [gi, rows, dim, cosine](uint32_t r) {
    const uint64_t lo = gi->lo[r], cnt = gi->lo[r + 1] - lo;
    const int s = validate_rows(rows + lo * dim, cnt, dim, cosine);
    return s == BBQ_OK ? s : fail(s, g_err, (int64_t)lo + g_err_vec, g_err_pos);
  });
  if (st == BBQ_OK && dim == 0) st = fail(BBQ_ERR_INVALID_ARG, "dim must be > 0");
  if (st == BBQ_OK && n > 0x7FFFFFF0ull) st = fail(BBQ_ERR_UNSUPPORTED, "more than 2^31 rows per shard (result ids are int32)");
  if (st == BBQ_OK && g->ctx[0]->cfg.index_bits > INDEX_BITS_MAX)
    st = fail(BBQ_ERR_UNSUPPORTED,
              "indexBits > 2: the reference's search cannot run any indexBits != 1 (createDirectPackedBuffer throws); "
              "this build searches 1-bit indexes (reference behaviour) and 2-bit ones (extension)");
  if (st != BBQ_OK) {
    gindex_free(gi);
    return st;
  }
  // 2. the sharded build on every rank: the chained reference centroid, each rank's rows, its base
  return gindex_make(gi, [gi, rows, dim, centroid](uint32_t r) {
    bbq_ctx* c = gi->g->ctx[r];
    const uint64_t lo = gi->lo[r];
    return build_sharded(c, rows + lo * dim, true, gi->lo[r + 1] - lo, dim, centroid, &gi->shards[r], /*rows_validated=*/true);
  }, out);
}

extern "C" int bbq_group_index_from_quantized(bbq_group* g, const uint8_t* packed, const double* corr4,
                                              const float* centroid, uint64_t n, uint32_t dim, bbq_group_index** out) {
  if (!g || !out) return fail(BBQ_ERR_NULL, "null ctx/out_index");
  *out = nullptr;
  TRY(group_usable(g));
  if (!packed || !corr4 || !centroid) return fail(BBQ_ERR_NULL, "null input");
  if (n == 0) return fail(BBQ_ERR_EMPTY, "vector set must not be empty");
  if (dim == 0) return fail(BBQ_ERR_INVALID_ARG, "dim must be > 0");
  if (g->ctx[0]->cfg.index_bits > INDEX_BITS_MAX) return fail(BBQ_ERR_UNSUPPORTED, "only 1- and 2-bit indexes can be adopted");
  const size_t P = caller_row_bytes(dim, (int)g->ctx[0]->cfg.index_bits);
  bbq_group_index* gi = gindex_new(g, n);
  return gindex_make(gi, [gi, packed, corr4, centroid, dim, P](uint32_t r) {
    bbq_ctx* c = gi->g->ctx[r];
    const uint64_t lo = gi->lo[r], cnt = gi->lo[r + 1] - lo;
    // an empty shard (n < devices) is an index of 0 rows with the centroid, as a sharded load gives
    const int s = cnt > 0 ? bbq_index_from_quantized(c, packed + lo * P, corr4 + lo * 4, centroid, cnt, dim, &gi->shards[r])
                          : bbq_index_reserve(c, 1, dim, centroid, &gi->shards[r]);
    return s == BBQ_OK ? bbq_index_set_base(gi->shards[r], lo) : s;
  }, out);
}

extern "C" int bbq_group_index_load(bbq_group* g, const char* veb_path, const char* vemb_path, bbq_group_index** out) {
  if (!g || !out) return fail(BBQ_ERR_NULL, "null ctx/out_index");
  *out = nullptr;
  TRY(group_usable(g));
  if (!veb_path || !vemb_path) return fail(BBQ_ERR_NULL, "null path");
  bbq_group_index* gi = gindex_new(g, 0);
  const int st = group_run(g, [gi, veb_path, vemb_path](uint32_t r) {
    return bbq_index_load_sharded(gi->g->ctx[r], veb_path, vemb_path, &gi->shards[r]);
  });
  if (st != BBQ_OK) {
    const std::string msg = g_err;
    gindex_free(gi);
    return fail(st, msg);
  }
  // the rows every rank loaded are the split of the image's N rows
  uint64_t n = 0;
  for (bbq_index* s : gi->shards) n += s->n;
  for (uint32_t r = 0; r <= g->size(); r++) gi->lo[r] = r < g->size() ? gi->shards[r]->base : n;
  gi->n = n;
  return gindex_publish(gi, out);
}

extern "C" int bbq_group_index_save(const bbq_group_index* gi, const char* veb_path, const char* vemb_path) {
  if (!gi || !veb_path || !vemb_path) return fail(BBQ_ERR_NULL, "null index/path");
  TRY(group_usable(gi->g));
  return group_run(gi->g, [gi, veb_path, vemb_path](uint32_t r) {
    return bbq_index_save_sharded(gi->shards[r], veb_path, vemb_path);
  });
}

extern "C" uint64_t bbq_group_index_size(const bbq_group_index* gi) { return gi ? gi->n : 0; }
extern "C" uint32_t bbq_group_index_dim(const bbq_group_index* gi) { return gi ? gi->dim : 0; }
extern "C" int bbq_group_index_centroid(const bbq_group_index* gi, float* out_centroid, double* out_cdp) {
  if (!gi) return fail(BBQ_ERR_NULL, "null index");
  if (out_centroid) memcpy(out_centroid, gi->centroid.data(), gi->dim * sizeof(float));
  if (out_cdp) *out_cdp = gi->cdp;
  return BBQ_OK;
}

// not collective: each piece of the range is exported by the shard that holds it
extern "C" int bbq_group_index_export(const bbq_group_index* gi, uint64_t first, uint64_t count, uint8_t* packed,
                                      double* corr4) {
  if (!gi) return fail(BBQ_ERR_NULL, "null index");
  if (first + count > gi->n || first + count < first) return fail(BBQ_ERR_INVALID_ARG, "row range out of bounds");
  if (count == 0) return BBQ_OK;
  TRY(group_usable(gi->g));
  const size_t P = caller_row_bytes(gi->dim, gi->ib);
  for (uint32_t r = 0; r < gi->g->size(); r++) {
    const uint64_t a = std::max(first, gi->lo[r]), b = std::min(first + count, gi->lo[r + 1]);
    if (a >= b) continue;
    TRY(bbq_index_export(gi->shards[r], a - gi->lo[r], b - a, packed ? packed + (a - first) * P : nullptr,
                         corr4 ? corr4 + (a - first) * 4 : nullptr));
  }
  return BBQ_OK;
}

extern "C" int bbq_group_index_attach_rows(bbq_group_index* gi, const float* rows) {
  if (!gi || !rows) return fail(BBQ_ERR_NULL, "null");
  TRY(group_usable(gi->g));
  gi->rows_attached = false;
  TRY(group_run(gi->g, [gi, rows](uint32_t r) {
    return bbq_index_attach_rows(gi->shards[r], rows + gi->lo[r] * gi->dim);
  }));
  gi->rows_attached = true;
  return BBQ_OK;
}

extern "C" int bbq_group_search(bbq_group_index* gi, const float* queries, uint32_t nq, int64_t k, int32_t* out_idx,
                                float* out_score, uint32_t* out_count) {
  // the checks of bbq_search, in its order, so that no argument error reaches a collective
  if (out_count) *out_count = 0;
  if (!queries) return fail(BBQ_ERR_NULL, "query vector must not be null");
  if (!gi) return fail(BBQ_ERR_NULL, "target vector set must not be null");
  if (k < 0) return fail(BBQ_ERR_NEGATIVE_K, "k must not be negative");
  if (k == 0 || nq == 0) return BBQ_OK;
  if (!out_idx || !out_score) return fail(BBQ_ERR_NULL, "output buffers must not be null");
  bbq_group* g = gi->g;
  TRY(group_usable(g));
  const uint32_t kk = (uint32_t)std::min<int64_t>(k, (int64_t)gi->n);
  if (kk > K_MAX) return fail(BBQ_ERR_UNSUPPORTED, "k > 4096 is not supported by the device top-k");
  // ranks >= 1 ask for kk (the same collective: the entry clamps k to the rows of all shards) into the group's scratch
  for (uint32_t r = 1; r < g->size(); r++) {
    g->h_idx[r].resize((size_t)nq * kk);
    g->h_score[r].resize((size_t)nq * kk);
  }
  uint32_t cnt0 = 0;
  TRY(group_run(g, [gi, g, queries, nq, k, kk, out_idx, out_score, &cnt0](uint32_t r) {
    if (r == 0) return bbq_search_sharded(gi->shards[0], queries, nq, k, out_idx, out_score, &cnt0);
    uint32_t cnt = 0;
    return bbq_search_sharded(gi->shards[r], queries, nq, kk, g->h_idx[r].data(), g->h_score[r].data(), &cnt);
  }));
  if (out_count) *out_count = cnt0;
  return BBQ_OK;
}

extern "C" int bbq_group_search_rerank(bbq_group_index* gi, const float* queries, uint32_t nq, uint32_t k,
                                       uint32_t factor, int32_t* out_idx, float* out_qscore, double* out_true,
                                       uint32_t* out_count) {
  // the checks of bbq_search_rerank, in its order
  if (out_count) *out_count = 0;
  if (!gi) return fail(BBQ_ERR_NULL, "target vector set must not be null");
  if (!queries) return fail(BBQ_ERR_NULL, "query vector must not be null");
  if (!gi->rows_attached) return fail(BBQ_ERR_INVALID_ARG, "no original rows attached (bbq_index_attach_rows)");
  if (nq == 0 || k == 0) return BBQ_OK;
  if (!out_idx || !out_qscore || !out_true) return fail(BBQ_ERR_NULL, "output buffers must not be null");
  if (factor == 0 || (uint64_t)k * factor > K_MAX) return fail(BBQ_ERR_UNSUPPORTED, "k * oversampleFactor must be in 1..4096");
  bbq_group* g = gi->g;
  TRY(group_usable(g));
  for (uint32_t r = 1; r < g->size(); r++) {  // the same k on every rank: it sets the size of the exchange
    g->h_idx[r].resize((size_t)nq * k);
    g->h_score[r].resize((size_t)nq * k);
    g->h_true[r].resize((size_t)nq * k);
  }
  uint32_t cnt0 = 0;
  TRY(group_run(g, [gi, g, queries, nq, k, factor, out_idx, out_qscore, out_true, &cnt0](uint32_t r) {
    if (r == 0) return bbq_search_rerank_sharded(gi->shards[0], queries, nq, k, factor, out_idx, out_qscore, out_true, &cnt0);
    uint32_t cnt = 0;
    return bbq_search_rerank_sharded(gi->shards[r], queries, nq, k, factor, g->h_idx[r].data(), g->h_score[r].data(),
                                     g->h_true[r].data(), &cnt);
  }));
  if (out_count) *out_count = cnt0;
  return BBQ_OK;
}

extern "C" void bbq_group_index_destroy(bbq_group_index* gi) {
  if (!gi) return;
  gi->g->live--;
  gindex_free(gi);
}
