/* bbq_napi.c — the N-API addon that sits between the reference's unchanged TypeScript surface
 * (createBinaryQuantizationFormat / quickQuantize / quickSearch, src/index.ts:20-139) and libbbq_b200.so.
 * Synchronous, like the reference (SURVEY §8b): every call blocks until the CUDA stream is idle.
 * Handles are napi externals with finalizers; the C library reference-counts the context, so the GC may
 * finalize the format and its indexes in any order.  Errors become `throw new Error(<reference message>)`
 * (the message table lives in ts/errors.ts; here the status code and (vector, position) are forwarded).
 *
 *   cc -shared -fPIC bbq_napi.c -I<node>/include/node -I../../../include -L../.. -lbbq_b200 -o bbq_b200.node
 * Without Node headers (this container): cc -fsyntax-only -I. -I../../../include bbq_napi.c  (compile check only). */
#ifdef BBQ_USE_REAL_NODE_API
#include <node_api.h>
#else
#include "node_api_min.h"
#endif
#include <stdio.h>
#include <string.h>
#include "bbq_b200.h"

#define ARGS(n)                                                          \
  size_t argc = (n);                                                     \
  napi_value argv[(n)];                                                  \
  if (napi_get_cb_info(env, info, &argc, argv, NULL, NULL) != napi_ok) return NULL

static napi_value throw_status(napi_env env, int status) {
  int64_t vec = -1, pos = -1;
  char code[64];
  bbq_last_error_pos(&vec, &pos);
  /* code = "BBQ:<status>:<vector>:<position>"; ts/errors.ts maps it to the reference's message text */
  snprintf(code, sizeof code, "BBQ:%d:%lld:%lld", status, (long long)vec, (long long)pos);
  napi_throw_error(env, code, bbq_last_error());
  return NULL;
}
static napi_value throw_invalid(napi_env env, const char* what) {
  char code[64];
  snprintf(code, sizeof code, "BBQ:%d:-1:-1", (int)BBQ_ERR_INVALID_ARG);
  napi_throw_error(env, code, what);
  return NULL;
}
/* every output buffer comes from here: NULL (and a pending JS exception) when the allocation fails */
static void* new_buffer(napi_env env, size_t bytes, napi_value* ab) {
  void* p = NULL;
  if (napi_create_arraybuffer(env, bytes ? bytes : 1, &p, ab) != napi_ok || !p) {
    napi_throw_error(env, "BBQ:102:-1:-1", "out of memory allocating a result buffer");
    return NULL;
  }
  return p;
}
static void fin_ctx(napi_env env, void* data, void* hint) { (void)env; (void)hint; bbq_destroy((bbq_ctx*)data); }
static void fin_index(napi_env env, void* data, void* hint) { (void)env; (void)hint; bbq_index_destroy((bbq_index*)data); }

static int get_f32(napi_env env, napi_value v, const float** p, size_t* len) {
  napi_typedarray_type t;
  void* data;
  if (napi_get_typedarray_info(env, v, &t, len, &data, NULL, NULL) != napi_ok || t != napi_float32_array) return 0;
  *p = (const float*)data;
  return 1;
}

/* create(queryBits, indexBits, similarity(0|1|2), lambda, iters, device) -> external ctx
 * replaces `new BinaryQuantizationFormat(config)`, src/binaryQuantizationFormat.ts:141-158 */
static napi_value n_create(napi_env env, napi_callback_info info) {
  ARGS(6);
  bbq_config cfg;
  memset(&cfg, 0, sizeof cfg);
  int64_t dev = -1;
  napi_get_value_uint32(env, argv[0], &cfg.query_bits);
  napi_get_value_uint32(env, argv[1], &cfg.index_bits);
  napi_get_value_uint32(env, argv[2], &cfg.similarity);
  napi_get_value_double(env, argv[3], &cfg.lambda);
  napi_get_value_uint32(env, argv[4], &cfg.iters);
  napi_get_value_int64(env, argv[5], &dev);
  cfg.device = (int32_t)dev;
  bbq_ctx* ctx = NULL;
  const int st = bbq_create(&cfg, &ctx);
  if (st != BBQ_OK) return throw_status(env, st);
  napi_value out;
  napi_create_external(env, ctx, fin_ctx, NULL, &out);
  return out;
}

/* build(ctx, rowsFlat Float32Array[n*dim], n, dim, centroid Float32Array|null) -> external index
 * replaces format.quantizeVectors(vectors), src/binaryQuantizationFormat.ts:165-263 (the TS side flattens
 * Float32Array[] and raises the ragged-dimension error itself, as :185-193 does) */
static napi_value n_build(napi_env env, napi_callback_info info) {
  ARGS(5);
  void* ctx;
  const float *rows, *cen = NULL;
  size_t len, clen;
  int64_t n;
  uint32_t dim;
  napi_valuetype ct;
  napi_get_value_external(env, argv[0], &ctx);
  if (!get_f32(env, argv[1], &rows, &len)) return throw_status(env, BBQ_ERR_INVALID_ARG);
  napi_get_value_int64(env, argv[2], &n);
  napi_get_value_uint32(env, argv[3], &dim);
  napi_typeof(env, argv[4], &ct);
  if (ct == napi_object && !get_f32(env, argv[4], &cen, &clen)) return throw_status(env, BBQ_ERR_INVALID_ARG);
  if (n < 0 || dim == 0 || (uint64_t)len != (uint64_t)n * dim || (cen && clen != dim)) return throw_invalid(env, "rows / centroid length does not match n * dim");
  bbq_index* ix = NULL;
  const int st = bbq_index_build((bbq_ctx*)ctx, rows, (uint64_t)n, dim, cen, &ix);
  if (st != BBQ_OK) return throw_status(env, st);
  napi_value out;
  napi_create_external(env, ix, fin_index, NULL, &out);
  return out;
}

/* buildSharded(ctx, rows: Float32Array, n, dim, centroid: Float32Array | null) -> index handle: this rank's rows of a
 * corpus split over the ranks of the communicator (bbq_index_build_sharded, collective).  n may be 0 (dim then too). */
static napi_value n_build_sharded(napi_env env, napi_callback_info info) {
  ARGS(5);
  void* ctx;
  const float *rows, *cen = NULL;
  size_t len, clen;
  int64_t n;
  uint32_t dim;
  napi_valuetype ct;
  napi_get_value_external(env, argv[0], &ctx);
  if (!get_f32(env, argv[1], &rows, &len)) return throw_status(env, BBQ_ERR_INVALID_ARG);
  napi_get_value_int64(env, argv[2], &n);
  napi_get_value_uint32(env, argv[3], &dim);
  napi_typeof(env, argv[4], &ct);
  if (ct == napi_object && !get_f32(env, argv[4], &cen, &clen)) return throw_status(env, BBQ_ERR_INVALID_ARG);
  if (n < 0 || (uint64_t)len != (uint64_t)n * dim || (cen && clen != dim)) return throw_invalid(env, "rows / centroid length does not match n * dim");
  bbq_index* ix = NULL;
  const int st = bbq_index_build_sharded((bbq_ctx*)ctx, rows, (uint64_t)n, dim, cen, &ix);
  if (st != BBQ_OK) return throw_status(env, st);
  napi_value out;
  napi_create_external(env, ix, fin_index, NULL, &out);
  return out;
}

/* info(index) -> {size, dimension, centroid: Float32Array, centroidDP}
 * BinarizedByteVectorValues.size()/dimension()/getCentroid()/getCentroidDP(), src/types.ts:32-49 */
static napi_value n_info(napi_env env, napi_callback_info info) {
  ARGS(1);
  void* ix;
  napi_get_value_external(env, argv[0], &ix);
  const uint32_t dim = bbq_index_dim((bbq_index*)ix);
  napi_value out, ab, cen, v;
  void* data;
  double cdp = 0;
  napi_create_object(env, &out);
  napi_create_arraybuffer(env, dim * sizeof(float), &data, &ab);
  bbq_index_centroid((bbq_index*)ix, (float*)data, &cdp);
  napi_create_typedarray(env, napi_float32_array, dim, ab, 0, &cen);
  napi_create_double(env, (double)bbq_index_size((bbq_index*)ix), &v);
  napi_set_named_property(env, out, "size", v);
  napi_create_uint32(env, dim, &v);
  napi_set_named_property(env, out, "dimension", v);
  napi_set_named_property(env, out, "centroid", cen);
  napi_create_double(env, cdp, &v);
  napi_set_named_property(env, out, "centroidDP", v);
  return out;
}

/* search(index, queriesFlat Float32Array[nq*dim], nq, k) -> {indices: Int32Array[nq*count], scores: Float32Array, count}
 * replaces format.searchNearestNeighbors(query, targetVectors, k), src/binaryQuantizationFormat.ts:308-412;
 * nq > 1 is the additive batched entry. */
static napi_value search_common(napi_env env, napi_callback_info info, int sharded) {
  ARGS(4);
  void* ix;
  const float* q;
  size_t len;
  uint32_t nq, count = 0;
  int64_t k;
  if (napi_get_value_external(env, argv[0], &ix) != napi_ok || !ix) return throw_status(env, BBQ_ERR_NULL);
  if (!get_f32(env, argv[1], &q, &len)) return throw_status(env, BBQ_ERR_NULL);
  if (napi_get_value_uint32(env, argv[2], &nq) != napi_ok || napi_get_value_int64(env, argv[3], &k) != napi_ok)
    return throw_invalid(env, "nq / k must be numbers");
  if (len != (size_t)nq * bbq_index_dim((bbq_index*)ix)) return throw_status(env, BBQ_ERR_DIM_MISMATCH);
  /* the reference accepts any k >= 0 and returns min(k, vectorCount) rows (:385); the device top-k serves 4096.
   * Size the buffers by what can come back, never by the caller's k (a negative k is rejected by the library). */
  int64_t kcap = k;
  if (!sharded && kcap > (int64_t)bbq_index_size((bbq_index*)ix)) kcap = (int64_t)bbq_index_size((bbq_index*)ix);
  if (kcap > 4096) kcap = 4096;
  if (k > 4096 && (sharded || bbq_index_size((bbq_index*)ix) > 4096)) return throw_status(env, BBQ_ERR_UNSUPPORTED);
  const int64_t kcall = k < 0 ? k : kcap;
  const size_t slots = (size_t)nq * (size_t)(kcap > 0 ? kcap : 0);
  napi_value out, abi, abs_, ti, ts, v;
  void* pi = new_buffer(env, slots * sizeof(int32_t), &abi);
  void* ps = pi ? new_buffer(env, slots * sizeof(float), &abs_) : NULL;
  if (!pi || !ps) return NULL;
  const int st = sharded ? bbq_search_sharded((bbq_index*)ix, q, nq, kcall, (int32_t*)pi, (float*)ps, &count)
                         : bbq_search((bbq_index*)ix, q, nq, kcall, (int32_t*)pi, (float*)ps, &count);
  if (st != BBQ_OK) return throw_status(env, st);
  napi_create_typedarray(env, napi_int32_array, slots, abi, 0, &ti);
  napi_create_typedarray(env, napi_float32_array, slots, abs_, 0, &ts);
  napi_create_object(env, &out);
  napi_set_named_property(env, out, "indices", ti);
  napi_set_named_property(env, out, "scores", ts);
  napi_create_uint32(env, count, &v);
  napi_set_named_property(env, out, "count", v);
  napi_create_uint32(env, (uint32_t)(kcap > 0 ? kcap : 0), &v);
  napi_set_named_property(env, out, "stride", v);   /* row i of the result starts at i * stride */
  return out;
}
static napi_value n_search(napi_env env, napi_callback_info info) { return search_common(env, info, 0); }
/* searchSharded(index, queriesFlat, nq, k): the same over ALL row shards of the box (collective; bbq_search_sharded) */
static napi_value n_search_sharded(napi_env env, napi_callback_info info) { return search_common(env, info, 1); }

/* rows(index, first, count) -> {packed: Uint8Array, corrections: Float64Array[count*4]}
 * vectorValue(ord) / getCorrectiveTerms(ord), src/types.ts:36-42 — lazy device->host copy */
static napi_value n_rows(napi_env env, napi_callback_info info) {
  ARGS(3);
  void* ix;
  int64_t first, count;
  napi_get_value_external(env, argv[0], &ix);
  napi_get_value_int64(env, argv[1], &first);
  napi_get_value_int64(env, argv[2], &count);
  if (first < 0 || count < 0 || (uint64_t)first + (uint64_t)count > bbq_index_size((bbq_index*)ix))
    return throw_invalid(env, "row range out of bounds");
  const size_t p = (bbq_index_dim((bbq_index*)ix) + 7) / 8;
  napi_value out, ab1, ab2, t1, t2;
  void* d1 = new_buffer(env, (size_t)count * p, &ab1);
  void* d2 = d1 ? new_buffer(env, (size_t)count * 4 * sizeof(double), &ab2) : NULL;
  if (!d1 || !d2) return NULL;
  const int st = bbq_index_export((bbq_index*)ix, (uint64_t)first, (uint64_t)count, (uint8_t*)d1, (double*)d2);
  if (st != BBQ_OK) return throw_status(env, st);
  napi_create_typedarray(env, napi_uint8_array, (size_t)count * p, ab1, 0, &t1);
  napi_create_typedarray(env, napi_float64_array, (size_t)count * 4, ab2, 0, &t2);
  napi_create_object(env, &out);
  napi_set_named_property(env, out, "packed", t1);
  napi_set_named_property(env, out, "corrections", t2);
  return out;
}

/* attachRows(index, rowsFlat Float32Array[n*dim]) — keeps the original rows on the device for the exact re-rank */
static napi_value n_attach_rows(napi_env env, napi_callback_info info) {
  ARGS(2);
  void* ix;
  const float* rows;
  size_t len;
  napi_get_value_external(env, argv[0], &ix);
  if (!get_f32(env, argv[1], &rows, &len)) return throw_status(env, BBQ_ERR_NULL);
  if (len != (size_t)bbq_index_size((bbq_index*)ix) * bbq_index_dim((bbq_index*)ix)) return throw_status(env, BBQ_ERR_DIM_MISMATCH);
  const int st = bbq_index_attach_rows((bbq_index*)ix, rows);
  if (st != BBQ_OK) return throw_status(env, st);
  napi_value u;
  napi_get_undefined(env, &u);
  return u;
}

/* searchRerank(index, queriesFlat, nq, k, oversampleFactor) -> {indices, quantizedScores, trueScores, count}
 * replaces getOversampledTopKWithSort / getOversampledTopKWithHeap, src/topKSelector.ts:29-114 */
static napi_value rerank_common(napi_env env, napi_callback_info info, int sharded) {
  ARGS(5);
  void* ix;
  const float* q;
  size_t len;
  uint32_t nq, k, factor, count = 0;
  napi_get_value_external(env, argv[0], &ix);
  if (!get_f32(env, argv[1], &q, &len)) return throw_status(env, BBQ_ERR_NULL);
  napi_get_value_uint32(env, argv[2], &nq);
  napi_get_value_uint32(env, argv[3], &k);
  napi_get_value_uint32(env, argv[4], &factor);
  if (len != (size_t)nq * bbq_index_dim((bbq_index*)ix)) return throw_status(env, BBQ_ERR_DIM_MISMATCH);
  if (k > 4096) return throw_status(env, BBQ_ERR_UNSUPPORTED);
  const size_t slots = (size_t)nq * k;
  napi_value out, a1, a2, a3, t1, t2, t3, v;
  void* p1 = new_buffer(env, slots * sizeof(int32_t), &a1);
  void* p2 = p1 ? new_buffer(env, slots * sizeof(float), &a2) : NULL;
  void* p3 = p2 ? new_buffer(env, slots * sizeof(double), &a3) : NULL;
  if (!p1 || !p2 || !p3) return NULL;
  const int st = sharded ? bbq_search_rerank_sharded((bbq_index*)ix, q, nq, k, factor, (int32_t*)p1, (float*)p2, (double*)p3, &count)
                         : bbq_search_rerank((bbq_index*)ix, q, nq, k, factor, (int32_t*)p1, (float*)p2, (double*)p3, &count);
  if (st != BBQ_OK) return throw_status(env, st);
  napi_create_typedarray(env, napi_int32_array, slots, a1, 0, &t1);
  napi_create_typedarray(env, napi_float32_array, slots, a2, 0, &t2);
  napi_create_typedarray(env, napi_float64_array, slots, a3, 0, &t3);
  napi_create_object(env, &out);
  napi_set_named_property(env, out, "indices", t1);
  napi_set_named_property(env, out, "quantizedScores", t2);
  napi_set_named_property(env, out, "trueScores", t3);
  napi_create_uint32(env, count, &v);
  napi_set_named_property(env, out, "count", v);
  return out;
}
static napi_value n_search_rerank(napi_env env, napi_callback_info info) { return rerank_common(env, info, 0); }
/* searchRerankSharded(index, queriesFlat, nq, k, oversampleFactor): the same over ALL row shards of the box
 * (collective; bbq_search_rerank_sharded), same result object */
static napi_value n_search_rerank_sharded(napi_env env, napi_callback_info info) { return rerank_common(env, info, 1); }

static int get_path(napi_env env, napi_value v, char* buf, size_t cap) {
  size_t n = 0;
  return napi_get_value_string_utf8(env, v, buf, cap, &n) == napi_ok && n + 1 < cap;
}

/* saveIndex(index, vebPath, vembPath) / loadIndex(ctx, vebPath, vembPath) -> external index
 * the on-disk form of serializeVectorData / deserializeVectorData, src/binaryQuantizationFormat.ts:483-560 */
static napi_value save_common(napi_env env, napi_callback_info info, int sharded) {
  ARGS(3);
  void* ix;
  char veb[4096], vemb[4096];
  napi_get_value_external(env, argv[0], &ix);
  if (!get_path(env, argv[1], veb, sizeof veb) || !get_path(env, argv[2], vemb, sizeof vemb)) return throw_status(env, BBQ_ERR_NULL);
  const int st = sharded ? bbq_index_save_sharded((bbq_index*)ix, veb, vemb) : bbq_index_save((bbq_index*)ix, veb, vemb);
  if (st != BBQ_OK) return throw_status(env, st);
  napi_value u;
  napi_get_undefined(env, &u);
  return u;
}
static napi_value load_common(napi_env env, napi_callback_info info, int sharded) {
  ARGS(3);
  void* ctx;
  char veb[4096], vemb[4096];
  napi_get_value_external(env, argv[0], &ctx);
  if (!get_path(env, argv[1], veb, sizeof veb) || !get_path(env, argv[2], vemb, sizeof vemb)) return throw_status(env, BBQ_ERR_NULL);
  bbq_index* ix = NULL;
  const int st = sharded ? bbq_index_load_sharded((bbq_ctx*)ctx, veb, vemb, &ix) : bbq_index_load((bbq_ctx*)ctx, veb, vemb, &ix);
  if (st != BBQ_OK) return throw_status(env, st);
  napi_value out;
  napi_create_external(env, ix, fin_index, NULL, &out);
  return out;
}
static napi_value n_save_index(napi_env env, napi_callback_info info) { return save_common(env, info, 0); }
static napi_value n_load_index(napi_env env, napi_callback_info info) { return load_common(env, info, 0); }
/* saveIndexSharded(index, vebPath, vembPath) / loadIndexSharded(ctx, vebPath, vembPath) -> external index (this rank's
 * row range, base set): one image of all row shards of the box (collective; bbq_index_save_sharded / _load_sharded) */
static napi_value n_save_index_sharded(napi_env env, napi_callback_info info) { return save_common(env, info, 1); }
static napi_value n_load_index_sharded(napi_env env, napi_callback_info info) { return load_common(env, info, 1); }

/* quantizeQuery(ctx, query Float32Array[dim], centroid Float32Array[dim]) -> {codes: Uint8Array[dim], corrections: Float64Array[4]}
 * replaces format.quantizeQueryVector(queryVector, centroid), src/binaryQuantizationFormat.ts:271-299 */
static napi_value n_quantize_query(napi_env env, napi_callback_info info) {
  ARGS(3);
  void* ctx;
  const float *q, *cen;
  size_t len, clen;
  napi_get_value_external(env, argv[0], &ctx);
  if (!get_f32(env, argv[1], &q, &len) || !get_f32(env, argv[2], &cen, &clen)) return throw_status(env, BBQ_ERR_NULL);
  if (len == 0 || len != clen) return throw_status(env, BBQ_ERR_DIM_MISMATCH);
  napi_value out, a1, a2, t1, t2;
  void* p1 = new_buffer(env, len, &a1);
  void* p2 = p1 ? new_buffer(env, 4 * sizeof(double), &a2) : NULL;
  if (!p1 || !p2) return NULL;
  const int st = bbq_quantize_query((bbq_ctx*)ctx, q, cen, (uint32_t)len, (uint8_t*)p1, (double*)p2);
  if (st != BBQ_OK) return throw_status(env, st);
  napi_create_typedarray(env, napi_uint8_array, len, a1, 0, &t1);
  napi_create_typedarray(env, napi_float64_array, 4, a2, 0, &t2);
  napi_create_object(env, &out);
  napi_set_named_property(env, out, "codes", t1);
  napi_set_named_property(env, out, "corrections", t2);
  return out;
}

/* accuracy(ctx, rowsFlat, queriesFlat, n, dim, targetOrd) -> Float64Array[5] {mean, max, min, std, correlation}
 * replaces format.computeQuantizationAccuracy, src/binaryQuantizationFormat.ts:420-475 */
static napi_value n_accuracy(napi_env env, napi_callback_info info) {
  ARGS(6);
  void* ctx;
  const float *rows, *qs;
  size_t len, qlen;
  int64_t n, target;
  uint32_t dim;
  napi_get_value_external(env, argv[0], &ctx);
  if (!get_f32(env, argv[1], &rows, &len) || !get_f32(env, argv[2], &qs, &qlen)) return throw_status(env, BBQ_ERR_NULL);
  napi_get_value_int64(env, argv[3], &n);
  napi_get_value_uint32(env, argv[4], &dim);
  napi_get_value_int64(env, argv[5], &target);
  if (n <= 0 || target < 0 || (uint64_t)len != (uint64_t)n * dim || qlen != len) return throw_invalid(env, "rows / queries length does not match n * dim");
  napi_value ab, t;
  void* p = new_buffer(env, 5 * sizeof(double), &ab);
  if (!p) return NULL;
  const int st = bbq_quantization_accuracy((bbq_ctx*)ctx, rows, qs, (uint64_t)n, dim, (uint64_t)target, (double*)p);
  if (st != BBQ_OK) return throw_status(env, st);
  napi_create_typedarray(env, napi_float64_array, 5, ab, 0, &t);
  return t;
}

/* fromQuantized(ctx, packed Uint8Array[n*ceil(dim/8)], corrections Float64Array[n*4], centroid Float32Array[dim], n, dim)
 * -> external index: the device side of deserializeVectorData, src/binaryQuantizationFormat.ts:533-560 */
static napi_value n_from_quantized(napi_env env, napi_callback_info info) {
  ARGS(6);
  void *ctx, *pk, *cr;
  const float* cen;
  size_t plen, clen, cenlen;
  napi_typedarray_type t1, t2;
  int64_t n;
  uint32_t dim;
  napi_get_value_external(env, argv[0], &ctx);
  if (napi_get_typedarray_info(env, argv[1], &t1, &plen, &pk, NULL, NULL) != napi_ok || t1 != napi_uint8_array ||
      napi_get_typedarray_info(env, argv[2], &t2, &clen, &cr, NULL, NULL) != napi_ok || t2 != napi_float64_array ||
      !get_f32(env, argv[3], &cen, &cenlen))
    return throw_status(env, BBQ_ERR_NULL);
  napi_get_value_int64(env, argv[4], &n);
  napi_get_value_uint32(env, argv[5], &dim);
  if (n <= 0 || cenlen != dim || (uint64_t)plen != (uint64_t)n * ((dim + 7) / 8) || (uint64_t)clen != (uint64_t)n * 4)
    return throw_invalid(env, "packed / corrections / centroid lengths do not match n and dim");
  bbq_index* ix = NULL;
  const int st = bbq_index_from_quantized((bbq_ctx*)ctx, (const uint8_t*)pk, (const double*)cr, cen, (uint64_t)n, dim, &ix);
  if (st != BBQ_OK) return throw_status(env, st);
  napi_value out;
  napi_create_external(env, ix, fin_index, NULL, &out);
  return out;
}

/* Sharded search bootstrap (one Node process per GPU; SURVEY §8e): commUniqueId() -> Uint8Array[128] on rank 0, shipped
 * to the other workers by the host (IPC message, env var, file); commInit(ctx, id, rank, world); setBase(index, base). */
static napi_value n_comm_unique_id(napi_env env, napi_callback_info info) {
  (void)info;
  napi_value ab, t;
  void* p = new_buffer(env, BBQ_COMM_ID_BYTES, &ab);
  if (!p) return NULL;
  const int st = bbq_comm_unique_id((uint8_t*)p);
  if (st != BBQ_OK) return throw_status(env, st);
  napi_create_typedarray(env, napi_uint8_array, BBQ_COMM_ID_BYTES, ab, 0, &t);
  return t;
}
static napi_value n_comm_init(napi_env env, napi_callback_info info) {
  ARGS(4);
  void *ctx, *id;
  size_t len;
  napi_typedarray_type t;
  int64_t rank, world;
  napi_get_value_external(env, argv[0], &ctx);
  if (napi_get_typedarray_info(env, argv[1], &t, &len, &id, NULL, NULL) != napi_ok || t != napi_uint8_array ||
      len != BBQ_COMM_ID_BYTES)
    return throw_invalid(env, "communicator id must be a Uint8Array of 128 bytes");
  napi_get_value_int64(env, argv[2], &rank);
  napi_get_value_int64(env, argv[3], &world);
  const int st = bbq_comm_init((bbq_ctx*)ctx, (const uint8_t*)id, (int)rank, (int)world);
  if (st != BBQ_OK) return throw_status(env, st);
  napi_value u;
  napi_get_undefined(env, &u);
  return u;
}
static napi_value n_set_base(napi_env env, napi_callback_info info) {
  ARGS(2);
  void* ix;
  int64_t base;
  napi_get_value_external(env, argv[0], &ix);
  napi_get_value_int64(env, argv[1], &base);
  if (base < 0) return throw_invalid(env, "base must be >= 0");
  const int st = bbq_index_set_base((bbq_index*)ix, (uint64_t)base);
  if (st != BBQ_OK) return throw_status(env, st);
  napi_value u;
  napi_get_undefined(env, &u);
  return u;
}

NAPI_MODULE_INIT() {
  const napi_property_descriptor props[] = {
      {"create", NULL, n_create, NULL, NULL, NULL, 0, NULL}, {"build", NULL, n_build, NULL, NULL, NULL, 0, NULL},
      {"buildSharded", NULL, n_build_sharded, NULL, NULL, NULL, 0, NULL},
      {"info", NULL, n_info, NULL, NULL, NULL, 0, NULL},     {"search", NULL, n_search, NULL, NULL, NULL, 0, NULL},
      {"rows", NULL, n_rows, NULL, NULL, NULL, 0, NULL},
      {"attachRows", NULL, n_attach_rows, NULL, NULL, NULL, 0, NULL},
      {"searchRerank", NULL, n_search_rerank, NULL, NULL, NULL, 0, NULL},
      {"searchRerankSharded", NULL, n_search_rerank_sharded, NULL, NULL, NULL, 0, NULL},
      {"saveIndex", NULL, n_save_index, NULL, NULL, NULL, 0, NULL},
      {"loadIndex", NULL, n_load_index, NULL, NULL, NULL, 0, NULL},
      {"saveIndexSharded", NULL, n_save_index_sharded, NULL, NULL, NULL, 0, NULL},
      {"loadIndexSharded", NULL, n_load_index_sharded, NULL, NULL, NULL, 0, NULL},
      {"quantizeQuery", NULL, n_quantize_query, NULL, NULL, NULL, 0, NULL},
      {"accuracy", NULL, n_accuracy, NULL, NULL, NULL, 0, NULL},
      {"fromQuantized", NULL, n_from_quantized, NULL, NULL, NULL, 0, NULL},
      {"searchSharded", NULL, n_search_sharded, NULL, NULL, NULL, 0, NULL},
      {"commUniqueId", NULL, n_comm_unique_id, NULL, NULL, NULL, 0, NULL},
      {"commInit", NULL, n_comm_init, NULL, NULL, NULL, 0, NULL},
      {"setBase", NULL, n_set_base, NULL, NULL, NULL, 0, NULL}};
  napi_define_properties(env, exports, sizeof props / sizeof props[0], props);
  return exports;
}
