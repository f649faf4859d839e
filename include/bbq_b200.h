/*
 * bbq_b200.h — C ABI of libbbq_b200.so, the B200-native (sm_100a) implementation of the brute-force
 * quantized search path of leolee9086/Better-Binary-Quantization.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch / C++ types.  The reference's
 * TypeScript classes keep their public surface (src/index.ts:20-139) and forward through an N-API
 * addon (better-binary-quantization_b200/bindings/napi/) to these entry points; INTEGRATION.md shows
 * the binding.  Each entry cites the reference interface (file:line, relative to the reference root)
 * it replaces.  The model for a flat-array interface is the reference's own wasm-bindgen surface,
 * rust-wasm/src/wasm_interface.rs:455-516 (WasmQuantizedIndex{new, build_index, search_nearest_neighbors}).
 *
 * All functions return a bbq_status; on failure bbq_last_error() holds a thread-local English
 * description and bbq_last_error_pos() the (vector, position) the reference would name in its message.
 * There is NO CPU fallback: without a usable sm_100 device bbq_create fails with BBQ_ERR_NO_DEVICE.
 *
 * Threading: a bbq_ctx and its indexes may be used from one host thread at a time (the reference is
 * synchronous single-threaded JS, SURVEY §8b).  Different contexts are independent.
 */
#ifndef BBQ_B200_H
#define BBQ_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BBQ_B200_ABI_VERSION 3

typedef struct bbq_ctx bbq_ctx;     /* one GPU: stream, scratch, config          */
typedef struct bbq_index bbq_index; /* device-resident index shard (a2 in SURVEY) */

/* src/types.ts:9-13 VectorSimilarityFunction (string enum in TS; the shim maps the strings) */
typedef enum {
  BBQ_SIM_EUCLIDEAN = 0,
  BBQ_SIM_COSINE = 1,
  BBQ_SIM_MAXIMUM_INNER_PRODUCT = 2
} bbq_similarity;

typedef enum {
  BBQ_OK = 0,
  /* input errors: each maps to one `throw new Error(...)` of the reference (see INTEGRATION.md table) */
  BBQ_ERR_QUERY_BITS = 1,    /* binaryQuantizationFormat.ts:143-145  'queryBits必须在1-8之间'            */
  BBQ_ERR_INDEX_BITS = 2,    /* binaryQuantizationFormat.ts:146-148  'indexBits必须在1-8之间'            */
  BBQ_ERR_EMPTY = 3,         /* binaryQuantizationFormat.ts:169-171  '向量集合不能为空'                   */
  BBQ_ERR_DIM_MISMATCH = 4,  /* binaryQuantizationFormat.ts:190-192, :327-329                            */
  BBQ_ERR_NAN = 5,           /* binaryQuantizationFormat.ts:202-204, optimizedScalarQuantizer.ts:141-143 */
  BBQ_ERR_INF = 6,           /* binaryQuantizationFormat.ts:205-207, optimizedScalarQuantizer.ts:144-146 */
  BBQ_ERR_NEGATIVE_K = 7,    /* binaryQuantizationFormat.ts:324-326  'k值不能为负数'                      */
  BBQ_ERR_NULL = 8,          /* binaryQuantizationFormat.ts:318-323  null query / targets                */
  BBQ_ERR_UNSUPPORTED = 9,   /* config outside what the reference's batch path can run (SURVEY §8 a5/a11) */
  BBQ_ERR_INVALID_ARG = 10,
  BBQ_ERR_IO = 11,           /* index image: open/read/write failed (message carries errno text)         */
  BBQ_ERR_FORMAT = 12,       /* index image: bad magic/version, other similarity, truncation, checksum   */
  /* runtime errors: never a silent fallback */
  BBQ_ERR_NO_DEVICE = 100,
  BBQ_ERR_CUDA = 101,
  BBQ_ERR_OOM = 102,
  BBQ_ERR_COMM = 103         /* NCCL could not be loaded / a collective failed (sharded search only)      */
} bbq_status;

/* src/types.ts:54-73 BinaryQuantizationConfig + QuantizerConfig; defaults src/index.ts:47-55,
 * src/constants.ts:9-30 (queryBits 4, indexBits 1, lambda 0.1, iters 5). */
typedef struct {
  uint32_t query_bits; /* 1..8 */
  uint32_t index_bits; /* 1..8 accepted as the reference does; search requires 1 (reference batch path) */
  uint32_t similarity; /* bbq_similarity */
  uint32_t iters;
  double lambda;
  int32_t device;      /* CUDA device ordinal; -1 = current device */
  uint32_t reserved;
} bbq_config;

/* -------- lifecycle ------------------------------------------------------------------------------ */

/* new BinaryQuantizationFormat(config) — src/binaryQuantizationFormat.ts:141-158 */
int bbq_create(const bbq_config* config, bbq_ctx** out_ctx);
void bbq_destroy(bbq_ctx* ctx);
const char* bbq_last_error(void);
void bbq_last_error_pos(int64_t* vector, int64_t* position);
int bbq_abi_version(void);

/* -------- index build (SURVEY a12, K5) ----------------------------------------------------------- */

/* format.quantizeVectors(vectors) — src/binaryQuantizationFormat.ts:165-263.
 * rows: n*dim f32, row-major, HOST memory.  centroid: NULL = reference-order centroid
 * (src/vectorOperations.ts:126-163: sequential f32 accumulation over the (normalised) rows);
 * non-NULL = explicit centroid (bench-scale corpora, SURVEY §7 hard-part 5).
 * Validates like the reference (empty, NaN, Inf). */
int bbq_index_build(bbq_ctx* ctx, const float* rows, uint64_t n, uint32_t dim, const float* centroid,
                    bbq_index** out_index);

/* Same, rows already in DEVICE memory (generated or uploaded by the caller; not validated). */
int bbq_index_build_device(bbq_ctx* ctx, const float* d_rows, uint64_t n, uint32_t dim,
                           const float* centroid_host_or_null, bbq_index** out_index);

/* Streaming build for corpora that never exist whole (SURVEY §7 hard-part 5): reserve `capacity` rows with an
 * EXPLICIT centroid (host pointer, required — the reference-order centroid needs every row first: one pass of
 * bbq_centroid_accumulate + bbq_centroid_finish below gives it), then append
 * row chunks (host or device memory) in order; each chunk is quantised exactly as quantizeVectors would with
 * that centroid (src/binaryQuantizationFormat.ts:221-249).  bbq_index_size() grows with each append. */
int bbq_index_reserve(bbq_ctx* ctx, uint64_t capacity, uint32_t dim, const float* centroid, bbq_index** out_index);
int bbq_index_append(bbq_index* index, const float* rows, uint64_t n);
int bbq_index_append_device(bbq_index* index, const float* d_rows, uint64_t n);

/* The reference-order centroid of a corpus that is streamed or split (src/vectorOperations.ts:126-163:
 * c = copy(V[0]); c = f32(c + V[j]) for j = 1 .. N-1 in row order; then f32(c / N)).  Not collective.
 * bbq_centroid_accumulate(_device): continues the running sum `running` (HOST, dim floats, read and written) over the
 *   n rows that follow the corpus's first rows_before rows; rows_before == 0: this slice starts the corpus (row 0 is
 *   copied, `running` is only written).  COSINE rows are normalised first, as bbq_index_build does.  Host rows are
 *   validated like bbq_index_build's (the vector index reported counts from the corpus's row 0); device rows are not.
 *   n == 0 leaves `running` unchanged.
 * bbq_centroid_finish: centroid[i] = f32((double)running[i] / (double)n_total), what bbq_index_build computes (dividing
 *   by float(N) instead is wrong once N > 2^24).  Host only, needs no device.
 * One pass of accumulate over all slices, finish, then bbq_index_reserve + bbq_index_append* of the slices gives the
 * index bbq_index_build gives for the whole corpus. */
int bbq_centroid_accumulate(bbq_ctx* ctx, const float* rows, uint64_t n, uint32_t dim, uint64_t rows_before,
                            float* running);
int bbq_centroid_accumulate_device(bbq_ctx* ctx, const float* d_rows, uint64_t n, uint32_t dim, uint64_t rows_before,
                                   float* running);
int bbq_centroid_finish(const float* running, uint32_t dim, uint64_t n_total, float* centroid);

/* quantizeVectors over row shards (collective: every rank of the communicator calls it with its own rows; see
 * bbq_comm_init).  Ranks hold consecutive row ranges in rank order; a rank may hold 0 rows (and pass dim 0, unless it
 * passes a centroid).  centroid: NULL on every rank = the reference-order centroid of the whole corpus, chained across
 * the ranks (rank r continues the running sum of ranks 0 .. r-1, one ncclAllReduce per non-empty rank); or the same
 * explicit centroid on every rank.  Each rank gets the index of rows [base, base + n) of bbq_index_build over the whole
 * corpus, byte for byte, with its base set (base = the rows of the ranks before it).
 * Every rank returns the same status and message: Σ n == 0 -> BBQ_ERR_EMPTY; a shard over 2^31 - 16 rows or Σ n over
 * 2^31 - 1 -> BBQ_ERR_UNSUPPORTED; dimensions, similarity, indexBits or centroids that differ -> BBQ_ERR_INVALID_ARG;
 * a NaN / Infinity in host rows -> the lowest such rank's status, with bbq_last_error_pos naming the vector in the
 * whole corpus; out of memory on any rank fails every rank.  Without a communicator (or world == 1) they are
 * bbq_index_build and bbq_index_build_device. */
int bbq_index_build_sharded(bbq_ctx* ctx, const float* rows, uint64_t n, uint32_t dim, const float* centroid,
                            bbq_index** out_index);
int bbq_index_build_sharded_device(bbq_ctx* ctx, const float* d_rows, uint64_t n, uint32_t dim,
                                   const float* centroid_host_or_null, bbq_index** out_index);

/* Adopt an index quantised elsewhere (e.g. by the reference itself): packed = n*ceil(dim/8) bytes,
 * MSB-first rows exactly as BinarizedByteVectorValuesImpl.vectors holds them
 * (src/binaryQuantizationFormat.ts:24-43, packAsBinary src/optimizedScalarQuantizer.ts:420-446);
 * corr4 = n*4 doubles {lowerInterval, upperInterval, additionalCorrection, quantizedComponentSum}
 * (src/types.ts:18-27).  HOST pointers. */
int bbq_index_from_quantized(bbq_ctx* ctx, const uint8_t* packed, const double* corr4,
                             const float* centroid, uint64_t n, uint32_t dim, bbq_index** out_index);

/* BinarizedByteVectorValues.size() / dimension() / getCentroid() / getCentroidDP() —
 * src/types.ts:32-49, src/binaryQuantizationFormat.ts:45-51,113-125 */
uint64_t bbq_index_size(const bbq_index* index);
uint32_t bbq_index_dim(const bbq_index* index);
int bbq_index_centroid(const bbq_index* index, float* out_centroid /* dim */, double* out_centroid_dp);

/* Index image on disk — the working form of serializeVectorData / deserializeVectorData
 * (src/binaryQuantizationFormat.ts:483-560) behind the reference's own file split: `veb_path` holds the vector data
 * (FILE_EXTENSIONS.VECTOR_DATA, one VectorDataFormat column per section: binaryValues, lowerInterval, upperInterval,
 * additionalCorrection, quantizedComponentSum — src/types.ts:78-90), `vemb_path` the MetadataFormat fields
 * (src/types.ts:95-113) plus the centroid.  Sections are the HBM arrays byte for byte, 4096-byte aligned, each with
 * a device-computed checksum; layout in csrc/bbq_io.cuh.  bbq_index_load requires a context with the same
 * similarity function and indexBits = 1 and returns BBQ_ERR_FORMAT otherwise (or on any corruption). */
int bbq_index_save(const bbq_index* index, const char* veb_path, const char* vemb_path);
int bbq_index_load(bbq_ctx* ctx, const char* veb_path, const char* vemb_path, bbq_index** out_index);

/* One image across row shards.  A section's checksum is Σ splitmix64(i << 32 | word_i) over its 32-bit words with i
 * counted from the image's row 0, so the checksums of disjoint row ranges add up (mod 2^64) to the section's.  The
 * shard-local primitives below are not collective; out_partial / checksums: {codes, lower, upper, additional,
 * componentSum}.
 * bbq_index_load_rows: rows [first, first + count) of an image into a new index whose base (bbq_index_set_base) is
 *   `first`, reading only that range of each section; the checks of bbq_index_load, plus first + count <= vectorCount
 *   (else BBQ_ERR_INVALID_ARG).  out_partial (may be NULL) receives the checksums of the rows uploaded; only when the
 *   range is the whole image are they compared with the header here.  count = 0 gives an index of 0 rows.
 * bbq_index_write_rows: this shard's rows at rows [base, base + n) of an image of total_rows rows (base + n <=
 *   total_rows, else BBQ_ERR_INVALID_ARG).  Opens the .veb with O_CREAT and without O_TRUNC and sets its length to the
 *   image's, so calls may come in any order from any process; start from a new (or truncated) file.
 * bbq_index_write_meta: the .vemb of an image of total_rows rows with the given checksums (the sums of every shard's
 *   partials) and this shard's dimension, similarity, centroid and centroidSquareMagnitude.
 * The files equal, byte for byte, what bbq_index_save writes for one index holding all the rows. */
int bbq_index_load_rows(bbq_ctx* ctx, const char* veb_path, const char* vemb_path, uint64_t first, uint64_t count,
                        bbq_index** out_index, uint64_t out_partial[5]);
int bbq_index_write_rows(const bbq_index* shard, const char* veb_path, uint64_t total_rows, uint64_t out_partial[5]);
int bbq_index_write_meta(const bbq_index* shard, const char* vemb_path, uint64_t total_rows, const uint64_t checksums[5]);

/* Collective (every rank of the communicator calls them; see bbq_comm_init below).  Without a communicator, or with
 * world == 1, they are bbq_index_save and bbq_index_load.
 * bbq_index_save_sharded: one all-gather of every rank's {base, rows, dim, similarity, indexBits, centroid}: shards
 *   that do not tile [0, N) exactly, a dimension, similarity or centroid other than rank 0's, or indexBits != 1 make
 *   every rank fail alike (empty shards may sit anywhere).  Rank 0 then removes the old .vemb and creates the .veb,
 *   every rank writes its rows, the partials are summed in one integer ncclAllReduce and rank 0 writes the .vemb.
 *   The files equal what bbq_index_save writes for one index holding the whole corpus.
 * bbq_index_load_sharded: rank r loads rows [r*per, min(N, (r+1)*per)), per = ceil(N / world) (host/sharded.py
 *   shard_bounds), with its base set; the partials are summed and checked against the header on every rank, and the
 *   ranks compare the headers they read, so a corrupted section, or paths naming different images, fail every rank
 *   with BBQ_ERR_FORMAT.
 * Every phase of both ends in an exchange of each rank's status: a rank that fails (open, read, out of memory, bad
 * header) makes every rank return the same status and message ("sharded save: rank r: ..."), none is left waiting. */
int bbq_index_save_sharded(const bbq_index* shard, const char* veb_path, const char* vemb_path);
int bbq_index_load_sharded(bbq_ctx* ctx, const char* veb_path, const char* vemb_path, bbq_index** out_index);

/* vectorValue(ord) / getCorrectiveTerms(ord) for ord in [first, first+count): lazy device->host copy.
 * packed: count*ceil(dim/8) bytes; corr4: count*4 doubles.  Either may be NULL. */
int bbq_index_export(const bbq_index* index, uint64_t first, uint64_t count, uint8_t* packed,
                     double* corr4);

/* Row-wise sharding (SURVEY §8e): global row id of this shard's row 0; reported ids = base + local. */
int bbq_index_set_base(bbq_index* index, uint64_t base);
void bbq_index_destroy(bbq_index* index);

/* -------- search (SURVEY a1..a10, K1-K4) ---------------------------------------------------------- */

/* format.searchNearestNeighbors(query, targetVectors, k) — src/binaryQuantizationFormat.ts:308-412 —
 * for nq queries at once (nq > 1 is additive: row i of the outputs equals the single-query call on
 * query i).  HOST pointers; blocks until done.  Per query the min(k, n) best under
 * (f32 score descending, row id ascending) are written, descending, to out_idx/out_score[i*k ...];
 * *out_count = min(k, n).  k == 0 -> *out_count = 0 (reference returns []). */
int bbq_search(bbq_index* index, const float* queries, uint32_t nq, int64_t k, int32_t* out_idx,
               float* out_score, uint32_t* out_count);

/* Device-resident variant: d_queries nq*dim f32, outputs nq*k each, all DEVICE memory; enqueued on
 * `stream` (a cudaStream_t; NULL = the context's stream).  The call may synchronise that stream internally (one
 * overflow-flag read per batch of <= 4096 queries) but its last kernels are left running.  Unused tail slots
 * (k > n) hold idx -1, score -inf.  All searches of a context share its scratch buffers: work given to a caller's
 * stream is ordered (by events) after what is already queued on the context's own stream and before what is queued
 * there later, so host-pointer entries (context stream) and device-pointer entries may follow each other freely; do
 * not run two caller streams on one context concurrently. */
int bbq_search_device(bbq_index* index, const float* d_queries, uint32_t nq, uint32_t k,
                      int32_t* d_out_idx, float* d_out_score, void* stream);

/* -------- the class members beside the search path ------------------------------------------------------- */

/* format.quantizeQueryVector(queryVector, centroid) — src/binaryQuantizationFormat.ts:271-299: COSINE normalises
 * ONCE (the search path normalises a second time, :337), then scalarQuantize(queryBits) against `centroid`.
 * codes: dim bytes; corr4: {lowerInterval, upperInterval, additionalCorrection, quantizedComponentSum}.  HOST. */
int bbq_quantize_query(bbq_ctx* ctx, const float* query, const float* centroid, uint32_t dim, uint8_t* codes,
                       double* corr4);

/* format.computeQuantizationAccuracy(originalVectors, queryVectors) — src/binaryQuantizationFormat.ts:420-475 with
 * the statistics of src/binaryQuantizedScorer.ts:524-617: quantises `rows` (n x dim, reference-order centroid), then
 * for every query i scores it against row `target_ord` (the reference: 0) through the single-vector quantised scorer
 * (src/binaryQuantizedScorer.ts:69-98; queryBits 1 or 4 only, else BBQ_ERR_UNSUPPORTED = its throw) and exactly
 * (computeOriginalScore :430-448), and reduces |orig - quant| to out5 = {meanError, maxError, minError, stdError,
 * correlation}.  rows and queries: n x dim each (the reference requires equal lengths).  HOST pointers. */
int bbq_quantization_accuracy(bbq_ctx* ctx, const float* rows, const float* queries, uint64_t n, uint32_t dim,
                              uint64_t target_ord, double* out5);

/* -------- sharded search over the GPUs of one box (SURVEY §8e) ------------------------------------------ */

/* The reference is single-process and has no counterpart; the model is its wasm surface, where ONE object owns build
 * and search (rust-wasm/src/wasm_interface.rs:455-516).  One process / bbq_ctx / communicator per GPU: every rank
 * builds (or loads) its contiguous row shard, sets its base (bbq_index_set_base), and calls bbq_search_sharded with
 * the SAME query batch; the per-shard top-k lists travel as 64-bit (score, id) keys in one ncclAllGather over NVLink
 * and every rank merges them with the canonical MinHeap rule of src/binaryQuantizationFormat.ts:383-411, so every
 * rank returns the same lists, identical to a single-shard search of the whole corpus.
 * Bootstrap: rank 0 calls bbq_comm_unique_id and ships the BBQ_COMM_ID_BYTES bytes to the other ranks by any means
 * (pipe, file, env var, torch.distributed store ...); then every rank calls bbq_comm_init(ctx, id, rank, world).
 * NCCL is loaded with dlopen("libnccl.so.2") on first use (override: env BBQ_NCCL_LIB); without it these entries
 * return BBQ_ERR_COMM and everything else keeps working. */
#define BBQ_COMM_ID_BYTES 128
int bbq_comm_unique_id(uint8_t* out_id /* BBQ_COMM_ID_BYTES */);
int bbq_comm_init(bbq_ctx* ctx, const uint8_t* id /* BBQ_COMM_ID_BYTES */, int rank, int world);
/* Collective, like bbq_comm_init: every rank calls it (ncclCommDestroy).  A context that is destroyed while it still
 * holds a communicator aborts it locally instead (ncclCommAbort), so finalizers never wait for a peer. */
int bbq_comm_destroy(bbq_ctx* ctx);
int bbq_comm_info(bbq_ctx* ctx, int* rank, int* world, int* nccl_version);

/* searchNearestNeighbors over ALL shards (same contract as bbq_search; *out_count = min(k, rows over all ranks)).
 * HOST pointers; collective: every rank of the communicator must call it with the same queries, nq and k.
 * Without a communicator (or world == 1) it is bbq_search. */
int bbq_search_sharded(bbq_index* index, const float* queries, uint32_t nq, int64_t k, int32_t* out_idx,
                       float* out_score, uint32_t* out_count);
/* Device-resident variant (collective), like bbq_search_device. */
int bbq_search_sharded_device(bbq_index* index, const float* d_queries, uint32_t nq, uint32_t k,
                              int32_t* d_out_idx, float* d_out_score, void* stream);

/* Page-locked host memory for query / result buffers (optional: any host pointer is accepted by bbq_search*, pinned
 * ones make the copies asynchronous DMA).  A Node host wraps these in external ArrayBuffers. */
void* bbq_host_alloc(size_t bytes);
void bbq_host_free(void* p);

/* -------- oversampled search + exact re-rank (SURVEY §8f rank 2) ---------------------------------------- */

/* Keeps a copy of the ORIGINAL f32 rows next to the index (device memory, n*dim*4 bytes) for the exact re-rank.
 * rows: HOST (bbq_index_attach_rows) or DEVICE (bbq_index_attach_rows_device) memory, n = bbq_index_size rows.
 * The copy covers the rows the index has at attach time: after a later bbq_index_append* the re-rank entries return
 * BBQ_ERR_INVALID_ARG ("rows attached for N rows, index has M") until the rows are attached again. */
int bbq_index_attach_rows(bbq_index* index, const float* rows);
int bbq_index_attach_rows_device(bbq_index* index, const float* d_rows);

/* getOversampledTopKWithSort(query, quantizedVectors, vectors, k, oversampleFactor, format) —
 * src/topKSelector.ts:90-114 (the heap form :29-78 returns the same set when no true score ties at the k-th place):
 * quantised search for k*factor candidates, exact computeCosineSimilarity (src/vectorSimilarity.ts:75-102, f64)
 * against the attached rows, the min(k, n) best by (trueScore desc, quantised rank asc).  HOST pointers; nq queries.
 * out_idx / out_qscore (the quantised f32 score) / out_true (f64): nq*k each; k*factor <= 4096. */
int bbq_search_rerank(bbq_index* index, const float* queries, uint32_t nq, uint32_t k, uint32_t factor,
                      int32_t* out_idx, float* out_qscore, double* out_true, uint32_t* out_count);

/* bbq_search_rerank over ALL row shards (the sharded search's setup: bbq_comm_init, bbq_index_set_base, and the
 * original rows of its own shard attached on every rank).  Collective: every rank calls it with the same queries, nq,
 * k and factor, and every rank gets, bit for bit, what bbq_search_rerank returns on one index holding the whole
 * corpus: m = min(k*factor, rows over all ranks) candidates per query, *out_count = min(k, m), k*factor <= 4096.
 * The candidates are the sharded search's global top m; the rank that holds a candidate's row scores it, and the f64
 * bits reach every rank in one integer-sum ncclAllReduce of nq*m words.  Before that exchange the ranks share
 * {base, rows, rows attached} in one small all-gather: a rank without rows attached for all its rows, or two ranks
 * whose id ranges overlap, make EVERY rank return BBQ_ERR_INVALID_ARG with the same message.  Query screening and
 * argument errors are those of bbq_search_rerank.  Without a communicator (or world == 1) it is bbq_search_rerank.
 * HOST pointers. */
int bbq_search_rerank_sharded(bbq_index* index, const float* queries, uint32_t nq, uint32_t k, uint32_t factor,
                              int32_t* out_idx, float* out_qscore, double* out_true, uint32_t* out_count);

/* The shard-local step of bbq_search_rerank_sharded on its own (not collective; a host with an exchange of its own
 * uses it the way it uses bbq_merge_topk_device): for [nq][m] GLOBAL candidate ids d_cand_idx (-1 = empty slot),
 * writes [nq][m] 64-bit words to d_true_bits: the bits of the f64 computeCosineSimilarity of query and row
 * (src/vectorSimilarity.ts:75-102, the same arithmetic as bbq_search_rerank) when this shard holds the row
 * (0 <= id - base < rows), else 0.  Summed as integers over all shards, the words are the exact scores' bits.
 * d_queries: the raw nq*dim f32 queries.  DEVICE pointers, enqueued on `stream` (NULL = the context's stream). */
int bbq_rerank_owned_device(bbq_index* index, const float* d_queries, uint32_t nq, const int32_t* d_cand_idx,
                            uint32_t m, uint64_t* d_true_bits, void* stream);

/* Deterministic merge of `lists` per-shard results (e.g. after an NCCL allgather, SURVEY §8e):
 * inputs [lists][nq][k] idx / score in DEVICE memory, output [nq][k].  Replaces nothing in the
 * reference (it has no sharding); the ordering rule is the MinHeap contract of
 * src/binaryQuantizationFormat.ts:383-411 made canonical. */
int bbq_merge_topk_device(bbq_ctx* ctx, const int32_t* d_idx, const float* d_score, uint32_t lists,
                          uint32_t nq, uint32_t k, int32_t* d_out_idx, float* d_out_score, void* stream);

/* -------- parity / debug taps (tests only) -------------------------------------------------------- */

/* format.quantizeQueryVector — src/binaryQuantizationFormat.ts:271-299 after the :337 normalisation.
 * codes: dim bytes (unpacked 0..2^queryBits-1), corr4: 4 doubles.  HOST pointers. */
int bbq_debug_quantize_query(bbq_index* index, const float* query, uint8_t* codes, double* corr4);
/* computeBatchFourBitDotProductDirectPacked / computeBatchDotProductDirectPacked over the whole index:
 * out_dots n int32 — src/utils/computeBatchFourBitDotProductDirectPacked.ts:10-53, src/batchDotProduct.ts:22-49 */
int bbq_debug_qcdist(bbq_index* index, const float* query, int32_t* out_dots);
/* The same integers from the TENSOR-CORE scan (tcgen05 accumulators >> 3, k_scan_mma<SCAN_DUMP>) for a batch:
 * out_dots [nq][n] int32, HOST.  BBQ_ERR_UNSUPPORTED where that engine cannot run (queryBits > 5, dim > 4096). */
int bbq_debug_qcdist_batch(bbq_index* index, const float* queries, uint32_t nq, int32_t* out_dots);
/* computeBatch{FourBit,OneBit}SimilarityScores + Float32Array store: out_scores n floats —
 * src/batchDotProduct.ts:478-541,554-617, src/binaryQuantizationFormat.ts:353,378 */
int bbq_debug_scores(bbq_index* index, const float* query, float* out_scores);

/* Counters: kernels launched by this context, and what the last search call did. */
typedef struct {
  uint64_t kernel_launches;   /* launches of THIS library's kernels since bbq_create */
  uint64_t last_candidates;   /* total candidates appended by the last filtered scan */
  uint32_t last_path;         /* 0 direct (dump+select), 1 sampled threshold + filtered scan, 2 exact chunked fallback */
  uint32_t last_overflow;     /* 1 if the candidate buffer overflowed and the fallback ran */
  uint32_t last_engine;       /* scan engine of the last filtered search: 1 popcount kernel, 2 tcgen05 kernel */
  uint32_t mma_layout;        /* last tensor-core scan: role layout, 0 wide-batch (8 epilogue warps + 1 expansion group), 1 narrow-batch (4 + 2) */
  /* with bbq_set_profiling(ctx, 1): CUDA-event time of the dominant (scan) kernel launches, on their stream */
  uint64_t scan_launches;
  double scan_ms;
  double quantize_ms;         /* query quantisation (K4) launches */
  double select_ms;           /* selection / merge (K3) launches */
  double sample_ms;           /* threshold-sample scan launches (not counted in scan_ms / scan_launches) */
  uint32_t mma_n_tile;        /* last tensor-core scan: queries resident per pass */
  uint32_t mma_passes;        /* ... and passes over the shard */
  uint64_t graph_replays;     /* bbq_search calls served by replaying the captured launch sequence (narrow batches) */
} bbq_stats;
int bbq_get_stats(bbq_ctx* ctx, bbq_stats* out);
/* Off by default.  When on, search calls bracket their kernel groups with CUDA events (recorded on the launch
 * stream); bbq_get_stats synchronises them and accumulates.  bbq_reset_profiling zeroes the accumulators. */
int bbq_set_profiling(bbq_ctx* ctx, int enabled);
/* Timeline of the tensor-core scan's hand-offs (clock64 stamps of CTA 0; only recorded with BBQ_MMA_DEBUG bit 32). */
int bbq_debug_trace(bbq_ctx* ctx, long long* out, uint32_t count);
int bbq_reset_profiling(bbq_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* BBQ_B200_H */
