// Index image on disk: <name>.vemb (metadata) + <name>.veb (vector data) — the two files the reference names in
// FILE_EXTENSIONS (src/constants.ts:52-57) and describes with MetadataFormat / VectorDataFormat
// (src/types.ts:78-113).  The reference's serializeVectorData / deserializeVectorData
// (src/binaryQuantizationFormat.ts:483-560) only build JS objects and never touch a file; this is the working
// format behind the same field names.
//
//   .vemb  little-endian: MetaHeader (144 bytes) followed by centroid f32[dimensions]
//   .veb   five sections, each starting on a 4096-byte boundary, stored exactly as they sit in HBM:
//            codes         [vectorCount][rowBytes]  packed MSB-first rows, zero-padded to a 16-byte stride
//            lower         f64[vectorCount]         VectorDataFormat.lowerInterval
//            upper         f64[vectorCount]         VectorDataFormat.upperInterval
//            additional    f64[vectorCount]         VectorDataFormat.additionalCorrection
//            componentSum  u32[vectorCount]         VectorDataFormat.quantizedComponentSum
//
// Each section carries a 64-bit checksum computed ON THE DEVICE (sum over 32-bit words of splitmix64(index, word)),
// at save time over the arrays being written and at load time over the arrays just uploaded, so it covers the whole
// disk -> host -> HBM path.  Transfers are double-buffered through pinned staging (file I/O overlaps the copies).
//
// Row ranges.  Every section has a fixed stride per row (rowBytes, 8, 8, 8, 4 bytes: all multiples of 4), so rows
// [r0, r1) of an image are one contiguous byte range of each section, at offset + r0 * stride.  The word index in the
// checksum counts from the section's start (row r0 starts at word r0 * stride / 4), so the checksums of disjoint row
// ranges add up, mod 2^64, to the checksum of the whole section.  One writer (io_write_rows: a shard's rows at its
// place in an image of N rows) and one reader (io_load: rows [first, first + count) of an image) serve the whole-index
// entries and the shard entries alike; the collective entries run them on every rank and exchange the partial sums.
// Included by bbq_api.cu (one translation unit), after the NCCL plumbing.
#pragma once
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

namespace bbqio {

constexpr char MAGIC[8] = {'B', 'V', 'E', 'C', 'b', '2', '0', '0'};  // COMPONENT_NAMES.BINARIZED_VECTOR + layout tag
constexpr uint32_t VERSION = 1;
constexpr uint64_t SECTION_ALIGN = 4096;
constexpr size_t STAGE_BYTES = 32u << 20;

struct MetaHeader {
  char magic[8];
  uint32_t version;
  uint32_t fieldNumber;              // MetadataFormat.fieldNumber (always 0, as the reference writes it)
  uint32_t vectorEncodingOrdinal;    // MetadataFormat.vectorEncodingOrdinal (0)
  uint32_t vectorSimilarityOrdinal;  // 0 EUCLIDEAN, 1 COSINE, 2 MAXIMUM_INNER_PRODUCT (bbq_similarity)
  uint32_t dimensions;
  uint32_t indexBits;
  uint32_t rowBytes;
  uint32_t reserved;
  uint64_t vectorCount;
  uint64_t vectorDataOffset;  // offset of the codes section in the .veb file
  uint64_t vectorDataLength;  // length of the .veb file
  uint64_t lowerOffset, upperOffset, additionalOffset, componentSumOffset;
  double centroidSquareMagnitude;  // getCentroidDP(): sum c_i*c_i, f64, index order
  uint64_t checksum[5];            // codes, lower, upper, additional, componentSum
};
static_assert(sizeof(MetaHeader) == 144, "on-disk header layout");

__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// out += sum_i splitmix64((first_word + i) << 32 | word_i): order-independent, position-dependent.  first_word is the
// position of words[0] in its section (the shift wraps mod 2^64 as it always did), so sums over disjoint ranges of a
// section add up to the sum over the whole section.
__global__ void __launch_bounds__(256) k_section_checksum(const uint32_t* __restrict__ words, uint64_t nwords,
                                                           uint64_t first_word, unsigned long long* __restrict__ out) {
  uint64_t acc = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x; i < nwords; i += (uint64_t)gridDim.x * 256)
    acc += splitmix64(((first_word + i) << 32) | (uint64_t)__ldg(words + i));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0 && acc != 0) atomicAdd(out, (unsigned long long)acc);
}

struct Section {
  const char* name;
  void* dev;        // this index's rows of the section
  uint64_t stride;  // bytes per row
  uint64_t offset;  // of the section in the image
};

struct Fd {
  int fd = -1;
  ~Fd() {
    if (fd >= 0) close(fd);
  }
};

struct Pinned {
  void* p[2] = {nullptr, nullptr};
  cudaEvent_t ev[2] = {nullptr, nullptr};
  ~Pinned() {
    for (int i = 0; i < 2; i++) {
      if (p[i]) cudaFreeHost(p[i]);
      if (ev[i]) cudaEventDestroy(ev[i]);
    }
  }
};

static inline uint64_t align_up(uint64_t v) { return (v + SECTION_ALIGN - 1) / SECTION_ALIGN * SECTION_ALIGN; }

// host-side fingerprint of a byte string of whole 32-bit words (a centroid, a header): every rank compares its own
// with rank 0's
static inline uint64_t fingerprint(const void* p, size_t bytes) {
  uint64_t h = splitmix64(bytes);
  for (size_t i = 0; i < bytes / 4; i++) {
    uint32_t w;
    memcpy(&w, (const char*)p + 4 * i, 4);
    h = splitmix64(h ^ (((uint64_t)i << 32) | w));
  }
  return h;
}

}  // namespace bbqio

static int io_fail(const std::string& what, const char* path) {
  return fail(BBQ_ERR_IO, what + " '" + path + "': " + strerror(errno));
}

// The five sections of an image of total_rows rows (offsets) holding this index's rows (dev); returns the image length.
static uint64_t io_sections(bbq_index* ix, uint64_t total_rows, bbqio::Section s[5]) {
  s[0] = {"codes", ix->codes, (uint64_t)ix->row_bytes, 0};
  s[1] = {"lower", ix->lower, sizeof(double), 0};
  s[2] = {"upper", ix->upper, sizeof(double), 0};
  s[3] = {"additional", ix->addc, sizeof(double), 0};
  s[4] = {"componentSum", ix->compsum, sizeof(uint32_t), 0};
  uint64_t off = 0, end = 0;
  for (int i = 0; i < 5; i++) {
    s[i].offset = off;
    end = off + total_rows * s[i].stride;
    off = bbqio::align_up(end);
  }
  return end;
}

// checksums of this index's rows, which sit at rows [first, first + n) of the image
static int io_checksums(bbq_index* ix, const bbqio::Section s[5], uint64_t first, uint64_t out[5]) {
  bbq_ctx* c = ix->ctx;
  TRY(c->cacc.reserve(5 * sizeof(uint64_t)));
  CU(cudaMemsetAsync(c->cacc.p, 0, 5 * sizeof(uint64_t), c->stream));
  for (int i = 0; i < 5; i++) {
    const uint64_t nwords = ix->n * s[i].stride / 4;
    const unsigned grid = (unsigned)std::min<uint64_t>((nwords + 255) / 256, (uint64_t)c->sm_count * 8);
    LAUNCH(c, bbqio::k_section_checksum, std::max(grid, 1u), 256, 0, c->stream, (const uint32_t*)s[i].dev, nwords,
           first * s[i].stride / 4, c->cacc.as<unsigned long long>() + i);
  }
  CU(cudaMemcpyAsync(out, c->cacc.p, 5 * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return BBQ_OK;
}

static int io_pinned(bbqio::Pinned& pin) {
  for (int i = 0; i < 2; i++) {
    CU(cudaHostAlloc(&pin.p[i], bbqio::STAGE_BYTES, cudaHostAllocDefault));
    CU(cudaEventCreateWithFlags(&pin.ev[i], cudaEventDisableTiming));
  }
  return BBQ_OK;
}

// The one writer: this index's rows at rows [first, first + n) of an image of total_rows rows.  Opens (creating) the
// .veb, truncating it first only when asked (a whole-index save; shards of one image must not), sets its length to
// the image length and writes nothing outside this range.  out: the checksums of the rows written.
static int io_write_rows(bbq_index* ix, const char* veb_path, uint64_t total_rows, uint64_t first, bool truncate,
                         uint64_t out[5]) {
  bbq_ctx* c = ix->ctx;
  CU(cudaSetDevice(c->device));
  bbqio::Section s[5];
  const uint64_t len = io_sections(ix, total_rows, s);
  TRY(io_checksums(ix, s, first, out));
  bbqio::Fd veb;
  veb.fd = open(veb_path, O_WRONLY | O_CREAT | (truncate ? O_TRUNC : 0), 0644);
  if (veb.fd < 0) return io_fail("cannot create", veb_path);
  if (ftruncate(veb.fd, (off_t)len) != 0) return io_fail("cannot set the length of", veb_path);
  bbqio::Pinned pin;
  if (ix->n > 0) TRY(io_pinned(pin));
  for (int i = 0; i < 5; i++) {
    // device -> pinned (async, buffer b) while the previous buffer is being written to the file
    const uint64_t bytes = ix->n * s[i].stride, at0 = s[i].offset + first * s[i].stride;
    uint64_t done = 0, issued = 0;
    int b = 0;
    uint64_t len_b[2] = {0, 0}, at[2] = {0, 0};
    auto issue = [&](int buf) -> int {
      len_b[buf] = std::min<uint64_t>(bbqio::STAGE_BYTES, bytes - issued);
      at[buf] = issued;
      CU(cudaMemcpyAsync(pin.p[buf], (const char*)s[i].dev + issued, len_b[buf], cudaMemcpyDeviceToHost, c->stream));
      CU(cudaEventRecord(pin.ev[buf], c->stream));
      issued += len_b[buf];
      return BBQ_OK;
    };
    if (bytes > 0) TRY(issue(b));
    while (done < bytes) {
      if (issued < bytes) TRY(issue(b ^ 1));
      CU(cudaEventSynchronize(pin.ev[b]));
      uint64_t w = 0;
      while (w < len_b[b]) {
        const ssize_t r = pwrite(veb.fd, (const char*)pin.p[b] + w, len_b[b] - w, (off_t)(at0 + at[b] + w));
        if (r < 0) return io_fail("write failed on", veb_path);
        w += (uint64_t)r;
      }
      done += len_b[b];
      b ^= 1;
    }
  }
  const int rc = close(veb.fd);
  veb.fd = -1;
  if (rc != 0) return io_fail("close failed on", veb_path);
  return BBQ_OK;
}

// The .vemb of an image of total_rows rows with the given section checksums; dimension, similarity, centroid and
// centroidSquareMagnitude are this index's.
static int io_write_meta(bbq_index* ix, const char* vemb_path, uint64_t total_rows, const uint64_t sums[5]) {
  bbq_ctx* c = ix->ctx;
  bbqio::Section s[5];
  const uint64_t len = io_sections(ix, total_rows, s);
  bbqio::MetaHeader h;
  memset(&h, 0, sizeof(h));
  memcpy(h.magic, bbqio::MAGIC, 8);
  h.version = bbqio::VERSION;
  h.vectorSimilarityOrdinal = (uint32_t)c->cfg.similarity;
  h.dimensions = ix->dim;
  h.indexBits = c->cfg.index_bits;
  h.rowBytes = (uint32_t)ix->row_bytes;
  h.vectorCount = total_rows;
  h.vectorDataOffset = s[0].offset;
  h.vectorDataLength = len;
  h.lowerOffset = s[1].offset;
  h.upperOffset = s[2].offset;
  h.additionalOffset = s[3].offset;
  h.componentSumOffset = s[4].offset;
  h.centroidSquareMagnitude = ix->cdp;
  memcpy(h.checksum, sums, sizeof(h.checksum));

  bbqio::Fd meta;
  meta.fd = open(vemb_path, O_WRONLY | O_CREAT | O_TRUNC, 0644);
  if (meta.fd < 0) return io_fail("cannot create", vemb_path);
  std::vector<char> blob(sizeof(h) + ix->dim * sizeof(float));
  memcpy(blob.data(), &h, sizeof(h));
  memcpy(blob.data() + sizeof(h), ix->centroid_h.data(), ix->dim * sizeof(float));
  size_t w = 0;
  while (w < blob.size()) {
    const ssize_t r = write(meta.fd, blob.data() + w, blob.size() - w);
    if (r < 0) return io_fail("write failed on", vemb_path);
    w += (size_t)r;
  }
  const int rc = close(meta.fd);
  meta.fd = -1;
  if (rc != 0) return io_fail("close failed on", vemb_path);
  return BBQ_OK;
}

// what every image writer refuses
static int io_check_writable(const bbq_index* ix, uint64_t total_rows, uint64_t first) {
  if (ix->ib != 1) return fail(BBQ_ERR_UNSUPPORTED, "only 1-bit index images can be saved");
  if (total_rows == 0) return fail(BBQ_ERR_EMPTY, "vector set must not be empty");
  if (first > total_rows || ix->n > total_rows - first)
    return fail(BBQ_ERR_INVALID_ARG, "rows [" + std::to_string(first) + ", " + std::to_string(first + ix->n) +
                                         ") lie outside an image of " + std::to_string(total_rows) + " rows");
  return BBQ_OK;
}

extern "C" int bbq_index_save(const bbq_index* cix, const char* veb_path, const char* vemb_path) {
  bbq_index* ix = const_cast<bbq_index*>(cix);
  if (!ix || !veb_path || !vemb_path) return fail(BBQ_ERR_NULL, "null index/path");
  if (ix->n == 0) return fail(BBQ_ERR_EMPTY, "vector set must not be empty");
  TRY(io_check_writable(ix, ix->n, 0));
  uint64_t sums[5];
  TRY(io_write_rows(ix, veb_path, ix->n, 0, /*truncate=*/true, sums));
  return io_write_meta(ix, vemb_path, ix->n, sums);
}

extern "C" int bbq_index_write_rows(const bbq_index* cix, const char* veb_path, uint64_t total_rows,
                                    uint64_t out_partial[5]) {
  bbq_index* ix = const_cast<bbq_index*>(cix);
  if (!ix || !veb_path) return fail(BBQ_ERR_NULL, "null index/path");
  TRY(io_check_writable(ix, total_rows, ix->base));
  uint64_t sums[5];
  TRY(io_write_rows(ix, veb_path, total_rows, ix->base, /*truncate=*/false, sums));
  if (out_partial) memcpy(out_partial, sums, sizeof sums);
  return BBQ_OK;
}

extern "C" int bbq_index_write_meta(const bbq_index* cix, const char* vemb_path, uint64_t total_rows,
                                    const uint64_t checksums[5]) {
  bbq_index* ix = const_cast<bbq_index*>(cix);
  if (!ix || !vemb_path || !checksums) return fail(BBQ_ERR_NULL, "null index/path/checksums");
  TRY(io_check_writable(ix, total_rows, ix->base));
  return io_write_meta(ix, vemb_path, total_rows, checksums);
}

// .vemb header, checked against this context (the checks of bbq_index_load, in its order)
static int io_read_header(bbq_ctx* c, int fd, const char* vemb_path, bbqio::MetaHeader* hp) {
  bbqio::MetaHeader& h = *hp;
  if (pread(fd, &h, sizeof(h), 0) != (ssize_t)sizeof(h)) return fail(BBQ_ERR_FORMAT, std::string("truncated metadata file '") + vemb_path + "'");
  if (memcmp(h.magic, bbqio::MAGIC, 8) != 0) return fail(BBQ_ERR_FORMAT, std::string("'") + vemb_path + "' is not a BVEC metadata file");
  if (h.version != bbqio::VERSION) return fail(BBQ_ERR_FORMAT, "unsupported index image version " + std::to_string(h.version));
  if (h.indexBits != 1 || c->cfg.index_bits != 1) return fail(BBQ_ERR_UNSUPPORTED, "only 1-bit index images can be loaded");
  if (h.vectorSimilarityOrdinal != (uint32_t)c->cfg.similarity)
    return fail(BBQ_ERR_FORMAT, "index image was built for similarity ordinal " + std::to_string(h.vectorSimilarityOrdinal) +
                                    ", this format uses " + std::to_string((int)c->cfg.similarity));
  if (h.vectorCount == 0 || h.dimensions == 0) return fail(BBQ_ERR_FORMAT, "empty index image");
  if (h.vectorCount > 0x7FFFFFFFull) return fail(BBQ_ERR_UNSUPPORTED, "row ids must fit in int32");
  if (h.rowBytes != (uint32_t)row_bytes_for(h.dimensions)) return fail(BBQ_ERR_FORMAT, "row stride does not match the dimension");
  return BBQ_OK;
}

// The one reader: rows [first, first + count) of an image (whole: the entire image, whatever its size) into a new
// index whose base is `first`.  Reads only that range of each section; out_sums: the checksums of what it uploaded,
// compared with the header only when the range is the whole image.
static int io_load(bbq_ctx* c, const char* veb_path, const char* vemb_path, bool whole, uint64_t first, uint64_t count,
                   bbq_index** out_index, uint64_t out_sums[5]) {
  if (!c || !out_index) return fail(BBQ_ERR_NULL, "null ctx/out_index");
  *out_index = nullptr;
  if (!veb_path || !vemb_path) return fail(BBQ_ERR_NULL, "null path");
  CU(cudaSetDevice(c->device));

  bbqio::Fd meta;
  meta.fd = open(vemb_path, O_RDONLY);
  if (meta.fd < 0) return io_fail("cannot open", vemb_path);
  bbqio::MetaHeader h;
  TRY(io_read_header(c, meta.fd, vemb_path, &h));
  if (whole) {
    first = 0;
    count = h.vectorCount;
  }
  if (first > h.vectorCount || count > h.vectorCount - first)
    return fail(BBQ_ERR_INVALID_ARG, "rows [" + std::to_string(first) + ", " + std::to_string(first + count) +
                                         ") lie outside an image of " + std::to_string(h.vectorCount) + " rows");
  std::vector<float> centroid(h.dimensions);
  if (pread(meta.fd, centroid.data(), centroid.size() * sizeof(float), sizeof(h)) != (ssize_t)(centroid.size() * sizeof(float)))
    return fail(BBQ_ERR_FORMAT, std::string("truncated metadata file '") + vemb_path + "'");

  bbqio::Fd veb;
  veb.fd = open(veb_path, O_RDONLY);
  if (veb.fd < 0) return io_fail("cannot open", veb_path);
  struct stat sb;
  if (fstat(veb.fd, &sb) != 0) return io_fail("cannot stat", veb_path);

  IndexGuard g;
  TRY(index_alloc(c, std::max<uint64_t>(count, 1), h.dimensions, &g.ix));  // (an empty range: no 0-byte allocations)
  bbq_index* ix = g.ix;
  ix->n = count;
  bbqio::Section s[5];
  const uint64_t len = io_sections(ix, h.vectorCount, s);
  const uint64_t want[5] = {h.vectorDataOffset, h.lowerOffset, h.upperOffset, h.additionalOffset, h.componentSumOffset};
  for (int i = 0; i < 5; i++)
    if (want[i] != s[i].offset) return fail(BBQ_ERR_FORMAT, std::string("unexpected offset of section ") + s[i].name);
  if ((uint64_t)sb.st_size < len || h.vectorDataLength != len)
    return fail(BBQ_ERR_FORMAT, std::string("truncated vector data file '") + veb_path + "'");
  bbqio::Pinned pin;
  if (count > 0) TRY(io_pinned(pin));
  bool busy[2] = {false, false};
  int b = 0;
  for (int i = 0; i < 5; i++) {
    const uint64_t bytes = count * s[i].stride, at0 = s[i].offset + first * s[i].stride;
    uint64_t done = 0;
    while (done < bytes) {
      if (busy[b]) CU(cudaEventSynchronize(pin.ev[b]));  // the copy that last used this buffer has drained
      const uint64_t len_b = std::min<uint64_t>(bbqio::STAGE_BYTES, bytes - done);
      uint64_t r = 0;
      while (r < len_b) {
        const ssize_t got = pread(veb.fd, (char*)pin.p[b] + r, len_b - r, (off_t)(at0 + done + r));
        if (got < 0) return io_fail("read failed on", veb_path);
        if (got == 0) return fail(BBQ_ERR_FORMAT, std::string("truncated vector data file '") + veb_path + "'");
        r += (uint64_t)got;
      }
      CU(cudaMemcpyAsync((char*)s[i].dev + done, pin.p[b], len_b, cudaMemcpyHostToDevice, c->stream));
      CU(cudaEventRecord(pin.ev[b], c->stream));
      busy[b] = true;
      done += len_b;
      b ^= 1;
    }
  }
  CU(cudaMemcpyAsync(ix->centroid, centroid.data(), centroid.size() * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  uint64_t sums[5];
  TRY(io_checksums(ix, s, first, sums));
  if (count == h.vectorCount)
    for (int i = 0; i < 5; i++)
      if (sums[i] != h.checksum[i]) return fail(BBQ_ERR_FORMAT, std::string("checksum mismatch in section ") + s[i].name);
  TRY(finish_centroid(ix));
  if (memcmp(&ix->cdp, &h.centroidSquareMagnitude, sizeof(double)) != 0)
    return fail(BBQ_ERR_FORMAT, "centroidSquareMagnitude does not match the stored centroid");
  ix->base = first;
  if (out_sums) memcpy(out_sums, sums, sizeof sums);
  *out_index = g.release();
  return BBQ_OK;
}

extern "C" int bbq_index_load(bbq_ctx* c, const char* veb_path, const char* vemb_path, bbq_index** out_index) {
  return io_load(c, veb_path, vemb_path, /*whole=*/true, 0, 0, out_index, nullptr);
}

extern "C" int bbq_index_load_rows(bbq_ctx* c, const char* veb_path, const char* vemb_path, uint64_t first,
                                   uint64_t count, bbq_index** out_index, uint64_t out_partial[5]) {
  return io_load(c, veb_path, vemb_path, /*whole=*/false, first, count, out_index, out_partial);
}

// ------------------------------------------------------------------------------------------------
// the image across row shards: collective save / load.  Every phase ends in an exchange that carries each rank's
// status, so a rank that fails (open, read, out of memory, a bad header) never leaves its peers waiting in a
// collective: every rank derives the same verdict from the same words and returns the same status and message.
// ------------------------------------------------------------------------------------------------
struct RankWord {  // one rank's contribution to an exchange: status, up to 7 words of state, and its error message
  uint64_t status;
  uint64_t w[7];
  char msg[192];
};
static_assert(sizeof(RankWord) == 256, "exchanged as 32 u64 words");

static RankWord rank_word(int status) {
  RankWord r;
  memset(&r, 0, sizeof r);
  r.status = (uint64_t)status;
  if (status != BBQ_OK) snprintf(r.msg, sizeof r.msg, "%s", g_err.c_str());
  return r;
}

// one ncclAllGather of every rank's RankWord
static int gather_ranks(bbq_ctx* c, const RankWord& mine, std::vector<RankWord>& all) {
  const int world = c->world;
  TRY(c->nglob.reserve(sizeof(RankWord) * (size_t)(1 + world)));
  char* d = c->nglob.as<char>();
  all.assign((size_t)world, RankWord{});
  CU(cudaMemcpyAsync(d, &mine, sizeof mine, cudaMemcpyHostToDevice, c->stream));
  NC(nccl_api()->AllGather(d, d + sizeof(RankWord), sizeof(RankWord) / 8, ncclUint64, c->comm, c->stream));
  CU(cudaMemcpyAsync(all.data(), d + sizeof(RankWord), all.size() * sizeof(RankWord), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return BBQ_OK;
}

// the verdict on an exchange: the status and message of the lowest failing rank, on every rank
static int first_failure(const std::vector<RankWord>& all, const char* what) {
  for (size_t r = 0; r < all.size(); r++)
    if (all[r].status != BBQ_OK)
      return fail((int)all[r].status, std::string(what) + ": rank " + std::to_string(r) + ": " + all[r].msg);
  return BBQ_OK;
}

// one integer-sum ncclAllReduce of the five partial checksums
static int sum_partials(bbq_ctx* c, uint64_t sums[5]) {
  TRY(c->nglob.reserve(5 * sizeof(uint64_t)));
  CU(cudaMemcpyAsync(c->nglob.p, sums, 5 * sizeof(uint64_t), cudaMemcpyHostToDevice, c->stream));
  NC(nccl_api()->AllReduce(c->nglob.p, c->nglob.p, 5, ncclUint64, ncclSum, c->comm, c->stream));
  CU(cudaMemcpyAsync(sums, c->nglob.p, 5 * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return BBQ_OK;
}

// The shards of a sharded save, from the gathered {base, n, dim, similarity, indexBits, centroid fingerprint,
// centroidSquareMagnitude bits}: 1-bit everywhere, rank 0's dimension, similarity and centroid everywhere, and the
// non-empty shards tiling [0, total) exactly.  The same words give the same verdict on every rank.
static int check_tiling(const std::vector<RankWord>& all, uint64_t* total) {
  const int world = (int)all.size();
  for (int r = 0; r < world; r++)
    if (all[r].w[4] != 1) return fail(BBQ_ERR_UNSUPPORTED, "only 1-bit index images can be saved");
  for (int r = 1; r < world; r++) {
    if (all[r].w[2] != all[0].w[2] || all[r].w[3] != all[0].w[3])
      return fail(BBQ_ERR_INVALID_ARG, "sharded save: rank " + std::to_string(r) + " has dimension " +
                                           std::to_string(all[r].w[2]) + " and similarity " + std::to_string(all[r].w[3]) +
                                           ", rank 0 has " + std::to_string(all[0].w[2]) + " and " + std::to_string(all[0].w[3]));
    if (all[r].w[5] != all[0].w[5] || all[r].w[6] != all[0].w[6])
      return fail(BBQ_ERR_INVALID_ARG, "sharded save: the centroid of rank " + std::to_string(r) + " differs from rank 0's");
  }
  std::vector<int> order;
  for (int r = 0; r < world; r++)
    if (all[r].w[1] > 0) order.push_back(r);
  std::sort(order.begin(), order.end(), [&](int a, int b) { return all[a].w[0] < all[b].w[0] || (all[a].w[0] == all[b].w[0] && a < b); });
  uint64_t next = 0;
  int prev = -1;
  for (int r : order) {
    const uint64_t base = all[r].w[0];
    if (base > next)
      return fail(BBQ_ERR_INVALID_ARG, "sharded save: rows [" + std::to_string(next) + ", " + std::to_string(base) +
                                           ") are held by no rank");
    if (base < next)
      return fail(BBQ_ERR_INVALID_ARG, "sharded save: the rows of rank " + std::to_string(r) + " [" + std::to_string(base) +
                                           ", " + std::to_string(base + all[r].w[1]) + ") overlap those of rank " +
                                           std::to_string(prev) + " (up to row " + std::to_string(next) + ")");
    next = base + all[r].w[1];
    prev = r;
  }
  if (next == 0) return fail(BBQ_ERR_EMPTY, "vector set must not be empty");
  *total = next;
  return BBQ_OK;
}

extern "C" int bbq_index_save_sharded(const bbq_index* cix, const char* veb_path, const char* vemb_path) {
  bbq_index* ix = const_cast<bbq_index*>(cix);
  if (!ix) return fail(BBQ_ERR_NULL, "null index/path");
  bbq_ctx* c = ix->ctx;
  TRY(group_guard(c));
  if (!c->comm || c->world == 1) return bbq_index_save(ix, veb_path, vemb_path);  // one shard: the plain entry
  CU(cudaSetDevice(c->device));
  std::vector<RankWord> all;
  // 1. who holds which rows, with which centroid
  RankWord mine = rank_word(veb_path && vemb_path ? BBQ_OK : fail(BBQ_ERR_NULL, "null index/path"));
  const uint64_t shape[7] = {ix->base, ix->n, ix->dim, (uint64_t)c->cfg.similarity, (uint64_t)ix->ib,
                             bbqio::fingerprint(ix->centroid_h.data(), ix->dim * sizeof(float)), 0};
  memcpy(mine.w, shape, sizeof shape);
  memcpy(&mine.w[6], &ix->cdp, sizeof(double));
  TRY(gather_ranks(c, mine, all));
  TRY(first_failure(all, "sharded save"));
  uint64_t total = 0;
  TRY(check_tiling(all, &total));
  // 2. rank 0 removes the old metadata first (a half-written image then never loads) and creates the vector data file
  int st = BBQ_OK;
  if (c->rank == 0) {
    bbqio::Section s[5];
    const uint64_t len = io_sections(ix, total, s);
    bbqio::Fd veb;
    if (unlink(vemb_path) != 0 && errno != ENOENT) st = io_fail("cannot remove", vemb_path);
    if (st == BBQ_OK && (veb.fd = open(veb_path, O_WRONLY | O_CREAT | O_TRUNC, 0644)) < 0) st = io_fail("cannot create", veb_path);
    if (st == BBQ_OK && ftruncate(veb.fd, (off_t)len) != 0) st = io_fail("cannot set the length of", veb_path);
  }
  // 3. barrier: no rank writes into a file rank 0 has not created yet
  TRY(gather_ranks(c, rank_word(st), all));
  TRY(first_failure(all, "sharded save"));
  // 4. every rank writes its rows
  uint64_t sums[5] = {0, 0, 0, 0, 0};
  st = io_write_rows(ix, veb_path, total, ix->base, /*truncate=*/false, sums);
  // 5. the partial checksums summed, and every rank's status
  TRY(sum_partials(c, sums));
  TRY(gather_ranks(c, rank_word(st), all));
  TRY(first_failure(all, "sharded save"));
  // 6. rank 0 writes the metadata; 7. every rank returns its verdict
  st = c->rank == 0 ? io_write_meta(ix, vemb_path, total, sums) : BBQ_OK;
  TRY(gather_ranks(c, rank_word(st), all));
  return first_failure(all, "sharded save");
}

extern "C" int bbq_index_load_sharded(bbq_ctx* c, const char* veb_path, const char* vemb_path, bbq_index** out_index) {
  if (!c || !out_index) return fail(BBQ_ERR_NULL, "null ctx/out_index");
  *out_index = nullptr;
  TRY(group_guard(c));
  if (!c->comm || c->world == 1) return bbq_index_load(c, veb_path, vemb_path, out_index);  // one shard: the plain entry
  CU(cudaSetDevice(c->device));
  // 1. the header this rank reads decides its range (the split of host/sharded.py:shard_bounds); 2. its rows
  bbqio::MetaHeader h;
  memset(&h, 0, sizeof h);
  int st = BBQ_OK;
  if (!veb_path || !vemb_path) {
    st = fail(BBQ_ERR_NULL, "null path");
  } else {
    bbqio::Fd meta;
    meta.fd = open(vemb_path, O_RDONLY);
    if (meta.fd < 0) st = io_fail("cannot open", vemb_path);
    else if (pread(meta.fd, &h, sizeof h, 0) != (ssize_t)sizeof h)
      st = fail(BBQ_ERR_FORMAT, std::string("truncated metadata file '") + vemb_path + "'");
  }
  IndexGuard g;
  uint64_t sums[5] = {0, 0, 0, 0, 0};
  if (st == BBQ_OK) {
    const uint64_t n = h.vectorCount, per = n / (uint64_t)c->world + (n % (uint64_t)c->world != 0);
    const uint64_t r0 = std::min(n, (uint64_t)c->rank * per), r1 = std::min(n, (uint64_t)(c->rank + 1) * per);
    st = io_load(c, veb_path, vemb_path, /*whole=*/false, r0, r1 - r0, &g.ix, sums);
  }
  // 3. the partial checksums summed; every rank's status and the fingerprint of the header it read
  TRY(sum_partials(c, sums));
  RankWord mine = rank_word(st);
  mine.w[0] = bbqio::fingerprint(&h, sizeof h);
  std::vector<RankWord> all;
  TRY(gather_ranks(c, mine, all));
  TRY(first_failure(all, "sharded load"));
  for (size_t r = 1; r < all.size(); r++)
    if (all[r].w[0] != all[0].w[0])
      return fail(BBQ_ERR_FORMAT, "sharded load: rank " + std::to_string(r) + " read another index image than rank 0");
  // 4. the whole image's checksums, checked on every rank against the same header
  static const char* names[5] = {"codes", "lower", "upper", "additional", "componentSum"};
  for (int i = 0; i < 5; i++)
    if (sums[i] != h.checksum[i]) return fail(BBQ_ERR_FORMAT, std::string("checksum mismatch in section ") + names[i]);
  *out_index = g.release();
  return BBQ_OK;
}
