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
// Included by bbq_api.cu (one translation unit).
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

__device__ __forceinline__ uint64_t splitmix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// out += sum_i splitmix64(i << 32 | word_i): order-independent, position-dependent
__global__ void __launch_bounds__(256) k_section_checksum(const uint32_t* __restrict__ words, uint64_t nwords,
                                                           unsigned long long* __restrict__ out) {
  uint64_t acc = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x; i < nwords; i += (uint64_t)gridDim.x * 256)
    acc += splitmix64((i << 32) | (uint64_t)__ldg(words + i));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0 && acc != 0) atomicAdd(out, (unsigned long long)acc);
}

struct Section {
  const char* name;
  void* dev;
  uint64_t bytes;
  uint64_t offset;
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

}  // namespace bbqio

static int io_fail(const std::string& what, const char* path) {
  return fail(BBQ_ERR_IO, what + " '" + path + "': " + strerror(errno));
}

static void io_sections(bbq_index* ix, bbqio::Section s[5]) {
  const uint64_t n = ix->n;
  s[0] = {"codes", ix->codes, n * (uint64_t)ix->row_bytes, 0};
  s[1] = {"lower", ix->lower, n * sizeof(double), 0};
  s[2] = {"upper", ix->upper, n * sizeof(double), 0};
  s[3] = {"additional", ix->addc, n * sizeof(double), 0};
  s[4] = {"componentSum", ix->compsum, n * sizeof(uint32_t), 0};
  uint64_t off = 0;
  for (int i = 0; i < 5; i++) {
    s[i].offset = off;
    off = bbqio::align_up(off + s[i].bytes);
  }
}

static int io_checksums(bbq_index* ix, const bbqio::Section s[5], uint64_t out[5]) {
  bbq_ctx* c = ix->ctx;
  TRY(c->cacc.reserve(5 * sizeof(uint64_t)));
  CU(cudaMemsetAsync(c->cacc.p, 0, 5 * sizeof(uint64_t), c->stream));
  for (int i = 0; i < 5; i++) {
    const uint64_t nwords = s[i].bytes / 4;
    const unsigned grid = (unsigned)std::min<uint64_t>((nwords + 255) / 256, (uint64_t)c->sm_count * 8);
    LAUNCH(c, bbqio::k_section_checksum, std::max(grid, 1u), 256, 0, c->stream, (const uint32_t*)s[i].dev, nwords,
           c->cacc.as<unsigned long long>() + i);
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

extern "C" int bbq_index_save(const bbq_index* cix, const char* veb_path, const char* vemb_path) {
  bbq_index* ix = const_cast<bbq_index*>(cix);
  if (!ix || !veb_path || !vemb_path) return fail(BBQ_ERR_NULL, "null index/path");
  if (ix->n == 0) return fail(BBQ_ERR_EMPTY, "vector set must not be empty");
  if (ix->ib != 1) return fail(BBQ_ERR_UNSUPPORTED, "only 1-bit index images can be saved");
  bbq_ctx* c = ix->ctx;
  CU(cudaSetDevice(c->device));
  bbqio::Section s[5];
  io_sections(ix, s);
  bbqio::MetaHeader h;
  memset(&h, 0, sizeof(h));
  memcpy(h.magic, bbqio::MAGIC, 8);
  h.version = bbqio::VERSION;
  h.vectorSimilarityOrdinal = (uint32_t)c->cfg.similarity;
  h.dimensions = ix->dim;
  h.indexBits = c->cfg.index_bits;
  h.rowBytes = (uint32_t)ix->row_bytes;
  h.vectorCount = ix->n;
  h.vectorDataOffset = s[0].offset;
  h.vectorDataLength = s[4].offset + s[4].bytes;
  h.lowerOffset = s[1].offset;
  h.upperOffset = s[2].offset;
  h.additionalOffset = s[3].offset;
  h.componentSumOffset = s[4].offset;
  h.centroidSquareMagnitude = ix->cdp;
  TRY(io_checksums(ix, s, h.checksum));

  bbqio::Pinned pin;
  TRY(io_pinned(pin));
  bbqio::Fd veb;
  veb.fd = open(veb_path, O_WRONLY | O_CREAT | O_TRUNC, 0644);
  if (veb.fd < 0) return io_fail("cannot create", veb_path);
  for (int i = 0; i < 5; i++) {
    // device -> pinned (async, buffer b) while the previous buffer is being written to the file
    uint64_t done = 0, issued = 0;
    int b = 0;
    uint64_t len[2] = {0, 0}, at[2] = {0, 0};
    auto issue = [&](int buf) -> int {
      len[buf] = std::min<uint64_t>(bbqio::STAGE_BYTES, s[i].bytes - issued);
      at[buf] = issued;
      CU(cudaMemcpyAsync(pin.p[buf], (const char*)s[i].dev + issued, len[buf], cudaMemcpyDeviceToHost, c->stream));
      CU(cudaEventRecord(pin.ev[buf], c->stream));
      issued += len[buf];
      return BBQ_OK;
    };
    if (s[i].bytes > 0) TRY(issue(b));
    while (done < s[i].bytes) {
      if (issued < s[i].bytes) TRY(issue(b ^ 1));
      CU(cudaEventSynchronize(pin.ev[b]));
      uint64_t w = 0;
      while (w < len[b]) {
        const ssize_t r = pwrite(veb.fd, (const char*)pin.p[b] + w, len[b] - w, (off_t)(s[i].offset + at[b] + w));
        if (r < 0) return io_fail("write failed on", veb_path);
        w += (uint64_t)r;
      }
      done += len[b];
      b ^= 1;
    }
  }
  if (close(veb.fd) != 0) {
    veb.fd = -1;
    return io_fail("close failed on", veb_path);
  }
  veb.fd = -1;

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
  if (close(meta.fd) != 0) {
    meta.fd = -1;
    return io_fail("close failed on", vemb_path);
  }
  meta.fd = -1;
  return BBQ_OK;
}

extern "C" int bbq_index_load(bbq_ctx* c, const char* veb_path, const char* vemb_path, bbq_index** out_index) {
  if (!c || !out_index) return fail(BBQ_ERR_NULL, "null ctx/out_index");
  *out_index = nullptr;
  if (!veb_path || !vemb_path) return fail(BBQ_ERR_NULL, "null path");
  CU(cudaSetDevice(c->device));

  bbqio::Fd meta;
  meta.fd = open(vemb_path, O_RDONLY);
  if (meta.fd < 0) return io_fail("cannot open", vemb_path);
  bbqio::MetaHeader h;
  if (pread(meta.fd, &h, sizeof(h), 0) != (ssize_t)sizeof(h)) return fail(BBQ_ERR_FORMAT, std::string("truncated metadata file '") + vemb_path + "'");
  if (memcmp(h.magic, bbqio::MAGIC, 8) != 0) return fail(BBQ_ERR_FORMAT, std::string("'") + vemb_path + "' is not a BVEC metadata file");
  if (h.version != bbqio::VERSION) return fail(BBQ_ERR_FORMAT, "unsupported index image version " + std::to_string(h.version));
  if (h.indexBits != 1 || c->cfg.index_bits != 1) return fail(BBQ_ERR_UNSUPPORTED, "only 1-bit index images can be loaded");
  if (h.vectorSimilarityOrdinal != (uint32_t)c->cfg.similarity)
    return fail(BBQ_ERR_FORMAT, "index image was built for similarity ordinal " + std::to_string(h.vectorSimilarityOrdinal) +
                                    ", this format uses " + std::to_string((int)c->cfg.similarity));
  if (h.vectorCount == 0 || h.dimensions == 0) return fail(BBQ_ERR_FORMAT, "empty index image");
  if (h.vectorCount > 0x7FFFFFFFull) return fail(BBQ_ERR_UNSUPPORTED, "row ids must fit in int32");
  if (h.rowBytes != (uint32_t)row_bytes_for(h.dimensions)) return fail(BBQ_ERR_FORMAT, "row stride does not match the dimension");
  std::vector<float> centroid(h.dimensions);
  if (pread(meta.fd, centroid.data(), centroid.size() * sizeof(float), sizeof(h)) != (ssize_t)(centroid.size() * sizeof(float)))
    return fail(BBQ_ERR_FORMAT, std::string("truncated metadata file '") + vemb_path + "'");

  bbqio::Fd veb;
  veb.fd = open(veb_path, O_RDONLY);
  if (veb.fd < 0) return io_fail("cannot open", veb_path);
  struct stat sb;
  if (fstat(veb.fd, &sb) != 0) return io_fail("cannot stat", veb_path);

  IndexGuard g;
  TRY(index_alloc(c, h.vectorCount, h.dimensions, &g.ix));
  bbq_index* ix = g.ix;
  bbqio::Section s[5];
  io_sections(ix, s);
  const uint64_t want[5] = {h.vectorDataOffset, h.lowerOffset, h.upperOffset, h.additionalOffset, h.componentSumOffset};
  for (int i = 0; i < 5; i++)
    if (want[i] != s[i].offset) return fail(BBQ_ERR_FORMAT, std::string("unexpected offset of section ") + s[i].name);
  if ((uint64_t)sb.st_size < s[4].offset + s[4].bytes || h.vectorDataLength != s[4].offset + s[4].bytes)
    return fail(BBQ_ERR_FORMAT, std::string("truncated vector data file '") + veb_path + "'");
  bbqio::Pinned pin;
  TRY(io_pinned(pin));
  bool busy[2] = {false, false};
  int b = 0;
  for (int i = 0; i < 5; i++) {
    uint64_t done = 0;
    while (done < s[i].bytes) {
      if (busy[b]) CU(cudaEventSynchronize(pin.ev[b]));  // the copy that last used this buffer has drained
      const uint64_t len = std::min<uint64_t>(bbqio::STAGE_BYTES, s[i].bytes - done);
      uint64_t r = 0;
      while (r < len) {
        const ssize_t got = pread(veb.fd, (char*)pin.p[b] + r, len - r, (off_t)(s[i].offset + done + r));
        if (got < 0) return io_fail("read failed on", veb_path);
        if (got == 0) return fail(BBQ_ERR_FORMAT, std::string("truncated vector data file '") + veb_path + "'");
        r += (uint64_t)got;
      }
      CU(cudaMemcpyAsync((char*)s[i].dev + done, pin.p[b], len, cudaMemcpyHostToDevice, c->stream));
      CU(cudaEventRecord(pin.ev[b], c->stream));
      busy[b] = true;
      done += len;
      b ^= 1;
    }
  }
  CU(cudaMemcpyAsync(ix->centroid, centroid.data(), centroid.size() * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  uint64_t sums[5];
  TRY(io_checksums(ix, s, sums));
  for (int i = 0; i < 5; i++)
    if (sums[i] != h.checksum[i]) return fail(BBQ_ERR_FORMAT, std::string("checksum mismatch in section ") + s[i].name);
  TRY(finish_centroid(ix));
  if (memcmp(&ix->cdp, &h.centroidSquareMagnitude, sizeof(double)) != 0)
    return fail(BBQ_ERR_FORMAT, "centroidSquareMagnitude does not match the stored centroid");
  *out_index = g.release();
  return BBQ_OK;
}
