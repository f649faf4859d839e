// bbq_kernels.cuh — sm_100a kernels of the brute-force quantized search path.
//
//   K5  k_osq_index      index-side OptimizedScalarQuantizer + MSB-first pack, SoA correctives
//   K4  k_osq_query      query-side quantiser (COSINE: double normalisation), k_query_planes bit-planes
//   K1  k_scan<NB,MODE>  4b x 1b scan: AND + POPC per query bit-plane, exact f64 corrective epilogue,
//                        fused threshold filter (candidates) or score dump
//   K3  k_select<MODE>   deterministic (score desc, row id asc) top-k: threshold / final / shard merge
//
// Reference lines each kernel replaces are cited at the kernel.  Compile with --fmad=false.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include "bbq_numerics.cuh"

namespace bbqk {

constexpr int TILE_ROWS = 128;     // rows per scan tile == threads per scan CTA
constexpr int SELECT_THREADS = 512;
constexpr int SELECT_MAX = 16384;  // max keys one select CTA sorts (128 KB of shared memory)

// ------------------------------------------------------------------------------------------------
// Staging: row-major f32 rows -> transposed scratch T[dim][ld] so that one thread per vector walks its
// components with coalesced loads (thread t reads T[i*ld + t]).
// ------------------------------------------------------------------------------------------------
__global__ void k_transpose(const float* __restrict__ rows, int64_t nrows, int dim, float* __restrict__ T,
                            int64_t ld) {
  __shared__ float tile[32][33];
  const int64_t r0 = (int64_t)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    const int64_t r = r0 + j;
    const int c = c0 + threadIdx.x;
    tile[j][threadIdx.x] = (r < nrows && c < dim) ? rows[r * dim + c] : 0.0f;
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    const int c = c0 + j;
    const int64_t r = r0 + threadIdx.x;
    if (c < dim && r < nrows) T[(int64_t)c * ld + r] = tile[threadIdx.x][j];
  }
}

struct TAcc {  // component accessor over the transposed scratch
  const float* p;
  int64_t ld;
  __device__ __forceinline__ float operator()(int i) const { return p[(int64_t)i * ld]; }
};
struct CAcc {  // centroid accessor (same address across the warp: one broadcast transaction)
  const float* p;
  __device__ __forceinline__ float operator()(int i) const { return __ldg(p + i); }
};

// normalizeVector, src/vectorOperations.ts:11-34, `times` times in place (queries: twice,
// src/binaryQuantizationFormat.ts:337 and :279).  One thread per vector, sequential f64 sum.
__global__ void k_normalize_T(float* __restrict__ T, int64_t ld, int64_t nrows, int dim, int times) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nrows) return;
  float* col = T + t;
  for (int rep = 0; rep < times; rep++) {
    TAcc v{col, ld};
    const double n = bbqn::l2norm_seq(v, dim);
    if (n == 0) {
      for (int i = 0; i < dim; i++) col[(int64_t)i * ld] = 0.0f;
    } else {
      for (int i = 0; i < dim; i++) col[(int64_t)i * ld] = (float)((double)col[(int64_t)i * ld] / n);
    }
  }
}

// The f64 norm of each row-major row, in bbqn::l2norm_seq order: the divisor k_normalize_T uses for COSINE.
struct RAcc {
  const float* p;
  __device__ __forceinline__ float operator()(int i) const { return p[i]; }
};
__global__ void k_row_norms(const float* __restrict__ rows, int64_t nrows, int dim, double* __restrict__ norms) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < nrows) norms[t] = bbqn::l2norm_seq(RAcc{rows + t * dim}, dim);
}

__device__ __forceinline__ void cp_async4(float* smem, const float* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// COSINE rows for the centroid chain, normalised into row-major scratch: out = f32((double)v / norm), or 0 when
// norm == 0, exactly as k_normalize_T computes it, with the norms of k_row_norms.  One thread per element, so that the
// f64 divisions run on the whole GPU instead of inside the chain.
__global__ void k_normalize_rows(const float* __restrict__ rows, int64_t nrows, int dim, const double* __restrict__ norms,
                                 float* __restrict__ out) {
  const int64_t total = nrows * dim;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const double nn = norms[e / dim];
    out[e] = nn == 0 ? 0.0f : (float)((double)rows[e] / nn);
  }
}

// computeCentroid, src/vectorOperations.ts:126-163: centroid = copy(V[0]); for j>=1: c_i = f32(c_i + V[j]_i) strictly in
// row order.  The running sum acc[0, dim) is continued over rows [0, nrows) (row-major, COSINE rows already normalised
// by k_normalize_rows); starts_corpus: rows[0] is the corpus's row 0 and is copied, otherwise every row is added.  Each
// step is __fadd_rn: for two f32 operands the correctly rounded f32 sum equals f32(f64 sum) (53 >= 2*24 + 2), the same
// bits for +-0, subnormals, +-Inf and NaN.  One warp per 32 components (grid: ceil(dim / 32) blocks of 32 threads): the
// lanes read one row's 128 contiguous bytes, and cp.async keeps CHAIN_GROUPS groups of CHAIN_ROWS rows in flight in
// shared memory, so the only dependent work per row is one shared load and one FADD.
constexpr int CHAIN_ROWS = 16;
constexpr int CHAIN_GROUPS = 16;
__global__ void __launch_bounds__(32) k_centroid_chain(const float* __restrict__ rows, int64_t nrows, int dim,
                                                       float* __restrict__ acc, int starts_corpus) {
  __shared__ float ring[CHAIN_GROUPS * CHAIN_ROWS][32];
  const int lane = threadIdx.x;
  const int i = blockIdx.x * 32 + lane;
  const bool on = i < dim;
  const float* col = rows + (on ? i : 0);
  const int64_t ngroups = (nrows + CHAIN_ROWS - 1) / CHAIN_ROWS;
  auto issue = [&](int64_t g) {  // one commit per call, empty past the end, so that wait_group counts uniformly
    if (g < ngroups) {
      const int slot = (int)(g % CHAIN_GROUPS) * CHAIN_ROWS;
      const int m = (int)min((int64_t)CHAIN_ROWS, nrows - g * CHAIN_ROWS);
      const float* src = col + g * CHAIN_ROWS * dim;
#pragma unroll
      for (int u = 0; u < CHAIN_ROWS; u++)
        if (on && u < m) cp_async4(&ring[slot + u][lane], src + (int64_t)u * dim);
    }
    cp_async_commit();
  };
#pragma unroll
  for (int g = 0; g < CHAIN_GROUPS - 1; g++) issue(g);
  float c = (on && !starts_corpus) ? acc[i] : 0.0f;
  for (int64_t g = 0; g < ngroups; g++) {
    issue(g + CHAIN_GROUPS - 1);  // into the slot group g - 1 used (each lane reads back only what it copied)
    cp_async_wait<CHAIN_GROUPS - 1>();
    const int slot = (int)(g % CHAIN_GROUPS) * CHAIN_ROWS;
    const int u0 = (g == 0 && starts_corpus) ? 1 : 0;
    const int m = (int)min((int64_t)CHAIN_ROWS, nrows - g * CHAIN_ROWS);
    if (u0) c = ring[slot][lane];
#pragma unroll
    for (int u = 0; u < CHAIN_ROWS; u++)
      if (u >= u0 && u < m) c = __fadd_rn(c, ring[slot + u][lane]);
  }
  cp_async_wait<0>();
  if (on) acc[i] = c;
}
__global__ void k_centroid_finish(float* __restrict__ acc, int dim, double n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < dim) acc[i] = (float)((double)acc[i] / n);
}
// getCentroidDP(undefined) = centroid . centroid, src/binaryQuantizationFormat.ts:113-121 (f64, sequential)
__global__ void k_centroid_dp(const float* __restrict__ c, int dim, double* __restrict__ out) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    double s = 0.0;
    for (int i = 0; i < dim; i++) s += (double)c[i] * (double)c[i];
    *out = s;
  }
}

// K5: scalarQuantize(indexBits) + packAsBinary, src/optimizedScalarQuantizer.ts:108-227,420-446,
// driven as src/binaryQuantizationFormat.ts:221-249 does.  One thread per vector.
// Device row layout (north-star item 1, "bit-plane-interleaved, 16-byte aligned"): the row is a sequence of 16-byte
// chunks; chunk rc * IB + p holds bit-plane p (p = 0: least significant) of the codes of dims [128 rc, 128 rc + 128),
// MSB-first inside each byte (dim 8j+t -> bit 7-t of byte j) exactly as packAsBinary writes a 1-bit row; zero padded.
// With IB = 1 this IS the reference's packed row (padded to 16 bytes).  With IB >= 2 (EXTENSION: the reference keeps
// such rows unpacked and cannot search them) a scan sees a 1-bit row of IB * 128 * chunks "virtual dims".
template <int IB>
__global__ void k_osq_index(const float* __restrict__ T, int64_t ld, int64_t nrows, int dim,
                            const float* __restrict__ centroid, int sim, double lambda, int iters,
                            uint8_t* __restrict__ codes, int row_bytes, int64_t row0,
                            double* __restrict__ lower, double* __restrict__ upper,
                            double* __restrict__ addc, uint32_t* __restrict__ compsum) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nrows) return;
  TAcc v{T + t, ld};
  CAcc c{centroid};
  const bbqn::OsqResult r = bbqn::osq_interval(v, c, dim, IB, sim, lambda, iters);
  uint4* out = reinterpret_cast<uint4*>(codes + (row0 + t) * (int64_t)row_bytes);
  uint32_t w[IB][4], cur[IB];
#pragma unroll
  for (int p = 0; p < IB; p++) {
    cur[p] = 0u;
#pragma unroll
    for (int j = 0; j < 4; j++) w[p][j] = 0u;
  }
  int nout = 0;
  auto flush_chunk = [&]() {
#pragma unroll
    for (int p = 0; p < IB; p++) {
      out[nout++] = make_uint4(w[p][0], w[p][1], w[p][2], w[p][3]);
#pragma unroll
      for (int j = 0; j < 4; j++) w[p][j] = 0u;
    }
  };
  const double qsum = bbqn::osq_codes(v, c, dim, IB, r.lower, r.upper, [&](int i, uint8_t q) {
    const int sh = 8 * ((i >> 3) & 3) + 7 - (i & 7);  // little-endian word of MSB-first bytes
#pragma unroll
    for (int p = 0; p < IB; p++) cur[p] |= (uint32_t)((q >> p) & 1u) << sh;
    if ((i & 31) == 31) {
      const int j = (i >> 5) & 3;
#pragma unroll
      for (int p = 0; p < IB; p++) {
        if (j == 0) w[p][0] = cur[p];
        else if (j == 1) w[p][1] = cur[p];
        else if (j == 2) w[p][2] = cur[p];
        else w[p][3] = cur[p];
        cur[p] = 0u;
      }
      if (j == 3) flush_chunk();
    }
  });
  if (dim & 31) {  // partial last word
    const int j = (dim >> 5) & 3;
#pragma unroll
    for (int p = 0; p < IB; p++) {
      if (j == 0) w[p][0] = cur[p];
      else if (j == 1) w[p][1] = cur[p];
      else if (j == 2) w[p][2] = cur[p];
      else w[p][3] = cur[p];
    }
  }
  if (dim & 127) flush_chunk();
  for (; nout < row_bytes / 16; nout++) out[nout] = make_uint4(0u, 0u, 0u, 0u);
  lower[row0 + t] = r.lower;
  upper[row0 + t] = r.upper;
  addc[row0 + t] = r.additional;
  compsum[row0 + t] = (uint32_t)qsum;
}

// K4: quantizeQueryVector, src/binaryQuantizationFormat.ts:271-299 (normalisation done by k_normalize_T).
// qcodes: [nq][code_ld] unpacked u8; qcorr: [nq][4] = lower, upper, additional, componentSum.
__global__ void k_osq_query(const float* __restrict__ T, int64_t ld, int nq, int dim,
                            const float* __restrict__ centroid, int sim, int bits, double lambda, int iters,
                            uint8_t* __restrict__ qcodes, int code_ld, double* __restrict__ qcorr) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nq) return;
  TAcc v{T + t, ld};
  CAcc c{centroid};
  const bbqn::OsqResult r = bbqn::osq_interval(v, c, dim, bits, sim, lambda, iters);
  uint8_t* out = qcodes + (int64_t)t * code_ld;
  const double qsum = bbqn::osq_codes(v, c, dim, bits, r.lower, r.upper, [&](int i, uint8_t q) { out[i] = q; });
  for (int i = dim; i < code_ld; i++) out[i] = 0;
  qcorr[4 * t + 0] = r.lower;
  qcorr[4 * t + 1] = r.upper;
  qcorr[4 * t + 2] = r.additional;
  qcorr[4 * t + 3] = qsum;
}

// K4, latency forms: ONE WARP per query, or ONE CTA per query.  The reference's sums are strictly sequential f64 (any
// re-association can flip a Math.round), so the per-component terms are computed in parallel and each chain is then
// accumulated in component order by ONE lane reading the staged terms from shared memory — up to 7 chains run side by
// side in lanes 0..6.  The coordinate descent is fused: the loss of a candidate interval and the grid sums of that same
// interval (needed only if it is accepted) share one pass.  Same arithmetic, same order, same bits as
// bbqn::osq_interval / osq_codes (tests compare all forms with the oracle).
//
// The two forms differ in who generates the terms (a "team" policy; the quantiser body below is shared):
//   * WarpTeam — the warp that owns the chain also generates: the generator's f64 math (~150 instructions per 32
//     components in the fused pass, a division among them) fills the latency slots of the 32 dependent adds, but both
//     share one warp's issue slots: ~400 cycles per 32 components.  Best throughput for large batches (4 queries per CTA).
//   * CtaTeam  — eight producer warps generate a 256-component super-block ahead while warp 0 does nothing but the
//     dependent adds: the pass runs at the latency of the add chain itself.  For a single query / a narrow batch,
//     where K4 is the longest kernel of the whole search.
struct WarpTeam {
  int lane;
  double (*terms)[33];  // [2 * 7][33]
  __device__ __forceinline__ int tid() const { return lane; }
  __device__ __forceinline__ int size() const { return 32; }
  __device__ __forceinline__ void sync() const { __syncwarp(); }
  template <int K, class Gen>
  __device__ __forceinline__ void seq_sums(int d, Gen gen, double (&result)[K]) const {
    // `terms` holds TWO buffers of K rows ([2*K][33]).  While the 32 dependent adds of block b run (every lane executes
    // them, lanes >= K on row 0 and unused), the terms of block b+1 are generated into the other buffer: the two are
    // independent, so the f64 math of the generator fills the latency slots of the serial chain.  Elements past d are
    // +0.0 terms: acc + 0.0 == acc bit for bit (acc is never -0.0: it starts at +0.0), so every block adds 32 terms and
    // the loop body has no branches.
    double acc = 0.0;
    const int nblk = (d + 31) >> 5;
    const int chain_row = lane < K ? lane : 0;
    auto generate = [&](int blk, int buf) {
      const int i = (blk << 5) + lane;
      double t[K];
#pragma unroll
      for (int k = 0; k < K; k++) t[k] = 0.0;
      if (i < d) gen(i, t);
#pragma unroll
      for (int k = 0; k < K; k++) terms[buf * K + k][lane] = t[k];
    };
    generate(0, 0);
    __syncwarp();
    for (int blk = 0; blk < nblk; blk++) {
      generate(blk + 1, (blk + 1) & 1);  // past the end: all zeros, never read
      const double* row = terms[(blk & 1) * K + chain_row];
#pragma unroll
      for (int m = 0; m < 32; m++) acc += row[m];
      __syncwarp();
    }
#pragma unroll
    for (int k = 0; k < K; k++) result[k] = __shfl_sync(0xffffffffu, acc, k);
  }
  __device__ __forceinline__ void minmax(double& mn, double& mx) const {
    for (int o = 16; o > 0; o >>= 1) {
      mn = bbqn::js_minz(mn, __shfl_xor_sync(0xffffffffu, mn, o));
      mx = bbqn::js_maxz(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
  }
  __device__ __forceinline__ double sum_integers(double v) const {  // integer-valued (or NaN) terms: any order is exact
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
  }
  __device__ __forceinline__ void min2(uint32_t& a, uint32_t& b) const {
    for (int o = 16; o > 0; o >>= 1) {
      a = min(a, __shfl_xor_sync(0xffffffffu, a, o));
      b = min(b, __shfl_xor_sync(0xffffffffu, b, o));
    }
  }
};

template <int K, class Gen>
__device__ __forceinline__ void warp_seq_sums(int d, int lane, double (*terms)[33], Gen gen, double (&result)[K]) {
  WarpTeam{lane, terms}.template seq_sums<K>(d, gen, result);
}

constexpr int OSQC_PRODUCERS = 8;                       // producer warps of the CTA form (warp 0 owns the chains)
constexpr int OSQC_THREADS = (OSQC_PRODUCERS + 1) * 32;
constexpr int OSQC_TERM_ROWS = 2 * OSQC_PRODUCERS * 7;  // two super-block buffers x producers x up to 7 chains
struct CtaTeam {
  int t, warp, lane;
  double (*terms)[33];  // [OSQC_TERM_ROWS][33]
  double* red;          // [2 * (OSQC_PRODUCERS + 1) + 8] cross-warp reductions and chain results
  __device__ __forceinline__ int tid() const { return t; }
  __device__ __forceinline__ int size() const { return OSQC_THREADS; }
  __device__ __forceinline__ void sync() const { __syncthreads(); }
  template <int K, class Gen>
  __device__ __forceinline__ void seq_sums(int d, Gen gen, double (&result)[K]) const {
    // Blocks of 32 components, super-blocks of OSQC_PRODUCERS blocks.  Producer warp w generates block sb * P + (w - 1)
    // of super-block sb + 1 while warp 0 adds the blocks of super-block sb in order: the same sequence of additions as
    // the warp form (and as the reference's loop), zero terms past d included.
    constexpr int P = OSQC_PRODUCERS;
    const int nblk = (d + 31) >> 5;
    const int nsb = (nblk + P - 1) / P;
    auto produce = [&](int sb) {
      const int blk = sb * P + (warp - 1);
      if (blk < nblk) {  // blocks past the end are never read
        const int i = (blk << 5) + lane;
        double tt[K];
#pragma unroll
        for (int k = 0; k < K; k++) tt[k] = 0.0;
        if (i < d) gen(i, tt);
#pragma unroll
        for (int k = 0; k < K; k++) terms[((sb & 1) * P + (warp - 1)) * K + k][lane] = tt[k];
      }
    };
    if (warp > 0) produce(0);
    __syncthreads();
    double acc = 0.0;
    const int chain_row = lane < K ? lane : 0;
    for (int sb = 0; sb < nsb; sb++) {
      if (warp > 0) {
        if (sb + 1 < nsb) produce(sb + 1);
      } else {
        const int nb = min(P, nblk - sb * P);
        for (int b = 0; b < nb; b++) {
          const double* row = terms[((sb & 1) * P + b) * K + chain_row];
#pragma unroll
          for (int m = 0; m < 32; m++) acc += row[m];
        }
      }
      __syncthreads();
    }
    double* res = red + 2 * (P + 1);
    if (warp == 0 && lane < K) res[lane] = acc;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < K; k++) result[k] = res[k];
    __syncthreads();  // (res is rewritten by the next call's last step only, but keep the hazard analysis trivial)
  }
  __device__ __forceinline__ void minmax(double& mn, double& mx) const {
    for (int o = 16; o > 0; o >>= 1) {
      mn = bbqn::js_minz(mn, __shfl_xor_sync(0xffffffffu, mn, o));
      mx = bbqn::js_maxz(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    constexpr int W = OSQC_PRODUCERS + 1;
    if (lane == 0) {
      red[warp] = mn;
      red[W + warp] = mx;
    }
    __syncthreads();
    mn = red[0];
    mx = red[W];
    for (int w = 1; w < W; w++) {  // same order in every thread
      mn = bbqn::js_minz(mn, red[w]);
      mx = bbqn::js_maxz(mx, red[W + w]);
    }
    __syncthreads();
  }
  __device__ __forceinline__ double sum_integers(double v) const {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    constexpr int W = OSQC_PRODUCERS + 1;
    if (lane == 0) red[warp] = v;
    __syncthreads();
    double s = red[0];
    for (int w = 1; w < W; w++) s += red[w];
    __syncthreads();
    return s;
  }
  __device__ __forceinline__ void min2(uint32_t& a, uint32_t& b) const {
    for (int o = 16; o > 0; o >>= 1) {
      a = min(a, __shfl_xor_sync(0xffffffffu, a, o));
      b = min(b, __shfl_xor_sync(0xffffffffu, b, o));
    }
    constexpr int W = OSQC_PRODUCERS + 1;
    uint32_t* r32 = reinterpret_cast<uint32_t*>(red);
    if (lane == 0) {
      r32[warp] = a;
      r32[W + warp] = b;
    }
    __syncthreads();
    for (int w = 0; w < W; w++) {
      a = min(a, r32[w]);
      b = min(b, r32[W + w]);
    }
    __syncthreads();
  }
};

// scalarQuantize of one query by one team (src/optimizedScalarQuantizer.ts:108-227, :280-407); `vec` = the team's
// staging copy of the query in shared memory.
//
// Input screening is fused in (bad != nullptr): the reference validates inside scalarQuantize
// (src/optimizedScalarQuantizer.ts:138-148, after the COSINE normalisation of src/binaryQuantizationFormat.ts:337).
// The team finds the query's first NaN / first Infinity while it stages the vector.  COSINE: a NaN anywhere makes the
// normalised vector all-NaN (reported at position 0); an Infinity makes the norm infinite, so the Infinity components
// become NaN — after ONE normalisation (quantizeQueryVector called directly, :271-299) that NaN sits at the position of
// the first Infinity; on the SEARCH path the query is normalised TWICE (:337, then :279), the second norm is NaN and
// everything is NaN: position 0.  (Observed by executing the reference: tests/golden/from_ts/errors.behaviour.json.)
// Otherwise the first non-finite component is reported as NaN or Infinity.  The lowest offending query wins: bad[0] = min over queries of (query << 34 | status << 32 | position),
// status 1 = NaN, 2 = Infinity (BBQ_ERR_NAN / BBQ_ERR_INF minus 4).  An offending query is ZEROED (staging copy and the
// device buffer it came from) so that the search already enqueued behind this kernel runs on harmless input; the host
// reads bad[0] at its one synchronisation point and reports the error instead of the results.
__device__ __forceinline__ unsigned long long query_verdict(long long q_global, int cosine, int normalize_times,
                                                            uint32_t first_nan, uint32_t first_inf) {
  uint32_t status, pos;
  if (cosine) {
    status = 1u;
    pos = (first_nan != 0xFFFFFFFFu || normalize_times >= 2) ? 0u : first_inf;
  } else if (first_nan < first_inf) {
    status = 1u;
    pos = first_nan;
  } else {
    status = 2u;
    pos = first_inf;
  }
  return ((unsigned long long)q_global << 34) | ((unsigned long long)status << 32) | pos;
}

template <class Team>
__device__ __forceinline__ void osq_query_team(const Team& T, float* __restrict__ src, float* vec, int dim,
                                               const float* __restrict__ centroid, int sim, int bits, double lambda,
                                               int iters, int normalize_times, uint8_t* __restrict__ out, int code_ld,
                                               double* __restrict__ qcorr4, unsigned long long* __restrict__ bad,
                                               long long q_global) {
  uint32_t first_nan = 0xFFFFFFFFu, first_inf = 0xFFFFFFFFu;
  for (int i = T.tid(); i < dim; i += T.size()) {
    const float x = src[i];
    vec[i] = x;
    if (x != x) first_nan = min(first_nan, (uint32_t)i);
    else if (fabsf(x) == INFINITY) first_inf = min(first_inf, (uint32_t)i);
  }
  if (bad != nullptr) {
    T.min2(first_nan, first_inf);
    if (first_nan != 0xFFFFFFFFu || first_inf != 0xFFFFFFFFu) {  // (uniform across the team)
      if (T.tid() == 0) atomicMin(bad, query_verdict(q_global, sim == bbqn::SIM_COSINE ? 1 : 0, normalize_times, first_nan, first_inf));
      for (int i = T.tid(); i < dim; i += T.size()) {
        vec[i] = 0.0f;
        src[i] = 0.0f;
      }
    }
  }
  T.sync();
  // normalizeVector (src/vectorOperations.ts:11-34), twice for COSINE queries (binaryQuantizationFormat.ts:337,279)
  for (int rep = 0; rep < normalize_times; rep++) {
    double r1[1];
    T.template seq_sums<1>(dim, [&](int i, double* t) { t[0] = (double)vec[i] * (double)vec[i]; }, r1);
    const double n = sqrt(r1[0]);
    T.sync();  // (every term has been read)
    for (int i = T.tid(); i < dim; i += T.size()) vec[i] = (n == 0) ? 0.0f : (float)((double)vec[i] / n);
    T.sync();
  }
  auto cen = [&](int i) { return (double)__ldg(centroid + i); };
  auto w_of = [&](int i) { return (double)(float)((double)vec[i] - cen(i)); };
  // statistics: centroidDot, mean, norm (three chains) + exact min/max
  double st[3];
  T.template seq_sums<3>(dim, [&](int i, double* t) {
    const double w = w_of(i);
    t[0] = (sim != bbqn::SIM_EUCLIDEAN) ? (double)vec[i] * cen(i) : 0.0;
    t[1] = w;
    t[2] = w * w;
  }, st);
  double mn = 1.7976931348623157e308, mx = -1.7976931348623157e308;
  for (int i = T.tid(); i < dim; i += T.size()) {
    const double cv = (double)vec[i] - cen(i);
    mn = bbqn::js_minz(mn, cv);
    mx = bbqn::js_maxz(mx, cv);
  }
  T.minmax(mn, mx);
  const double centroidDot = (sim != bbqn::SIM_EUCLIDEAN) ? st[0] : 0.0;
  const double mean = st[1] / (double)dim;
  const double nrm = sqrt(st[2]);
  double r1[1];
  T.template seq_sums<1>(dim, [&](int i, double* t) {
    const double diff = w_of(i) - mean;
    t[0] = diff * diff;
  }, r1);
  const double sd = sqrt(r1[0] / (double)dim);
  const double g = bbqn::mse_grid(bits);
  double a = bbqn::js_clamp(-g * sd + mean, mn, mx);
  double b = bbqn::js_clamp(g * sd + mean, mn, mx);
  const int points = 1 << bits;
  const double pm1 = (double)(points - 1);
  // one pass: loss(ai, bi) [chains 0,1] and the grid sums of (ai, bi) [chains 2..6]
  auto fused_pass = [&](double ai, double bi, double (&res)[7]) {
    const double step = (bi - ai) / pm1;      // computeLoss: step, 1/step
    const double stepInvL = 1.0 / step;
    const double stepInvG = pm1 / (bi - ai);  // optimizeIntervals: (points-1)/(b-a)
    T.template seq_sums<7>(dim, [&](int i, double* t) {
      const double xi = w_of(i);
      const double clamped = bbqn::js_clamp(xi, ai, bi);
      const double kl = bbqn::js_round((clamped - ai) * stepInvL);
      const double xiq = ai + step * kl;
      const double diff = xi - xiq;
      t[0] = xi * diff;
      t[1] = diff * diff;
      const double kg = bbqn::js_round((clamped - ai) * stepInvG);
      const double s = kg / pm1;
      const double oms = 1.0 - s;
      t[2] = oms * oms;
      t[3] = oms * s;
      t[4] = s * s;
      t[5] = xi * oms;
      t[6] = xi * s;
    }, res);
  };
  double ps[7];
  fused_pass(a, b, ps);
  double loss0 = (1.0 - lambda) * ps[0] * ps[0] / nrm + lambda * ps[1];
  const double scale = (1.0 - lambda) / nrm;
  if (bbqn::js_isfinite(scale)) {
    for (int iter = 0; iter < iters; iter++) {  // (every branch below is uniform across the team)
      const double daa = ps[2], dab = ps[3], dbb = ps[4], dax = ps[5], dbx = ps[6];
      const double m0 = scale * dax * dax + lambda * daa;
      const double m1 = scale * dax * dbx + lambda * dab;
      const double m2 = scale * dbx * dbx + lambda * dbb;
      const double det = m0 * m2 - m1 * m1;
      if (fabs(det) < 1e-12) break;
      const double aOpt = (m2 * dax - m1 * dbx) / det;
      const double bOpt = (m0 * dbx - m1 * dax) / det;
      if (fabs(a - aOpt) < 1e-8 && fabs(b - bOpt) < 1e-8) break;
      double pn[7];
      fused_pass(aOpt, bOpt, pn);
      const double loss1 = (1.0 - lambda) * pn[0] * pn[0] / nrm + lambda * pn[1];
      if (loss1 > loss0) break;
      a = aOpt;
      b = bOpt;
      loss0 = loss1;
#pragma unroll
      for (int k = 0; k < 7; k++) ps[k] = pn[k];
    }
  }
  // codes (src/optimizedScalarQuantizer.ts:192-216); the component sum is a sum of integers (or NaN): any order is exact
  const int nSteps = points - 1;
  const double step = nSteps > 0 ? (b - a) / (double)nSteps : 0.0;
  const double stepInv = step > 0 ? 1.0 / step : 0.0;
  const double threshold = (a + b) / 2;
  double qsum = 0.0;
  for (int i = T.tid(); i < code_ld; i += T.size()) {
    uint8_t code = 0;
    if (i < dim) {
      const double clamped = bbqn::js_clamp(w_of(i), a, b);
      if (bits == 1) {
        const int c1 = clamped >= threshold ? 1 : 0;
        code = (uint8_t)c1;
        qsum += (double)c1;
      } else {
        const double assignment = bbqn::js_round((clamped - a) * stepInv);
        const double stored = bbqn::js_min(assignment, (double)nSteps);
        code = (stored != stored) ? (uint8_t)0 : (uint8_t)(((long long)stored) & 0xFF);
        qsum += assignment;
      }
    }
    out[i] = code;
  }
  qsum = T.sum_integers(qsum);
  if (T.tid() == 0) {
    qcorr4[0] = a;
    qcorr4[1] = b;
    qcorr4[2] = (sim == bbqn::SIM_EUCLIDEAN) ? nrm : centroidDot;
    qcorr4[3] = qsum;
  }
}

constexpr int OSQW_WARPS = 4;  // queries per CTA of the warp form

__global__ void __launch_bounds__(OSQW_WARPS * 32) k_osq_query_warp(
    float* __restrict__ queries, int nq, int dim, const float* __restrict__ centroid, int sim, int bits,
    double lambda, int iters, int normalize_times, uint8_t* __restrict__ qcodes, int code_ld,
    double* __restrict__ qcorr, unsigned long long* __restrict__ bad, int q_base) {
  extern __shared__ __align__(16) uint8_t osqw_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = blockIdx.x * OSQW_WARPS + warp;
  const size_t per_warp = (size_t)((dim + 3) & ~3) * sizeof(float) + 14 * 33 * sizeof(double);
  WarpTeam T{lane, reinterpret_cast<double(*)[33]>(osqw_smem + warp * per_warp)};
  float* vec = reinterpret_cast<float*>(osqw_smem + warp * per_warp + 14 * 33 * sizeof(double));
  if (q >= nq) return;  // whole warp
  osq_query_team(T, queries + (int64_t)q * dim, vec, dim, centroid, sim, bits, lambda, iters, normalize_times,
                 qcodes + (int64_t)q * code_ld, code_ld, qcorr + 4 * (int64_t)q, bad, (long long)q_base + q);
}

__global__ void __launch_bounds__(OSQC_THREADS) k_osq_query_cta(
    float* __restrict__ queries, int nq, int dim, const float* __restrict__ centroid, int sim, int bits,
    double lambda, int iters, int normalize_times, uint8_t* __restrict__ qcodes, int code_ld,
    double* __restrict__ qcorr, unsigned long long* __restrict__ bad, int q_base) {
  extern __shared__ __align__(16) uint8_t osqc_smem[];
  // layout: [terms OSQC_TERM_ROWS x 33 f64][red 2*(P+1)+8 f64][vec dim f32]
  double(*terms)[33] = reinterpret_cast<double(*)[33]>(osqc_smem);
  double* red = reinterpret_cast<double*>(osqc_smem) + OSQC_TERM_ROWS * 33;
  float* vec = reinterpret_cast<float*>(red + 2 * (OSQC_PRODUCERS + 1) + 8);
  const int q = blockIdx.x;  // one CTA per query (grid = nq)
  CtaTeam T{(int)threadIdx.x, (int)(threadIdx.x >> 5), (int)(threadIdx.x & 31), terms, red};
  osq_query_team(T, queries + (int64_t)q * dim, vec, dim, centroid, sim, bits, lambda, iters, normalize_times,
                 qcodes + (int64_t)q * code_ld, code_ld, qcorr + 4 * (int64_t)q, bad, (long long)q_base + q);
}

// Threshold from the sample: tau[q] = k-th largest of the maxima of BINS disjoint bins of the sampled scores (bin b
// holds the scores i with i % BINS == b).  The k largest maxima belong to k distinct rows, so tau is a valid lower
// bound of the final k-th best score — and almost as tight as the exact k-th of the sample while k is small against
// BINS (the top few rarely share a bin), at a fraction of the cost of sorting the whole sample.  Requires k <= BINS;
// BINS > TAU_THREADS takes its BINS keys as dynamic shared memory.  tau = -inf when fewer than k bins hold a finite score.
constexpr int TAU_THREADS = 512;     // k <= 512: one bin per thread
constexpr int TAU_BINS_MAX = 16384;  // k > 512: even at k = 4096 the k-th maximum is about the 1.15 k-th score of the sample
template <int BINS>
__global__ void __launch_bounds__(TAU_THREADS) k_tau_from_sample(const float* __restrict__ scores, int64_t ld, uint32_t m,
                                                                  uint32_t k, float* __restrict__ tau) {
  __shared__ uint32_t tau_keys_s[BINS <= TAU_THREADS ? BINS : 1];
  extern __shared__ uint32_t tau_keys_d[];
  uint32_t* const tau_keys = BINS <= TAU_THREADS ? tau_keys_s : tau_keys_d;
  const int q = blockIdx.x, tid = threadIdx.x;
  for (uint32_t b = tid; b < (uint32_t)BINS; b += TAU_THREADS) {
    uint32_t best = 0u;  // ordered-score key; 0 = nothing / NaN
    for (uint32_t i = b; i < m; i += BINS) best = max(best, (uint32_t)(bbqn::topk_key(scores[(int64_t)q * ld + i], 0u) >> 32));
    tau_keys[b] = best;
  }
  for (uint32_t size = 2; size <= (uint32_t)BINS; size <<= 1) {
    for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      for (uint32_t t = tid; t < (uint32_t)BINS / 2; t += TAU_THREADS) {
        const uint32_t i = 2 * t - (t & (stride - 1)), j = i + stride;
        const uint32_t x = tau_keys[i], y = tau_keys[j];
        const bool desc = (i & size) == 0;
        if (desc ? (x < y) : (x > y)) {
          tau_keys[i] = y;
          tau_keys[j] = x;
        }
      }
    }
  }
  __syncthreads();
  if (tid == 0) {
    float t = -INFINITY;
    if (k >= 1 && k <= (uint32_t)BINS && tau_keys[k - 1] != 0u) t = bbqn::topk_key_score((uint64_t)tau_keys[k - 1] << 32);
    tau[q] = t;
  }
}

// Query bit-planes in the index's bit order: plane b, word w holds bit b of codes[32w .. 32w+31],
// dim 8j+t at bit 7-t of byte j (so `plane & row` pairs equal dims).  Layout [nq][nbv][words].
// With an IB-bit index (plane-interleaved rows, see k_osq_index) the row is a 1-bit row of virtual dims and the query
// gets nbv = nb + IB - 1 VIRTUAL planes of weight 2^b': at a position of index plane p, virtual plane b' holds bit
// b' - p of the code, so that  sum_b' 2^b' popc(vplane_b' & row) = sum_d code[d] * x[d]  (x = sum_p 2^p bit_p).
// Also hoists the per-query score terms (src/batchDotProduct.ts:497-502,573-578).
__global__ void k_query_planes(const uint8_t* __restrict__ qcodes, int code_ld, const double* __restrict__ qcorr,
                               int nq, int nb, int ib, int words, uint32_t* __restrict__ planes,
                               bbqn::QueryTerms* __restrict__ qterms) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int nbv = nb + ib - 1;
  const int64_t total = (int64_t)nq * nbv * words;
  if (g < total) {
    const int w = (int)(g % words);
    const int b = (int)((g / words) % nbv);
    const int q = (int)(g / ((int64_t)words * nbv));
    const int chunk = w >> 2, rc = chunk / ib, p = chunk - rc * ib;  // virtual chunk -> (real 128-dim chunk, index plane)
    const int bit = b - p;
    uint32_t word = 0;
    if (bit >= 0 && bit < nb) {
      const uint8_t* cd = qcodes + (int64_t)q * code_ld + 128 * rc + 32 * (w & 3);
#pragma unroll
      for (int j = 0; j < 4; j++)
#pragma unroll
        for (int t = 0; t < 8; t++) word |= (uint32_t)((cd[8 * j + t] >> bit) & 1) << (8 * j + 7 - t);
    }
    planes[g] = word;
  }
  if (g < nq) {
    const double* c = qcorr + 4 * g;
    qterms[g] = bbqn::make_query_terms(c[0], c[1], c[2], c[3], nb, ib);
  }
}

// ------------------------------------------------------------------------------------------------
// K1: the scan.  Replaces createDirectPackedBuffer + computeBatchFourBitDotProductDirectPacked +
// computeBatchFourBitSimilarityScores (+ the 1-bit pair) — src/batchDotProduct.ts:420-436,22-49,478-617,
// src/utils/computeBatchFourBitDotProductDirectPacked.ts:10-53 — and the admission test of the heap
// loop, src/binaryQuantizationFormat.ts:383-400.
//
// One CTA = one tile of 128 index rows x one block of queries.  Rows are staged once into shared
// memory with 128-bit coalesced loads (padded stride: conflict-free LDS.128 per thread-row); query
// bit-planes sit in shared memory and are read as warp broadcasts.  dot = sum_b 2^b popc(plane_b & row)
// is the reference's integer exactly; the epilogue replays the f64 formula and rounds to f32.
// ------------------------------------------------------------------------------------------------
enum { SCAN_DUMP = 0, SCAN_FILTER = 1 };

struct ScanParams {
  const uint8_t* codes;   // [n][row_bytes]
  const double* lower;
  const double* upper;
  const double* addc;
  const uint32_t* compsum;
  int64_t n;
  int row_bytes;          // multiple of 16
  const uint32_t* planes; // [nq][nb][row_bytes/4]
  const bbqn::QueryTerms* qterms;
  int nq;
  int q_block;            // queries per CTA (blockIdx.y)
  double dim;
  double cdp;
  int sim;
  int one_bit_query;      // bbqn::SCORE_REF_MULTIBIT / SCORE_REF_ONEBIT / SCORE_EXT
  double lx_div;          // 2^indexBits - 1: lx = (upper - lower) / lx_div
  int64_t ntiles;         // k_scan_stream (persistent): number of tiles to cover
  uint32_t base;          // global id of row 0
  // tile mapping: CTA x handles tile (tile_first + blockIdx.x * tile_stride)
  int64_t tile_first;
  int64_t tile_stride;
  // SCAN_DUMP: scores[q * dump_ld + blockIdx.x*128 + tid]; optional dots for query 0
  float* dump;
  int64_t dump_ld;
  int32_t* dots;
  // SCAN_FILTER
  const float* tau;       // [nq]
  uint64_t* cand;         // [nq][cap]
  uint32_t* cand_cnt;     // [nq]
  uint32_t cap;
  uint32_t* overflow;
};

template <int NB, int MODE>
__global__ void __launch_bounds__(TILE_ROWS) k_scan(const ScanParams p) {
  extern __shared__ uint4 smem4[];
  const int w4 = p.row_bytes >> 4;   // 16-byte chunks per row
  const int s4 = w4 | 1;             // padded row stride (odd => conflict-free LDS.128)
  uint4* rows_s = smem4;                                   // [128][s4]
  uint4* planes_s = rows_s + TILE_ROWS * s4;               // [q_block][NB][w4]
  bbqn::QueryTerms* qt_s = reinterpret_cast<bbqn::QueryTerms*>(planes_s + (size_t)p.q_block * NB * w4);
  float* tau_s = reinterpret_cast<float*>(qt_s + p.q_block);

  const int tid = threadIdx.x;
  const int64_t tile = p.tile_first + (int64_t)blockIdx.x * p.tile_stride;
  const int64_t row0 = tile * TILE_ROWS;
  const int q0 = blockIdx.y * p.q_block;
  const int nql = min(p.q_block, p.nq - q0);

  // stage the tile's rows (contiguous in HBM): 128-bit coalesced loads
  {
    const uint4* src = reinterpret_cast<const uint4*>(p.codes + row0 * (int64_t)p.row_bytes);
    const int64_t rows_here = min((int64_t)TILE_ROWS, p.n - row0);
    const int total = TILE_ROWS * w4;
    for (int c = tid; c < total; c += TILE_ROWS) {
      const int r = c / w4, j = c - r * w4;
      rows_s[r * s4 + j] = (r < rows_here) ? __ldg(src + c) : make_uint4(0u, 0u, 0u, 0u);
    }
    const uint4* psrc = reinterpret_cast<const uint4*>(p.planes) + (size_t)q0 * NB * w4;
    const int ptotal = nql * NB * w4;
    for (int c = tid; c < ptotal; c += TILE_ROWS) planes_s[c] = __ldg(psrc + c);
    for (int c = tid; c < nql; c += TILE_ROWS) {
      qt_s[c] = p.qterms[q0 + c];
      if (MODE == SCAN_FILTER) tau_s[c] = p.tau[q0 + c];
    }
  }
  const int64_t row = row0 + tid;
  const bool valid = row < p.n;
  double ax = 0, lx = 0, addx = 0, x1 = 0;
  if (valid) {
    ax = p.lower[row];
    lx = (p.upper[row] - ax) / p.lx_div;  // `indexCorrections.upperInterval - ax`, src/batchDotProduct.ts:499,575 (/1 there)
    addx = p.addc[row];
    x1 = (double)p.compsum[row];
  }
  __syncthreads();

  const uint4* myrow = rows_s + tid * s4;
  const uint32_t id = p.base + (uint32_t)row;
  for (int ql = 0; ql < nql; ql++) {
    int acc[NB];
#pragma unroll
    for (int b = 0; b < NB; b++) acc[b] = 0;
    const uint4* pl = planes_s + (size_t)ql * NB * w4;
    for (int j = 0; j < w4; j++) {
      const uint4 x = myrow[j];
#pragma unroll
      for (int b = 0; b < NB; b++) {
        const uint4 q = pl[b * w4 + j];
        acc[b] += __popc(x.x & q.x) + __popc(x.y & q.y) + __popc(x.z & q.z) + __popc(x.w & q.w);
      }
    }
    int dot = 0;
#pragma unroll
    for (int b = 0; b < NB; b++) dot += acc[b] << b;
    const float score = bbqn::score_f32((double)dot, ax, lx, addx, x1, qt_s[ql], p.dim, p.cdp, p.sim,
                                        p.one_bit_query);
    const int q = q0 + ql;
    if (MODE == SCAN_DUMP) {
      if (valid) {
        p.dump[(int64_t)q * p.dump_ld + (int64_t)blockIdx.x * TILE_ROWS + tid] = score;
        if (p.dots != nullptr && q == 0) p.dots[row] = dot;
      }
    } else {
      if (valid && score >= tau_s[ql]) {
        const uint32_t pos = atomicAdd(p.cand_cnt + q, 1u);
        if (pos < p.cap) p.cand[(size_t)q * p.cap + pos] = bbqn::topk_key(score, id);
        else *p.overflow = 1u;
      }
    }
  }
}


// Carry-save form of sum_b 2^b * popc(x & plane_b) over one 16-byte chunk and four query bit-planes: the 16 masks
// are added as bit-vectors (full adder = 2 LOP3) plane by plane, carries moving up one weight, so 6 POPC (weights
// 1..32) replace 16.  The scan is bound by the quarter-rate POPC pipe otherwise.  Same integer.
__device__ __forceinline__ void csa_fa(uint32_t a, uint32_t b, uint32_t c, uint32_t& s, uint32_t& k) {
  asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(s) : "r"(a), "r"(b), "r"(c));
  asm("lop3.b32 %0, %1, %2, %3, 0xE8;" : "=r"(k) : "r"(a), "r"(b), "r"(c));
}
__device__ __forceinline__ int csa_dot4(const uint4 x, const uint4 p0, const uint4 p1, const uint4 p2, const uint4 p3) {
  uint32_t s, t, o1, o2, o4, o8, o16, o32, k1a, k1b, k2a, k2b, k2c, k4a, k4b, k4c, k8a, k8b, k8c;
  csa_fa(x.x & p0.x, x.y & p0.y, x.z & p0.z, s, k1a);
  {  // half adder with the raw fourth mask: sum = s ^ (x & p), carry = s & x & p — one LOP3 each
    asm("lop3.b32 %0, %1, %2, %3, 0x78;" : "=r"(o1) : "r"(s), "r"(x.w), "r"(p0.w));   // a ^ (b & c)
    asm("lop3.b32 %0, %1, %2, %3, 0x80;" : "=r"(k1b) : "r"(s), "r"(x.w), "r"(p0.w));  // a & b & c
  }
  csa_fa(x.x & p1.x, x.y & p1.y, x.z & p1.z, s, k2a);
  csa_fa(x.w & p1.w, k1a, k1b, t, k2b);
  o2 = s ^ t;
  k2c = s & t;
  csa_fa(x.x & p2.x, x.y & p2.y, x.z & p2.z, s, k4a);
  csa_fa(x.w & p2.w, k2a, k2b, t, k4b);
  csa_fa(s, t, k2c, o4, k4c);
  csa_fa(x.x & p3.x, x.y & p3.y, x.z & p3.z, s, k8a);
  csa_fa(x.w & p3.w, k4a, k4b, t, k8b);
  csa_fa(s, t, k4c, o8, k8c);
  csa_fa(k8a, k8b, k8c, o16, o32);
  return __popc(o1) + 2 * __popc(o2) + 4 * __popc(o4) + 8 * __popc(o8) + 16 * __popc(o16) + 32 * __popc(o32);
}

// ------------------------------------------------------------------------------------------------
// K1s: the streaming form of the scan for ONE (or a few) queries — the HBM-bound regime.  No shared memory:
// persistent warps walk 32-row units (4 KB of codes at D=1024); a lane loads 16 bytes of a row per instruction
// (fully coalesced) and the NEXT unit's loads are issued before the current one is reduced, so every warp always
// has a unit in flight.  The query's bit-planes for a lane's fixed 128-dim segment sit in registers, the partial
// dots of the lanes that share a row are combined by a butterfly exchange (power-of-two rows: w4-1 shuffles
// per unit) and the exact f64 epilogue then runs with one row per lane.
// Same integers, same scores, same outputs as k_scan; tiles/dump layout identical.
// ------------------------------------------------------------------------------------------------
template <int NB, int MODE, int W4>
__global__ void __launch_bounds__(TILE_ROWS, 4) k_scan_stream(const ScanParams p) {
  constexpr int w4 = W4;                  // 16-byte chunks per row (compile-time: 1..16)
  constexpr int R = 32 / w4;              // rows per load instruction
  constexpr int iters = (32 + R - 1) / R; // load instructions per 32-row unit
  constexpr bool POW2 = (w4 & (w4 - 1)) == 0;  // then iters == w4 and the butterfly applies
  const int lane = threadIdx.x & 31;
  const int seg = lane % w4, grp = lane / w4;      // this lane's segment of a row / which row of the instruction
  const bool lane_on = lane < R * w4;
  // row (within the unit) whose dot this lane holds after the reduction, hence the row of its epilogue
  const int out_rl = POW2 ? seg * R + grp : lane;
  const int src_lane = (lane % R) * w4;            // !POW2: leader lane of the group that held this lane's row
  const int64_t nunits = p.ntiles * (TILE_ROWS / 32);
  const int64_t ustride = (int64_t)gridDim.x * (TILE_ROWS / 32);
  int64_t u = (int64_t)blockIdx.x * (TILE_ROWS / 32) + (threadIdx.x >> 5);

  auto unit_row0 = [&](int64_t uu) -> int64_t {
    return (p.tile_first + (uu >> 2) * p.tile_stride) * TILE_ROWS + (uu & 3) * 32;
  };
  // query-side constants live in shared memory: inside the unit loop the ONLY global loads are the prefetches, so
  // nothing else waits on the scoreboard they occupy (a predicated-off plane reload there cost 20% of the kernel)
  constexpr int QMAX = 4;
  __shared__ uint4 planes_s[QMAX * NB * w4];
  __shared__ bbqn::QueryTerms qt_s[QMAX];
  __shared__ float tau_s[QMAX];
  for (int i = threadIdx.x; i < p.nq * NB * w4; i += TILE_ROWS) planes_s[i] = __ldg(reinterpret_cast<const uint4*>(p.planes) + i);
  if (threadIdx.x < p.nq) {
    qt_s[threadIdx.x] = p.qterms[threadIdx.x];
    tau_s[threadIdx.x] = MODE == SCAN_FILTER ? p.tau[threadIdx.x] : 0.f;
  }
  __syncthreads();
  if (u >= nunits) return;
  uint4 pl[NB];
#pragma unroll
  for (int b = 0; b < NB; b++) pl[b] = lane_on ? planes_s[b * w4 + seg] : make_uint4(0u, 0u, 0u, 0u);

  uint4 x[iters], xn[iters];
  double lo_n = 0, up_n = 0, add_n = 0;
  uint32_t cs_n = 0;
  auto fetch = [&](int64_t uu) {
    const int64_t r0 = unit_row0(uu);
#pragma unroll
    for (int it = 0; it < iters; it++) {
      xn[it] = make_uint4(0u, 0u, 0u, 0u);
      const int rl = it * R + grp;  // row within the unit
      const int64_t row = r0 + rl;
      if (lane_on && rl < 32 && row < p.n)
        xn[it] = __ldg(reinterpret_cast<const uint4*>(p.codes + row * (int64_t)p.row_bytes) + seg);
    }
    const int64_t er = r0 + out_rl;
    lo_n = up_n = add_n = 0;
    cs_n = 0;
    if (er < p.n) {
      lo_n = __ldg(p.lower + er);
      up_n = __ldg(p.upper + er);
      add_n = __ldg(p.addc + er);
      cs_n = __ldg(p.compsum + er);
    }
  };
  fetch(u);
  for (; u < nunits; u += ustride) {
#pragma unroll
    for (int it = 0; it < iters; it++) x[it] = xn[it];
    const double ax = lo_n, lx = (up_n - lo_n) / p.lx_div, addx = add_n, x1 = (double)cs_n;
    const int64_t my_row = unit_row0(u) + out_rl;
    const bool valid = my_row < p.n;
    if (u + ustride < nunits) fetch(u + ustride);  // next unit in flight while this one is reduced

    const uint32_t id = p.base + (uint32_t)my_row;
    for (int q = 0; q < p.nq; q++) {
      if (p.nq > 1) {
        const uint4* psrc = planes_s + q * NB * w4;
#pragma unroll
        for (int b = 0; b < NB; b++) pl[b] = lane_on ? psrc[b * w4 + seg] : make_uint4(0u, 0u, 0u, 0u);
      }
      int part[iters];
#pragma unroll
      for (int it = 0; it < iters; it++) {
        if (NB == 4) {
          part[it] = csa_dot4(x[it], pl[0], pl[1 % NB], pl[2 % NB], pl[3 % NB]);
        } else {
          int acc = 0;
#pragma unroll
          for (int b = 0; b < NB; b++) {
            const int c = __popc(x[it].x & pl[b].x) + __popc(x[it].y & pl[b].y) + __popc(x[it].z & pl[b].z) +
                          __popc(x[it].w & pl[b].w);
            acc += c << b;
          }
          part[it] = acc;
        }
      }
      int mydot = 0;
      if (POW2) {
        // butterfly: at distance s a lane keeps half of its values (the upper half iff seg & s) and receives the
        // partner's partial sums of the same rows; after log2(w4) steps part[0] is the dot of row seg*R + grp
#pragma unroll
        for (int s = w4 / 2; s > 0; s >>= 1) {
          const bool hi = (seg & s) != 0;
#pragma unroll
          for (int j = 0; j < s; j++) {
            const int a = part[j], b = part[j + s];
            const int send = hi ? a : b, keep = hi ? b : a;
            part[j] = keep + __shfl_xor_sync(0xffffffffu, send, s);
          }
        }
        mydot = part[0];
      } else {
#pragma unroll
        for (int it = 0; it < iters; it++) {
          int v = part[it];
          // sum over the w4 lanes of a row (lanes of a row are contiguous)
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            if (o < w4) {
              const int other = __shfl_down_sync(0xffffffffu, v, o);
              if (seg + o < w4) v += other;
            }
          }
          const int got = __shfl_sync(0xffffffffu, v, src_lane);
          if (lane / R == it) mydot = got;  // row (it*R + lane%R) == lane
        }
      }
      const float score = bbqn::score_f32((double)mydot, ax, lx, addx, x1, qt_s[q], p.dim, p.cdp, p.sim, p.one_bit_query);
      if (MODE == SCAN_DUMP) {
        if (valid) {
          p.dump[(int64_t)q * p.dump_ld + (u >> 2) * TILE_ROWS + (u & 3) * 32 + out_rl] = score;
          if (p.dots != nullptr && q == 0) p.dots[my_row] = mydot;
        }
      } else if (valid && score >= tau_s[q]) {
        const uint32_t pos = atomicAdd(p.cand_cnt + q, 1u);
        if (pos < p.cap) p.cand[(size_t)q * p.cap + pos] = bbqn::topk_key(score, id);
        else *p.overflow = 1u;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// K3: deterministic selection.  One CTA per query sorts up to SELECT_MAX 64-bit keys
// (ordered f32 score << 32 | ~row id) in shared memory (bitonic, descending) and emits the k best —
// the canonical form of the MinHeap loop, src/binaryQuantizationFormat.ts:383-411 / src/minHeap.ts.
// ------------------------------------------------------------------------------------------------
enum { SEL_DENSE = 0, SEL_KEYS = 1, SEL_PAIRS = 2, SEL_KLISTS = 3 };

struct SelectParams {
  int nq;
  uint32_t k;
  // SEL_DENSE: scores[q*ld + i], i < m; id = base + (tile_first + (i/128)*tile_stride)*128 + i%128
  const float* scores;
  int64_t ld;
  uint32_t m;
  int64_t tile_first;
  int64_t tile_stride;
  uint32_t base;
  // SEL_KEYS: keys[q*cap + i], i < min(cnt[q], cap)
  const uint64_t* keys;
  const uint32_t* cnt;
  uint32_t cap;
  // SEL_PAIRS: lists x [nq][k_in] idx/score; idx < 0 = empty slot.  SEL_KLISTS: the same lists as 64-bit keys
  // (`keys` = [lists][nq][k_in], 0 = empty slot) — what the NCCL all-gather of the sharded search delivers
  const int32_t* in_idx;
  const float* in_score;
  uint32_t lists;
  uint32_t k_in;
  // outputs (any may be null)
  uint64_t* out_keys; // [nq][k] the selected keys themselves (0 = empty slot)
  int32_t* out_idx;   // [nq][k]
  float* out_score;   // [nq][k]
};

template <int MODE>
__global__ void __launch_bounds__(SELECT_THREADS) k_select(const SelectParams p, uint32_t m2_max) {
  extern __shared__ uint64_t keys_s[];
  const int q = blockIdx.x;
  const int tid = threadIdx.x;
  uint32_t m;
  if (MODE == SEL_DENSE) m = p.m;
  else if (MODE == SEL_KEYS) m = min(p.cnt[q], p.cap);
  else m = p.lists * p.k_in;  // SEL_PAIRS, SEL_KLISTS
  // sort size: smallest power of two covering the keys and the k outputs (block-uniform)
  uint32_t m2 = 2;
  while (m2 < m || m2 < p.k) m2 <<= 1;
  m2 = min(m2, m2_max);
  for (uint32_t i = tid; i < m2; i += SELECT_THREADS) {
    uint64_t key = 0ull;
    if (i < m) {
      if (MODE == SEL_DENSE) {
        const uint32_t id = p.base + (uint32_t)((p.tile_first + (int64_t)(i / TILE_ROWS) * p.tile_stride) * TILE_ROWS + (i % TILE_ROWS));
        key = bbqn::topk_key(p.scores[(int64_t)q * p.ld + i], id);
      } else if (MODE == SEL_KEYS) {
        key = p.keys[(size_t)q * p.cap + i];
      } else if (MODE == SEL_KLISTS) {
        const uint32_t l = i / p.k_in, j = i - l * p.k_in;
        key = p.keys[((size_t)l * p.nq + q) * p.k_in + j];
      } else {
        const uint32_t l = i / p.k_in, j = i - l * p.k_in;
        const size_t off = ((size_t)l * p.nq + q) * p.k_in + j;
        const int32_t idx = p.in_idx[off];
        key = idx < 0 ? 0ull : bbqn::topk_key(p.in_score[off], (uint32_t)idx);
      }
    }
    keys_s[i] = key;
  }
  for (uint32_t size = 2; size <= m2; size <<= 1) {
    for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      for (uint32_t t = tid; t < (m2 >> 1); t += SELECT_THREADS) {
        const uint32_t i = 2 * t - (t & (stride - 1));
        const uint32_t j = i + stride;
        const uint64_t a = keys_s[i], b = keys_s[j];
        const bool desc = (i & size) == 0;
        if (desc ? (a < b) : (a > b)) {
          keys_s[i] = b;
          keys_s[j] = a;
        }
      }
    }
  }
  __syncthreads();
  if (p.out_keys != nullptr)
    for (uint32_t j = tid; j < p.k; j += SELECT_THREADS) p.out_keys[(size_t)q * p.k + j] = j < m2 ? keys_s[j] : 0ull;
  if (p.out_idx != nullptr) {
    for (uint32_t j = tid; j < p.k; j += SELECT_THREADS) {
      const uint64_t key = j < m2 ? keys_s[j] : 0ull;
      const size_t off = (size_t)q * p.k + j;
      if (key == 0ull) {
        p.out_idx[off] = -1;
        p.out_score[off] = -INFINITY;
      } else {
        p.out_idx[off] = (int32_t)bbqn::topk_key_id(key);
        p.out_score[off] = bbqn::topk_key_score(key);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Oversampled search + exact re-rank ("next" row of the scope table): src/topKSelector.ts:29-114.
// The quantised search returns k*factor candidates per query; each is then scored EXACTLY against the original
// f32 row with computeCosineSimilarity (src/vectorSimilarity.ts:75-102: three interleaved sequential f64 sums),
// and the k best true scores are kept — (trueScore desc, quantised rank asc), i.e. the stable sort of
// getOversampledTopKWithSort.
// kOwnedOnly (a row shard, global candidate ids): only candidates with 0 <= idx - base < rows_n are scored; every other
// slot, empty ones included, gets +0.0, whose bits are 0, so that an integer sum of all shards' outputs delivers each
// owner's f64 bits unchanged.
// ------------------------------------------------------------------------------------------------
constexpr int RERANK_WARPS = 4;
template <bool kOwnedOnly>
__global__ void __launch_bounds__(RERANK_WARPS * 32) k_rerank_scores(const float* __restrict__ rows, int dim,
                                                                    const float* __restrict__ queries, int nq, int m,
                                                                    const int32_t* __restrict__ cand_idx,
                                                                    uint32_t base, uint32_t rows_n,
                                                                    double* __restrict__ true_scores) {
  __shared__ double terms_s[RERANK_WARPS][6][33];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t pair = (int64_t)blockIdx.x * RERANK_WARPS + warp;
  if (pair >= (int64_t)nq * m) return;
  const int q = (int)(pair / m);
  const int32_t idx = cand_idx[pair];
  // base + rows_n < 2^31 (bbq_index_set_base), so an id below base wraps to >= 2^31 and fails the unsigned test too
  const bool skip = idx < 0 || (kOwnedOnly && (uint32_t)idx - base >= rows_n);
  if (skip) {
    if (lane == 0) true_scores[pair] = kOwnedOnly ? 0.0 : -INFINITY;  // empty slot (fewer than k*factor rows) / not ours
    return;
  }
  const float* a = queries + (int64_t)q * dim;
  const float* b = rows + (int64_t)((uint32_t)idx - base) * dim;
  double r[3];
  warp_seq_sums<3>(dim, lane, terms_s[warp], [&](int i, double* t) {
    const double av = (double)a[i], bv = (double)__ldg(b + i);
    t[0] = av * bv;
    t[1] = av * av;
    t[2] = bv * bv;
  }, r);
  if (lane == 0) true_scores[pair] = (r[1] == 0 || r[2] == 0) ? 0.0 : r[0] / (sqrt(r[1]) * sqrt(r[2]));
}

// one CTA per query: rank by (trueScore desc, quantised rank asc); NaN ranks last; O(m^2 / threads), m <= 4096
__global__ void __launch_bounds__(256) k_rerank_select(const double* __restrict__ true_scores, const int32_t* __restrict__ cand_idx,
                                                       const float* __restrict__ cand_score, int m, uint32_t k,
                                                       int32_t* __restrict__ out_idx, float* __restrict__ out_qscore,
                                                       double* __restrict__ out_true) {
  const int q = blockIdx.x;
  const double* t = true_scores + (size_t)q * m;
  const int32_t* ci = cand_idx + (size_t)q * m;
  for (uint32_t j = threadIdx.x; j < k; j += blockDim.x) {
    out_idx[(size_t)q * k + j] = -1;
    out_qscore[(size_t)q * k + j] = -INFINITY;
    out_true[(size_t)q * k + j] = -INFINITY;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < m; i += blockDim.x) {
    if (ci[i] < 0) continue;
    const double ti = t[i];
    const bool nani = ti != ti;
    uint32_t rank = 0;
    for (int j = 0; j < m; j++) {
      if (ci[j] < 0 || j == i) continue;
      const double tj = t[j];
      const bool nanj = tj != tj;
      const bool better = nani ? (!nanj || j < i) : (!nanj && (tj > ti || (tj == ti && j < i)));
      rank += better ? 1u : 0u;
    }
    if (rank < k) {
      out_idx[(size_t)q * k + rank] = ci[i];
      out_qscore[(size_t)q * k + rank] = cand_score[(size_t)q * m + i];
      out_true[(size_t)q * k + rank] = ti;
    }
  }
}

// Input screening as a kernel of its own (one warp per query), for the thread-per-query form of K4 only — the warp and
// CTA forms do it while they stage the query (osq_query_team, where the rules are stated).
__global__ void k_validate_queries(float* __restrict__ queries, int nq, int dim, int cosine, int normalize_times,
                                   unsigned long long* __restrict__ bad, int q_base) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= nq) return;
  float* v = queries + (int64_t)warp * dim;
  uint32_t first_nan = 0xFFFFFFFFu, first_inf = 0xFFFFFFFFu;
  for (int i = lane; i < dim; i += 32) {
    const float x = v[i];
    if (x != x) first_nan = min(first_nan, (uint32_t)i);
    else if (fabsf(x) == INFINITY) first_inf = min(first_inf, (uint32_t)i);
  }
  for (int o = 16; o > 0; o >>= 1) {
    first_nan = min(first_nan, __shfl_xor_sync(0xffffffffu, first_nan, o));
    first_inf = min(first_inf, __shfl_xor_sync(0xffffffffu, first_inf, o));
  }
  if (first_nan == 0xFFFFFFFFu && first_inf == 0xFFFFFFFFu) return;
  if (lane == 0) atomicMin(bad, query_verdict((long long)q_base + warp, cosine, normalize_times, first_nan, first_inf));
  for (int i = lane; i < dim; i += 32) v[i] = 0.0f;
}

// ------------------------------------------------------------------------------------------------
// computeQuantizationAccuracy on the device (SURVEY §8f rank 4): src/binaryQuantizationFormat.ts:420-475 scores every
// query against ONE target row (the reference uses row 0) twice — through the single-vector quantised scorer
// (src/binaryQuantizedScorer.ts:69-98) and exactly (computeOriginalScore :430-448 -> src/vectorSimilarity.ts) — and
// src/binaryQuantizedScorer.ts:524-617 reduces the two score arrays to error statistics.
// k_accuracy_scores: one warp per query; the exact score's sums are sequential f64 (warp_seq_sums keeps the order).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(RERANK_WARPS * 32) k_accuracy_scores(
    const uint8_t* __restrict__ qcodes, int code_ld, const double* __restrict__ qcorr, int nq, int one_bit_query,
    const uint8_t* __restrict__ row_codes, const double* __restrict__ lower, const double* __restrict__ upper,
    const double* __restrict__ addc, const uint32_t* __restrict__ compsum, const float* __restrict__ queries,
    const float* __restrict__ target_row, int dim, int sim, double cdp, double* __restrict__ orig_out,
    double* __restrict__ quant_out) {
  __shared__ double terms_s[RERANK_WARPS][6][33];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = blockIdx.x * RERANK_WARPS + warp;
  if (q >= nq) return;
  // quantised: qcDist = sum_d code[d] * bit_d(row)  (computeInt4BitDotProduct / computeInt1BitDotProduct on the
  // unpacked row, src/bitwiseDotProduct.ts:41-55) — an integer, any order
  const uint8_t* cd = qcodes + (int64_t)q * code_ld;
  int dot = 0;
  for (int i = lane; i < dim; i += 32) dot += (int)cd[i] * (int)((row_codes[i >> 3] >> (7 - (i & 7))) & 1);
  for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
  // exact: computeSimilarity(query, originalVectors[target]) on the ORIGINAL (un-normalised) f32 vectors
  const float* a = queries + (int64_t)q * dim;
  double r[3];
  warp_seq_sums<3>(dim, lane, terms_s[warp], [&](int i, double* t) {
    const double av = (double)a[i], bv = (double)__ldg(target_row + i);
    if (sim == bbqn::SIM_EUCLIDEAN) {
      const double d = av - bv;
      t[0] = d * d;
      t[1] = t[2] = 0.0;
    } else {
      t[0] = av * bv;
      t[1] = av * av;
      t[2] = bv * bv;
    }
  }, r);
  if (lane == 0) {
    const double* c = qcorr + 4 * q;
    quant_out[q] = bbqn::score_single_f64((double)dot, lower[0], upper[0], addc[0], (double)compsum[0], c[0], c[1], c[2],
                                          c[3], (double)dim, cdp, sim, one_bit_query != 0);
    double o;
    if (sim == bbqn::SIM_EUCLIDEAN) o = 1.0 / (1.0 + sqrt(r[0]));                                  // vectorSimilarity.ts:38-67
    else if (sim == bbqn::SIM_COSINE) o = (r[1] == 0 || r[2] == 0) ? 0.0 : r[0] / (sqrt(r[1]) * sqrt(r[2]));  // :75-102
    else o = r[0];                                                                                 // :110-120
    orig_out[q] = o;
  }
}
__global__ void k_accuracy_stats(const double* __restrict__ orig, const double* __restrict__ quant, int64_t n,
                                 double* __restrict__ out5) {
  if (blockIdx.x == 0 && threadIdx.x == 0) bbqn::accuracy_stats(orig, quant, n, out5);
}

// (idx, score) lists -> 64-bit selection keys (idx < 0 = empty slot = key 0): what a shard contributes to the
// NCCL all-gather of the sharded search (SURVEY §8e) — 8 bytes per entry, one collective instead of two.
__global__ void k_pack_keys(const int32_t* __restrict__ idx, const float* __restrict__ score, int64_t count,
                            uint64_t* __restrict__ keys) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) keys[i] = idx[i] < 0 ? 0ull : bbqn::topk_key(score[i], (uint32_t)idx[i]);
}

}  // namespace bbqk
