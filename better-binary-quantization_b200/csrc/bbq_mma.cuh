// bbq_mma.cuh — K2: the batched scan on the 5th-generation tensor cores (tcgen05, sm_100a only).
//
// For a batch of queries the scan is the integer contraction  dot[v][q] = sum_d bit_d(x_v) * q_code[q][d]
// (src/utils/computeBatchFourBitDotProductDirectPacked.ts:10-53, one call per query in the reference).
// Here it is ONE persistent, warp-specialised kernel per query batch (512 threads, one CTA per SM):
//
//   * B operand  = a block of <= 224 accumulator columns (one per query; two for codes wider than 5 bits), resident
//                  in shared memory for a whole pass over the index shard (no-swizzle K-major core-matrix image,
//                  loaded with cp.async.bulk by warp 0);
//   * A operand  = the 1-bit index rows, expanded on the fly by one or two "expansion" groups of 4 warps (one thread
//                  per row, 1 SHF + 8 LOP3 per 32 dims) and written STRAIGHT INTO TENSOR MEMORY with tcgen05.st —
//                  the packed index is the only thing streamed from HBM (128 B/row), the expanded bytes never touch
//                  shared memory;
//   * D          = s32 accumulators in TMEM, double buffered: tcgen05.mma.kind::i8 (M=128, N<=224, K=32) issued by two
//                  or three elected threads on alternate 128-dim chunks; exact integers (<= 15*8*dim, far below 2^31);
//   * epilogue   = 8 (wide batches) or 4 (narrow batches) warps read D with tcgen05.ld (thread = index row, columns =
//                  queries), screen the pairs — COSINE / MIP first with an integer test on the accumulators against a
//                  per-block envelope, then with a 4-FMA fp32 bound against the query's running k-th score — and PARK
//                  the few pairs the screens cannot exclude; a drainer warp replays those with the reference's f64
//                  corrective formula (src/batchDotProduct.ts:554-617) and appends survivors to the candidate lists.
//   Role layouts: MmaLayout<0> "wide" = 8 epilogue warps + 1 expansion group + 2 issuers, MmaLayout<1> "narrow" = 4 + 2
//   + 3 issuers (the B loader's warp takes a third share), picked per launch by the width of the resident block.
//
// A is expanded with weights: K position 32g + 4u + j (u = 4s + b) holds  2^b * bit(4s+b of packed byte j of
// word g)  and B holds  code[dim] * 2^(3-b), so every product is 8 * code * bit and D = 8 * dot exactly;
// this lets one shift serve eight masks.  Requires code * 8 <= 255, i.e. queryBits <= 5.
#pragma once
#include <cuda_runtime.h>
#include <climits>
#include <cstdint>
#include "bbq_kernels.cuh"

namespace bbqk {

// Role layout of the 16 warps of a CTA: warp 0 B loader, 1-2 MMA issuers (2 also allocates TMEM), 3 drainer,
// 4.. expansion groups of 4 warps (one warp per TMEM lane quarter, alternating hand-offs), then the epilogue (one or two
// warps per TMEM lane quarter, alternating accumulator chunks).  Two layouts are compiled into the library:
//   0 "wide batch"  : 8 epilogue warps + 1 expansion group — the per-pair screen is the load;
//   1 "narrow batch": 4 epilogue warps + 2 expansion groups, same 512 threads / 128 registers — with few resident
//                     queries the epilogue has almost nothing to do and the serial operand feed of ONE group is the bound.
// mma_plan picks by the number of accumulator columns (measured crossover, profiles/r02_k2_narrow_layout.txt).
template <int L>
struct MmaLayout {
  static constexpr int EPI_WARPS = L == 0 ? 8 : 4;
  static constexpr int EXP_GROUPS = L == 0 ? 1 : 2;
  static constexpr int EPI_WARP0 = 4 + 4 * EXP_GROUPS;
  static constexpr int THREADS = (EPI_WARP0 + EPI_WARPS) * 32;
};
constexpr int MMA_N_MAX = 224;        // 2 accumulators + >= 2 A stages must fit the 512 TMEM columns
constexpr int MMA_CHUNK_DIMS = 128;   // dims per A stage (32 TMEM columns)

// per-query constants of the fp32 screen (see k_query_screen)
struct __align__(16) QScreen {
  float ly8;    // ly / 8          (D = 8 * dot)
  float aq;     // A_q = ay * dim + ly * y1
  float ay;
  float negl;   // -(L - margin)
  float wadj;   // EUCLIDEAN: upper bound U + margin of (s - addx/2) — the pole 1+e = 0 — INDEPENDENT of tau; +inf otherwise
  float tau;
  float negl0;  // negl at the sampled threshold — what the first-level offset qoff0 and the block envelope were made from
  int qoff0;    // first-level offset at the sampled threshold (k_query_screen); the running one lives in MmaParams::qoff
};

struct IndexBounds {  // maxima over the shard's correctives, for the screen's error margin ...
  float lx, ax, mv, wv;
  // ... and the sums of the per-row screen constants (rv, x1, gv, iv) over the rows that have them, from which the
  // "typical row" rho0 of the first-level screen is taken (any rho0 is valid; a central one is tight)
  double sum[4];
  unsigned long long cnt, pad;
};

// First-level screen, per resident query block (pass): see k_query_screen.
struct __align__(16) QEnv {
  float rho0[4];   // typical row constants (rv, x1, gv, iv)
  float cbar[4];   // centre of the queries' threshold gradients
  float hdev[4];   // max deviation of a query's gradient from cbar, rounded up
  float pad[4];
};

// ---- small PTX wrappers ------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done;
  do {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
  } while (!done);
}
// wait with a suspend-time hint: for producers that run far ahead and should not steal issue slots by polling
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done;
  do {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(done)
        : "r"(addr), "r"(parity), "r"(20000u)
        : "memory");
  } while (!done);
}
__device__ __forceinline__ bool mbar_try(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(done)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return done != 0;
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem desc], kind::i8, cta_group::1
__device__ __forceinline__ void tc_mma_i8_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t"
      "}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(0u)
      : "memory");
}
__device__ __forceinline__ void tc_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_ld16(uint32_t taddr, int (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, "
      "[%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ int tc_ld1(uint32_t taddr) {
  int r;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r) : "r"(taddr) : "memory");
  return r;
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// packed fp32 pairs (Blackwell FFMA2 / FMUL2): two independent IEEE fp32 operations per instruction
__device__ __forceinline__ uint64_t f2_pack(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void f2_unpack(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t f2_sub(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
// max of three (one FMNMX3); a NaN operand is ignored, like fmaxf
__device__ __forceinline__ float f_max3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}
__device__ __forceinline__ uint64_t f2_mul(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}

// no-swizzle K-major shared-memory matrix descriptor (cute::UMMA::SmemDescriptor, version 1):
// core matrix = 8 rows x 16 B contiguous; LBO = byte step between K-adjacent core matrices,
// SBO = byte step between row-adjacent core matrices.
__device__ __forceinline__ uint64_t make_kmajor_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
// cute::UMMA::InstrDescriptor for kind::i8: u8 x u8 -> s32, both operands K-major
__host__ __device__ inline uint32_t make_idesc_i8(int m, int n) {
  return (2u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// ---- operand / constant preparation ------------------------------------------------------------
// B image of pass p: element (n, kpos) at (kpos/16)*(n_tile*16) + (n/8)*128 + (n%8)*16 + kpos%16, where
// kpos = 32g + 4u + j  <->  virtual dim 32g + 8j + 7 - u, weight 2^(3 - u%4)  (see file header).
// Virtual dims: with an IB-bit index the row is plane-interleaved (k_osq_index): 16-byte chunk c of the row is index
// plane p = c % IB of real dims [128 (c / IB), +128), and the B element there is code << p.
// Columns: one per query while (2^queryBits - 1) * 2^(IB-1) * 8 <= 255, otherwise TWO per query (cpq = 2): column 2q
// carries the high nibble of the code, column 2q+1 the low one, and the epilogue recombines 16 * D_hi + D_lo — that is
// how 6..8-bit queries (and the 8b x 2b extension) run on kind::i8.  Columns beyond the batch: 0.
__global__ void k_query_tiles(const uint8_t* __restrict__ qcodes, int code_ld, int nq, int n_tile, int kbytes, int ib,
                              int cpq, uint8_t* __restrict__ images) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // one thread per (pass, n, 16-byte k group)
  const int k16s = kbytes / 16;
  const int ncols = nq * cpq;
  const int passes = (ncols + n_tile - 1) / n_tile;
  if (g >= (int64_t)passes * n_tile * k16s) return;
  const int n = (int)(g % n_tile);
  const int k16 = (int)((g / n_tile) % k16s);
  const int p = (int)(g / ((int64_t)n_tile * k16s));
  const int col = p * n_tile + n;
  uint32_t w[4] = {0u, 0u, 0u, 0u};
  if (col < ncols) {
    const int q = col / cpq, half = col - q * cpq;
    const uint8_t* cd = qcodes + (int64_t)q * code_ld;
#pragma unroll
    for (int i = 0; i < 16; i++) {
      const int kpos = k16 * 16 + i;
      const int grp = kpos >> 5, u = (kpos >> 2) & 7, j = kpos & 3;
      const int chunk = grp >> 2, rc = chunk / ib, plane = chunk - rc * ib;
      uint32_t code = cd[128 * rc + 32 * (grp & 3) + 8 * j + 7 - u];
      if (cpq == 2) code = half == 0 ? (code >> 4) : (code & 15u);
      const uint32_t v = (code << plane) << (3 - (u & 3));
      w[i >> 2] |= (v & 0xFFu) << (8 * (i & 3));
    }
  }
  uint4* dst = reinterpret_cast<uint4*>(images + (size_t)p * n_tile * kbytes + (size_t)k16 * n_tile * 16 +
                                        (size_t)(n >> 3) * 128 + (size_t)(n & 7) * 16);
  *dst = make_uint4(w[0], w[1], w[2], w[3]);
}

// One pass over the shard's correctives: (1) maxima of lx, |ax|, lx*x1, |addx| (finite rows with lx > 0) for the
// screen's error margin; (2) the per-row screen constants {ax/lx, x1, c*addx/lx, 1/lx} as one float4 per row
// (c = -1/2 for EUCLIDEAN, 1 otherwise).  A row whose correctives are degenerate gets 1/lx = 0, which the scan
// reads as "send every pair of this row to the exact replay".
__global__ void k_index_bounds(const double* __restrict__ lower, const double* __restrict__ upper,
                               const double* __restrict__ addc, const uint32_t* __restrict__ compsum, int64_t n,
                               int sim, double lx_div, uint32_t* __restrict__ out4, float4* __restrict__ rscreen) {
  float m0 = 0.f, m1 = 0.f, m2 = 0.f, m3 = 0.f;
  double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
  unsigned long long cnt = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double ax = lower[i], lx = (upper[i] - ax) / lx_div, ad = addc[i];
    float4 rs = make_float4(0.f, 0.f, 0.f, 0.f);
    if (lx > 0 && bbqn::js_isfinite(lx) && bbqn::js_isfinite(ax) && bbqn::js_isfinite(ad)) {
      m0 = fmaxf(m0, __double2float_ru(lx));
      m1 = fmaxf(m1, __double2float_ru(fabs(ax)));
      m2 = fmaxf(m2, __double2float_ru(lx * (double)compsum[i]));
      m3 = fmaxf(m3, __double2float_ru(fabs(ad)));
      const double inv = 1.0 / lx;
      const float rv = (float)(ax * inv), gv = (float)((sim == bbqn::SIM_EUCLIDEAN ? -0.5 * ad : ad) * inv),
                  iv = (float)inv;
      if (bbqn::js_isfinite((double)rv) && bbqn::js_isfinite((double)gv) && bbqn::js_isfinite((double)iv) && iv > 0.f) {
        rs = make_float4(rv, (float)compsum[i], gv, iv);
        s0 += (double)rs.x;
        s1 += (double)rs.y;
        s2 += (double)rs.z;
        s3 += (double)rs.w;
        cnt++;
      }
    }
    rscreen[i] = rs;
  }
  for (int o = 16; o > 0; o >>= 1) {
    m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, o));
    m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, o));
    m2 = fmaxf(m2, __shfl_xor_sync(0xffffffffu, m2, o));
    m3 = fmaxf(m3, __shfl_xor_sync(0xffffffffu, m3, o));
  }
  for (int o = 16; o > 0; o >>= 1) {
    s0 += __shfl_xor_sync(0xffffffffu, s0, o);
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    s3 += __shfl_xor_sync(0xffffffffu, s3, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  if ((threadIdx.x & 31) == 0) {  // non-negative floats order like their bit patterns
    atomicMax(out4 + 0, __float_as_uint(m0));
    atomicMax(out4 + 1, __float_as_uint(m1));
    atomicMax(out4 + 2, __float_as_uint(m2));
    atomicMax(out4 + 3, __float_as_uint(m3));
    IndexBounds* b = reinterpret_cast<IndexBounds*>(out4);  // (the order of these additions only moves rho0: harmless)
    atomicAdd(&b->sum[0], s0);
    atomicAdd(&b->sum[1], s1);
    atomicAdd(&b->sum[2], s2);
    atomicAdd(&b->sum[3], s3);
    atomicAdd(&b->cnt, cnt);
  }
}

// The screen.  With s = ax*A_q + (lx*x1)*ay + lx*ly*dot (the reference's base score, regrouped) every
// similarity's admission test "f32(score) >= tau" is, over the reals, a window on s:
//   EUCLIDEAN  (addq+1-1/tau)/2 <= s - addx/2 <  (addq+1)/2          (pole at 1+e = 0, clamp below it)
//   COSINE     s + addx >= 2 tau - 1 - addq + cdp
//   MIP        s + addx >= g(tau) - addq + cdp,  g = (tau-1)*S for tau >= 1 else (1-1/tau)*S,  S = 1/15 (1 if queryBits==1)
// Dividing by lx > 0:  F0 = ly*dot + (ax/lx)*A_q + x1*ay + (c*addx)/lx;  F0 - L/lx >= 0  [and F0 <= U/lx, U = L + W].
// F is evaluated in fp32; `margin` (in s units) bounds every rounding in that chain and the f32 rounding
// of the score itself, so the screen only ever errs towards admitting a pair to the exact f64 replay.
__device__ __forceinline__ QScreen make_qscreen(const bbqn::QueryTerms& t, float tau, double dim, double cdp, int sim,
                                                int one_bit_query, const IndexBounds& b) {
  QScreen s;
  s.ly8 = s.aq = s.ay = 0.f;
  s.negl = INFINITY;  // admit everything unless a finite lower bound can be derived
  s.wadj = INFINITY;
  s.tau = tau;
  s.negl0 = s.negl;
  s.qoff0 = 0;
  const double tq = (double)tau;
  const double aq = t.ay * dim + t.ly * t.y1;
  double L = 0, W = INFINITY;
  bool ok = tq > 0 && bbqn::js_isfinite(tq) && bbqn::js_isfinite(aq) && bbqn::js_isfinite(t.ay) &&
            bbqn::js_isfinite(t.ly) && bbqn::js_isfinite(t.addq);
  if (ok) {
    if (sim == bbqn::SIM_EUCLIDEAN) {
      L = (t.addq + 1.0 - 1.0 / tq) / 2;
      W = 1.0 / (2 * tq);
    } else if (sim == bbqn::SIM_COSINE) {
      L = 2 * tq - 1.0 - t.addq + cdp;
    } else {
      const double S = one_bit_query ? 1.0 : (1.0 / 15.0);
      L = (tq >= 1 ? (tq - 1.0) * S : (1.0 - 1.0 / tq) * S) - t.addq + cdp;
    }
    const double eps = 1.0 / 16777216.0;  // 2^-24
    const double wv = (sim == bbqn::SIM_EUCLIDEAN) ? 0.5 * b.wv : b.wv;
    const double terms = (double)b.lx * fabs(t.ly) * fabs(t.y1) + (double)b.ax * fabs(aq) + (double)b.mv * fabs(t.ay) + wv;
    const double margin = 32.0 * eps * (terms + fabs(L)) + 16.0 * eps * (fabs(L) + 1.0 + fabs(t.addq) + fabs(cdp));
    // EUCLIDEAN upper bound: s - addx/2 < U = (addq + 1)/2 (= L + W for every tau).  It must NOT move with tau: the
    // fields of a QScreen are re-published one by one while the scan runs, and an upper bound tied to a newer tau
    // combined with a lower offset of an older one would cut off the pairs next to the pole — the best ones.
    const double U = (t.addq + 1.0) / 2;
    const double margin_u = 32.0 * eps * (terms + fabs(U)) + 16.0 * eps * (fabs(U) + 1.0 + fabs(t.addq));
    if (bbqn::js_isfinite(margin) && bbqn::js_isfinite(L) && bbqn::js_isfinite(margin_u)) {
      s.ly8 = (float)(t.ly / 8);
      s.aq = (float)aq;
      s.ay = (float)t.ay;
      s.negl = __double2float_ru(-(L - margin));
      s.wadj = (W == INFINITY) ? INFINITY : __double2float_ru(U + margin_u);
    }
  }
  s.negl0 = s.negl;
  return s;
}

// Per resident query block (= pass; one CTA each): the fp32 screen constants of every query (QScreen, second-level
// screen) and the FIRST-LEVEL screen, an integer test on the accumulators themselves.
//
// In exact arithmetic on the fp32 constants the second-level test  g = negl*iv + ly8*D + rv*aq + x1*ay + gv >= 0
// is  D >= theta_q(rho) = c_q . rho  with the row vector rho = (rv, x1, gv, iv) and the query's gradient
// c_q = -(aq, ay, 1, negl) / ly8.  Around a typical row rho0 (the shard mean):  theta_q(rho) = b_q + c_q . (rho - rho0),
// b_q = c_q . rho0, and for every query of the block  c_q . d >= cbar . d - sum_i hdev_i |d_i|.  So a pair can only
// pass if   D + qoff[q]  >=  S(row) = cbar . d - hdev . |d|   (d = rho - rho0),  qoff[q] = -(floor(b_q) - 1),
// an INTEGER test: the epilogue adds the (warp-uniform) offsets to the 16 accumulators of a chunk, takes the maximum
// and compares it with the row's integer T = floor(S - guard) — 16 IADD + 8 VIMNMX3 + 1 ISETP for 16 pairs.
// (Pre-loading the accumulators with qoff through tcgen05.st instead — so that the tensor core delivers D + qoff —
// was built and measured: correct, but 2.2x slower; tensor-memory stores are the scarce resource while MMAs run.)
// Only chunks that pass go on to the per-pair fp32 screen (about 1-2 % of them: the thresholds here are the SAMPLED
// ones, constant during the scan; the running threshold acts at the second level).
// qoff = +2^30: no usable bound for this query (always second level); -2^30: padding column (never passes).
// COSINE and MAXIMUM_INNER_PRODUCT only: the EUCLIDEAN window is two-sided and too narrow for any block envelope.
constexpr int QOFF_ALWAYS = 1 << 30;
__global__ void __launch_bounds__(256) k_query_screen(const bbqn::QueryTerms* __restrict__ qterms,
                                                      const float* __restrict__ tau, int nq, int n_tile, double dim,
                                                      double cdp, int sim, int one_bit_query,
                                                      const IndexBounds* __restrict__ bounds, QScreen* __restrict__ out,
                                                      uint32_t* __restrict__ tau_bits, int32_t* __restrict__ qoff,
                                                      QEnv* __restrict__ qenv) {
  __shared__ double red_lo[4][8], red_hi[4][8];
  __shared__ float cbar_s[4];
  const int pass = blockIdx.x, t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int q = pass * n_tile + t;
  const bool live = t < n_tile;
  QScreen s;
  s.ly8 = s.aq = s.ay = 0.f;
  s.negl = -INFINITY;  // padding column of the last query block: admits nothing
  s.wadj = INFINITY;
  s.tau = INFINITY;
  s.negl0 = s.negl;
  s.qoff0 = 0;
  if (live) {
    if (q < nq) {
      s = make_qscreen(qterms[q], tau[q], dim, cdp, sim, one_bit_query, *bounds);
      tau_bits[q] = (uint32_t)(bbqn::topk_key(tau[q], 0u) >> 32);
    } else {
      tau_bits[q] = 0xFFFFFFFFu;
    }
  }
  float rho0[4] = {0.f, 0.f, 0.f, 1.f};
  if (bounds->cnt > 0) {
#pragma unroll
    for (int i = 0; i < 4; i++) rho0[i] = (float)(bounds->sum[i] / (double)bounds->cnt);
  }
  const bool has = live && q < nq && s.ly8 > 0.f && bbqn::js_isfinite((double)s.negl) &&
                   bbqn::js_isfinite((double)s.aq) && bbqn::js_isfinite((double)s.ay);
  double c[4] = {0, 0, 0, 0};
  if (has) {
    const double inv = 1.0 / (double)s.ly8;
    c[0] = -(double)s.aq * inv;
    c[1] = -(double)s.ay * inv;
    c[2] = -inv;
    c[3] = -(double)s.negl * inv;
  }
  // block-wide min / max of every gradient component over the queries that have one
#pragma unroll
  for (int i = 0; i < 4; i++) {
    double lo = has ? c[i] : INFINITY, hi = has ? c[i] : -INFINITY;
    for (int o = 16; o > 0; o >>= 1) {
      lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o));
      hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if (lane == 0) {
      red_lo[i][warp] = lo;
      red_hi[i][warp] = hi;
    }
  }
  __syncthreads();
  if (t < 4) {
    double lo = INFINITY, hi = -INFINITY;
    for (int w = 0; w < 8; w++) {
      lo = fmin(lo, red_lo[t][w]);
      hi = fmax(hi, red_hi[t][w]);
    }
    const float cb = (lo <= hi) ? (float)((lo + hi) / 2) : 0.f;
    cbar_s[t] = bbqn::js_isfinite((double)cb) ? cb : 0.f;
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; i++) {
    double dev = has ? fabs(c[i] - (double)cbar_s[i]) : 0.0;
    for (int o = 16; o > 0; o >>= 1) dev = fmax(dev, __shfl_xor_sync(0xffffffffu, dev, o));
    if (lane == 0) red_hi[i][warp] = dev;
  }
  __syncthreads();
  if (t == 0) {
    QEnv e;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      double dev = 0;
      for (int w = 0; w < 8; w++) dev = fmax(dev, red_hi[i][w]);
      e.rho0[i] = rho0[i];
      e.cbar[i] = cbar_s[i];
      e.hdev[i] = __double2float_ru(dev * (1.0 + 1e-6));
      e.pad[i] = 0.f;
    }
    qenv[pass] = e;
  }
  if (live) {
    int off = QOFF_ALWAYS;
    if (q >= nq) {
      off = -QOFF_ALWAYS;
    } else if (has) {
      const double b = c[0] * (double)rho0[0] + c[1] * (double)rho0[1] + c[2] * (double)rho0[2] + c[3] * (double)rho0[3];
      const double fl = floor(b) - 1.0;  // one unit of slack for the f64 rounding of b itself
      if (fabs(fl) < 1.0e9) off = -(int)fl;
    }
    qoff[q] = off;
    s.negl0 = s.negl;
    s.qoff0 = off;
    out[q] = s;
  }
}

// ---- the kernel ----------------------------------------------------------------------------------
struct MmaParams {
  const uint8_t* codes;
  const double* lower;
  const double* upper;
  const double* addc;
  const uint32_t* compsum;
  int64_t n;
  int row_bytes;           // packed bytes per row (multiple of 16)
  int kbytes;              // expanded K bytes per row = row_bytes * 8
  const uint8_t* images;   // [passes][n_tile * kbytes]
  QScreen* qscreen;        // [passes * n_tile]; tightened in place while the scan runs (see mma_retighten)
  uint32_t* tau_bits;      // [passes * n_tile] ordered-key form of tau, atomicMax'ed
  const IndexBounds* bounds;
  uint32_t k;              // top-k size (dynamic tightening needs k <= RETIGHTEN_KMAX)
  const float4* rscreen;   // [n] per-row screen constants (k_index_bounds)
  const int32_t* qoff;     // [passes * n_tile] per-query offsets of the first-level screen (nullptr in SCAN_DUMP)
  const QEnv* qenv;        // [passes] first-level envelope of each resident query block
  const bbqn::QueryTerms* qterms;
  int nq, n_tile, passes, nstage;
  int nissuers;            // MMA issuing threads (2; 3 = the B loader's warp takes a third share: narrow batches are issue-bound)
  double dim, cdp;
  int sim, one_bit_query;  // one_bit_query: bbqn::SCORE_* mode
  double lx_div;           // 2^indexBits - 1
  uint32_t base;
  int64_t tile_first, tile_stride, ntiles;  // tiles handled: tile_first + i*tile_stride, i < ntiles
  // SCAN_DUMP: exact score of every pair -> dump[q*dump_ld + i*128 + row]
  float* dump;
  int64_t dump_ld;
  int32_t* dots;           // optional parity tap: the integer dot (accumulator >> 3) of every pair, same layout as dump
  // SCAN_FILTER
  uint64_t* cand;
  uint32_t* cand_cnt;
  uint32_t cap;
  uint32_t* overflow;
};

// The exact replay of one (row, query) pair the screen could not exclude — deliberately out of line: it runs for
// ~0.1% of the pairs and must not bloat (or serialise) the branch-free screen loop.  `p` points at the kernel's
// __grid_constant__ parameter block; the row's f64 correctives are fetched here, only when needed.
struct RowTerms {  // the row's f64 correctives, loaded once per tile (asynchronously) for the rare exact replays
  double ax, ux, addx;
  uint32_t x1;
};

// everything the (rare, out-of-line) hit path needs, kept in shared memory so that calling it costs no
// per-chunk parameter marshalling in the hot screen loop
struct HitCtx {
  double dim, cdp;
  uint64_t* cand;
  uint32_t* cand_cnt;
  uint32_t* overflow;
  QScreen* qscreen;
  uint32_t* tau_bits;
  const bbqn::QueryTerms* qterms;
  const IndexBounds* bounds;
  const double* lower;
  const double* upper;
  const double* addc;
  const uint32_t* compsum;
  uint32_t cap, k, base;
  int nq, one_bit_query;
  double lx_div;
  int32_t* qoff;   // running first-level offsets (nullptr: no first level)
};

constexpr uint32_t RETIGHTEN_KMAX = 128;   // k up to which the running threshold is tightened inside the scan (k rounds over a 256-key window)
constexpr uint32_t RETIGHTEN_EVERY = 16;   // ... once per this many appended candidates of a query
constexpr uint32_t RETIGHTEN_ZCAP = 4096;  // leading slots of every candidate list that the host zeroes before a scan
constexpr uint32_t HIT_RING = 512;         // CTA-wide ring of parked hits (8 B each)

// ---- hits: parked by the epilogue warps, replayed by a dedicated "drainer" warp -------------------------------
// A lane that replayed its own hit would serialise its whole warp behind a ~100-instruction f64 routine plus two
// dependent global round trips (measured: 1.0 ms of a 2.2 ms scan).  Instead the epilogue lanes only PARK a hit —
// one 64-bit word (row+1 | query | dot) into a CTA-wide shared-memory ring — and warp 3 drains the ring,
// one lane per hit: exact f64 replay, comparison with the query's CURRENT threshold, candidate append, and the
// threshold tightening below.  A ring word is published by a single 64-bit store and consumed in order.
// ring word: row + 1 (31 bits: a shard holds < 2^31 - 16 rows) | query (12 bits) | integer dot (21 bits)
constexpr int HIT_DOT_BITS = 21;
__device__ __forceinline__ uint64_t hit_pack(uint32_t row, uint32_t q, uint32_t dot) {
  return ((uint64_t)(row + 1u) << 33) | ((uint64_t)(q & 0xFFFu) << HIT_DOT_BITS) | (uint64_t)(dot & 0x1FFFFFu);
}

__device__ __noinline__ void mma_park_hits(uint64_t* ring, uint32_t* tail_s, const uint32_t* head_s, uint32_t mask,
                                           uint32_t row, int q0c0, int a0, int a1, int a2, int a3, int a4, int a5, int a6,
                                           int a7, int a8, int a9, int a10, int a11, int a12, int a13, int a14, int a15) {
  const int acc[16] = {a0, a1, a2, a3, a4, a5, a6, a7, a8, a9, a10, a11, a12, a13, a14, a15};
  while (mask) {
    const int j = __ffs(mask) - 1;
    mask &= mask - 1;
    const uint32_t slot = atomicAdd(tail_s, 1u);
    while (slot - *((volatile const uint32_t*)head_s) >= HIT_RING) __nanosleep(100);  // ring full: wait for the drainer
    *((volatile uint64_t*)(ring + (slot % HIT_RING))) = hit_pack(row, (uint32_t)(q0c0 + j), (uint32_t)acc[j] >> 3);
  }
}

// The running threshold.  tau[q] starts as a lower bound of the final k-th best score taken from a sample; while
// the scan runs, whenever a query's candidate count passes a multiple of 16 the drainer warp recomputes the k-th
// best key among (up to 256 of) the candidates appended so far — every one of them is a real row, so that key's
// score is again a valid lower bound — raises tau[q] with an atomicMax and rewrites the query's screen constants
// in global memory; every CTA re-reads them once per tile.  Published values only ever tighten and each 32-bit
// field is a valid bound by itself, so readers need no synchronisation.  Cuts the exact replays ~10x.
template <int SIM>
__device__ void mma_retighten_warp(const HitCtx* cx, int q, int lane) {  // whole warp, convergent
  const uint32_t k = cx->k;
  uint32_t n = 0;
  if (lane == 0) n = min(*((volatile uint32_t*)(cx->cand_cnt + q)), cx->cap);
  n = __shfl_sync(0xffffffffu, n, 0);  // one read, so that every lane takes the same branches below
  // Only the zero-initialised prefix of the list may be read: a slot that has been reserved (count bumped) but not
  // written yet must read as 0 = "absent".  A stale key there (e.g. the same row from the previous search) would be
  // counted twice and push the bound ABOVE the true k-th best.
  if (n < k || n > RETIGHTEN_ZCAP) return;
  const uint32_t first = n > 256u ? n - 256u : 0u;  // any subset gives a valid bound; the latest are the best
  const uint64_t* list = cx->cand + (size_t)q * cx->cap;
  uint64_t mine[8];
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const uint32_t e = first + (uint32_t)(i * 32 + lane);
    mine[i] = e < n ? __ldcg(list + e) : 0ull;  // 0 = slot reserved but not written yet: ranks below everything
  }
  uint64_t bound = ~0ull;
  for (uint32_t t = 0; t < k; t++) {  // k-th largest by k rounds of "largest key below the previous one"
    uint64_t m = 0ull;
#pragma unroll
    for (int i = 0; i < 8; i++)
      if (mine[i] < bound && mine[i] > m) m = mine[i];
    for (int o = 16; o > 0; o >>= 1) {
      const uint64_t other = __shfl_xor_sync(0xffffffffu, m, o);
      m = other > m ? other : m;
    }
    bound = m;
    if (m == 0ull) return;  // fewer than k visible candidates
  }
  const uint32_t bits = (uint32_t)(bound >> 32);
  if (bits == 0u) return;  // NaN-scored k-th: no bound
  if (lane == 0) {
    const uint32_t old = atomicMax(cx->tau_bits + q, bits);
    if (bits > old) {
      const float tnew = bbqn::topk_key_score(bound);
      const QScreen s = make_qscreen(cx->qterms[q], tnew, cx->dim, cx->cdp, SIM, cx->one_bit_query, *cx->bounds);
      QScreen* dst = cx->qscreen + q;
      if (s.ly8 == dst->ly8 && s.aq == dst->aq && s.ay == dst->ay) {  // same query terms: only the bounds move
        dst->negl = fminf(dst->negl, s.negl);
        dst->tau = fmaxf(dst->tau, tnew);
        // The first level follows: theta_q(rho) grows by delta * iv(row), delta = (negl0 - negl) / ly8 >= 0, and
        // iv(row) >= 1 / max lx over the shard — so the integer offset may drop by floor(delta / lx_max), whatever
        // the row (k_query_screen's envelope was built from negl0 and stays as it is).  One 32-bit atomicMin.
        const int q0off = dst->qoff0;
        if (cx->qoff != nullptr && q0off > -QOFF_ALWAYS && q0off < QOFF_ALWAYS && s.ly8 > 0.f && cx->bounds->lx > 0.f) {
          const double delta = ((double)dst->negl0 - (double)s.negl) / (double)s.ly8;
          const double drop = floor(delta / (double)cx->bounds->lx * (1.0 - 1.0e-6));
          if (drop >= 1.0 && drop < 1.0e9) atomicMin(cx->qoff + q, q0off - (int)drop);
        }
      }
    }
  }
}

template <int SIM>
__device__ void mma_drain_ring(const HitCtx* cx, uint64_t* ring, const uint32_t* tail_s, uint32_t* head_s,
                               const uint32_t* done_s, uint32_t epi_warps, int lane) {
  uint32_t head = 0;
  for (;;) {
    const uint64_t e = *((volatile uint64_t*)(ring + ((head + (uint32_t)lane) % HIT_RING)));
    const uint32_t valid = __ballot_sync(0xffffffffu, e != 0ull);
    const uint32_t n = (valid == 0xffffffffu) ? 32u : (uint32_t)(__ffs(~valid) - 1);  // contiguous published prefix
    if (n == 0u) {
      if (*((volatile const uint32_t*)done_s) == epi_warps && head == *((volatile const uint32_t*)tail_s)) break;
      __nanosleep(200);
      continue;
    }
    int tighten_q = -1;
    if ((uint32_t)lane < n) {
      const int64_t row = (int64_t)((uint32_t)(e >> 33) - 1u);
      const int q = (int)((e >> HIT_DOT_BITS) & 0xFFFu);
      const int dot = (int)(e & 0x1FFFFFu);
      float score = 0.f, tau = INFINITY;
      if (q < cx->nq) {  // (a degenerate row parks the padding columns of the last query block too)
        const double ax = __ldg(cx->lower + row), ux = __ldg(cx->upper + row), addx = __ldg(cx->addc + row);
        const double x1 = (double)__ldg(cx->compsum + row);
        const bbqn::QueryTerms qt = cx->qterms[q];
        tau = __ldcg(&cx->qscreen[q].tau);
        score = bbqn::score_f32((double)dot, ax, (ux - ax) / cx->lx_div, addx, x1, qt, cx->dim, cx->cdp, SIM,
                                cx->one_bit_query);
      }
      if (q < cx->nq && score >= tau) {
        const uint32_t pos = atomicAdd(cx->cand_cnt + q, 1u);
        if (pos < cx->cap) {
          cx->cand[(size_t)q * cx->cap + pos] = bbqn::topk_key(score, cx->base + (uint32_t)row);
          if (cx->k <= RETIGHTEN_KMAX && pos + 1 >= 2 * cx->k && (pos + 1) % RETIGHTEN_EVERY == 0) tighten_q = q;
        } else {
          *cx->overflow = 1u;
        }
      }
      *((volatile uint64_t*)(ring + ((head + (uint32_t)lane) % HIT_RING))) = 0ull;  // slot is free again
    }
    __threadfence_block();
    __syncwarp();
    head += n;
    if (lane == 0) *((volatile uint32_t*)head_s) = head;
    // tightening requests of this batch, one query at a time, the whole warp on each
    uint32_t want = __ballot_sync(0xffffffffu, tighten_q >= 0);
    if (want) __threadfence();
    while (want) {
      const int src = __ffs(want) - 1;
      want &= want - 1;
      mma_retighten_warp<SIM>(cx, __shfl_sync(0xffffffffu, tighten_q, src), lane);
    }
  }
}

// ---- the expansion role (warps 4 .. 4 + 4 G): packed 1-bit row -> weighted u8 A operand, straight into TMEM ----------
// The (tile, chunk) sequence of a pass is one flat stream of chunks f = 0 .. total-1, handed over CH at a time (all
// CH tcgen05.st in flight before the single wait::st); hand-off h belongs to group h % G.  Every group prefetches its
// own chunks PF deep across tile boundaries, and group 0 asks L2 for each row four tiles ahead (the 16-byte loads
// themselves come too late to hide an HBM round trip under a busy SM).
template <int G, int CH>
__device__ __forceinline__ void mma_expansion(const MmaParams& p, uint64_t* a_full, uint64_t* a_empty, uint32_t tmem_base,
                                              uint32_t a_col, int nstage, int nchunks, int warp, int lane) {
  const int grp = (warp - 4) >> 2;
  const int r = ((warp - 4) & 3) * 32 + lane;  // row within the tile == TMEM lane
  const uint32_t lane_addr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
  constexpr int PF = 4;
  constexpr int L2_AHEAD = 4;
  static_assert(PF % CH == 0, "the prefetch queue holds whole hand-offs");
  const int64_t my_tiles = (p.ntiles > blockIdx.x) ? (p.ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const int64_t total = my_tiles * nchunks;
  const int64_t hands = (total + CH - 1) / CH;  // hand-offs of the pass
  // cursor of the NEXT chunk of this group to load: tile ordinal + chunk in tile + a row pointer per tile
  int64_t pf_tile = 0;
  int pf_kc = 0;
  int pf_in = 0;                  // position of the cursor inside its hand-off (0 .. CH-1)
  const uint4* pf_ptr = nullptr;  // nullptr: the row lies past the end of the shard (zero chunks)
  auto row_ptr = [&](int64_t t) -> const uint8_t* {
    if (t >= my_tiles) return nullptr;
    const int64_t row = (p.tile_first + (blockIdx.x + t * gridDim.x) * p.tile_stride) * TILE_ROWS + r;
    return row < p.n ? p.codes + row * (int64_t)p.row_bytes : nullptr;
  };
  auto pf_set_tile = [&]() {
    pf_ptr = reinterpret_cast<const uint4*>(row_ptr(pf_tile));
    if (grp == 0) {
      const uint8_t* far = row_ptr(pf_tile + L2_AHEAD);
      if (far != nullptr)
        for (int b = 0; b < p.row_bytes; b += 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(far + b));
    }
  };
  auto pf_advance = [&](int k) {
    pf_kc += k;
    bool moved = false;
    while (pf_kc >= nchunks) {
      pf_kc -= nchunks;
      pf_tile++;
      moved = true;
    }
    if (moved) pf_set_tile();
  };
  auto load_next = [&]() -> uint4 {  // the chunk under the cursor; then on to this group's next chunk
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (pf_ptr != nullptr) v = __ldg(pf_ptr + pf_kc);
    if (++pf_in == CH) {
      pf_in = 0;
      pf_advance((G - 1) * CH + 1);
    } else {
      pf_advance(1);
    }
    return v;
  };
  auto expand = [&](const uint4& x, uint32_t (&e)[32]) {
    const uint32_t ws[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
    for (int g = 0; g < 4; g++) {
      const uint32_t lo = ws[g], hi = ws[g] >> 4;
#pragma unroll
      for (int b = 0; b < 4; b++) {
        e[8 * g + b] = lo & (0x01010101u << b);      // u = b     : bit b   of each packed byte, weight 2^b
        e[8 * g + 4 + b] = hi & (0x01010101u << b);  // u = 4 + b : bit 4+b of each packed byte, weight 2^b
      }
    }
  };
  // (stage, phase) of the first chunk of this group's current hand-off; chunks are numbered through all passes
  uint32_t stage = 0, sphase = 0;
  auto stage_inc = [&](uint32_t& st_, uint32_t& ph_) {
    if (++st_ == (uint32_t)nstage) {
      st_ = 0;
      ph_ ^= 1u;
    }
  };
  for (int k = 0; k < CH * grp; k++) stage_inc(stage, sphase);
  for (int pass = 0; pass < p.passes; pass++) {
    uint4 q[PF];
    pf_tile = 0;
    pf_kc = 0;
    pf_in = 0;
    pf_set_tile();
    pf_advance(CH * grp);
#pragma unroll
    for (int i = 0; i < PF; i++) q[i] = load_next();
    for (int64_t h0 = grp; h0 < hands; h0 += (PF / CH) * G) {
#pragma unroll
      for (int i = 0; i < PF; i += CH) {
        const int64_t h = h0 + (i / CH) * G;  // this group's hand-off
        if (h < hands) {
          uint32_t e[2][32];
          uint32_t sid[CH];
          uint32_t st_ = stage, ph_ = sphase;
          const int nval = (int)min((int64_t)CH, total - CH * h);  // chunks of this hand-off that exist (the stream may end short)
#pragma unroll
          for (int c = 0; c < CH; c++) {
            expand(q[i + c], e[c & 1]);  // (a zero chunk past the end of the stream: loaded, never stored)
            q[i + c] = load_next();
            sid[c] = st_;
            if (c < nval) {
              mbar_wait_relaxed(a_empty + st_, ph_ ^ 1u);
              tc_fence_after();
              tc_st32(lane_addr + a_col + st_ * 32u, e[c & 1]);
            }
            stage_inc(st_, ph_);
          }
          tc_wait_st();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {  // one arrival per expansion warp and stage
#pragma unroll
            for (int c = 0; c < CH; c++)
              if (c < nval) mbar_arrive(a_full + sid[c]);
          }
          for (int k = 0; k < CH * G; k++) stage_inc(stage, sphase);  // on to this group's next hand-off
        }
      }
    }
    // chunk numbers run on through the passes: re-base this group's (stage, phase) for the next pass.  The loop
    // above advanced it in steps of CH * G from CH * grp; the next pass starts at total + CH * grp.
    {
      const int64_t mine = hands > grp ? (hands - grp + G - 1) / G : 0;  // hand-offs this group handled
      const int64_t at = CH * grp + mine * CH * G;                        // where the stepping left off
      const int64_t want = total + CH * grp;                              // first chunk of the next pass
      for (int64_t k = at; k < want; k++) stage_inc(stage, sphase);
      for (int64_t k = want; k < at; k++) {  // (a few positions at most)
        if (stage == 0u) {
          stage = (uint32_t)nstage - 1u;
          sphase ^= 1u;
        } else {
          stage--;
        }
      }
    }
  }
}

// CPQ = accumulator columns per query: 1, or 2 when the query code is split into nibbles (k_query_tiles); then the
// epilogue works on val = 16 * D_hi + D_lo = 8 * dot and every per-query table is indexed by column / 2.
template <int MODE, int SIM, int CPQ, int LAYOUT>
__global__ void __launch_bounds__(MmaLayout<LAYOUT>::THREADS, 1) k_scan_mma(const __grid_constant__ MmaParams p) {
  constexpr int MMA_EPI_WARPS = MmaLayout<LAYOUT>::EPI_WARPS, MMA_EXP_GROUPS = MmaLayout<LAYOUT>::EXP_GROUPS,
                MMA_EPI_WARP0 = MmaLayout<LAYOUT>::EPI_WARP0, MMA_THREADS = MmaLayout<LAYOUT>::THREADS;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // layout: [B image n_tile*kbytes][QScreen n_tile][QueryTerms n_tile][barriers][tmem ptr]
  uint8_t* b_smem = smem_raw;
  // per-pass screen constants, interleaved by query PAIR so that one LDS.128 feeds a packed FFMA2 operand pair:
  //   qpa[j] = (ly8_2j, ly8_2j+1, aq_2j, aq_2j+1)   qpb[j] = (ay_2j, ay_2j+1, negl_2j, negl_2j+1)   qw[j] = wadj pair
  float4* qpa_s = reinterpret_cast<float4*>(b_smem + (size_t)p.n_tile * p.kbytes);
  float4* qpb_s = qpa_s + p.n_tile / 2;
  float2* qw_s = reinterpret_cast<float2*>(qpb_s + p.n_tile / 2);
  bbqn::QueryTerms* qt_s = reinterpret_cast<bbqn::QueryTerms*>(qw_s + p.n_tile / 2);  // DUMP mode only
  int32_t* qoff_s = reinterpret_cast<int32_t*>(qt_s + p.n_tile);   // [n_tile] this pass's first-level offsets (16 B aligned)
  uint64_t* bars = reinterpret_cast<uint64_t*>(qoff_s + p.n_tile + 16);  // (+16: never-passing offsets past the block)
  uint64_t* a_full = bars;            // [8]
  uint64_t* a_empty = bars + 8;       // [8]
  uint64_t* acc_full = bars + 16;     // [2]
  uint64_t* acc_empty = bars + 18;    // [2]
  uint64_t* b_full = bars + 20;
  uint64_t* b_empty = bars + 21;
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(bars + 22);
  uint64_t* tile_go = bars + 24;      // [2] first MMA of a tile has overwritten the accumulator (issuer 0 -> issuer 1)
  HitCtx* hit_s = reinterpret_cast<HitCtx*>(bars + 26);
  uint64_t* ring_s = reinterpret_cast<uint64_t*>(hit_s + 1);            // [HIT_RING] parked hits
  uint32_t* ring_ctl_s = reinterpret_cast<uint32_t*>(ring_s + HIT_RING);  // tail, head, done

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nstage = p.nstage;
  const int nchunks = p.kbytes / MMA_CHUNK_DIMS;  // A stages per tile

  if (threadIdx.x == 0) {
    for (int i = 0; i < 8; i++) {
      mbar_init(a_full + i, 4);
      mbar_init(a_empty + i, 1);
    }
    const uint32_t nissuers = (uint32_t)max(1, min(p.nissuers, min(nchunks, 3)));  // every issuer commits its own MMAs
    for (int i = 0; i < 2; i++) {
      mbar_init(acc_full + i, nissuers);
      mbar_init(acc_empty + i, MMA_EPI_WARPS * 32);
      mbar_init(tile_go + i, 1);
    }
    mbar_init(b_full, 1);
    mbar_init(b_empty, nissuers);
    hit_s->dim = p.dim;
    hit_s->cdp = p.cdp;
    hit_s->cand = p.cand;
    hit_s->cand_cnt = p.cand_cnt;
    hit_s->overflow = p.overflow;
    hit_s->qscreen = p.qscreen;
    hit_s->tau_bits = p.tau_bits;
    hit_s->qterms = p.qterms;
    hit_s->bounds = p.bounds;
    hit_s->lower = p.lower;
    hit_s->upper = p.upper;
    hit_s->addc = p.addc;
    hit_s->compsum = p.compsum;
    hit_s->cap = p.cap;
    hit_s->k = p.k;
    hit_s->base = p.base;
    hit_s->nq = p.nq;
    hit_s->one_bit_query = p.one_bit_query;
    hit_s->lx_div = p.lx_div;
    hit_s->qoff = const_cast<int32_t*>(p.qoff);
    ring_ctl_s[0] = ring_ctl_s[1] = ring_ctl_s[2] = 0u;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (uint32_t i = threadIdx.x; i < HIT_RING; i += MMA_THREADS) ring_s[i] = 0ull;
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_s)),
                 "r"(512u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_s;
  const uint32_t acc_col = 0;                              // accumulators: columns [0, 2*n_tile)
  const uint32_t a_col = 2u * (uint32_t)p.n_tile;          // A stages: 32 columns each

  // ===== MMA issuers =====
  // One thread needs ~99 cycles to issue a tcgen05.mma (tools/probe/mma_issue_probe.cu: independent of N and of
  // TS/SS), so 4 issues + the per-chunk hand-off (barrier wait, fence, commit: ~260 cycles) exceed the ~420
  // cycles the tensor pipe needs for the chunk, and the pipe idles.  NI issuers take the chunks round-robin (warp 1
  // chunks 0, NI, ..; warp 2 chunks 1, NI + 1, ..; with NI = 3 the B loader, idle for the whole of a pass, takes the
  // third share); integer accumulation commutes, and the one ordering that matters — the overwriting first MMA of a
  // tile before anything else — is enforced by a commit-signalled barrier.
  const int NI = max(1, min(p.nissuers, min(nchunks, 3)));
  uint32_t gchunk = 0;  // running chunk count of this CTA: stage = gchunk % nstage, phase = (gchunk / nstage) & 1
  uint32_t tcount_i = 0;
  auto issue_pass = [&](int pass, int me) {  // whole warp; me = 0 issues the tile's first (overwriting) MMA
    const uint32_t idesc = make_idesc_i8(128, p.n_tile);
    const uint32_t lbo = (uint32_t)p.n_tile * 16u;
    const uint32_t b_addr = smem_u32(b_smem);
    mbar_wait(b_full, (uint32_t)(pass & 1));
    for (int64_t i = blockIdx.x; i < p.ntiles; i += gridDim.x) {
      const uint32_t buf = tcount_i & 1u, bphase = (tcount_i >> 1) & 1u;
      if (me == 0) mbar_wait(acc_empty + buf, bphase ^ 1u);  // epilogue has drained this accumulator
      else mbar_wait(tile_go + buf, bphase);                 // ... and issuer 0's overwriting MMA has completed
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc_col + buf * (uint32_t)p.n_tile;
      for (int kc = me; kc < nchunks; kc += NI) {
        const uint32_t g = gchunk + (uint32_t)kc;
        const uint32_t stage = g % (uint32_t)nstage, sphase = (g / (uint32_t)nstage) & 1u;
        mbar_wait(a_full + stage, sphase);
        tc_fence_after();
        if (lane == 0) {
#pragma unroll
          for (int j = 0; j < 4; j++) {
            const uint32_t a_tmem = tmem_base + a_col + stage * 32u + (uint32_t)j * 8u;
            const uint64_t bdesc = make_kmajor_desc(b_addr + (uint32_t)((kc * 4 + j) * 2) * lbo, lbo, 128u);
            tc_mma_i8_ts(d_tmem, a_tmem, bdesc, idesc, (kc | j) != 0 ? 1u : 0u);
            if (kc == 0 && j == 0 && NI > 1) tc_commit(tile_go + buf);
          }
          tc_commit(a_empty + stage);  // frees the A stage once these MMAs have read it
        }
        __syncwarp();
      }
      gchunk += (uint32_t)nchunks;
      if (lane == 0) tc_commit(acc_full + buf);
      __syncwarp();
      tcount_i++;
    }
    if (lane == 0) tc_commit(b_empty);  // this issuer's MMAs of the pass are done -> B may be replaced
    __syncwarp();
  };

  if (warp == 0) {
    // ===== B loader: one resident query block per pass (and, with three issuers, the third share of the MMAs) =====
    const uint32_t bytes = (uint32_t)p.n_tile * (uint32_t)p.kbytes;
    for (int pass = 0; pass < p.passes; pass++) {
      if (lane == 0) {
        // previous pass's MMAs have drained (a whole pass away: poll lazily, do not steal issue slots)
        while (!mbar_try(b_empty, (uint32_t)((pass & 1) ^ 1))) __nanosleep(NI == 3 ? 100 : 1000);
        mbar_expect_tx(b_full, bytes);
        const uint8_t* src = p.images + (size_t)pass * bytes;
        for (uint32_t off = 0; off < bytes; off += 32768u) {
          const uint32_t sz = min(32768u, bytes - off);
          bulk_g2s(b_smem + off, src + off, sz, b_full);
        }
      }
      __syncwarp();
      if (NI == 3) issue_pass(pass, 2);
    }
  } else if (warp == 1 || (warp == 2 && NI > 1)) {
    for (int pass = 0; pass < p.passes; pass++) issue_pass(pass, warp - 1);
  } else if (warp == 3) {
    // ===== drainer: exact replay of the parked hits, candidate append, threshold tightening =====
    if (MODE == SCAN_FILTER) mma_drain_ring<SIM>(hit_s, ring_s, ring_ctl_s + 0, ring_ctl_s + 1, ring_ctl_s + 2, (uint32_t)MMA_EPI_WARPS, lane);
  } else if (warp >= 4 && warp < MMA_EPI_WARP0) {
    // ===== expansion: packed 1-bit row -> weighted u8 A operand, straight into TMEM (mma_expansion above) =====
    // Chunks per hand-off: one group pairs them; with 8 A stages (<= 128 accumulator columns per buffer: small and
    // medium batches, wide rows) it hands over FOUR at a time — the tcgen05.wait::st round trip, not the ALU work,
    // bounds the feed, and four stores in flight amortise it twice as well; two groups alternate pairs of chunks when 8
    // stages exist, single chunks otherwise.
    if (MMA_EXP_GROUPS == 2 && nstage >= 8)
      mma_expansion<2, 2>(p, a_full, a_empty, tmem_base, a_col, nstage, nchunks, warp, lane);
    else if (MMA_EXP_GROUPS == 2)
      mma_expansion<2, 1>(p, a_full, a_empty, tmem_base, a_col, nstage, nchunks, warp, lane);
    else if (nstage >= 8)
      mma_expansion<1, 4>(p, a_full, a_empty, tmem_base, a_col, nstage, nchunks, warp, lane);
    else
      mma_expansion<1, 2>(p, a_full, a_empty, tmem_base, a_col, nstage, nchunks, warp, lane);
  } else if (warp >= MMA_EPI_WARP0) {
    // ===== epilogue: first-level integer screen on the accumulators, second level + parking for what passes =====
    const int ew = warp - MMA_EPI_WARP0;           // 0 .. MMA_EPI_WARPS-1
    const int quarter = ew & 3;                    // TMEM lane quarter this warp may touch (== warp % 4)
    const int sub = ew >> 2;                       // which of the quarter's warps: takes chunks sub, sub+NSUB, ...
    constexpr int NSUB = MMA_EPI_WARPS / 4;
    const int r = quarter * 32 + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(quarter * 32) << 16);
    const int et = threadIdx.x - MMA_EPI_WARP0 * 32;  // 0 .. MMA_EPI_WARPS*32-1 within the epilogue group
    uint32_t tcount = 0;
    for (int pass = 0; pass < p.passes; pass++) {
      // per-pass query constants -> shared memory (epilogue warps only: named barrier 1)
      asm volatile("bar.sync 1, %0;" ::"n"(MMA_EPI_WARPS * 32) : "memory");
      const int q0 = pass * p.n_tile;                     // first accumulator COLUMN of the pass (all passes)
      const int nv = min(p.n_tile, p.nq * CPQ - q0);      // valid columns of this pass
      const int nq_pass = p.n_tile / CPQ;                 // query slots per pass: every per-query table is indexed by slot
      const int q0q = pass * nq_pass, nvq = nv / CPQ;     // first query slot of the pass / valid queries in it
      for (int c = et; c < nq_pass; c += MMA_EPI_WARPS * 32) {
        if (MODE == SCAN_FILTER) {
          const QScreen qs = p.qscreen[q0q + c];
          float* pa = reinterpret_cast<float*>(qpa_s + (c >> 1));
          float* pb = reinterpret_cast<float*>(qpb_s + (c >> 1));
          float* pw = reinterpret_cast<float*>(qw_s + (c >> 1));
          pa[c & 1] = qs.ly8;
          pa[2 + (c & 1)] = qs.aq;
          pb[c & 1] = qs.ay;
          pb[2 + (c & 1)] = qs.negl;
          pw[c & 1] = qs.wadj;
        }
        qoff_s[c] = p.qoff != nullptr ? p.qoff[q0q + c] : 0;
        if (c < 16) qoff_s[nq_pass + c] = -QOFF_ALWAYS;  // slots past the block: never pass
        if (MODE == SCAN_DUMP && c < nvq) qt_s[c] = p.qterms[q0q + c];
      }
      // first-level envelope of this query block (registers; warp-uniform)
      float e_r0 = 0.f, e_r1 = 0.f, e_r2 = 0.f, e_r3 = 1.f, e_c0 = 0.f, e_c1 = 0.f, e_c2 = 0.f, e_c3 = 0.f, e_h0 = 0.f,
            e_h1 = 0.f, e_h2 = 0.f, e_h3 = 0.f;
      if (MODE == SCAN_FILTER && p.qenv != nullptr) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(p.qenv + pass));
        const float4 b = __ldg(reinterpret_cast<const float4*>(p.qenv + pass) + 1);
        const float4 h = __ldg(reinterpret_cast<const float4*>(p.qenv + pass) + 2);
        e_r0 = a.x; e_r1 = a.y; e_r2 = a.z; e_r3 = a.w;
        e_c0 = b.x; e_c1 = b.y; e_c2 = b.z; e_c3 = b.w;
        e_h0 = h.x; e_h1 = h.y; e_h2 = h.z; e_h3 = h.w;
      }
      asm volatile("bar.sync 1, %0;" ::"n"(MMA_EPI_WARPS * 32) : "memory");
      auto row_of = [&](int64_t ti) { return (p.tile_first + ti * p.tile_stride) * TILE_ROWS + r; };
      // per-row screen constants: prefetched one tile ahead (placeholders for rows past the end of the shard).
      const float4 rs_none = make_float4(0.f, 0.f, -INFINITY, 1.f);
      auto load_rs = [&](int64_t ti) -> float4 {
        if (MODE != SCAN_FILTER || ti >= p.ntiles) return rs_none;
        const int64_t rw = row_of(ti);
        return rw < p.n ? __ldg(p.rscreen + rw) : rs_none;
      };
      float4 rs_next = load_rs(blockIdx.x);
      for (int64_t i = blockIdx.x; i < p.ntiles; i += gridDim.x) {
        const int64_t row = row_of(i);
        const bool valid = row < p.n;
        const float4 rs = rs_next;
        rs_next = load_rs(i + gridDim.x);
        const float rv = rs.x, x1f = rs.y, gv = rs.z, iv = rs.w;
        const bool always = valid && !(iv > 0.f);  // degenerate correctives: every pair goes to the exact replay
        // first level: T = floor(cbar . d - hdev . |d| - guard), d = rho(row) - rho0; a pair can only pass the second
        // level if its pre-loaded accumulator reaches T (see k_query_screen).  The guard covers the fp32 rounding of
        // this very expression (a few ulp of each product; 2^-19 of their absolute sum is ample) plus one unit.
        int T;
        {
          const float d0 = rv - e_r0, d1 = x1f - e_r1, d2 = gv - e_r2, d3 = iv - e_r3;
          const float a0 = fabsf(d0), a1 = fabsf(d1), a2 = fabsf(d2), a3 = fabsf(d3);
          const float S = fmaf(e_c0, d0, fmaf(e_c1, d1, fmaf(e_c2, d2, e_c3 * d3)));
          const float H = fmaf(e_h0, a0, fmaf(e_h1, a1, fmaf(e_h2, a2, e_h3 * a3)));
          const float A = fmaf(fabsf(e_c0), a0, fmaf(fabsf(e_c1), a1, fmaf(fabsf(e_c2), a2, fabsf(e_c3) * a3))) + H;
          const float Sl = S - H - fmaf(A, 1.9073486328125e-06f, 1.0f);
          T = (Sl > -1.0e9f && Sl < 1.0e9f) ? (int)floorf(Sl) : INT_MIN;  // NaN / out of range: everything passes on
          if (!valid) T = INT_MAX;
          if (always || MODE != SCAN_FILTER || p.qenv == nullptr) T = INT_MIN;
        }
        const uint64_t rv2 = f2_pack(rv, rv), x1f2 = f2_pack(x1f, x1f), gv2 = f2_pack(gv, gv), iv2 = f2_pack(iv, iv);
        // f64 correctives: issued now, consumed only by the dump
        RowTerms rt{0.0, 0.0, 0.0, 0u};
        if (MODE == SCAN_DUMP && valid) {
          rt.ax = __ldg(p.lower + row);
          rt.ux = __ldg(p.upper + row);
          rt.addx = __ldg(p.addc + row);
          rt.x1 = __ldg(p.compsum + row);
        }
        const uint32_t buf = tcount & 1u, bphase = (tcount >> 1) & 1u;
        mbar_wait(acc_full + buf, bphase);
        tc_fence_after();
        const uint32_t d_addr = lane_addr + buf * (uint32_t)p.n_tile;
        // this tile's refresh of the (possibly tightened) second-level constants: loads issued now, stored after the tile
        constexpr int ET = MMA_EPI_WARPS * 32;  // 128 or 256 threads refresh up to 224 queries: one or two each
        const bool refresh = MODE == SCAN_FILTER && p.k <= RETIGHTEN_KMAX && et < nvq;
        const bool refresh2 = MODE == SCAN_FILTER && p.k <= RETIGHTEN_KMAX && ET < MMA_N_MAX && et + ET < nvq;
        float4 fr0 = make_float4(0.f, 0.f, 0.f, 0.f), fr1 = fr0;
        int fo0 = 0, fo1 = 0;
        if (refresh) fr0 = __ldcg(reinterpret_cast<const float4*>(p.qscreen + q0q + et));
        if (refresh2) fr1 = __ldcg(reinterpret_cast<const float4*>(p.qscreen + q0q + et + ET));
        if (refresh && p.qoff != nullptr) fo0 = __ldcg(p.qoff + q0q + et);
        if (refresh2 && p.qoff != nullptr) fo1 = __ldcg(p.qoff + q0q + et + ET);
        // software pipeline over this warp's 16-column chunks: the next chunk's TMEM load is in flight while the
        // current one is reduced; the chunk just read is re-armed for the tile two positions ahead
        constexpr int W = 16;  // accumulator columns per TMEM load (tcgen05.ld .x16)
        int acc[W], nxt[W];
        int c0 = sub * W;
        if (c0 < nv) {
          tc_ld16(d_addr + (uint32_t)c0, acc);
          tc_wait_ld();
        }
        auto chunk = [&](int (&cur)[W], int (&nx)[W], int cc) -> bool {
          const int c1 = cc + NSUB * W;
          if (c1 < nv) tc_ld16(d_addr + (uint32_t)c1, nx);
          // per QUERY from here on: val = 8 * dot (split codes: 16 * D_hi + D_lo), qc = the chunk's first query slot
          constexpr int NVC = W / CPQ;
          int val[NVC];
#pragma unroll
          for (int j = 0; j < NVC; j++) val[j] = CPQ == 1 ? cur[j] : cur[2 * j] * 16 + cur[2 * j + 1];
          const int qc = cc / CPQ;
          if (MODE == SCAN_DUMP) {
            if (valid) {
#pragma unroll
              for (int j = 0; j < NVC; j++) {
                const int c = qc + j;
                if (c < nvq) {
                  const int64_t off = (int64_t)(q0q + c) * p.dump_ld + i * TILE_ROWS + r;
                  if (p.dump != nullptr)
                    p.dump[off] = bbqn::score_f32((double)(val[j] >> 3), rt.ax, (rt.ux - rt.ax) / p.lx_div, rt.addx, (double)rt.x1,
                                                  qt_s[c], p.dim, p.cdp, SIM, p.one_bit_query);
                  if (p.dots != nullptr) p.dots[off] = val[j] >> 3;  // D = 8 * dot exactly (file header)
                }
              }
            }
          } else {
            // Second level (EUCLIDEAN: the only level): the packed fp32 screen of every pair of the chunk against the
            // query's CURRENT threshold — 4 FFMA2 (+ 1 FMUL2 + 1 FADD2 for the EUCLIDEAN window) per two pairs.
            // EUCLIDEAN has no first level: its admission window is TWO-sided (the pole 1 + e = 0) and, on the corpora
            // this path meets, only a few accumulator units wide in the dense part of the distribution — no envelope
            // over a block of queries is that sharp (measured: a one-sided first level passes 88 % of the chunks).
            bool go = true;
            if (SIM != bbqn::SIM_EUCLIDEAN) {
              // first level: max_j (8*dot_j + qoff_j) against the row's T; the 16 offsets are warp-uniform (4 broadcast
              // LDS.128).  A warp goes on if ANY of its 32 rows passes, so the per-row rate has to be well below 1/32:
              // the offsets follow the running threshold (mma_retighten_warp), not just the sampled one.
              const int4* o4 = reinterpret_cast<const int4*>(qoff_s + qc);
              int mm[4] = {INT_MIN, INT_MIN, INT_MIN, INT_MIN};  // four independent VIMNMX3 chains
#pragma unroll
              for (int g = 0; g < NVC / 4; g++) {
                const int4 o = o4[g];
                mm[g & 3] = max(max(mm[g & 3], val[4 * g] + o.x), val[4 * g + 1] + o.y);
                mm[(g + 2) & 3] = max(max(mm[(g + 2) & 3], val[4 * g + 2] + o.z), val[4 * g + 3] + o.w);
              }
              const int m = max(max(mm[0], mm[1]), max(mm[2], mm[3]));
              go = m >= T;
            }
            uint32_t mask = 0u;
            if (go) {
#pragma unroll
              for (int j = 0; j < NVC / 2; j++) {  // two queries per step
                const int pj = (qc >> 1) + j;
                const float4 qa = qpa_s[pj], qb = qpb_s[pj];
                // f0 = (s + c*addx) / lx for the two queries; lower test: f0 + negl/lx >= 0; upper: f0 <= wadj/lx
                uint64_t t = f2_fma(x1f2, f2_pack(qb.x, qb.y), gv2);
                t = f2_fma(rv2, f2_pack(qa.z, qa.w), t);
                const uint64_t f0 = f2_fma(f2_pack(qa.x, qa.y), f2_pack((float)val[2 * j], (float)val[2 * j + 1]), t);
                float g0, g1;
                f2_unpack(f2_fma(f2_pack(qb.z, qb.w), iv2, f0), g0, g1);
                if (SIM == bbqn::SIM_EUCLIDEAN) {
                  float d0, d1;
                  const float2 w = qw_s[pj];
                  f2_unpack(f2_sub(f2_mul(f2_pack(w.x, w.y), iv2), f0), d0, d1);  // wadj * iv - f0
                  g0 = fminf(g0, d0);
                  g1 = fminf(g1, d1);
                }
                if (g0 >= 0.f) mask |= (1u << (2 * j));
                if (g1 >= 0.f) mask |= (1u << (2 * j + 1));
              }
            }
            const uint32_t vmask = (nvq - qc >= 32) ? 0xFFFFFFFFu : ((1u << (nvq - qc)) - 1u);  // never a padding slot: its query id would alias
            if (always) mask = 0xFFFFFFFFu;
            // a row past the end of the shard never parks: with tau = -inf its placeholder constants make the EUCLIDEAN
            // lower test NaN, and fminf returns the (+inf) window test instead
            if (!valid) mask = 0u;
            mask &= vmask;
            auto v_at = [&](int j) { return j < NVC ? val[j < NVC ? j : 0] : 0; };
            if ((mask & 0xFFFFu) != 0u)  // park the hits for the drainer warp
              mma_park_hits(ring_s, ring_ctl_s + 0, ring_ctl_s + 1, mask & 0xFFFFu, (uint32_t)row, q0q + qc, v_at(0), v_at(1),
                            v_at(2), v_at(3), v_at(4), v_at(5), v_at(6), v_at(7), v_at(8), v_at(9), v_at(10), v_at(11),
                            v_at(12), v_at(13), v_at(14), v_at(15));
          }
          if (c1 >= nv) return false;
          tc_wait_ld();
          return true;
        };
        while (c0 < nv) {  // ping-pong between the two register sets (no copies)
          if (!chunk(acc, nxt, c0)) break;
          c0 += NSUB * W;
          if (!chunk(nxt, acc, c0)) break;
          c0 += NSUB * W;
        }
        if (refresh) {  // fr0 = (ly8, aq, ay, negl) of query et: only the lower offset moves with the threshold
          float* pb = reinterpret_cast<float*>(qpb_s + (et >> 1));
          pb[2 + (et & 1)] = fr0.w;
          if (p.qoff != nullptr) qoff_s[et] = fo0;
        }
        if (refresh2) {
          float* pb = reinterpret_cast<float*>(qpb_s + ((et + ET) >> 1));
          pb[2 + ((et + ET) & 1)] = fr1.w;
          if (p.qoff != nullptr) qoff_s[et + ET] = fo1;
        }
        tc_fence_before();
        mbar_arrive(acc_empty + buf);
        tcount++;
      }
    }
    __syncwarp();
    if (lane == 0) atomicAdd(ring_ctl_s + 2, 1u);  // this epilogue warp will park nothing more
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

}  // namespace bbqk
