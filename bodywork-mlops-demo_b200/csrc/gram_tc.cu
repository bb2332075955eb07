// gram_tc.cu -- the hot kernel: row-block streaming Gram accumulator on tcgen05 (sm_100a).
//
// Replaces the pass over the training rows inside LinearRegression.fit
// (stage_1_train_model.py:105-106 -> sklearn/linear_model/_base.py: centre + LAPACK gelsd).
//
// Data flow per CTA (persistent, one CTA per SM, contiguous range of 64-row tiles):
//
//   HBM --TMA (cp.async.bulk.tensor, evict-first)--> smem raw tile [64 rows][D] (+ y, + row mask)
//     --16 transform warps: v = x - c (per-column shift), bf16 split v = hi + lo
//     -- 1 "E" warp: extra columns E = [1, y'_hi, y'_lo] (y' = y - c_y), CUDA-core sums of y', y'^2, rows
//     --> operands, K-major canonical layout (8 x 16 B core matrices, no swizzle; one 16-byte chunk =
//         8 consecutive rows of X for one feature):
//            smem  rows j = 0..127 hi | 128..143 E                      (B = [hi | E], and A = hi)
//            D = 128:  A = lo goes to TENSOR MEMORY (tcgen05.st, lane = feature, 4 packed columns per 8 rows);
//            D < 128:  lo is a third smem block (rows 144..271), A = lo read through a descriptor
//     --tcgen05.mma.cta_group::1.kind::f16 (bf16 x bf16 -> fp32 in TMEM), M=128, N=144, K=16, two per K-step:
//            D1[i][j] += sum_r hi[r][i] * [hi | E][r][j]      TMEM columns 0..143 / 144..287 (double buffered)
//            D2[i][j] += sum_r lo[r][i] * [hi | E][r][j]      TMEM columns 288..431 (never drained mid-kernel)
//        so D1[:, :128] = hi^T hi, D2[:, :128] = lo^T hi, column 128 = sum v, columns 129/130 = sum v*y'.
//        (TMEM columns 432..495: the two stages of the A = lo operand.)
//     --every `drain_rows` rows: epilogue warps tcgen05.ld the D1 buffer just finished and fold it into this
//        CTA's fp64 partial in global memory while the MMAs continue into the other D1 buffer; D2 holds
//        only the small zero-mean lo terms, so its fp32 sums are drained once at the end.
//
// Why the shift and the split: the tensor core accumulates fp32 with truncation, so raw (uncentred)
// second moments cannot reach the 1e-4 coefficient tolerance; after the shift the Gram is ~diagonal and
// the centring in the solve subtracts almost nothing.  hi+lo carries 16 mantissa bits, i.e. products are
// accurate to ~2^-17 relative (lo*lo is dropped).
//
// tc_reduce_kernel sums the per-CTA partials in a fixed order (deterministic); tc_fold_kernel undoes the shift
// in fp64 and adds the result to the context's raw statistic S = [X 1 y]^T [X 1 y].
#include <cuda_bf16.h>
#include <stdlib.h>

#include "b2_internal.cuh"
#include "b2_ptx.cuh"
#include "b2_xchg.cuh"

namespace b2 {
namespace {

// ------------------------------------------------------------------------------------------
// geometry
// ------------------------------------------------------------------------------------------
constexpr int kRawStages = 4;
constexpr int kOpStages = 2;
constexpr int kXformWarps = 16;
constexpr int kThreads = 32 * (8 + kXformWarps);  // warps: 0 TMA, 1 MMA(+TMEM alloc), 2-3 E, 4-7 epilogue, 8.. transform
constexpr int kProducers = kXformWarps + 2;        // warps that fill an operand stage (transform + 2 E warps)
constexpr int kKGroups = kTcRows / 8;              // 8-row K groups per stage
constexpr uint32_t kRawStageBytes = kTcRows * kMaxD * 4;      // 32768 (fp32, D = 128)
constexpr uint32_t kOpSBO = 128;                              // bytes between 8-row j groups (core matrices along M/N)
constexpr uint32_t kOpLBO_SS = (16 + 2 + 16) * kOpSBO;        // 4352: hi | E | lo groups per K group (operands all in smem)
constexpr uint32_t kOpLBO_TS = (16 + 2) * kOpSBO;             // 2304: hi | E only; A = lo is staged in TMEM (D = 128 path)
constexpr uint32_t kOpEOff = 16 * kOpSBO;                     // E block inside a K group
constexpr uint32_t kOpLoOff = 18 * kOpSBO;                    // lo block inside a K group (SS layout only)
constexpr uint32_t kOpStageBytes = kKGroups * kOpLBO_SS;      // 34816 (sized for the SS layout)
constexpr uint32_t kTmemALoCol = 432;                         // TS: A = lo operand, 2 stages x 32 columns (432..495)
constexpr uint32_t kOffRaw = 0;
constexpr uint32_t kOffOp = kOffRaw + kRawStages * kRawStageBytes;     // 131072
constexpr uint32_t kOffY = kOffOp + kOpStages * kOpStageBytes;         // 200704
constexpr int kMaxPack = 5;                                             // original rows per 128-wide super-row (3 E columns each)
constexpr uint32_t kYStageBytes = kTcRows * kMaxPack * 4;               // 1280
constexpr uint32_t kMStageBytes = 384;                                  // 64 * kMaxPack = 320 mask bytes, padded: TMA
                                                                        // destinations are 128-byte aligned
static_assert(kMStageBytes >= kTcRows * kMaxPack && kMStageBytes % 128 == 0 && kYStageBytes % 128 == 0, "stage alignment");
constexpr uint32_t kOffMask = kOffY + kRawStages * kYStageBytes;
constexpr uint32_t kOffBar = kOffMask + kRawStages * kMStageBytes;
constexpr int kNumBars = 2 * kRawStages + 2 * kOpStages + 4;
constexpr uint32_t kOffTmemPtr = kOffBar + kNumBars * 8;
constexpr uint32_t kOffShift = kOffTmemPtr + 16;
constexpr uint32_t kSmemBytes = kOffShift + (kMaxD + 4) * 4 + 1024;    // + alignment slack (~204 KB)
static_assert(kSmemBytes <= 227 * 1024, "shared memory budget");
constexpr uint32_t kTmemD1Stride = 144;   // D1 (A = hi) is double buffered: columns 0..143 and 144..287
constexpr uint32_t kTmemD2Col = 288;      // D2 (A = lo): columns 288..431, accumulates for the whole kernel

// instruction descriptor: D=f32, A=B=bf16, both K-major, N=144, M=128 (cute::UMMA::InstrDescriptor layout)
constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kTcN >> 3) << 17) |
                            ((uint32_t)(kTcM >> 4) << 24);

// ------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

constexpr uint64_t kEvictFirst = 0x12F0000000000000ull;  // L2 cache hint: streaming data, read once

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "l"(kEvictFirst)
      : "memory");
}
__device__ __forceinline__ void tma_load_1d(uint32_t dst, const CUtensorMap* tm, int c0, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.1d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3}], [%2], %4;" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "l"(kEvictFirst)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}

// K-major, no-swizzle shared-memory matrix descriptor (cute::UMMA::SmemDescriptor, version 1)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t addr, uint32_t lbo) {
  return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) |
         ((uint64_t)(kOpSBO >> 4) << 32) | (1ull << 46);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(kIdesc), "r"(accumulate)
      : "memory");
}
// A operand from tensor memory (128 lanes x 8 columns of packed bf16 pairs per K = 16)
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(kIdesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t (&v)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(v[0]), "r"(v[1]),
               "r"(v[2]), "r"(v[3])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void st_shared_v4(uint32_t addr, const uint32_t (&v)[4]) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3])
               : "memory");
}
__device__ __forceinline__ void st_shared_u16(uint32_t addr, uint32_t v) {
  asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"((unsigned short)v) : "memory");
}
// bf16 split of two fp32 values: hi = rn(v), lo = rn(v - hi), packed (element 0 in the low half)
__device__ __forceinline__ void split2(float v0, float v1, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(v0, v1);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  const float h0 = __uint_as_float(hi << 16), h1 = __uint_as_float(hi & 0xffff0000u);
  const __nv_bfloat162 l = __floats2bfloat162_rn(v0 - h0, v1 - h1);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

// ------------------------------------------------------------------------------------------
// per-column shift c: mean of a strided sample of the rows the statistic keeps (any value near the column mean will
// do; the algebra in tc_fold_kernel is exact for every c)
// ------------------------------------------------------------------------------------------
constexpr int kShiftBlocks = 64;                 // partial sums of the row sample, one per block
constexpr int kShiftStride = kMaxD + 2;          // floats per partial: features, y (slot kMaxD), rows sampled (kMaxD + 1)
static_assert(kShiftBlocks * kShiftStride <= kShiftFloats, "b2_ctx::shift holds the partials");

__host__ __device__ __forceinline__ int64_t shift_samples(int64_t n) { return n < 2048 ? n : 2048; }

// c_j from the column's sum over the sampled rows and their count (no row sampled: c = 0).  fp32 rows take the fp32
// mean: x - c is exact when the offset dominates (Sterbenz) and rounds at 2^-24 |x - c| otherwise, far below the hi/lo
// split's 2^-17 -- whereas a bf16-rounded c leaves a residual mean - c of up to half a bf16 spacing (32 for a column
// at 10016), and every shifted value carries it into the fp32 sums.  The bf16-storage kernels need c on the bf16 grid
// (they subtract it in bf16; the single-operand kernel feeds the raw tile to the tensor core): `bf16_grid`.
__device__ __forceinline__ float shift_from_sums(float sum, float rows, bool bf16_grid) {
  const float c = rows > 0.f ? sum / rows : 0.f;
  return bf16_grid ? __bfloat162float(__float2bfloat16_rn(c)) : c;
}
// Called with identical arguments by the Gram kernels and (on its shared-memory copy of the partials, same order of
// the 64 additions) by tc_finalize_kernel -> identical c.
__device__ __forceinline__ float shift_value(const float* __restrict__ sp, int j, bool bf16_grid) {
  float acc = 0.f, rows = 0.f;
#pragma unroll 8
  for (int b = 0; b < kShiftBlocks; ++b) {
    acc += sp[b * kShiftStride + j];
    rows += sp[b * kShiftStride + kMaxD + 1];
  }
  return shift_from_sums(acc, rows, bf16_grid);
}

// 64 blocks x (4 row groups x 160 columns): a thread sums 8 sample rows (one batch of loads in flight -- the rows are
// megabytes apart, every load is a DRAM round trip), the 4 groups are combined in a fixed order.  Column d + 1 counts
// the sampled rows the mask keeps; a dropped row contributes nothing, whatever it holds.
constexpr int kShiftCols = 160;                  // >= kMaxD + 2, a multiple of 32
constexpr int kShiftGroups = 4;

template <typename T>
__global__ void __launch_bounds__(kShiftCols * kShiftGroups)
tc_shift_kernel(const T* __restrict__ X, const float* __restrict__ y, const uint8_t* __restrict__ mask, int keep,
                int64_t n, int d, int64_t ldx, float* __restrict__ sp) {
  __shared__ float sub[kShiftGroups][kShiftCols];
  const int j = threadIdx.x % kShiftCols, g = threadIdx.x / kShiftCols;
  const int64_t samples = shift_samples(n);
  const int64_t stride = n / samples;
  const int64_t per = (samples + kShiftBlocks - 1) / kShiftBlocks;
  const int64_t s0 = blockIdx.x * per;
  const int64_t s1 = (s0 + per < samples) ? s0 + per : samples;
  float acc = 0.f;
  if (j <= d + 1) {
#pragma unroll 8
    for (int64_t s = s0 + g; s < s1; s += kShiftGroups) {
      const int64_t row = s * stride;
      if (mask != nullptr && mask[row] != (uint8_t)keep) continue;
      const float v = (j < d) ? raw_ld_global<T>(X + row * ldx + j) : (j == d ? __ldg(y + row) : 1.f);
      acc += (fabsf(v) <= 3.0e38f) ? v : 0.f;     // a kept non-finite value makes the statistic non-finite anyway
    }
  }
  sub[g][j] = acc;
  __syncthreads();
  if (g == 0 && j <= d + 1)
    sp[blockIdx.x * kShiftStride + (j < d ? j : kMaxD + (j - d))] = ((sub[0][j] + sub[1][j]) + sub[2][j]) + sub[3][j];
}

// ------------------------------------------------------------------------------------------
// finalize, shared by the stand-alone kernels (tc_reduce_kernel / tc_fold_kernel: the b2_gram_accumulate path) and
// by the fused tail of the Gram kernel (b2_fit): the same summation order in both, so the two paths agree bit for bit.
//   red[col * 128 + i], col in [0, 288):  col < 144: D1 (A = hi), col >= 144: D2 (A = lo), columns of [hi | E]
//   red[kTcAccElems + 0..2]            : sum y', sum y'^2, rows used
// ------------------------------------------------------------------------------------------
constexpr int kRedElems = kTcAccElems + 3;

// Sum over the CTAs of elements [e0, e1) of the per-CTA partials.  4 threads per element: thread (e, q) sums the q-th
// quarter of the CTAs with 8 loads in flight (the loads are the latency), the quarters are combined in the fixed order
// 0..3 -> deterministic.  `quarter`: shared scratch of 4 * (blockDim.x / 4) doubles.  Call with the whole block.
__device__ __forceinline__ void tc_reduce_range(const double* part, const double* side, int n_ctas, double* red,
                                                int e0, int e1, double* quarter) {
  const int epb = blockDim.x >> 2;                 // elements per pass
  const int e = threadIdx.x % epb, q = threadIdx.x / epb;
  const int per = (n_ctas + 3) / 4;
  const int c0 = q * per, c1 = (c0 + per < n_ctas) ? c0 + per : n_ctas;
  for (int base = e0; base < e1; base += epb) {
    const int idx = base + e;
    if (idx < e1 && idx < kTcAccElems) {
      double acc[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
      int c = c0;
      for (; c + 8 <= c1; c += 8) {
#pragma unroll
        for (int u = 0; u < 8; ++u) acc[u] += __ldcg(part + (size_t)(c + u) * kTcAccElems + idx);
      }
      for (; c < c1; ++c) acc[0] += __ldcg(part + (size_t)c * kTcAccElems + idx);
      quarter[q * epb + e] = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
    } else if (idx < e1 && idx < kRedElems) {
      // the three CUDA-core sums (sum y', sum y'^2, rows): same quarter scheme, loads 8 deep (a serial walk over the
      // CTAs costs one L2 round trip each: 148 x ~140 ns was most of this phase)
      const int k = idx - kTcAccElems;
      double acc[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
      int c = c0;
      for (; c + 8 <= c1; c += 8) {
#pragma unroll
        for (int u = 0; u < 8; ++u)
          acc[u] += __ldcg(side + (size_t)(c + u) * kTcSideDoubles + k) + __ldcg(side + (size_t)(c + u) * kTcSideDoubles + 3 + k);
      }
      for (; c < c1; ++c) acc[0] += __ldcg(side + (size_t)c * kTcSideDoubles + k) + __ldcg(side + (size_t)c * kTcSideDoubles + 3 + k);
      quarter[q * epb + e] = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
    }
    __syncthreads();
    if (q == 0 && idx < e1 && idx < kRedElems)
      red[idx] = ((quarter[e] + quarter[epb + e]) + quarter[2 * epb + e]) + quarter[3 * epb + e];
    __syncthreads();
  }
}

// Grid-wide barrier of a co-resident (cooperatively launched) grid: arrive on a counter, wait until all CTAs have.
// The counter is zeroed again by the kernel's final ticket.  Bounded: a protocol bug traps instead of hanging.
__device__ __forceinline__ void grid_barrier(unsigned int* ctr) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(ctr, 1u);
    const uint64_t t0 = globaltimer_ns();
    unsigned int seen;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(ctr) : "memory");
      if (seen < gridDim.x) {
        __nanosleep(40);
        if (globaltimer_ns() - t0 > 4000000000ull) __trap();
      }
    } while (seen < gridDim.x);
    __threadfence();
  }
  __syncthreads();
}

// `pack` original rows share one 128-wide super-row (d * pack == 128 when pack > 1): original feature a of
// sub-row blk is super-feature blk*d + a, and its E columns are 128 + 3*blk (+0 ones, +1 y'_hi, +2 y'_lo).
// The true statistic is the sum over blk of the diagonal (blk, blk) blocks.
// Returns the contribution of this launch to S[idx]; c[j] = the shift of feature j, c[kMaxD] = the shift of y
// (fp64 copy in `red` for the stand-alone kernel, the CTA's fp32 smem copy in the fused tail -- the same values).
template <typename CT>
__device__ __forceinline__ double tc_fold_value(const double* red, const CT* c, int d, int pack, int idx) {
  const int dp = d + 2;
  const int r = idx / dp, q = idx % dp;
  const int a = r < q ? r : q, b = r < q ? q : r;   // (a, b) and (b, a) evaluate the same expression: S stays bit-symmetric
  // D1[i][j] = red[j*128 + i], D2[i][j] = red[(144 + j)*128 + i]
  auto D1 = [&](int i, int j) { return __ldcg(red + (size_t)j * kTcM + i); };
  auto D2 = [&](int i, int j) { return __ldcg(red + (size_t)(kTcN + j) * kTcM + i); };
  auto s1 = [&](int i) {                                                     // sum (x_i - c_i)
    double t = 0.0;
    for (int blk = 0; blk < pack; ++blk) t += D1(blk * d + i, 128 + 3 * blk) + D2(blk * d + i, 128 + 3 * blk);
    return t;
  };
  auto sxy = [&](int i) {                                                    // sum (x_i - c_i) y'
    double t = 0.0;
    for (int blk = 0; blk < pack; ++blk) {
      const int r = blk * d + i, e = 128 + 3 * blk;
      t += D1(r, e + 1) + D1(r, e + 2) + D2(r, e + 1) + D2(r, e + 2);
    }
    return t;
  };
  const double sy = __ldcg(red + kTcAccElems + 0);
  const double syy = __ldcg(red + kTcAccElems + 1);
  const double n = __ldcg(red + kTcAccElems + 2);
  const double cy = (double)c[kMaxD];
  double val;
  if (a < d && b < d) {
    const double ca = (double)c[a], cb = (double)c[b];
    // G'(a,b) = sum (x_a-c_a)(x_b-c_b) ~= hi.hi + lo.hi + hi.lo   (lo.lo dropped, ~2^-18 relative)
    double g = 0.0;
    for (int blk = 0; blk < pack; ++blk) {
      const int ia = blk * d + a, ib = blk * d + b;
      g += 0.5 * (D1(ia, ib) + D1(ib, ia)) + D2(ia, ib) + D2(ib, ia);
    }
    val = g + ca * s1(b) + cb * s1(a) + n * ca * cb;
  } else if (a < d || b < d) {
    const int i = a < d ? a : b;
    const int o = a < d ? b : a;  // d (ones) or d+1 (y)
    const double ci = (double)c[i];
    if (o == d) val = s1(i) + n * ci;
    else val = sxy(i) + cy * s1(i) + ci * sy + n * ci * cy;
  } else if (a == d && b == d) {
    val = n;
  } else if (a == d + 1 && b == d + 1) {
    val = syy + 2.0 * cy * sy + n * cy * cy;
  } else {
    val = sy + n * cy;
  }
  return val;
}


// ------------------------------------------------------------------------------------------
// the Gram kernel
// ------------------------------------------------------------------------------------------
// DFIX = 128: feature count known at compile time (immediate smem offsets, no index arithmetic in
// the transform loop); DFIX = 0: runtime d (any multiple of 4 / 8 up to 128).
// SPLIT = true : operands hi + lo (16 mantissa bits, the default);
// SPLIT = false: single bf16 operand hi = rn(x - c) ("bf16-accum" mode of BASELINE.json configs[1]): half the MMAs,
//                no lo arithmetic; the operand rounding error (2^-9 relative, zero mean) averages out as 1/sqrt(n).
template <typename T, int DFIX, bool SPLIT>
__global__ void __launch_bounds__(kThreads, 1)
gram_tc_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmY,
               const __grid_constant__ CUtensorMap tmM, int y_map_2d, int has_mask, int keep,
               int64_t n_rows, int d_arg, int pack, int d_orig, const float* __restrict__ shift,
               int chunk_tiles,
               double* __restrict__ part, double* __restrict__ side, uint32_t wait_ns, uint32_t dbg_arg) {
#ifdef B2_DEV_KNOBS
  const uint32_t dbg = dbg_arg;      // ablation switches (tools/build_dev.sh): results are WRONG when non-zero
#else
  constexpr uint32_t dbg = 0u;       // product build: the ablation branches compile away
  (void)dbg_arg;
#endif
  const int d = DFIX ? DFIX : d_arg;
  constexpr bool kTS = (DFIX == 128);                         // A = lo from TMEM (needs warp%4 == feature quad)
  constexpr uint32_t kLBO = kTS ? kOpLBO_TS : kOpLBO_SS;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (sbase - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  const uint32_t bar_raw_full = sbase + kOffBar;                       // [kRawStages]
  const uint32_t bar_raw_empty = bar_raw_full + 8 * kRawStages;        // [kRawStages]
  const uint32_t bar_op_full = bar_raw_empty + 8 * kRawStages;         // [kOpStages]
  const uint32_t bar_op_empty = bar_op_full + 8 * kOpStages;           // [kOpStages]
  const uint32_t bar_acc_full = bar_op_empty + 8 * kOpStages;          // [2]
  const uint32_t bar_acc_empty = bar_acc_full + 16;                    // [2]
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem + kOffTmemPtr);
  float* shift_s = reinterpret_cast<float*>(smem + kOffShift);

  // contiguous tile range of this CTA
  const int64_t total_tiles = (n_rows + kTcRows - 1) / kTcRows;
  const int64_t tile_begin = (int64_t)blockIdx.x * total_tiles / gridDim.x;
  const int64_t tile_end = (int64_t)(blockIdx.x + 1) * total_tiles / gridDim.x;
  const int my_tiles = (int)(tile_end - tile_begin);
  const int n_chunks = (my_tiles + chunk_tiles - 1) / chunk_tiles;

  // ---- one-time setup --------------------------------------------------------------------
  if (threadIdx.x == 0) {
    for (int s = 0; s < kRawStages; ++s) {
      mbar_init(bar_raw_full + 8 * s, 1);
      mbar_init(bar_raw_empty + 8 * s, kProducers);
    }
    for (int s = 0; s < kOpStages; ++s) {
      mbar_init(bar_op_full + 8 * s, kProducers);
      mbar_init(bar_op_empty + 8 * s, 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(bar_acc_full + 8 * b, 1);
      mbar_init(bar_acc_empty + 8 * b, 4);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmY);
    if (has_mask) tma_prefetch_desc(&tmM);
  }
  if (warp == 1) {  // TMEM: 512 columns (D1 x2 at 0 / 144, D2 at 288, TS operand A = lo at 432)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(sbase + kOffTmemPtr)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // zero the operand stages once: feature rows >= d, the unused E rows and the lo/hi padding read as 0
  for (uint32_t o = threadIdx.x * 16; o < kOpStages * kOpStageBytes; o += kThreads * 16)
    *reinterpret_cast<uint4*>(smem + kOffOp + o) = make_uint4(0, 0, 0, 0);
  // packed rows (pack > 1): super-row feature i < pack * d_orig is original feature i % d_orig -> the shift repeats;
  // the columns from pack * d_orig to 127 are TMA out-of-bounds zero fill and keep shift 0 (they contribute nothing)
  for (int j = threadIdx.x; j <= kMaxD; j += kThreads)
    shift_s[j] = (j == kMaxD) ? shift_value(shift, kMaxD, false)
                              : (j < pack * d_orig ? shift_value(shift, j % d_orig, false) : 0.f);
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  // ---- warp roles --------------------------------------------------------------------------
  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      const uint32_t tx = (uint32_t)(kTcRows * d * sizeof(T)) + kTcRows * pack * 4 + (has_mask ? kTcRows * pack : 0);
      int s = 0;
      uint32_t ph = 0;
      for (int it = 0; it < my_tiles; ++it) {
        mbar_wait(bar_raw_empty + 8 * s, ph ^ 1, wait_ns);
        const uint32_t full = bar_raw_full + 8 * s;
        mbar_expect_tx(full, tx);
        const int64_t row0 = (tile_begin + it) * kTcRows;
        tma_load_2d(sbase + kOffRaw + s * kRawStageBytes, &tmX, 0, (int)row0, full);
        const int sub0 = (int)row0 * pack;                               // first original row of the tile
        if (y_map_2d) tma_load_2d(sbase + kOffY + s * kYStageBytes, &tmY, 0, sub0 >> 2, full);
        else tma_load_1d(sbase + kOffY + s * kYStageBytes, &tmY, sub0, full);
        if (has_mask == 2) tma_load_2d(sbase + kOffMask + s * kMStageBytes, &tmM, 0, sub0 >> 4, full);
        else if (has_mask) tma_load_1d(sbase + kOffMask + s * kMStageBytes, &tmM, sub0, full);
        if (++s == kRawStages) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (one elected thread: straight-line UTCHMMA, see elect_one) =====
    if (elect_one()) {
      int os = 0;
      uint32_t oph = 0;
      int in_chunk = 0, chunk = 0;
      for (int it = 0; it < my_tiles; ++it) {
        const int b = chunk & 1;
        if (in_chunk == 0) {  // this D1 buffer must have been drained (two chunks ago)
          mbar_wait(bar_acc_empty + 8 * b, ((chunk >> 1) & 1) ^ 1);
          tc_fence_after();
        }
        mbar_wait(bar_op_full + 8 * os, oph, wait_ns);
        tc_fence_after();
        const uint32_t op_addr = sbase + kOffOp + os * kOpStageBytes;
        const uint32_t tmem_d1 = tmem_base + (uint32_t)b * kTmemD1Stride;
#pragma unroll
        for (int k2 = 0; k2 < kTcRows / 16; ++k2) {
          const uint64_t b_desc = make_smem_desc(op_addr + k2 * 2 * kLBO, kLBO);            // [hi | E], also A = hi
          if (!(dbg & 2u)) umma_bf16(tmem_d1, b_desc, b_desc, (in_chunk > 0 || k2 > 0) ? 1u : 0u);
          if (SPLIT && !(dbg & 3u)) {
            if constexpr (kTS) {
              umma_bf16_ts(tmem_base + kTmemD2Col, tmem_base + kTmemALoCol + (uint32_t)(os * 32 + k2 * 8), b_desc,
                           (it > 0 || k2 > 0) ? 1u : 0u);
            } else {
              const uint64_t lo_desc = make_smem_desc(op_addr + k2 * 2 * kLBO + kOpLoOff, kLBO);   // A = lo
              umma_bf16(tmem_base + kTmemD2Col, lo_desc, b_desc, (it > 0 || k2 > 0) ? 1u : 0u);
            }
          }
        }
        umma_commit(bar_op_empty + 8 * os);  // frees the operand stage when these MMAs retire
        const bool last = (in_chunk == chunk_tiles - 1) || (it == my_tiles - 1);
        if (last) { umma_commit(bar_acc_full + 8 * b); in_chunk = 0; ++chunk; }
        else ++in_chunk;
        if (++os == kOpStages) { os = 0; oph ^= 1; }
      }
    }
  } else if (warp == 2 || warp == 3) {
    // ===== E warps: extra operand columns [1, y'_hi, y'_lo] and the CUDA-core sums of y' =====
    const float c_y = shift_s[kMaxD];
    double sy = 0.0, syy = 0.0, cnt = 0.0;
    int rs = 0, os = 0;
    uint32_t rph = 0, oph = 0;
    for (int it = 0; it < my_tiles; ++it) {
      mbar_wait(bar_raw_full + 8 * rs, rph, wait_ns);
      mbar_wait(bar_op_empty + 8 * os, oph ^ 1, wait_ns);
      tc_fence_after();
      const int64_t row0 = (tile_begin + it) * kTcRows;
      const uint32_t y_addr = sbase + kOffY + rs * kYStageBytes;
      const uint32_t m_addr = sbase + kOffMask + rs * kMStageBytes;
      const uint32_t e_addr = sbase + kOffOp + os * kOpStageBytes + kOpEOff;
      const int64_t left = n_rows - row0;
      const int rows_valid = left < kTcRows ? (int)left : kTcRows;
      // warp 2 covers super-rows 0..31 of the tile, warp 3 covers 32..63: one super-row per lane
      float a = 0.f, b = 0.f, c = 0.f;
      {
        const int rr = lane + 32 * (warp - 2);      // super-row inside the tile
        const uint32_t dst = e_addr + (rr >> 3) * kLBO + (rr & 7) * 2;
        for (int bl = 0; bl < pack; ++bl) {         // original row rr * pack + bl -> E columns 3*bl .. 3*bl+2
          const int sub = rr * pack + bl;
          bool use = rr < rows_valid;
          if (use && has_mask) use = (ld_shared_u8(m_addr + sub) == (uint32_t)keep);
          const float yv = use ? ld_shared_f32(y_addr + sub * 4) - c_y : 0.f;
          uint32_t yh, yl;
          split2(yv, 0.f, yh, yl);
          st_shared_u16(dst + (3 * bl) * 16, use ? 0x3F80u : 0u);   // bf16(1.0): row-validity ("ones") column
          st_shared_u16(dst + (3 * bl + 1) * 16, yh);
          st_shared_u16(dst + (3 * bl + 2) * 16, yl);
          a += yv;
          b = fmaf(yv, yv, b);
          c += use ? 1.f : 0.f;
        }
      }
      sy += (double)a; syy += (double)b; cnt += (double)c;
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(bar_op_full + 8 * os);
        mbar_arrive(bar_raw_empty + 8 * rs);
      }
      if (++rs == kRawStages) { rs = 0; rph ^= 1; }
      if (++os == kOpStages) { os = 0; oph ^= 1; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      sy += __shfl_xor_sync(0xffffffffu, sy, o);
      syy += __shfl_xor_sync(0xffffffffu, syy, o);
      cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    }
    if (lane == 0) {
      double* ys = side + (size_t)blockIdx.x * kTcSideDoubles + 3 * (warp - 2);
      ys[0] = sy; ys[1] = syy; ys[2] = cnt;
    }
  } else if (warp >= 4 && warp < 8) {
    // ===== epilogue: TMEM -> registers -> fp64 partial in global (column-major [col][feature]) =====
    const int w = warp & 3;  // TMEM lane quadrant this warp may access
    double* my_part = part + (size_t)blockIdx.x * kTcAccElems + w * 32 + lane;
    const uint32_t lane_base = tmem_base + ((uint32_t)(w * 32) << 16);
    for (int chunk = 0; chunk < n_chunks; ++chunk) {
      const int b = chunk & 1;
      mbar_wait(bar_acc_full + 8 * b, (chunk >> 1) & 1);
      tc_fence_after();
      // D1 (A = hi) of this chunk: fold into partial columns [0, 144)
#pragma unroll 1
      for (int p = 0; p < kTcN / 16; ++p) {
        uint32_t r[16];
        tmem_ld16(lane_base + (uint32_t)b * kTmemD1Stride + (uint32_t)(p * 16), r);
        tmem_ld_wait();
        double* dst = my_part + (size_t)(p * 16) * kTcM;
        if (chunk == 0) {
#pragma unroll
          for (int j = 0; j < 16; ++j) dst[(size_t)j * kTcM] = (double)__uint_as_float(r[j]);
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) dst[(size_t)j * kTcM] += (double)__uint_as_float(r[j]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_acc_empty + 8 * b);
    }
    // D2 (A = lo) accumulated over the whole range (small zero-mean sums): partial columns [144, 288)
    tc_fence_after();
#pragma unroll 1
    for (int p = 0; p < kTcN / 16; ++p) {
      uint32_t r[16];
      if constexpr (SPLIT) {
        tmem_ld16(lane_base + kTmemD2Col + (uint32_t)(p * 16), r);
        tmem_ld_wait();
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) r[j] = 0u;     // no lo accumulator in single-operand mode
      }
      double* dst = my_part + (size_t)(kTcN + p * 16) * kTcM;
#pragma unroll
      for (int j = 0; j < 16; ++j) dst[(size_t)j * kTcM] = (double)__uint_as_float(r[j]);
    }
  } else if (warp >= 8) {
    // ===== transform: shift, bf16 hi/lo split, K-major operand store =====
    // A task = (feature quad q, 8-row group g) of a tile; nq * 8 tasks per tile, at most 2 per warp.
    const int t = warp - 8;
    const int nq = (d + 31) >> 5;
    const uint32_t esz = sizeof(T);
    const uint32_t pitch = (uint32_t)d * esz;       // raw tile row pitch in bytes
    bool tv[2];
    float tc[2];
    uint32_t tsrc[2], tdst[2];
    int tr0[2], tblk[2];
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      const int tt = t + kXformWarps * s;
      const bool valid = tt < nq * kKGroups;
      const int q = valid ? tt % nq : 0, g = valid ? tt / nq : 0;
      const int i = q * 32 + lane;
      tv[s] = valid && (i < d);
      tc[s] = shift_s[tv[s] ? i : 0];
      tr0[s] = g * 8;
      tblk[s] = (tv[s] ? i : 0) / d_orig;           // which original row of the super-row this feature belongs to
      tsrc[s] = (uint32_t)(g * 8) * pitch + (uint32_t)(tv[s] ? i : 0) * esz;
      tdst[s] = (uint32_t)g * kLBO + (uint32_t)((i >> 3) * kOpSBO + (i & 7) * 16);
    }
    int rs = 0, os = 0;
    uint32_t rph = 0, oph = 0;
    for (int it = 0; it < my_tiles; ++it) {
      mbar_wait(bar_raw_full + 8 * rs, rph, wait_ns);
      mbar_wait(bar_op_empty + 8 * os, oph ^ 1, wait_ns);
      tc_fence_after();
      const int64_t row0 = (tile_begin + it) * kTcRows;
      const int64_t left = n_rows - row0;
      const int rows_valid = left < kTcRows ? (int)left : kTcRows;
      const bool full_tile = (!has_mask) && (rows_valid == kTcRows);
      const uint32_t raw_addr = sbase + kOffRaw + rs * kRawStageBytes;
      const uint32_t m_addr = sbase + kOffMask + rs * kMStageBytes;
      const uint32_t op_addr = sbase + kOffOp + os * kOpStageBytes;
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        if (tv[s]) {
          float v[8];
          const uint32_t src = raw_addr + tsrc[s];
          const float c_i = tc[s];
#pragma unroll
          for (int k = 0; k < 8; ++k)
            v[k] = ((dbg & 8u) ? __uint_as_float(src + k) : raw_ld_shared<T>(src + (uint32_t)k * pitch)) - c_i;
          if (!full_tile) {
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              bool use = (tr0[s] + k) < rows_valid;
              if (use && has_mask) use = (ld_shared_u8(m_addr + (tr0[s] + k) * pack + tblk[s]) == (uint32_t)keep);
              if (!use) v[k] = 0.f;
            }
          }
          uint32_t hp[4], lp[4];
#pragma unroll
          for (int p = 0; p < 4; ++p) {
            if constexpr (SPLIT) {
              split2(v[2 * p], v[2 * p + 1], hp[p], lp[p]);
            } else {
              const __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * p], v[2 * p + 1]);
              hp[p] = *reinterpret_cast<const uint32_t*>(&h);
              lp[p] = 0u;
            }
          }
          if (!(dbg & 4u)) {
            st_shared_v4(op_addr + tdst[s], hp);
            if constexpr (!SPLIT) {
              // single-operand mode: no lo block / TMEM operand
            } else if constexpr (kTS) {
              // lane l of this warp owns TMEM lane 32*(warp%4)+l == feature i; K group g -> 4 packed columns
              tmem_st4(tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + kTmemALoCol +
                           (uint32_t)(os * 32 + (tr0[s] >> 3) * 4), lp);
            } else {
              st_shared_v4(op_addr + tdst[s] + kOpLoOff, lp);
            }
          }
        }
      }
      if constexpr (kTS && SPLIT) {
        tmem_st_wait();
        tc_fence_before();
      }
      if (!(dbg & 32u)) fence_proxy_async_smem();  // generic-proxy stores -> visible to the tensor core (async proxy)
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(bar_op_full + 8 * os);
        mbar_arrive(bar_raw_empty + 8 * rs);
      }
      if (++rs == kRawStages) { rs = 0; rph ^= 1; }
      if (++os == kOpStages) { os = 0; oph ^= 1; }
    }
  }

  // ---- teardown ---------------------------------------------------------------------------
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
  }
}

#include "gram_tc_b16.cuh"
#include "gram_tc_b16_split.cuh"

// ------------------------------------------------------------------------------------------
// finalize: tc_reduce_kernel sums the per-CTA partials in CTA order (deterministic)
//   red[col * 128 + i], col in [0, 288):  col < 144: D1 (A = hi), col >= 144: D2 (A = lo), columns of [hi | E]
//   red[kTcAccElems + 0..2]            : sum y', sum y'^2, rows used
// tc_fold_kernel undoes the shift in fp64 and adds the result into the raw statistic S ((d+2)^2, stride d+2).
// ------------------------------------------------------------------------------------------

// What tc_finalize_kernel does after the reduce + fold (passed by value).
struct TcFinal {
  int assign;                 // S = value instead of S += value (fresh statistic: no memset launch)
  int n_ranks, rank;          // n_ranks > 1: store S into the exchange slot of every rank and publish the flags
  unsigned int epoch;
  PeerPtrs peers;
};

// ONE launch behind the Gram kernel: reduce the per-CTA partials (fixed order: deterministic), grid barrier, undo the
// shift in fp64 and fold into S, store S into the peers' exchange slots (b2_fit with an attached peer exchange), and
// -- through a last-block ticket -- publish the exchange flags and re-arm the barrier.  Cooperative launch: every CTA
// is resident, so the counter barrier is safe.  This work deliberately does NOT live in the Gram kernel's tail: with
// it there (even out of line) the hot role loops lost 5 % (same box: 0.807 ms without, 0.849 ms with, 10 M x 128
// rows) -- more than the launch it saves.
constexpr int kFinalizeThreads = 1024;                           // 4 threads per element of the partials
constexpr int kFinalizeCtas = (kRedElems + kFinalizeThreads / 4 - 1) / (kFinalizeThreads / 4);   // 145: one pass

__global__ void __launch_bounds__(kFinalizeThreads, 1)
tc_finalize_kernel(const double* part, const double* side, int n_ctas, double* red, const float* __restrict__ shift,
                   int bf16_grid, int d, int pack, double* S, unsigned int* sync, const TcFinal fin) {
  __shared__ double quarter[kFinalizeThreads];
  __shared__ double c_s[kMaxD + 1];                              // the shift as fp64 (c_s[kMaxD]: c_y)
  __shared__ float c_part[kShiftBlocks * kShiftStride];          // the 64 partial sums of the shift sample (33 KB)
  // the same values shift_value() gives the Gram kernel -- same operands, same order of the 64 additions -- but with
  // all loads of the CTA in flight at once: the serial walk (8 batches of dependent-latency loads by 129 threads while
  // 895 wait at the next barrier) was 40 % of this kernel (profiles/r02_tc_finalize_summary.txt)
  for (int idx = threadIdx.x; idx < kShiftBlocks * kShiftStride; idx += blockDim.x) c_part[idx] = __ldg(shift + idx);
  __syncthreads();
  for (int j = threadIdx.x; j <= kMaxD; j += blockDim.x) {
    float acc = 0.f, rows = 0.f;
#pragma unroll 8
    for (int b = 0; b < kShiftBlocks; ++b) {
      acc += c_part[b * kShiftStride + j];
      rows += c_part[b * kShiftStride + kMaxD + 1];
    }
    c_s[j] = (j < d || j == kMaxD) ? (double)shift_from_sums(acc, rows, bf16_grid != 0 && j < kMaxD) : 0.0;
  }
  {
    constexpr int epb = kFinalizeThreads / 4;                    // elements per pass of a CTA
    const int per = (((kRedElems + (int)gridDim.x - 1) / (int)gridDim.x) + epb - 1) / epb * epb;
    const int e0 = (int)blockIdx.x * per;
    const int e1 = e0 + per < kRedElems ? e0 + per : kRedElems;
    if (e0 < kRedElems) tc_reduce_range(part, side, n_ctas, red, e0, e1, quarter);
  }
  grid_barrier(sync + 0);
  {
    const int dp = d + 2;
    const int total = dp * dp;
    const size_t slot = xchg_slot_offset(fin.epoch, fin.rank);
    for (int idx = (int)(blockIdx.x * blockDim.x + threadIdx.x); idx < total; idx += (int)(gridDim.x * blockDim.x)) {
      const double val = tc_fold_value(red, c_s, d, pack, idx);
      const double sv = fin.assign ? val : S[idx] + val;
      S[idx] = sv;
      if (fin.n_ranks > 1) xchg_store_all(fin.peers, fin.n_ranks, slot, idx, sv);
    }
    if (fin.n_ranks > 1) __threadfence_system();
  }
  __syncthreads();
  __shared__ bool last_cta;
  if (threadIdx.x == 0) {
    __threadfence();
    last_cta = (atomicAdd(sync + 2, 1u) == gridDim.x - 1);
    if (last_cta) {                       // every CTA has passed the barrier: re-arm it for the next launch
      sync[0] = 0u; sync[2] = 0u;
      __threadfence();
    }
  }
  __syncthreads();
  if (last_cta && fin.n_ranks > 1) xchg_publish(fin.peers, fin.n_ranks, fin.rank, fin.epoch);
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (fn == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

}  // namespace

bool gram_tc_supported(const void* X, int x_dtype, const float* y, int64_t n, int d, int64_t ldx) {
  const int es = x_dtype == B2_F32 ? 4 : 2;
  if (d < 4 || d > kMaxD) return false;
  if ((d * es) % 16 != 0) return false;
  if ((ldx * es) % 16 != 0) return false;
  if ((reinterpret_cast<uintptr_t>(X) & 15) != 0 || (reinterpret_cast<uintptr_t>(y) & 15) != 0) return false;
  if (n < kTcRows) return false;
  if (n > (int64_t)0x7fffffff) return false;  // TMA coordinates are int32
  return true;
}

// d: inner extent of the (super-)row tensor; d_box: inner extent of the smem tile (> d: the rest is zero fill)
// swz64: the bf16 D = 128 kernel's raw layout -- [64 rows][64 features] boxes (128-byte rows) with SWIZZLE_128B
static int encode_maps(PFN_encodeTiled encode, const void* X, int x_dtype, int es, const float* y, int64_t n, int d,
                       int d_box, int64_t ldx, int64_t n_y, int pack, const uint8_t* mask, bool swz64, CUtensorMap* tmX_out,
                       CUtensorMap* tmY_out, CUtensorMap* tmM_out, int* y_map_2d_out, int* m_map_2d_out) {
  const cuuint32_t y_box = (cuuint32_t)(kTcRows * pack);   // original rows per tile
  CUtensorMap& tmX = *tmX_out; CUtensorMap& tmY = *tmY_out; CUtensorMap& tmM = *tmM_out;
  memset(&tmM, 0, sizeof(tmM));
  {
    cuuint64_t dims[2] = {(cuuint64_t)d, (cuuint64_t)n};
    cuuint64_t strides[1] = {(cuuint64_t)ldx * es};
    cuuint32_t box[2] = {(cuuint32_t)(swz64 ? 64 : d_box), (cuuint32_t)kTcRows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = encode(&tmX, x_dtype == B2_F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16,
                        2, const_cast<void*>(X), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        swz64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      set_error("cuTensorMapEncodeTiled(X) failed with %d (n=%lld d=%d box=%d ldx=%lld)", (int)r, (long long)n, d, d_box,
                (long long)ldx);
      return B2_E_CUDA;
    }
  }
  int y_map_2d = 0;
  {
    cuuint64_t dims[1] = {(cuuint64_t)n_y};
    cuuint64_t strides[1] = {0};
    cuuint32_t box[1] = {y_box};
    cuuint32_t estr[1] = {1};
    CUresult r = CUDA_ERROR_INVALID_VALUE;
    if (y_box <= 256)
      r = encode(&tmY, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 1, const_cast<float*>(y), dims, strides, box, estr,
                 CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                 CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      // rank-1 maps refused: view y as [ceil(n/4)][4] (16-byte rows) -- the same bytes land in smem
      cuuint64_t dims2[2] = {4, (cuuint64_t)((n_y + 3) / 4)};
      cuuint64_t strides2[1] = {16};
      cuuint32_t box2[2] = {4, y_box / 4};
      cuuint32_t estr2[2] = {1, 1};
      r = encode(&tmY, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(y), dims2, strides2, box2, estr2,
                 CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                 CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      y_map_2d = 1;
      if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled(y) failed with %d", (int)r);
        return B2_E_CUDA;
      }
    }
  }
  if (mask != nullptr && (reinterpret_cast<uintptr_t>(mask) & 15) != 0) {
    set_error("row_mask must be 16-byte aligned for the tcgen05 path");
    return B2_E_ARG;
  }
  int m_map_2d = 0;
  if (mask != nullptr) {
    cuuint64_t dims[1] = {(cuuint64_t)n_y};
    cuuint64_t strides[1] = {0};
    cuuint32_t box[1] = {y_box};
    cuuint32_t estr[1] = {1};
    CUresult r = CUDA_ERROR_INVALID_VALUE;
    if (y_box <= 256)
      r = encode(&tmM, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, const_cast<uint8_t*>(mask), dims, strides, box, estr,
                 CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                 CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS && n_y % 16 == 0) {
      // box extents stop at 256: view the mask as [n/16][16] (16-byte rows) -- the same bytes land in smem
      cuuint64_t dims2[2] = {16, (cuuint64_t)(n_y / 16)};
      cuuint64_t strides2[1] = {16};
      cuuint32_t box2[2] = {16, y_box / 16};
      cuuint32_t estr2[2] = {1, 1};
      r = encode(&tmM, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<uint8_t*>(mask), dims2, strides2, box2, estr2,
                 CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                 CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      m_map_2d = 1;
    }
    if (r != CUDA_SUCCESS) {
      set_error("cuTensorMapEncodeTiled(mask) failed with %d", (int)r);
      return B2_E_CUDA;
    }
  }

  *m_map_2d_out = m_map_2d;
  *y_map_2d_out = y_map_2d;
  return B2_OK;
}

// Row packing rule: how many of the n rows the tensor-core launch covers (the rest, < 80 rows, take the CUDA-core kernel)
int64_t gram_tc_main_rows(int64_t n_in, int d_in, int64_t ldx_in, int* pack_out) {
  int pack = 1;
  if (d_in > 16 && d_in <= 64 && ldx_in == d_in) {
    pack = 128 / d_in;
    if (pack > kMaxPack) pack = kMaxPack;
    if (n_in < (int64_t)2 * kTcRows * pack) pack = 1;
  }
  const int group = pack == 1 ? 1 : (pack == 3 ? 48 : (pack == 5 ? 80 : 16));
  if (pack_out != nullptr) *pack_out = pack;
  return n_in - n_in % group;
}

int launch_gram_tc(b2_ctx* ctx, const void* X, int x_dtype, const float* y, int64_t n_in, int d_in, int64_t ldx_in,
                   const uint8_t* mask, int keep, const TcFuse* fuse) {
  PFN_encodeTiled encode = get_encode();
  if (encode == nullptr) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return B2_E_CUDA;
  }
  const int es = x_dtype == B2_F32 ? 4 : 2;
  // Row packing: `pack` contiguous rows of 17..64 features are viewed as one super-row of pack * d_in <= 128 columns
  // ([n / pack][pack * d_in], zero-filled by TMA to the 128-wide tile) and run on the D = 128 fast path; the diagonal
  // d_in x d_in blocks of the 128 x 128 Gram sum to the true statistic (tc_fold_kernel).  The tensor maps cover a
  // multiple of lcm(pack, 16) rows (the y / mask views are 16-byte rows); the < 80 leftover rows go through the
  // CUDA-core kernel.
  int pack = 1;
  const int64_t n_main = gram_tc_main_rows(n_in, d_in, ldx_in, &pack);   // original rows handled here
  const int64_t n = n_main / pack;                      // super-rows
  const int d = pack > 1 ? 128 : d_in;                  // kernel feature count (DFIX = 128 when packed)
  const int d_tensor = d_in * pack;                     // columns that exist; the tile is zero-filled beyond them
  const int64_t ldx = ldx_in * pack;
  const int64_t n_y = n_main;                           // y / mask elements covered by the tensor maps
  // bf16-stored rows with D = 128 take their own kernels (gram_tc_b16.cuh: single operand, gram_tc_b16_split.cuh: hi + lo); B2_TC_B16_GENERIC=1 keeps them on the generic
  // kernel (diagnostic switch for same-box A/B runs)
  static const bool b16_generic = []() { const char* e = getenv("B2_TC_B16_GENERIC"); return e != nullptr && e[0] == '1'; }();
  const bool b16 = x_dtype == B2_BF16 && d_in == 128 && pack == 1 && !b16_generic;
  CUtensorMap tmX, tmY, tmM;
  int y_map_2d = 0, m_map_2d = 0;
  b2_ctx::TmCache& tc = ctx->tm_cache;
  const bool cached = tc.X == X && tc.y == y && tc.mask == mask && tc.n == n_in && tc.ldx == ldx_in && tc.d == d_in &&
                      tc.x_dtype == x_dtype;
  if (cached) {
    memcpy(&tmX, tc.tmX, sizeof(tmX)); memcpy(&tmY, tc.tmY, sizeof(tmY)); memcpy(&tmM, tc.tmM, sizeof(tmM));
    y_map_2d = tc.y_map_2d & 1; m_map_2d = (tc.y_map_2d >> 1) & 1;
  } else {
    if (int r = encode_maps(encode, X, x_dtype, es, y, n, d_tensor, d, ldx, n_y, pack, mask, b16, &tmX, &tmY, &tmM, &y_map_2d,
                            &m_map_2d))
      return r;
    tc.X = X; tc.y = y; tc.mask = mask; tc.n = n_in; tc.ldx = ldx_in; tc.d = d_in; tc.x_dtype = x_dtype;
    tc.y_map_2d = y_map_2d | (m_map_2d << 1);
    memcpy(tc.tmX, &tmX, sizeof(tmX)); memcpy(tc.tmY, &tmY, sizeof(tmY)); memcpy(tc.tmM, &tmM, sizeof(tmM));
  }

  const int64_t total_tiles = (n + kTcRows - 1) / kTcRows;
  const int sms = (ctx->sm_limit > 0 && ctx->sm_limit < ctx->sm_count) ? ctx->sm_limit : ctx->sm_count;
  const int grid = (int)(total_tiles < sms ? total_tiles : sms);
  int chunk_tiles = ctx->drain_rows / kTcRows;
  if (chunk_tiles < 1) chunk_tiles = 1;

  if (!ctx->tc_attr_set) {
#define B2_SET_SMEM(T, DF, SP) \
  B2_CUDA(cudaFuncSetAttribute(gram_tc_kernel<T, DF, SP>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes))
    B2_SET_SMEM(float, 128, true); B2_SET_SMEM(float, 0, true);
    B2_SET_SMEM(float, 128, false); B2_SET_SMEM(float, 0, false);
    B2_SET_SMEM(__nv_bfloat16, 128, true); B2_SET_SMEM(__nv_bfloat16, 0, true);
    B2_SET_SMEM(__nv_bfloat16, 128, false); B2_SET_SMEM(__nv_bfloat16, 0, false);
#undef B2_SET_SMEM
    B2_CUDA(cudaFuncSetAttribute(b16::sp::gram_b16_split_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, b16::sp::kSmem));
    B2_CUDA(cudaFuncSetAttribute(b16::gram_b16_single_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, b16::kSmem));
    ctx->tc_attr_set = true;
  }

  // S: a fresh statistic is overwritten by the finalize kernel (no memset launch); otherwise it must be cleared first
  const bool assign = fuse != nullptr && fuse->assign != 0;
  if (!assign) {
    if (int r = ensure_s_cleared(ctx)) return r;
  }
  if (x_dtype == B2_F32)
    tc_shift_kernel<float><<<kShiftBlocks, kShiftCols * kShiftGroups, 0, ctx->stream>>>(static_cast<const float*>(X), y, mask, keep,
                                                                                          n_in, d_in, ldx_in, ctx->shift);
  else
    tc_shift_kernel<__nv_bfloat16><<<kShiftBlocks, kShiftCols * kShiftGroups, 0, ctx->stream>>>(
        static_cast<const __nv_bfloat16*>(X), y, mask, keep, n_in, d_in, ldx_in, ctx->shift);
  B2_CUDA(cudaGetLastError());

#ifdef B2_DEV_KNOBS
  static const uint32_t wait_ns = []() {   // development knob: suspend-time hint of the pipeline waits
    const char* e = getenv("B2_WAIT_HINT_NS");
    return e ? (uint32_t)atoi(e) : 20000u;
  }();
#else
  constexpr uint32_t wait_ns = 20000u;     // try_wait suspend hint (ns); measured insensitive 0..20000 (r01)
#endif
#ifdef B2_DEV_KNOBS
  static const uint32_t dbg = []() {       // ablations: bit0 skip MMA2, bit1 skip all MMAs, bit2 skip STS, bit3 skip LDS, bit5 skip proxy fence
    const char* e = getenv("B2_TC_DEBUG");
    return e ? (uint32_t)atoi(e) : 0u;
  }();
#else
  constexpr uint32_t dbg = 0u;
#endif
  const int pair = ctx->k_pairs % kKernelEventPairs;
  B2_CUDA(cudaEventRecord(ctx->ev_k[pair][0], ctx->stream));
#define B2_LAUNCH_TC(T, DF, SP)                                                                          \
  gram_tc_kernel<T, DF, SP><<<grid, kThreads, kSmemBytes, ctx->stream>>>(                                \
      tmX, tmY, tmM, y_map_2d, mask != nullptr ? 1 + m_map_2d : 0, keep, n, d, pack, d_in, ctx->shift,       \
      chunk_tiles,                                                                                        \
      ctx->tc_part, ctx->tc_side, wait_ns, dbg)
#define B2_LAUNCH_TC_D(T, SP) \
  do { if (d == 128) B2_LAUNCH_TC(T, 128, SP); else B2_LAUNCH_TC(T, 0, SP); } while (0)
  const bool split = ctx->precision == B2_PRECISION_SPLIT;
  if (b16) {
    const int hm = mask != nullptr ? 1 + m_map_2d : 0;
    if (split)
      b16::sp::gram_b16_split_kernel<<<grid, kThreads, b16::sp::kSmem, ctx->stream>>>(tmX, tmY, tmM, y_map_2d, hm, keep, n,
                                                                                      ctx->shift, chunk_tiles, ctx->tc_part, ctx->tc_side);
    else
      b16::gram_b16_single_kernel<<<grid, kThreads, b16::kSmem, ctx->stream>>>(tmX, tmY, tmM, y_map_2d, hm, keep, n, ctx->shift,
                                                                               chunk_tiles, ctx->tc_part, ctx->tc_side);
  } else if (x_dtype == B2_F32) {
    if (split) B2_LAUNCH_TC_D(float, true); else B2_LAUNCH_TC_D(float, false);
  } else {
    if (split) B2_LAUNCH_TC_D(__nv_bfloat16, true); else B2_LAUNCH_TC_D(__nv_bfloat16, false);
  }
#undef B2_LAUNCH_TC_D
#undef B2_LAUNCH_TC
  B2_CUDA(cudaGetLastError());
  B2_CUDA(cudaEventRecord(ctx->ev_k[pair][1], ctx->stream));
  ctx->k_pairs += 1;

  // finalize: reduce + fold (+ peer scatter) in one cooperative launch
  TcFinal fin;
  memset(&fin, 0, sizeof(fin));
  fin.assign = assign ? 1 : 0;
  fin.n_ranks = 1;
  if (fuse != nullptr && fuse->scatter) {
    fin.n_ranks = ctx->n_ranks; fin.rank = ctx->rank; fin.epoch = fuse->epoch;
    for (int r = 0; r < kMaxRanks; ++r) fin.peers.p[r] = ctx->xchg_peer[r];
  }
  {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(kFinalizeCtas < sms ? kFinalizeCtas : sms);
    cfg.blockDim = dim3(kFinalizeThreads); cfg.dynamicSmemBytes = 0; cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    const double* part_arg = ctx->tc_part; const double* side_arg = ctx->tc_side;
    const float* shift_arg = ctx->shift;
    B2_CUDA(cudaLaunchKernelEx(&cfg, tc_finalize_kernel, part_arg, side_arg, grid, ctx->tc_red, shift_arg, b16 ? 1 : 0, d_in,
                               pack, ctx->S, ctx->tc_sync, fin));
  }
  ctx->launches += 3;
  ctx->k_launches += 3;
  ctx->s_zero_pending = false;
  const bool fused = fuse != nullptr;
  if (n_main < n_in && !fused) {   // the n % pack leftover rows (the fused caller accumulates them first)
    const char* Xt = static_cast<const char*>(X) + (size_t)n_main * ldx_in * es;
    return launch_gram_simt(ctx, Xt, x_dtype, y + n_main, n_in - n_main, d_in, ldx_in,
                            mask != nullptr ? mask + n_main : nullptr, keep);
  }
  return B2_OK;
}

}  // namespace b2
