// gram_narrow.cu -- Gram accumulator for narrow rows (D <= 16): CUDA cores behind a TMA bulk-copy pipeline.
//
// Replaces the pass over the training rows inside LinearRegression.fit (stage_1_train_model.py:105-106) for the
// reference's own shape (one feature, `X.reshape(-1, 1)`, stage_1_train_model.py:95) and its narrow generalisations.
//
// Why not the tcgen05 kernel: a D x D Gram with D <= 16 is 1..17 products per loaded float -- HBM-bound on CUDA
// cores with room to spare -- while zero-padding D to the MMA's M = 128 caps the tensor path at its tile rate
// (0.08 of the HBM roofline at D = 8).  So: stream, do not reshape.
//
// Data flow per CTA (persistent; tiles of kRows contiguous rows, interleaved over the grid):
//
//   HBM --cp.async.bulk (1-D, evict-first; X tile, y tile, row-mask tile)--> smem stage (6 stages, mbarrier full/empty)
//     consumer lane = one row (D <= 8) or half a row (D = 9..16, two lanes share a row and split the products):
//       v = x - c (per-column shift), y' = y - c_y; fp32 FMA into register accumulators
//          sum v_a v_b (a <= b), sum v_a y', sum v_a, sum y'^2, sum y', rows
//     every kFlushRows rows per lane (and at the end): warp butterfly -> per-warp fp64 matrix in smem
//   end: per-CTA fp64 partial (fixed warp order) -> global;  narrow_fold_kernel sums the CTAs in order, undoes the
//   shift in fp64 and adds into the context's raw statistic S = [X 1 y]^T [X 1 y].
//
// Precision: products are fp32 FMAs (round to nearest, 2^-24) of shifted values, chains are at most kFlushRows long
// before they are folded into fp64, and the rounding errors are zero-mean across ~10^5 lanes: the statistic is
// accurate to ~1e-7 relative, coefficient error vs the fp64 oracle ~1e-7 (tests/test_gpu_parity.py).
#include <cuda_bf16.h>

#include "b2_internal.cuh"
#include "b2_ptx.cuh"

namespace b2 {
namespace {

constexpr int kNwStages = 6;
constexpr int kNwMaxDP = 16;
constexpr int kNwM = kNwMaxDP + 2;            // side of the per-CTA partial (features | ones | y)
constexpr int kNwMM = kNwM * kNwM;            // doubles per CTA partial (row stride DP + 2 inside)
constexpr int kNwFlushRows = 2048;            // rows per lane between fp32 -> fp64 folds
constexpr int kNwShiftSamples = 2048;
constexpr int kNwCY = kNwMaxDP;               // slot of c_y in the shift vector

template <int DP>
struct NwGeom {
  static constexpr int TPR = DP > 8 ? 2 : 1;                      // lanes sharing one row
  static constexpr int kConsumerWarps = DP > 8 ? 11 : 7;       // + 1 producer warp = a multiple of 4 warps (ptxas sizes the register cap by that)
  static constexpr int kConsumers = 32 * kConsumerWarps;
  static constexpr int kThreads = kConsumers + 32;                // + the producer warp
  static constexpr int RPT = DP <= 2 ? 4 : (DP == 4 ? 2 : 1);     // rows per lane per stage
  static constexpr int kLaneRows = kConsumers / TPR;              // rows covered by one sweep of the consumers
  static constexpr int kRows = kLaneRows * RPT;                   // rows per stage
  static constexpr int NP = DP > 8 ? 8 : DP;                      // size of the lane's "P" group
  static constexpr int kMinBlocks = DP > 8 ? 1 : 2;
  static constexpr uint32_t kXStage = kRows * DP * 4;             // sized for fp32
  static constexpr uint32_t kYStage = kRows * 4;
  static constexpr uint32_t kMStage = kRows;
  static constexpr uint32_t kOffY = kNwStages * kXStage;
  static constexpr uint32_t kOffM = kOffY + kNwStages * kYStage;
  static constexpr uint32_t kOffBar = kOffM + kNwStages * kMStage;
  static constexpr uint32_t kOffShift = kOffBar + 2 * kNwStages * 8 + 16;         // shift vector (20 floats, 16-byte aligned)
  static constexpr uint32_t kOffAcc = kOffShift + 96;                             // per-warp fp64 matrices
  static constexpr uint32_t kSmem = kOffAcc + kConsumerWarps * (DP + 2) * (DP + 2) * 8 + 128;
};

// butterfly step as a volatile asm: the folds of successive accumulators stay sequential, so the (cold) flush does
// not double the live registers of the (hot) accumulate loop
__device__ __forceinline__ float shfl_bfly_ordered(float v, int off) {
  float r;
  asm volatile("shfl.sync.bfly.b32 %0, %1, %2, 0x1f, 0xffffffff;" : "=f"(r) : "f"(v), "r"(off));
  return r;
}

// ---- per-column shift: mean of a strided sample of the kept rows (any c is algebraically exact, see
// narrow_fold_kernel).  Dropped rows and non-finite values are skipped and the mean divides by what was summed (nothing
// summed: c = 0): a masked-out row may hold anything, and a NaN there must not become c. ----------------------------
template <typename T>
__global__ void narrow_shift_kernel(const T* __restrict__ X, const float* __restrict__ y, const uint8_t* __restrict__ mask,
                                    int keep, int64_t n, int d, float* __restrict__ cvec) {
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;   // warp w: feature w (w < d), warp d: y
  if (w > kNwMaxDP) return;
  if (w > d) { if (lane == 0 && w < kNwMaxDP) cvec[w] = 0.f; return; }
  const int64_t samples = n < kNwShiftSamples ? n : kNwShiftSamples;
  const int64_t stride = n / samples;
  float acc = 0.f, cnt = 0.f;
  for (int64_t s = lane; s < samples; s += 32) {
    const int64_t row = s * stride;
    if (mask != nullptr && mask[row] != (uint8_t)keep) continue;
    const float v = (w < d) ? raw_ld_global<T>(X + row * d + w) : __ldg(y + row);
    if (fabsf(v) <= 3.0e38f) { acc += v; cnt += 1.f; }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    acc += __shfl_xor_sync(0xffffffffu, acc, off);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
  }
  if (lane == 0) {
    cvec[w < d ? w : kNwCY] = cnt > 0.f ? acc / cnt : 0.f;
    if (w == d && d < kNwMaxDP) cvec[d] = 0.f;
  }
}

// ---- packed fp32 pairs: FFMA2 / FADD2 do two lanes of arithmetic per issue slot and are the only way to the full fp32
// rate on sm_100 (a 3-register FFMA issues every other cycle); a pack2(v, v) operand compiles to the scalar-broadcast form
__device__ __forceinline__ uint64_t pack2(float a, float b) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ void unpack2(uint64_t v, float& a, float& b) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}

// ---- the kernel ----------------------------------------------------------------------------------------------
// MODE 2: d == DP (a power of two): vector row loads.  MODE 1: d < DP but the row pitch is a multiple of 16 bytes: the
// same vector loads (they run into the next row), features >= d zeroed.  MODE 0: any d < DP, element loads.
//
// Accumulators are fp32 pairs.  With v the shifted row (features P of this lane, NP of them; Q = NP / 2 pairs):
//   tri2[(b, q)]  += (v_2q, v_2q+1) * v_b      for 2q <= b        -> sum v_a v_b, a <= b (the a = b + 1 lane is a duplicate)
//   py2[q]        += (v_2q, v_2q+1) * y'        p12[q] += (v_2q, v_2q+1)
//   ys2           += (y', 1) * y'               cnt += 1
// and for the two-lane split (D = 9..16; lane half h): P = features 8h..8h+7, plus the cross block
//   ab2[(i, b)]   += (v_2i, v_2i+1) * v_(8+4h+b)   i < 4, b < 4    (features 0..7 against 8+4h..11+4h)
template <typename T, int DP, int MODE>
__global__ void __launch_bounds__(NwGeom<DP>::kThreads, NwGeom<DP>::kMinBlocks)
gram_narrow_kernel(const T* __restrict__ X, const float* __restrict__ y, const uint8_t* __restrict__ mask, int keep,
                   int n_tiles, int d, const float* __restrict__ cvec, double* __restrict__ part) {
  using G = NwGeom<DP>;
  constexpr int TPR = G::TPR, NP = G::NP, RPT = G::RPT;
  constexpr int NQ = NP >= 2 ? NP / 2 : 1;                  // pairs in the P group
  constexpr int NA = TPR == 2 ? 8 : 2, NB = TPR == 2 ? 4 : 1;
  constexpr int NT2 = NP >= 2 ? (NP / 2) * (NP / 2 + 1) : 1;   // sum over b < NP of (b / 2 + 1)
  constexpr int MS = DP + 2;                        // stride of the partial matrix; DP = ones, DP + 1 = y
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const uint32_t sbase = smem_u32(smem_raw);
  const uint32_t bar_full = sbase + G::kOffBar, bar_empty = bar_full + 8 * kNwStages;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool has_mask = mask != nullptr;
  const uint32_t row_bytes = (uint32_t)d * sizeof(T);
  const uint32_t x_bytes = (uint32_t)G::kRows * row_bytes;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kNwStages; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, G::kConsumerWarps);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (warp == G::kConsumerWarps) {
    // ---- producer: one elected lane feeds the ring ----
    if (lane == 0) {
      const uint32_t tx = x_bytes + G::kYStage + (has_mask ? G::kMStage : 0u);
      int it = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
        const int s = it % kNwStages;
        if (it >= kNwStages) mbar_wait(bar_empty + 8 * s, (uint32_t)((it / kNwStages - 1) & 1));
        const uint32_t full = bar_full + 8 * s;
        mbar_expect_tx(full, tx);
        const int64_t row0 = (int64_t)tile * G::kRows;
        bulk_load_1d(sbase + s * G::kXStage, reinterpret_cast<const char*>(X) + (size_t)row0 * row_bytes, x_bytes, full);
        bulk_load_1d(sbase + G::kOffY + s * G::kYStage, y + row0, G::kYStage, full);
        if (has_mask) bulk_load_1d(sbase + G::kOffM + s * G::kMStage, mask + row0, G::kMStage, full);
      }
    }
    return;
  }

  // ---- consumers ----
  const int ctid = threadIdx.x;                    // 0 .. kConsumers-1
  const int h = TPR == 2 ? (lane & 1) : 0;         // which half of the products this lane owns
  const int lrow = ctid / TPR;                     // row of this lane inside one sweep
  const int startP = TPR == 2 ? 8 * h : 0;
  const int startB = 8 + 4 * h;                    // TPR == 2 only

  // minus the shift: registers when a lane owns the whole row; for the two-lane split they would not fit beside the
  // accumulators, so the row loop re-reads them from shared memory (broadcast loads)
  const uint32_t cs = sbase + G::kOffShift;
  if (ctid < 20) reinterpret_cast<float*>(smem_raw + G::kOffShift)[ctid] = ctid <= kNwCY ? -cvec[ctid] : 0.f;
  asm volatile("bar.sync 1, %0;" ::"n"(G::kConsumers) : "memory");
  uint64_t ncP[NQ];
  if constexpr (TPR == 1) {
#pragma unroll
    for (int q = 0; q < NQ; ++q) ncP[q] = pack2(-cvec[2 * q], NP >= 2 ? -cvec[2 * q + 1] : 0.f);
  }
  const float cy = cvec[kNwCY];
  const float cvec_c0 = cvec[0];

  uint64_t tri2[NT2], py2[NQ], p12[NQ], ab2[(NA / 2) * NB], ys2 = 0ull;
  uint64_t y12 = 0ull;                              // DP == 1 only: the pair lanes are two rows (see the row loop)
  float cnt = 0.f;
#pragma unroll
  for (int k = 0; k < NT2; ++k) tri2[k] = 0ull;
#pragma unroll
  for (int k = 0; k < NQ; ++k) { py2[k] = 0ull; p12[k] = 0ull; }
#pragma unroll
  for (int k = 0; k < (NA / 2) * NB; ++k) ab2[k] = 0ull;

  double* Mw = reinterpret_cast<double*>(smem_raw + G::kOffAcc) + warp * (MS * MS);
  for (int k = lane; k < MS * MS; k += 32) Mw[k] = 0.0;
  __syncwarp();

  // fold one fp32 accumulator of every lane into the warp's fp64 matrix (lanes of the same half are summed; the five
  // fp32 butterfly adds are noise next to the <= kNwFlushRows roundings already in the chain)
  auto fold = [&](float v, int idx, bool mine) {
#pragma unroll
    for (int off = 16; off >= TPR; off >>= 1) v += shfl_bfly_ordered(v, off);
    if (lane < TPR && mine) Mw[idx] += (double)v;
  };
  auto fold2 = [&](uint64_t& acc, int idx_lo, int idx_hi, bool hi_valid) {
    float lo, hi;
    unpack2(acc, lo, hi);
    acc = 0ull;
    fold(lo, idx_lo, true);
    if (hi_valid) fold(hi, idx_hi, true);       // hi_valid is a compile-time fact at every call site
  };
  auto flush = [&]() {
    if constexpr (DP == 1) {          // both lanes of every pair carry the same statistic (two rows at a time)
      auto both = [&](uint64_t& acc, int idx) {
        float lo, hi;
        unpack2(acc, lo, hi);
        acc = 0ull;
        fold(lo + hi, idx, true);
      };
      both(tri2[0], 0);
      both(p12[0], DP);
      both(py2[0], DP + 1);
      both(y12, DP * MS + DP + 1);
      both(ys2, (DP + 1) * MS + DP + 1);
      fold(cnt, DP * MS + DP, true);
      cnt = 0.f;
      __syncwarp();
      return;
    }
    int k = 0;
#pragma unroll
    for (int b = 0; b < NP; ++b)
#pragma unroll
      for (int q = 0; q <= b / 2; ++q)
        fold2(tri2[k++], (startP + 2 * q) * MS + startP + b, (startP + 2 * q + 1) * MS + startP + b, 2 * q + 1 <= b);
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
      fold2(p12[q], (startP + 2 * q) * MS + DP, (startP + 2 * q + 1) * MS + DP, NP >= 2);
      fold2(py2[q], (startP + 2 * q) * MS + DP + 1, (startP + 2 * q + 1) * MS + DP + 1, NP >= 2);
    }
    if constexpr (TPR == 2) {
#pragma unroll
      for (int i = 0; i < NA / 2; ++i)
#pragma unroll
        for (int b = 0; b < NB; ++b)
          fold2(ab2[i * NB + b], (2 * i) * MS + startB + b, (2 * i + 1) * MS + startB + b, true);
    }
    float yy, y1;
    unpack2(ys2, yy, y1);
    ys2 = 0ull;
    fold(cnt, DP * MS + DP, h == 0);
    cnt = 0.f;
    fold(y1, DP * MS + DP + 1, h == 0);
    fold(yy, (DP + 1) * MS + DP + 1, h == 0);
    __syncwarp();
  };

  int rows_since_flush = 0;
  int s = 0;
  uint32_t phase = 0;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    mbar_wait(bar_full + 8 * s, phase);
    const uint32_t xs = sbase + s * G::kXStage, ys = sbase + G::kOffY + s * G::kYStage,
                   ms = sbase + G::kOffM + s * G::kMStage;
    if constexpr (DP == 1) {
      // one feature: the two lanes of a pair are two rows, (x, x') and (y, y') -- 8 packed operations per 2 rows
      const uint64_t ncy2 = pack2(-cy, -cy);
#pragma unroll
      for (int rr = 0; rr < RPT; rr += 2) {
        const int r0 = rr * G::kLaneRows + lrow, r1 = r0 + G::kLaneRows;
        float x0[1], x1[1];
        ld_vals_vec<T, 1>(xs + (uint32_t)r0 * (uint32_t)sizeof(T), x0);
        ld_vals_vec<T, 1>(xs + (uint32_t)r1 * (uint32_t)sizeof(T), x1);
        uint64_t Xp = add2(pack2(x0[0], x1[0]), pack2(-cvec_c0, -cvec_c0));
        uint64_t Yp = add2(pack2(ld_shared_f32(ys + 4 * r0), ld_shared_f32(ys + 4 * r1)), ncy2);
        if (has_mask) {
          const bool u0 = ld_shared_u8(ms + r0) == (uint32_t)keep, u1 = ld_shared_u8(ms + r1) == (uint32_t)keep;
          float a, b, e, f;
          unpack2(Xp, a, b);
          unpack2(Yp, e, f);
          Xp = pack2(u0 ? a : 0.f, u1 ? b : 0.f);
          Yp = pack2(u0 ? e : 0.f, u1 ? f : 0.f);
          cnt += (u0 ? 1.f : 0.f) + (u1 ? 1.f : 0.f);
        } else {
          cnt += 2.f;
        }
        tri2[0] = fma2(Xp, Xp, tri2[0]);
        py2[0] = fma2(Xp, Yp, py2[0]);
        p12[0] = add2(p12[0], Xp);
        ys2 = fma2(Yp, Yp, ys2);
        y12 = add2(y12, Yp);
      }
    } else {
#pragma unroll
    for (int rr = 0; rr < RPT; ++rr) {
      const int r = rr * G::kLaneRows + lrow;
      const bool use = !has_mask || ld_shared_u8(ms + r) == (uint32_t)keep;
      const uint32_t row_addr = xs + (uint32_t)r * row_bytes;
      float P[NP], A[NA], B[NB];
      if constexpr (MODE >= 1) {
        ld_vals_vec<T, NP>(row_addr + startP * (uint32_t)sizeof(T), P);
        if constexpr (TPR == 2) {
          ld_vals_vec<T, NA>(row_addr, A);
          ld_vals_vec<T, NB>(row_addr + startB * (uint32_t)sizeof(T), B);
        }
        if constexpr (MODE == 1) {
#pragma unroll
          for (int k = 0; k < NP; ++k) P[k] = startP + k < d ? P[k] : 0.f;
          if constexpr (TPR == 2) {
#pragma unroll
            for (int k = 0; k < NA; ++k) A[k] = k < d ? A[k] : 0.f;
#pragma unroll
            for (int k = 0; k < NB; ++k) B[k] = startB + k < d ? B[k] : 0.f;
          }
        }
      } else {
        ld_vals_any<T, NP>(row_addr, startP, d, P);
        if constexpr (TPR == 2) {
          ld_vals_any<T, NA>(row_addr, 0, d, A);
          ld_vals_any<T, NB>(row_addr, startB, d, B);
        }
      }
      const float yv = ld_shared_f32(ys + 4 * r) - cy;
      if (use) {
        // shifted values as pairs (and, aliased, as scalars for the broadcast operand)
        uint64_t Pp[NQ];
        if constexpr (TPR == 1) {
#pragma unroll
          for (int q = 0; q < NQ; ++q) Pp[q] = add2(pack2(P[2 * q], NP >= 2 ? P[2 * q + 1] : 0.f), ncP[q]);
        } else {
          float c8[8];
          ld_vals_vec<float, 8>(cs + startP * 4u, c8);
#pragma unroll
          for (int q = 0; q < NQ; ++q) Pp[q] = add2(pack2(P[2 * q], P[2 * q + 1]), pack2(c8[2 * q], c8[2 * q + 1]));
        }
        float v[2 * NQ];
#pragma unroll
        for (int q = 0; q < NQ; ++q) unpack2(Pp[q], v[2 * q], v[2 * q + 1]);
        int k = 0;
#pragma unroll
        for (int b = 0; b < NP; ++b) {
          const uint64_t vb = pack2(v[b], v[b]);
#pragma unroll
          for (int q = 0; q <= b / 2; ++q) { tri2[k] = fma2(Pp[q], vb, tri2[k]); ++k; }
        }
        const uint64_t yb = pack2(yv, yv);
#pragma unroll
        for (int q = 0; q < NQ; ++q) { py2[q] = fma2(Pp[q], yb, py2[q]); p12[q] = add2(p12[q], Pp[q]); }
        if constexpr (TPR == 2) {
          float cA[8], cB[4];
          ld_vals_vec<float, 8>(cs, cA);
          ld_vals_vec<float, 4>(cs + startB * 4u, cB);
          uint64_t Ap[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) Ap[i] = add2(pack2(A[2 * i], A[2 * i + 1]), pack2(cA[2 * i], cA[2 * i + 1]));
#pragma unroll
          for (int b = 0; b < NB; ++b) {
            const float vbs = B[b] + cB[b];
            const uint64_t vb = pack2(vbs, vbs);
#pragma unroll
            for (int i = 0; i < 4; ++i) ab2[i * NB + b] = fma2(Ap[i], vb, ab2[i * NB + b]);
          }
        }
        ys2 = fma2(pack2(yv, 1.f), yb, ys2);
        cnt += 1.f;
      }
    }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(bar_empty + 8 * s);
    if (++s == kNwStages) { s = 0; phase ^= 1u; }
    rows_since_flush += RPT;
    if (rows_since_flush >= kNwFlushRows) { flush(); rows_since_flush = 0; }
  }
  flush();

  // ---- per-CTA partial: warps summed in a fixed order ----
  asm volatile("bar.sync 1, %0;" ::"n"(G::kConsumers) : "memory");
  const double* M0 = reinterpret_cast<const double*>(smem_raw + G::kOffAcc);
  double* out = part + (size_t)blockIdx.x * kNwMM;
  for (int k = ctid; k < MS * MS; k += G::kConsumers) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < G::kConsumerWarps; ++w) t += M0[w * (MS * MS) + k];
    out[k] = t;
  }
}

// ---- finalize: sum the CTA partials in order, undo the shift in fp64, S += ------------------------------------
// m(i, j), i <= j over internal indices (features 0..DP-1, DP = ones, DP + 1 = y'), row stride DP + 2.
__global__ void __launch_bounds__(384)
narrow_fold_kernel(const double* __restrict__ part, int n_ctas, int DP, int d, const float* __restrict__ cvec,
                   double* __restrict__ S) {
  __shared__ double m[kNwMM];
  const int MS = DP + 2;
  for (int k = threadIdx.x; k < MS * MS; k += blockDim.x) {
    double s0 = 0.0, s1 = 0.0;
    int c = 0;
    for (; c + 1 < n_ctas; c += 2) { s0 += part[(size_t)c * kNwMM + k]; s1 += part[(size_t)(c + 1) * kNwMM + k]; }
    if (c < n_ctas) s0 += part[(size_t)c * kNwMM + k];
    m[k] = s0 + s1;
  }
  __syncthreads();
  const int dp = d + 2;
  auto M = [&](int i, int j) { return i <= j ? m[i * MS + j] : m[j * MS + i]; };
  const int ONE = DP, Y = DP + 1;
  const double n = M(ONE, ONE), sy = M(ONE, Y), syy = M(Y, Y), cy = (double)cvec[kNwCY];
  for (int idx = threadIdx.x; idx < dp * dp; idx += blockDim.x) {
    const int r = idx / dp, q = idx % dp;
    const int a = r < q ? r : q, b = r < q ? q : r;   // (a, b) and (b, a) evaluate the same expression: S stays bit-symmetric
    double val;
    if (b < d) {
      const double ca = (double)cvec[a], cb = (double)cvec[b];
      val = M(a, b) + ca * M(b, ONE) + cb * M(a, ONE) + n * ca * cb;
    } else if (a < d) {
      const double ci = (double)cvec[a];
      if (b == d) val = M(a, ONE) + n * ci;
      else val = M(a, Y) + cy * M(a, ONE) + ci * sy + n * ci * cy;
    } else if (a == d && b == d) {
      val = n;
    } else if (a == d + 1) {
      val = syy + 2.0 * cy * sy + n * cy * cy;
    } else {
      val = sy + n * cy;
    }
    S[idx] += val;
  }
}

template <typename T, int DP>
int launch_narrow_dp(b2_ctx* ctx, const T* X, const float* y, const uint8_t* mask, int keep, int n_tiles, int d,
                     int* grid_out) {
  using G = NwGeom<DP>;
  const int mode = d == DP ? 2 : ((d * (int)sizeof(T)) % 16 == 0 ? 1 : 0);
  const int cap = ctx->sm_count * G::kMinBlocks;
  const int grid = n_tiles < cap ? n_tiles : cap;
  *grid_out = grid;
#define B2_LAUNCH_NW(MODE)                                                                                          \
  do {                                                                                                              \
    B2_CUDA(cudaFuncSetAttribute(gram_narrow_kernel<T, DP, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,      \
                                 G::kSmem));                                                                        \
    gram_narrow_kernel<T, DP, MODE><<<grid, G::kThreads, G::kSmem, ctx->stream>>>(X, y, mask, keep, n_tiles, d,     \
                                                                                  ctx->shift, ctx->simt_part);      \
  } while (0)
  if (mode == 2) {
    B2_LAUNCH_NW(2);
  } else if (mode == 1) {
    if constexpr (DP == 16 && sizeof(T) == 4) B2_LAUNCH_NW(1);   // fp32 d = 12 is the only such shape
    else B2_LAUNCH_NW(0);
  } else {
    B2_LAUNCH_NW(0);
  }
#undef B2_LAUNCH_NW
  B2_CUDA(cudaGetLastError());
  return B2_OK;
}

template <typename T>
int launch_narrow_t(b2_ctx* ctx, const T* X, const float* y, const uint8_t* mask, int keep, int64_t n, int d,
                    int64_t* rows_done) {
  const int DP = d <= 1 ? 1 : d <= 2 ? 2 : d <= 4 ? 4 : d <= 8 ? 8 : 16;
  const int rows = DP == 1 ? NwGeom<1>::kRows : DP == 2 ? NwGeom<2>::kRows : DP == 4 ? NwGeom<4>::kRows
                 : DP == 8 ? NwGeom<8>::kRows : NwGeom<16>::kRows;
  const int n_tiles = (int)(n / rows);            // n <= INT32_MAX rows (gram_narrow_supported)
  *rows_done = (int64_t)n_tiles * rows;
  if (n_tiles == 0) return B2_OK;
  narrow_shift_kernel<T><<<1, 32 * (kNwMaxDP + 1), 0, ctx->stream>>>(X, y, mask, keep, n, d, ctx->shift);
  B2_CUDA(cudaGetLastError());
  const int pair = ctx->k_pairs % kKernelEventPairs;
  B2_CUDA(cudaEventRecord(ctx->ev_k[pair][0], ctx->stream));
  int grid = 0, rc = B2_OK;
  switch (DP) {
    case 1: rc = launch_narrow_dp<T, 1>(ctx, X, y, mask, keep, n_tiles, d, &grid); break;
    case 2: rc = launch_narrow_dp<T, 2>(ctx, X, y, mask, keep, n_tiles, d, &grid); break;
    case 4: rc = launch_narrow_dp<T, 4>(ctx, X, y, mask, keep, n_tiles, d, &grid); break;
    case 8: rc = launch_narrow_dp<T, 8>(ctx, X, y, mask, keep, n_tiles, d, &grid); break;
    default: rc = launch_narrow_dp<T, 16>(ctx, X, y, mask, keep, n_tiles, d, &grid); break;
  }
  if (rc != B2_OK) return rc;
  B2_CUDA(cudaEventRecord(ctx->ev_k[pair][1], ctx->stream));
  ctx->k_pairs += 1;
  narrow_fold_kernel<<<1, 384, 0, ctx->stream>>>(ctx->simt_part, grid, DP, d, ctx->shift, ctx->S);
  B2_CUDA(cudaGetLastError());
  ctx->launches += 3;
  ctx->k_launches += 3;
  return B2_OK;
}

}  // namespace

// rows contiguous (ldx == d), X / y / mask 16-byte aligned; full tiles here, the < kRows leftover rows on the fp64 kernel
bool gram_narrow_supported(const void* X, int x_dtype, const float* y, int64_t n, int d, int64_t ldx,
                           const uint8_t* mask) {
  (void)x_dtype;
  if (d < 1 || d > kNwMaxDP || ldx != d || n < 1 || n > (int64_t)0x7fffffff) return false;
  if ((reinterpret_cast<uintptr_t>(X) & 15) != 0 || (reinterpret_cast<uintptr_t>(y) & 15) != 0) return false;
  if (mask != nullptr && (reinterpret_cast<uintptr_t>(mask) & 15) != 0) return false;
  return true;
}

int launch_gram_narrow(b2_ctx* ctx, const void* X, int x_dtype, const float* y, int64_t n, int d, int64_t ldx,
                       const uint8_t* mask, int keep) {
  static_assert(2 * kNwMM <= kMaxS * kMaxS, "two CTAs per SM of partials fit the CUDA-core scratch (simt_part)");
  int64_t done = 0;
  int rc;
  if (x_dtype == B2_F32)
    rc = launch_narrow_t<float>(ctx, static_cast<const float*>(X), y, mask, keep, n, d, &done);
  else
    rc = launch_narrow_t<__nv_bfloat16>(ctx, static_cast<const __nv_bfloat16*>(X), y, mask, keep, n, d, &done);
  if (rc != B2_OK) return rc;
  if (done < n) {
    const int es = x_dtype == B2_F32 ? 4 : 2;
    const char* Xt = static_cast<const char*>(X) + (size_t)done * ldx * es;
    return launch_gram_simt(ctx, Xt, x_dtype, y + done, n - done, d, ldx, mask != nullptr ? mask + done : nullptr, keep);
  }
  return B2_OK;
}

}  // namespace b2
