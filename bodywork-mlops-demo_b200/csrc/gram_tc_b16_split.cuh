// gram_tc_b16_split.cuh -- bf16-stored rows, D = 128, DEFAULT hi + lo operand mode (16 mantissa bits per operand).
// Included by gram_tc.cu after gram_tc_b16.cuh (helpers: ldmatrix / tcgen05.st.16x128b / mixed-precision FMA wrappers).
//
// Same front end as the single-operand kernel (swizzled TMA boxes -> ldmatrix.x4.trans -> A operands into tensor memory),
// but the B operand is the CENTRED hi, written to shared memory in the K-major canonical layout (one STS.32 per pair, a
// warp writes a whole 128-byte core matrix): with the raw tile as B (the single-operand kernel's trick) every accumulator
// entry carries c_j * sum_r v_i, and the fp32 truncation of that term costs a factor 3 in coefficient accuracy
// (3.6e-5 instead of 1.2e-5 at 1 M rows) -- acceptable when the operand itself has 8 bits, not in the 16-bit mode.
//   The operand stage holds [E | hi | E] per 8-row K group (two copies of the 16 E columns around the 128 hi columns), the
//   accumulator is 160 columns [Ea | G | Eb], and both MMAs of a K = 16 step have the SAME shape (M 128, N 144):
//       [G | Eb] += hi^T     [hi | E]      B descriptor starts at hi, D at column 16
//       [Ea | G] += (2 lo)^T [E | hi]      B descriptor starts at the first E copy, D at column 0
//   so G = hi.hi + 2 lo.hi in ONE accumulator, Eb = hi^T E, Ea = 2 lo^T E.  One accumulator is enough because the fold
//   symmetrises: 0.5 (G[a][b] + G[b][a]) = hi.hi + lo.hi + hi.lo, which is what tc_fold_value computes from the partials
//   (this kernel writes [G | Eb] into the "A = hi" half of the partial, zeros and 0.5 Ea into the "A = lo" half).  Same
//   flops as the generic kernel's two MMAs, and the 144 tensor-memory columns that a second full accumulator would take
//   hold a three-deep ring of both A operands instead.
//   lo arithmetic: 2 lo = rn(2x - 2c - 2 hi) with two mixed-precision FMAs per element (fma.rn.f32.bf16).
#pragma once

namespace b16 {
namespace sp {

constexpr int kRaw = 6;                                   // raw tile stages (16 KB each)
constexpr int kOpsMax = 3;                                // operand stages: smem B ring + tensor-memory A rings (192 columns)
constexpr uint32_t kRawBytes = kTcRows * 128 * 2;         // 16384
constexpr uint32_t kRawHalf = kTcRows * 128;              // 8192: one [64][64] bf16 box
constexpr uint32_t kLBO = (2 + 16 + 2) * kOpSBO;          // 2560: E | hi | E groups per 8-row K group
constexpr uint32_t kHiOff = 2 * kOpSBO;                   // hi groups inside a K group
constexpr uint32_t kE1Off = (2 + 16) * kOpSBO;            // the E copy behind hi (B = [hi | E])
constexpr uint32_t kOpBytes = kKGroups * kLBO;            // 20480
constexpr uint32_t kOffRaw = 0;
constexpr uint32_t kOffOp = kOffRaw + kRaw * kRawBytes;   // 98304
constexpr uint32_t kOffY = kOffOp + kOpsMax * kOpBytes;   // 159744
constexpr uint32_t kYBytes = kTcRows * 4;                 // 256
constexpr uint32_t kMBytes = 128;                         // 64 mask bytes, padded (TMA destinations are 128-byte aligned)
constexpr uint32_t kOffMask = kOffY + kRaw * kYBytes;
constexpr uint32_t kOffBar = kOffMask + kRaw * kMBytes;
constexpr int kBars = 2 * kRaw + 2 * kOpsMax + 4;
constexpr uint32_t kOffTmemPtr = kOffBar + kBars * 8;
constexpr uint32_t kOffShift = kOffTmemPtr + 16;
constexpr uint32_t kSmem = kOffShift + (kMaxD + 4) * 4 + 1024;
static_assert(kSmem <= 227 * 1024, "shared memory budget");
// tensor memory: accumulator [Ea 16 | G 128 | Eb 16] double buffered at 0 / 160, A = hi ring at 320 + 32 s, A = 2 lo ring
// at 416 + 32 s
constexpr uint32_t kAccStride = 160;
constexpr uint32_t kTmemAHi = 320;
constexpr uint32_t kTmemALo = 416;

// K-major operand of this kernel: instruction descriptor without the B-transpose bit
__host__ __device__ constexpr uint32_t idesc_k(int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kTcM >> 4) << 24);
}
__device__ __forceinline__ void tmem_st16_zero(uint32_t taddr) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};"
               ::"r"(taddr), "r"(0u) : "memory");
}

// One tile of the issue thread in a single asm block: 8 MMAs (stage OS), the commit that frees the stage, and -- after
// the first K step -- a NON-BLOCKING probe of the next tile's `full` barrier whose result is consumed only after the last
// MMA: mbarrier.test_wait takes 150-250 cycles here, and every cycle this thread waits between two MMAs is a cycle the
// tensor core idles (tools/ubench_umma.cu), so the probe has to be in flight while the MMAs issue.
template <uint32_t DESC_HI, uint32_t IDESC>
__device__ __forceinline__ bool issue_tile(uint32_t tmem_acc, uint32_t tmem_a, uint32_t desc_hi, uint32_t desc_e,
                                           uint32_t first_accumulates, uint32_t bar_empty, uint32_t bar_next, uint32_t par_next) {
  uint32_t ready;
  constexpr uint32_t kSK = (uint32_t)((2 * kLBO) >> 4);          // descriptor step of one K = 16 step
  asm volatile(
      "{\n\t"
      ".reg .pred pa, pt, pr;\n\t"
      ".reg .b32 dl, ta, td;\n\t"
      ".reg .b64 dd;\n\t"
      "setp.ne.b32 pa, %4, 0;\n\t"
      "setp.eq.b32 pt, %4, %4;\n\t"
      "add.u32 td, %1, 16;\n\t"
      // K step 0
      "mov.b64 dd, {%2, %9};\n\t add.u32 ta, %5, %11;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [td], [ta], dd, %10, pa;\n\t"
      "mov.b64 dd, {%3, %9};\n\t add.u32 ta, %5, %15;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%1], [ta], dd, %10, pt;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 pr, [%6], %7;\n\t"
      // K step 1
      "add.u32 dl, %2, %19;\n\t mov.b64 dd, {dl, %9};\n\t add.u32 ta, %5, %12;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [td], [ta], dd, %10, pt;\n\t"
      "add.u32 dl, %3, %19;\n\t mov.b64 dd, {dl, %9};\n\t add.u32 ta, %5, %16;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%1], [ta], dd, %10, pt;\n\t"
      // K step 2
      "add.u32 dl, %2, %20;\n\t mov.b64 dd, {dl, %9};\n\t add.u32 ta, %5, %13;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [td], [ta], dd, %10, pt;\n\t"
      "add.u32 dl, %3, %20;\n\t mov.b64 dd, {dl, %9};\n\t add.u32 ta, %5, %17;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%1], [ta], dd, %10, pt;\n\t"
      // K step 3
      "add.u32 dl, %2, %21;\n\t mov.b64 dd, {dl, %9};\n\t add.u32 ta, %5, %14;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [td], [ta], dd, %10, pt;\n\t"
      "add.u32 dl, %3, %21;\n\t mov.b64 dd, {dl, %9};\n\t add.u32 ta, %5, %18;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%1], [ta], dd, %10, pt;\n\t"
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%8];\n\t"
      "selp.u32 %0, 1, 0, pr;\n\t"
      "}"
      : "=r"(ready)
      : "r"(tmem_acc), "r"(desc_hi), "r"(desc_e), "r"(first_accumulates), "r"(tmem_a), "r"(bar_next), "r"(par_next),
        "r"(bar_empty), "n"(DESC_HI), "n"(IDESC),
        "n"(kTmemAHi), "n"(kTmemAHi + 8), "n"(kTmemAHi + 16), "n"(kTmemAHi + 24),
        "n"(kTmemALo), "n"(kTmemALo + 8), "n"(kTmemALo + 16), "n"(kTmemALo + 24),
        "n"(kSK), "n"(2 * kSK), "n"(3 * kSK)
      : "memory");
  return ready != 0;
}

__global__ void __launch_bounds__(kThreads, 1)
gram_b16_split_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmY,
                const __grid_constant__ CUtensorMap tmM, int y_map_2d, int has_mask, int keep, int64_t n_rows,
                const float* __restrict__ shift, int chunk_tiles, double* __restrict__ part,
                double* __restrict__ side) {
  constexpr int kOps = 3;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (sbase - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  const uint32_t bar_raw_full = sbase + kOffBar;                 // [kRaw]
  const uint32_t bar_raw_empty = bar_raw_full + 8 * kRaw;        // [kRaw]
  const uint32_t bar_op_full = bar_raw_empty + 8 * kRaw;         // [kOps]
  const uint32_t bar_op_empty = bar_op_full + 8 * kOpsMax;       // [kOps]
  const uint32_t bar_acc_full = bar_op_empty + 8 * kOpsMax;      // [2]
  const uint32_t bar_acc_empty = bar_acc_full + 16;              // [2]
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem + kOffTmemPtr);
  float* shift_s = reinterpret_cast<float*>(smem + kOffShift);

  const int64_t total_tiles = (n_rows + kTcRows - 1) / kTcRows;
  const int64_t tile_begin = (int64_t)blockIdx.x * total_tiles / gridDim.x;
  const int64_t tile_end = (int64_t)(blockIdx.x + 1) * total_tiles / gridDim.x;
  const int my_tiles = (int)(tile_end - tile_begin);
  const int n_chunks = (my_tiles + chunk_tiles - 1) / chunk_tiles;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kRaw; ++s) {
      mbar_init(bar_raw_full + 8 * s, 1);
      mbar_init(bar_raw_empty + 8 * s, kProducers);
    }
    for (int s = 0; s < kOps; ++s) {
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
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(sbase + kOffTmemPtr) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // the unused E rows of the operand stages read as 0
  for (uint32_t o = threadIdx.x * 16; o < kOpsMax * kOpBytes; o += kThreads * 16)
    *reinterpret_cast<uint4*>(smem + kOffOp + o) = make_uint4(0, 0, 0, 0);
  for (int j = threadIdx.x; j <= kMaxD; j += kThreads) shift_s[j] = shift_value(shift, j, j < kMaxD);   // c_y: fp32
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  if (warp >= 4 && warp < 8) {     // Ea is only ever accumulated into (the first MMA of a chunk initialises [G | Eb])
    tmem_st16_zero(tmem_base + ((uint32_t)((warp & 3) * 32) << 16));
    tmem_st16_zero(tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + kAccStride);
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  if (warp == 0) {
    // ===== TMA producer (the whole warp runs the loop, one elected lane issues) =====
    const uint32_t tx = kRawBytes + kTcRows * 4 + (has_mask ? kTcRows : 0);
    int s = 0;
    uint32_t ph = 0;
    for (int it = 0; it < my_tiles; ++it) {
      wait_lean(bar_raw_empty + 8 * s, ph ^ 1);
      if (elect_one()) {
        const uint32_t full = bar_raw_full + 8 * s;
        mbar_expect_tx(full, tx);
        const int row0 = (int)((tile_begin + it) * kTcRows);
        tma_load_2d(sbase + kOffRaw + s * kRawBytes, &tmX, 0, row0, full);
        tma_load_2d(sbase + kOffRaw + s * kRawBytes + kRawHalf, &tmX, 64, row0, full);
        if (y_map_2d) tma_load_2d(sbase + kOffY + s * kYBytes, &tmY, 0, row0 >> 2, full);
        else tma_load_1d(sbase + kOffY + s * kYBytes, &tmY, row0, full);
        if (has_mask == 2) tma_load_2d(sbase + kOffMask + s * kMBytes, &tmM, 0, row0 >> 4, full);
        else if (has_mask) tma_load_1d(sbase + kOffMask + s * kMBytes, &tmM, row0, full);
      }
      __syncwarp();
      if (++s == kRaw) { s = 0; ph ^= 1; }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: ONE elected thread runs the whole loop.  The tensor core does not queue: every cycle the issuing
    // thread spends between two tcgen05.mma beyond ~one MMA time is a cycle the tensor core idles (tools/ubench_umma.cu).
    // So the loop is unrolled over the operand stages (descriptors, tensor-memory and barrier addresses are constants
    // off loop-invariant registers) and the readiness of the NEXT tile is probed between the MMAs of the current one =====
    if (elect_one()) {
      uint32_t oph = 0;
      int in_chunk = 0, chunk = 0, it = 0;
      bool ready = false;
      const uint32_t desc_e0 = (uint32_t)make_smem_desc(sbase + kOffOp, kLBO), desc_hi0 = (uint32_t)make_smem_desc(sbase + kOffOp + kHiOff, kLBO);
      constexpr uint32_t kDescHi = (uint32_t)((((uint64_t)(kOpSBO >> 4) << 32) | (1ull << 46)) >> 32);   // high word: constant
      while (it < my_tiles) {
#pragma unroll
        for (int os = 0; os < kOps; ++os) {
          if (it < my_tiles) {
            const int b = chunk & 1;
            if (in_chunk == 0) wait_lean(bar_acc_empty + 8 * b, ((chunk >> 1) & 1) ^ 1);
            if (!ready) wait_lean(bar_op_full + 8 * os, oph);
            tc_fence_after();
            const bool last = (in_chunk == chunk_tiles - 1) || (it == my_tiles - 1);
            const uint32_t tmem_acc = tmem_base + (uint32_t)b * kAccStride;
            const int osn = (os + 1 == kOps) ? 0 : os + 1;
            const uint32_t ophn = (os + 1 == kOps) ? (oph ^ 1u) : oph;
            // descriptors of other stages / K steps differ by a constant in the address field (no carry: addresses < 2^18)
            ready = issue_tile<kDescHi, idesc_k(144)>(tmem_acc, tmem_base + (uint32_t)(os * 32), desc_hi0 + (uint32_t)((os * kOpBytes) >> 4),
                                                     desc_e0 + (uint32_t)((os * kOpBytes) >> 4), in_chunk > 0 ? 1u : 0u,
                                                     bar_op_empty + 8 * os, bar_op_full + 8 * osn, ophn);
            if (last) { umma_commit(bar_acc_full + 8 * b); in_chunk = 0; ++chunk; }
            else ++in_chunk;
            ++it;
          }
        }
        oph ^= 1;
      }
    }
    __syncwarp();
  } else if (warp == 2 || warp == 3) {
    // ===== E warps: operand columns [1, y'_hi, y'_lo] and the CUDA-core sums of y' (one row per lane) =====
    const float c_y = shift_s[kMaxD];
    double sy = 0.0, syy = 0.0, cnt = 0.0;
    int rs = 0, os = 0;
    uint32_t rph = 0, oph = 0;
    const int rr = lane + 32 * (warp - 2);
    for (int it = 0; it < my_tiles; ++it) {
      wait_lean2(bar_raw_full + 8 * rs, rph, bar_op_empty + 8 * os, oph ^ 1);
      tc_fence_after();
      const int64_t left = n_rows - (tile_begin + it) * kTcRows;
      bool use = rr < left;
      if (use && has_mask) use = (ld_shared_u8(sbase + kOffMask + rs * kMBytes + rr) == (uint32_t)keep);
      const float yv = use ? ld_shared_f32(sbase + kOffY + rs * kYBytes + rr * 4) - c_y : 0.f;
      uint32_t yh, yl;
      split2(yv, 0.f, yh, yl);
      const uint32_t dst = sbase + kOffOp + os * kOpBytes + (rr >> 3) * kLBO + (rr & 7) * 2;
      st_shared_u16(dst + kE1Off, use ? 0x3F80u : 0u);
      st_shared_u16(dst + kE1Off + 16, yh);
      st_shared_u16(dst + kE1Off + 32, yl);
      {                  // the copy in front of hi: B = [E | hi] of the A = 2 lo MMA
        st_shared_u16(dst, use ? 0x3F80u : 0u);
        st_shared_u16(dst + 16, yh);
        st_shared_u16(dst + 32, yl);
      }
      sy += (double)yv; syy += (double)(yv * yv); cnt += use ? 1.0 : 0.0;
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(bar_op_full + 8 * os);
        mbar_arrive(bar_raw_empty + 8 * rs);
      }
      if (++rs == kRaw) { rs = 0; rph ^= 1; }
      if (++os == kOps) { os = 0; oph ^= 1; }
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
  } else if (warp < 8) {
    // ===== epilogue: TMEM -> fp64 partial in global (column-major [col][feature]) =====
    const int w = warp & 3;
    double* my_part = part + (size_t)blockIdx.x * kTcAccElems + w * 32 + lane;
    const uint32_t lane_base = tmem_base + ((uint32_t)(w * 32) << 16);
    for (int chunk = 0; chunk < n_chunks; ++chunk) {
      const int b = chunk & 1;
      wait_lean(bar_acc_full + 8 * b, (chunk >> 1) & 1);
      tc_fence_after();
      // accumulator columns [Ea | G | Eb] -> partial columns: G, Eb -> [0, 144) (the "A = hi" half), 0.5 Ea -> the E
      // columns of the "A = lo" half
#pragma unroll 1
      for (int p = 0; p < (int)kAccStride / 16; ++p) {
        uint32_t r[16];
        tmem_ld16(lane_base + (uint32_t)b * kAccStride + (uint32_t)(p * 16), r);
        tmem_ld_wait();
        double* dst = my_part + (size_t)(p == 0 ? kTcN + 128 : (p - 1) * 16) * kTcM;
        const double scale = p == 0 ? 0.5 : 1.0;
        if (chunk == 0) {
#pragma unroll
          for (int j = 0; j < 16; ++j) dst[(size_t)j * kTcM] = scale * (double)__uint_as_float(r[j]);
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) dst[(size_t)j * kTcM] += scale * (double)__uint_as_float(r[j]);
        }
      }
      {                  // Ea starts the next chunk of this buffer from zero
        tmem_st16_zero(lane_base + (uint32_t)b * kAccStride);
        tmem_st_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_acc_empty + 8 * b);
    }
    // the rest of the "A = lo" half: lo.hi is already inside G (twice: the fold halves the symmetrised sum)
#pragma unroll 1
    for (int p = 0; p < kTcN / 16 - 1; ++p) {
      double* dst = my_part + (size_t)(kTcN + p * 16) * kTcM;
#pragma unroll
      for (int j = 0; j < 16; ++j) dst[(size_t)j * kTcM] = 0.0;
    }
  } else {
    // ===== transform: warp (q, s) owns features 32q .. 32q+31 (its tensor-memory lane quadrant) x rows 16s .. 16s+15 =====
    const int t = warp - 8;
    const int q = t & 3, s = t >> 2;
    const int j4 = lane & 3, f8 = lane >> 2;
    // ldmatrix row address of lane L: matrix b = L / 8 (features 32q + 8b ..), row L % 8 of the 8-row group; the 16-byte
    // chunk index is XORed with the row (SWIZZLE_128B; the rows of a box are 128 bytes apart)
    const uint32_t lm_off = (uint32_t)(q >> 1) * kRawHalf + (uint32_t)(lane & 7) * 128u +
                            ((uint32_t)((4 * (q & 1) + (lane >> 3)) ^ (lane & 7)) << 4);
    uint32_t cc[4];      // (c, c) as packed bf16 of this thread's four features 32q + 8b + lane/4
    float m2c[4];        // -2 c
    constexpr uint32_t kTwo = 0x40004000u, kMinusTwo = 0xC000C000u;      // bf16 pairs (2, 2) and (-2, -2)
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const float c = shift_s[32 * q + 8 * b + f8];
      const __nv_bfloat162 cp = __floats2bfloat162_rn(c, c);     // exact: c is bf16-representable
      cc[b] = *reinterpret_cast<const uint32_t*>(&cp);
      m2c[b] = -2.f * c;
    }
    const uint32_t st_off = (uint32_t)(2 * s) * kLBO + kHiOff + (uint32_t)(4 * q) * kOpSBO + (uint32_t)lane * 4u;
    const uint32_t tm_lane = tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(8 * s);
    int rs = 0, os = 0;
    uint32_t rph = 0, oph = 0;
    for (int it = 0; it < my_tiles; ++it) {
      wait_lean2(bar_raw_full + 8 * rs, rph, bar_op_empty + 8 * os, oph ^ 1);
      tc_fence_after();
      const uint32_t raw_addr = sbase + kOffRaw + rs * kRawBytes + lm_off + (uint32_t)(2 * s) * 1024u;
      uint32_t R[2][4];
      ldsm_x4_trans(raw_addr, R[0]);
      ldsm_x4_trans(raw_addr + 1024u, R[1]);
      const int64_t left = n_rows - (tile_begin + it) * kTcRows;
      uint32_t H[2][4], L[2][4];
#pragma unroll
      for (int g = 0; g < 2; ++g) {
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          const uint32_t raw = R[g][b];
          const uint32_t hp = sub_bf16x2(raw, cc[b]);                  // hi = rn(x - c), both rows of the pair
          H[g][b] = hp;
          {
            // 2 lo = rn(2x - 2c - 2 hi): both FMAs are exact in fp32 (lo has at most 16 significant bits)
            const float l0 = fma_bf16_lo(hp, kMinusTwo, fma_bf16_lo(raw, kTwo, m2c[b]));
            const float l1 = fma_bf16_hi(hp, kMinusTwo, fma_bf16_hi(raw, kTwo, m2c[b]));
            const __nv_bfloat162 lp = __floats2bfloat162_rn(l0, l1);
            L[g][b] = *reinterpret_cast<const uint32_t*>(&lp);
          }
        }
      }
      if (has_mask || left < kTcRows) {          // rows 16s + 8g + 2 j4 (low half of the pair) and + 1 (high half)
        const uint32_t m_addr = sbase + kOffMask + rs * kMBytes;
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          const int r0 = 16 * s + 8 * g + 2 * j4;
          bool u0 = r0 < left, u1 = (r0 + 1) < left;
          if (has_mask) {
            u0 = u0 && (ld_shared_u8(m_addr + r0) == (uint32_t)keep);
            u1 = u1 && (ld_shared_u8(m_addr + r0 + 1) == (uint32_t)keep);
          }
          const uint32_t keep32 = (u0 ? 0x0000ffffu : 0u) | (u1 ? 0xffff0000u : 0u);
#pragma unroll
          for (int b = 0; b < 4; ++b) {
            H[g][b] &= keep32;
            L[g][b] &= keep32;
          }
        }
      }
#pragma unroll
      for (int g = 0; g < 2; ++g) {
#pragma unroll
        for (int b = 0; b < 4; ++b)
          st_shared_b32(sbase + kOffOp + os * kOpBytes + st_off + (uint32_t)g * kLBO + (uint32_t)b * kOpSBO, H[g][b]);
      }
      const uint32_t ta = tm_lane + (uint32_t)(os * 32);
      tmem_st_16x128b_x2(ta + kTmemAHi, H[0][0], H[0][1], H[1][0], H[1][1]);
      tmem_st_16x128b_x2(ta + kTmemAHi + (16u << 16), H[0][2], H[0][3], H[1][2], H[1][3]);
      {
        tmem_st_16x128b_x2(ta + kTmemALo, L[0][0], L[0][1], L[1][0], L[1][1]);
        tmem_st_16x128b_x2(ta + kTmemALo + (16u << 16), L[0][2], L[0][3], L[1][2], L[1][3]);
      }
      tmem_st_wait();
      tc_fence_before();
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(bar_op_full + 8 * os);
        mbar_arrive(bar_raw_empty + 8 * rs);
      }
      if (++rs == kRaw) { rs = 0; rph ^= 1; }
      if (++os == kOps) { os = 0; oph ^= 1; }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
  }
}

}  // namespace sp
}  // namespace b16
