// gram_tc_b16.cuh -- Gram kernels for bf16-STORED rows with D = 128 (BASELINE.json configs[1]: "10 M x 128 bf16-accum").
// Included by gram_tc.cu inside its anonymous namespace (same PTX wrappers, same partial / finalize format).  This file:
// the shared device helpers and the SINGLE-OPERAND kernel (B2_PRECISION_BF16, the literal "bf16-accum" mode); the default
// hi + lo mode is gram_tc_b16_split.cuh.
//
// Why these kernels: at 260 B / row the generic kernel is bound by the shared-memory pipe, not by HBM
// (profiles/r02_gram_tc_10Mx128_bf16_*: per 64-row tile 256 half-empty LDS.U16 wavefronts + 128 STS + 411 wavefronts of
// MMA operand reads + 128 of TMA writes = 88 % of the pipe).  Here every byte crosses shared memory as few times as the
// data flow allows -- the B operand of the MMA is THE RAW TILE AS TMA DEPOSITED IT, never rewritten:
//
//   HBM --TMA, two [64 rows][64 features] boxes, SWIZZLE_128B--> raw tile (16 KB)                       128 wavefronts
//     B = [x | E]: the raw tile read by the tensor core as an MN-major SWIZZLE_128B operand (three 64-column atoms:
//         features 0..63, 64..127, and a third atom whose first 3 columns hold E = [1, y'_hi, y'_lo], written by the E
//         warps with the same swizzle)                                                          MMA operand reads: 144
//     A : ldmatrix.x4.trans of the same raw tile -- an 8 x 8 block comes back TRANSPOSED: thread t holds feature f0 + t/4,
//         rows 2(t%4), 2(t%4)+1 as one packed bf16 pair (conflict-free through the swizzle)                           128
//         hi = rn(x - c): ONE packed sub.rn.bf16x2 per pair
//         --> TENSOR MEMORY: tcgen05.st.16x128b.x2 takes the ldmatrix fragments as they are (register k of thread t ->
//         lane t/4 (+8), column t%4 (+4)): no shuffles, and no shared-memory stores at all in the transform
//   tcgen05.mma per K = 16 step (M 128, N 144, A from tensor memory, B MN-major from shared memory):  D += hi^T [x | E]
//   so D[i][j] = sum_r hi_i x_j with x the STORED value (exact in bf16).  The epilogue turns it into the centred product
//   the fold expects,   sum_r hi_i v_j = D[i][j] - c_j * D[i][ones column]      (per-CTA partial, linear, fp64)
//   and writes it into the "A = hi" half of the partial; the "A = lo" half is zero.  The fold symmetrises as always.
//   One accumulator (x2 buffers) = 288 tensor-memory columns; 128 more hold a 4-deep ring of A operands.
//   (With hi + lo operands the same scheme gives 0.61 of the roofline but every accumulator entry then carries
//   c_j * sum_r v_i, whose fp32 truncation costs a factor 3 in coefficient accuracy -- hence the separate split kernel.)
//   Measured on the way here (profiles/r02_b16_ablations.txt): a third N = 16 MMA per K step costs 58 cycles (an MMA
//   costs max(58, N / 2) cycles whatever its N: tools/ubench_umma.cu); unpacking bf16 pairs with shifts and masks made
//   the lo arithmetic 150 instructions per warp and tile; MMAs issued under `lane == 0` are wrapped in waterfall loops.
#pragma once

namespace b16 {

constexpr int kRaw = 6;                                   // raw tile stages
constexpr int kOpsMax = 4;                                // tensor-memory A-operand stages
constexpr uint32_t kRawHalf = kTcRows * 128;              // 8192: one [64 rows][64 columns] bf16 atom
constexpr uint32_t kRawX = 2 * kRawHalf;                  // 16384: the two feature atoms TMA fills
constexpr uint32_t kRawBytes = 3 * kRawHalf;              // 24576: + the E atom
constexpr uint32_t kOffRaw = 0;
constexpr uint32_t kOffY = kOffRaw + kRaw * kRawBytes;    // 147456
constexpr uint32_t kYBytes = kTcRows * 4;                 // 256
constexpr uint32_t kMBytes = 128;                         // 64 mask bytes, padded (TMA destinations are 128-byte aligned)
constexpr uint32_t kOffMask = kOffY + kRaw * kYBytes;
constexpr uint32_t kOffBar = kOffMask + kRaw * kMBytes;
constexpr int kBars = 2 * kRaw + 2 * kOpsMax + 4;
constexpr uint32_t kOffTmemPtr = kOffBar + kBars * 8;
constexpr uint32_t kOffShift = kOffTmemPtr + 16;
constexpr uint32_t kSmem = kOffShift + (kMaxD + 4) * 4 + 1024;
static_assert(kSmem <= 227 * 1024, "shared memory budget");
// tensor memory: accumulator [G 128 | E 16] double buffered at 0 / 144, A = hi ring at 288 + 32 s
constexpr uint32_t kAccStride = 144;
constexpr uint32_t kTmemAHi = 288;

// MN-major SWIZZLE_128B operand (cute::UMMA::SmemDescriptor, version 1): 64-column atoms `kRawHalf` bytes apart (leading
// byte offset), 8-row K groups 1024 bytes apart (stride byte offset), layout type 2
__device__ __forceinline__ uint64_t make_desc_mn128(uint32_t addr) {
  return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)(kRawHalf >> 4) << 16) | ((uint64_t)(1024u >> 4) << 32) |
         (1ull << 46) | (2ull << 61);
}
// instruction descriptor: D = f32, A = B = bf16, A K-major (tensor memory), B MN-major (bit 16), N, M = 128
__host__ __device__ constexpr uint32_t idesc(int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kTcM >> 4) << 24);
}

__device__ __forceinline__ void ldsm_x4_trans(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
// registers (a, b, c, d) of thread t -> [lane t/4][col t%4], [lane t/4 + 8][col t%4], [lane t/4][col 4 + t%4],
// [lane t/4 + 8][col 4 + t%4] of the 16-lane x 8-column block at `taddr`
__device__ __forceinline__ void tmem_st_16x128b_x2(uint32_t taddr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("tcgen05.st.sync.aligned.16x128b.x2.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(a), "r"(b), "r"(c), "r"(d)
               : "memory");
}
__device__ __forceinline__ uint32_t sub_bf16x2(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("sub.rn.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}
// d = a.lo * b.lo + c  /  d = a.hi * b.lo + c: bf16 operands taken from the halves of packed registers, fp32 accumulate
__device__ __forceinline__ float fma_bf16_lo(uint32_t a2, uint32_t b2, float c) {
  float d;
  asm("{\n\t.reg .b16 al, ah, bl, bh;\n\tmov.b32 {al, ah}, %1;\n\tmov.b32 {bl, bh}, %2;\n\tfma.rn.f32.bf16 %0, al, bl, %3;\n\t}"
      : "=f"(d) : "r"(a2), "r"(b2), "f"(c));
  return d;
}
__device__ __forceinline__ float fma_bf16_hi(uint32_t a2, uint32_t b2, float c) {
  float d;
  asm("{\n\t.reg .b16 al, ah, bl, bh;\n\tmov.b32 {al, ah}, %1;\n\tmov.b32 {bl, bh}, %2;\n\tfma.rn.f32.bf16 %0, ah, bl, %3;\n\t}"
      : "=f"(d) : "r"(a2), "r"(b2), "f"(c));
  return d;
}
__device__ __forceinline__ void st_shared_zero16(uint32_t addr) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(addr), "r"(0u) : "memory");
}
__device__ __forceinline__ void st_shared_b32(uint32_t addr, uint32_t v) {
  asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
// pipeline wait: the suspend hint lets the warp sleep inside try_wait; the timer (a protocol bug must trap, never hang)
// is read once per 1024 failed polls, so a failed poll costs three instructions, not fourteen
__device__ __forceinline__ void wait_lean(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  uint64_t t0 = 0;
  while (true) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity), "r"(20000u)
        : "memory");
    if (done) break;
    if ((++spins & 1023u) == 0u) {
      const uint64_t now = globaltimer_ns();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000ull) __trap();
    }
  }
}

// Wait for two barriers at once: both try_wait are in flight together (an already-complete try_wait still takes ~90+
// cycles; two in a row were ~a fifth of a transform warp's tile time).  Bounded like wait_lean.
__device__ __forceinline__ void wait_lean2(uint32_t bar_a, uint32_t par_a, uint32_t bar_b, uint32_t par_b) {
  uint32_t da, db;
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%2], %3, %6;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 q, [%4], %5, %6;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "selp.u32 %1, 1, 0, q;\n\t}"
      : "=r"(da), "=r"(db)
      : "r"(bar_a), "r"(par_a), "r"(bar_b), "r"(par_b), "r"(20000u)
      : "memory");
  if (!da) wait_lean(bar_a, par_a);
  if (!db) wait_lean(bar_b, par_b);
}
// One tile of the issue thread in a single asm block: 4 MMAs, the two commits that free the A stage and the raw stage,
// and -- after the first MMA -- a NON-BLOCKING probe of the next tile's `full` barrier whose result is consumed only after
// the last MMA (mbarrier.test_wait takes 150-250 cycles here; every cycle this thread waits between two MMAs is a cycle
// the tensor core idles, tools/ubench_umma.cu, so the probe has to be in flight while the MMAs issue).
template <uint32_t DESC_HI, uint32_t IDESC>
__device__ __forceinline__ bool issue_tile_single(uint32_t tmem_acc, uint32_t tmem_a, uint32_t desc, uint32_t first_accumulates,
                                                  uint32_t bar_op_empty, uint32_t bar_raw_empty, uint32_t bar_next,
                                                  uint32_t par_next) {
  uint32_t ready;
  asm volatile(
      "{\n\t"
      ".reg .pred pa, pt, pr;\n\t"
      ".reg .b32 dl, ta;\n\t"
      ".reg .b64 dd;\n\t"
      "setp.ne.b32 pa, %4, 0;\n\t"
      "setp.eq.b32 pt, %4, %4;\n\t"
      "mov.b64 dd, {%3, %9};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%1], [%2], dd, %10, pa;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 pr, [%7], %8;\n\t"
      "add.u32 dl, %3, 128;\n\t mov.b64 dd, {dl, %9};\n\t add.u32 ta, %2, 8;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%1], [ta], dd, %10, pt;\n\t"
      "add.u32 dl, %3, 256;\n\t mov.b64 dd, {dl, %9};\n\t add.u32 ta, %2, 16;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%1], [ta], dd, %10, pt;\n\t"
      "add.u32 dl, %3, 384;\n\t mov.b64 dd, {dl, %9};\n\t add.u32 ta, %2, 24;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%1], [ta], dd, %10, pt;\n\t"
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%5];\n\t"
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%6];\n\t"
      "selp.u32 %0, 1, 0, pr;\n\t"
      "}"
      : "=r"(ready)
      : "r"(tmem_acc), "r"(tmem_a), "r"(desc), "r"(first_accumulates), "r"(bar_op_empty), "r"(bar_raw_empty), "r"(bar_next),
        "r"(par_next), "n"(DESC_HI), "n"(IDESC)
      : "memory");
  return ready != 0;
}

__global__ void __launch_bounds__(kThreads, 1)
gram_b16_single_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmY,
                const __grid_constant__ CUtensorMap tmM, int y_map_2d, int has_mask, int keep, int64_t n_rows,
                const float* __restrict__ shift, int chunk_tiles, double* __restrict__ part,
                double* __restrict__ side) {
  constexpr int kOps = kOpsMax;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (sbase - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  const uint32_t bar_raw_full = sbase + kOffBar;                 // [kRaw]  TMA bytes landed
  const uint32_t bar_raw_empty = bar_raw_full + 8 * kRaw;        // [kRaw]  the MMAs that read the stage as B have retired
  const uint32_t bar_op_full = bar_raw_empty + 8 * kRaw;         // [kOps]  A operands in tensor memory + E columns written
  const uint32_t bar_op_empty = bar_op_full + 8 * kOpsMax;       // [kOps]  the MMAs that read the A stage have retired
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
      mbar_init(bar_raw_empty + 8 * s, 1);
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
  // the E atoms: only 3 of their 64 columns are ever written; the MMA reads the first 16
  for (int st = 0; st < kRaw; ++st)
    for (uint32_t o = threadIdx.x * 16; o < kRawHalf; o += kThreads * 16)
      *reinterpret_cast<uint4*>(smem + kOffRaw + st * kRawBytes + kRawX + o) = make_uint4(0, 0, 0, 0);
  for (int j = threadIdx.x; j <= kMaxD; j += kThreads) shift_s[j] = shift_value(shift, j, j < kMaxD);   // c_y: fp32
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // ===== TMA producer (the whole warp runs the loop, one elected lane issues) =====
    const uint32_t tx = kRawX + kTcRows * 4 + (has_mask ? kTcRows : 0);
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
    // ===== MMA issuer: ONE elected thread runs the whole loop.  The tensor core does not queue: tools/ubench_umma.cu shows
    // that every cycle the issuing thread spends between two tcgen05.mma beyond ~one MMA time is a cycle the tensor core
    // idles (bursts of 8 MMAs + commit + d cycles of other work take 648 + d cycles).  So the loop is unrolled over the
    // stages (descriptors, tensor-memory and barrier addresses are constants off loop-invariant registers) and the
    // readiness of the NEXT tile is probed between the MMAs of the current one, where the latency is free =====
    if (elect_one()) {
      uint32_t oph = 0;
      int in_chunk = 0, chunk = 0, it = 0, os = 0;
      bool ready = false;
      const uint32_t desc00 = (uint32_t)make_desc_mn128(sbase + kOffRaw);      // low word; the high word is a constant
      constexpr uint32_t kDescHi = (uint32_t)((((uint64_t)(1024u >> 4) << 32) | (1ull << 46) | (2ull << 61)) >> 32);
      while (it < my_tiles) {
#pragma unroll
        for (int rs = 0; rs < kRaw; ++rs) {
          if (it < my_tiles) {
            const int b = chunk & 1;
            if (in_chunk == 0) wait_lean(bar_acc_empty + 8 * b, ((chunk >> 1) & 1) ^ 1);
            if (!ready) wait_lean(bar_op_full + 8 * os, oph);     // implies raw_full of this tile (the producers waited for it)
            tc_fence_after();
            const bool last = (in_chunk == chunk_tiles - 1) || (it == my_tiles - 1);
            const uint32_t tmem_acc = tmem_base + (uint32_t)b * kAccStride;
            const uint32_t a_hi = tmem_base + kTmemAHi + (uint32_t)(os * 32);
            const int osn = (os + 1 == kOps) ? 0 : os + 1;
            const uint32_t ophn = (os + 1 == kOps) ? (oph ^ 1u) : oph;
            // K steps of 16 rows are 2048 bytes (128 descriptor units) apart inside the atoms, stages kRawBytes apart
            ready = issue_tile_single<kDescHi, idesc(144)>(tmem_acc, a_hi, desc00 + (uint32_t)((rs * kRawBytes) >> 4),
                                                          in_chunk > 0 ? 1u : 0u, bar_op_empty + 8 * os, bar_raw_empty + 8 * rs,
                                                          bar_op_full + 8 * osn, ophn);
            if (last) { umma_commit(bar_acc_full + 8 * b); in_chunk = 0; ++chunk; }
            else ++in_chunk;
            ++it;
            os = osn; oph = ophn;
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 2 || warp == 3) {
    // ===== E warps: B columns 128..130 = [1, y'_hi, y'_lo] in the third atom of the raw stage (row r: 128-byte rows, the
    // 16-byte chunk index XORed with r % 8 like the TMA swizzle), and the CUDA-core sums of y' (one row per lane) =====
    const float c_y = shift_s[kMaxD];
    double sy = 0.0, syy = 0.0, cnt = 0.0;
    int rs = 0, os = 0;
    uint32_t rph = 0, oph = 0;
    const int rr = lane + 32 * (warp - 2);
    const uint32_t e_off = kRawX + (uint32_t)rr * 128u + ((uint32_t)(rr & 7) << 4);
    for (int it = 0; it < my_tiles; ++it) {
      wait_lean2(bar_raw_full + 8 * rs, rph, bar_op_empty + 8 * os, oph ^ 1);
      const int64_t left = n_rows - (tile_begin + it) * kTcRows;
      bool use = rr < left;
      if (use && has_mask) use = (ld_shared_u8(sbase + kOffMask + rs * kMBytes + rr) == (uint32_t)keep);
      const float yv = use ? ld_shared_f32(sbase + kOffY + rs * kYBytes + rr * 4) - c_y : 0.f;
      uint32_t yh, yl;
      split2(yv, 0.f, yh, yl);
      const uint32_t dst = sbase + kOffRaw + rs * kRawBytes + e_off;
      st_shared_u16(dst, use ? 0x3F80u : 0u);
      st_shared_u16(dst + 2, yh);
      st_shared_u16(dst + 4, yl);
      sy += (double)yv; syy += (double)(yv * yv); cnt += use ? 1.0 : 0.0;
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_op_full + 8 * os);
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
    // ===== epilogue: TMEM -> fp64 partial in global (column-major [col][feature]); lane = feature i =====
    const int w = warp & 3;
    double* my_part = part + (size_t)blockIdx.x * kTcAccElems + w * 32 + lane;
    const uint32_t lane_base = tmem_base + ((uint32_t)(w * 32) << 16);
    for (int chunk = 0; chunk < n_chunks; ++chunk) {
      const int b = chunk & 1;
      wait_lean(bar_acc_full + 8 * b, (chunk >> 1) & 1);
      tc_fence_after();
      // E block first: column 128 = sum_r v_i (the ones column), 129 / 130 = sum_r v_i y'
      uint32_t re[16];
      tmem_ld16(lane_base + (uint32_t)b * kAccStride + 128u, re);
      tmem_ld_wait();
      const double s1 = (double)__uint_as_float(re[0]);
      {
        double* dst = my_part + (size_t)128 * kTcM;
        if (chunk == 0) {
#pragma unroll
          for (int j = 0; j < 16; ++j) dst[(size_t)j * kTcM] = (double)__uint_as_float(re[j]);
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) dst[(size_t)j * kTcM] += (double)__uint_as_float(re[j]);
        }
      }
      // G: D[i][j] = sum_r v_i x_j  ->  sum_r v_i v_j = D[i][j] - c_j sum_r v_i   (x_j = v_j + c_j exactly on the B side)
#pragma unroll 1
      for (int p = 0; p < 8; ++p) {
        uint32_t r[16];
        tmem_ld16(lane_base + (uint32_t)b * kAccStride + (uint32_t)(p * 16), r);
        tmem_ld_wait();
        double* dst = my_part + (size_t)(p * 16) * kTcM;
        if (chunk == 0) {
#pragma unroll
          for (int j = 0; j < 16; ++j)
            dst[(size_t)j * kTcM] = fma(-(double)shift_s[p * 16 + j], s1, (double)__uint_as_float(r[j]));
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j)
            dst[(size_t)j * kTcM] += fma(-(double)shift_s[p * 16 + j], s1, (double)__uint_as_float(r[j]));
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_acc_empty + 8 * b);
    }
    // the "A = lo" half of the partial format stays empty: both operand halves went into the one accumulator
#pragma unroll 1
    for (int p = 0; p < kTcN / 16; ++p) {
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
    // chunk index is XORed with the row (SWIZZLE_128B; the rows of an atom are 128 bytes apart)
    const uint32_t lm_off = (uint32_t)(q >> 1) * kRawHalf + (uint32_t)(lane & 7) * 128u +
                            ((uint32_t)((4 * (q & 1) + (lane >> 3)) ^ (lane & 7)) << 4);
    uint32_t cc[4];      // (c, c) as packed bf16 of this thread's four features 32q + 8b + lane/4
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const float c = shift_s[32 * q + 8 * b + f8];
      const __nv_bfloat162 cp = __floats2bfloat162_rn(c, c);     // exact: c is bf16-representable
      cc[b] = *reinterpret_cast<const uint32_t*>(&cp);
    }
    const uint32_t tm_lane = tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(8 * s);
    int rs = 0, os = 0;
    uint32_t rph = 0, oph = 0;
    for (int it = 0; it < my_tiles; ++it) {
      wait_lean2(bar_raw_full + 8 * rs, rph, bar_op_empty + 8 * os, oph ^ 1);
      tc_fence_after();
      const uint32_t stage = sbase + kOffRaw + rs * kRawBytes;
      const uint32_t raw_addr = stage + lm_off + (uint32_t)(2 * s) * 1024u;
      uint32_t R[2][4];
      ldsm_x4_trans(raw_addr, R[0]);
      ldsm_x4_trans(raw_addr + 1024u, R[1]);
      const int64_t left = n_rows - (tile_begin + it) * kTcRows;
      uint32_t H[2][4];
#pragma unroll
      for (int g = 0; g < 2; ++g) {
#pragma unroll
        for (int b = 0; b < 4; ++b) H[g][b] = sub_bf16x2(R[g][b], cc[b]);      // hi = rn(x - c), both rows of the pair
      }
      const bool masked = has_mask || left < kTcRows;
      if (masked) {
        __syncwarp();                            // the ldmatrix reads above vs the clearing stores below (other lanes' rows)
        const uint32_t m_addr = sbase + kOffMask + rs * kMBytes;
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          // A side: rows 16s + 8g + 2 j4 (low half of the pair) and + 1 (high half) of this thread's fragments
          const int r0 = 16 * s + 8 * g + 2 * j4;
          bool u0 = r0 < left, u1 = (r0 + 1) < left;
          if (has_mask) {
            u0 = u0 && (ld_shared_u8(m_addr + r0) == (uint32_t)keep);
            u1 = u1 && (ld_shared_u8(m_addr + r0 + 1) == (uint32_t)keep);
          }
          const uint32_t keep32 = (u0 ? 0x0000ffffu : 0u) | (u1 ? 0xffff0000u : 0u);
#pragma unroll
          for (int b = 0; b < 4; ++b) H[g][b] &= keep32;
          // B side: a dropped row multiplies A = 0, but 0 * (NaN or Inf) would still poison the sums, so the warp also
          // clears its 64-byte segment of every dropped row of the raw tile (row 16s + 8g + lane / 4, chunk lane % 4)
          const int rz = 16 * s + 8 * g + f8;
          bool uz = rz < left;
          if (uz && has_mask) uz = (ld_shared_u8(m_addr + rz) == (uint32_t)keep);
          if (!uz)
            st_shared_zero16(stage + (uint32_t)(q >> 1) * kRawHalf + (uint32_t)rz * 128u +
                             ((uint32_t)((4 * (q & 1) + j4) ^ (rz & 7)) << 4));
        }
      }
      const uint32_t ta = tm_lane + (uint32_t)(os * 32);
      tmem_st_16x128b_x2(ta + kTmemAHi, H[0][0], H[0][1], H[1][0], H[1][1]);
      tmem_st_16x128b_x2(ta + kTmemAHi + (16u << 16), H[0][2], H[0][3], H[1][2], H[1][3]);
      tmem_st_wait();
      tc_fence_before();
      if (masked) fence_proxy_async_smem();      // the cleared rows (generic proxy) -> the MMA's operand reads (async proxy)
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_op_full + 8 * os);
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

}  // namespace b16
