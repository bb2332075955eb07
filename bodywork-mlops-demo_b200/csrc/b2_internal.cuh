// b2_internal.cuh -- shared declarations of libb2gram.so (not part of the public C-ABI).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/b2gram.h"

namespace b2 {

constexpr int kMaxD = B2_MAX_D;          // 128 features
constexpr int kMaxS = kMaxD + 2;         // 130: features, ones, y
constexpr int kKernelEventPairs = 64;
constexpr int kMaxRanks = 8;
constexpr size_t kXchgSlotDoubles = (size_t)kMaxS * kMaxS;                 // one rank's S
constexpr size_t kXchgDataDoubles = 2 * kMaxRanks * kXchgSlotDoubles;       // two epochs (parity) x ranks
constexpr size_t kXchgBytes = kXchgDataDoubles * sizeof(double) + 256;      // + flags[8] (u32) + ticket

// ---- tcgen05 Gram kernel geometry (gram_tc.cu) ------------------------------------------
constexpr int kTcRows = 64;              // rows of X per pipeline stage (4 MMA K-steps of 16)
constexpr int kTcM = 128;                // MMA M: feature index (zero padded)
constexpr int kTcN = 144;                // MMA N: 128 feature columns (hi) + 16 extra columns [1, y_hi, y_lo, 0...]
constexpr int kTcAccCols = 2 * kTcN;     // two accumulators: A = hi and A = lo against the same B = [hi | E]
constexpr int kTcAccElems = kTcM * kTcAccCols;  // fp32 accumulators drained per chunk (36 864)
constexpr int kTcSideDoubles = 8;        // per-CTA CUDA-core sums: sum y', sum y'^2, rows used
constexpr int kShiftFloats = 64 * (kMaxD + 2);   // b2_ctx::shift: 64 partials of the shift sample (features, y, rows)

void set_error(const char* fmt, ...);

#define B2_CUDA(call)                                                                      \
  do {                                                                                     \
    cudaError_t e_ = (call);                                                               \
    if (e_ != cudaSuccess) {                                                               \
      b2::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
      return B2_E_CUDA;                                                                    \
    }                                                                                      \
  } while (0)

}  // namespace b2

struct b2_ctx {
  int device = 0;
  int sm_count = 0;
  size_t hbm_bytes = 0;
  char name[128] = {0};
  cudaStream_t stream = nullptr;       // compute stream (all kernels)
  cudaStream_t copy_stream = nullptr;  // H2D staging for B2_MEM_HOST
  cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;
  cudaEvent_t ev_k[b2::kKernelEventPairs][2];
  int k_pairs = 0;                     // pairs recorded since the last b2_last_kernel_ms
  int k_launches = 0;                  // kernels launched by the most recent accumulate
  int64_t launches = 0;                // kernels launched since ctx creation

  int kernel_mode = B2_KERNEL_AUTO;
  int drain_rows = 8192;
  int precision = B2_PRECISION_SPLIT;

  int d = 0;                           // feature count of the current statistic (0 = not reset)
  int s_kernels = 0;                   // 1 << B2_KERNEL_* of every kernel that added to S since the last reset / import
  double* S = nullptr;                 // device, kMaxS*kMaxS (only (d+2)^2 used, row stride d+2)

  // tcgen05 path scratch
  double* tc_part = nullptr;           // [sm_count][kTcAccElems]   per-CTA fp64 partial Gram (col-major)
  double* tc_side = nullptr;           // [sm_count][kTcSideDoubles]
  double* tc_red = nullptr;            // [kTcAccElems + 16 + 129 + pad]: reduced partials, y sums, barrier slot, shift
  float* shift = nullptr;              // [kShiftFloats] partial sums of the row sample -> per-column shift c
  bool tc_attr_set = false;
  bool solve_attr_set = false;
  double* solve_host = nullptr;        // pinned mirror of solve_out (D2H without a staging copy)
  // tensor-map cache of the most recent tcgen05 launch (a refit of resident rows re-uses the same maps)
  struct TmCache {
    const void* X = nullptr; const float* y = nullptr; const uint8_t* mask = nullptr;
    int64_t n = 0, ldx = 0; int d = 0, x_dtype = -1, y_map_2d = 0;
    alignas(64) unsigned char tmX[128], tmY[128], tmM[128];
  } tm_cache;
  // SIMT path scratch
  double* simt_part = nullptr;         // [simt_ctas][kMaxS*kMaxS]
  int simt_ctas = 0;
  // scoring scratch
  double* score_part = nullptr;        // [score_ctas][6]
  int score_ctas = 0;
  double* coef_dev = nullptr;          // [kMaxD + 1]
  double* coef_host = nullptr;         // pinned [2][kMaxD + 1]: upload slots of b2_score's coefficients
  cudaEvent_t ev_coef[2] = {nullptr, nullptr};
  int coef_slot = 0;
  long long* synth_count = nullptr;    // device counter of b2_synth_tranche (rows kept by the y >= 0 filter)
  // solve scratch
  double* solve_out = nullptr;         // [kMaxD + 2 + kMaxD]: coef, intercept, info, singular
  double* solve_work = nullptr;        // [2 * kMaxD * kMaxD] eigenvectors etc.
  // host staging ring (B2_MEM_HOST)
  void* stage_x[2] = {nullptr, nullptr};
  float* stage_y[2] = {nullptr, nullptr};
  uint8_t* stage_m[2] = {nullptr, nullptr};
  size_t stage_bytes_x = 0;
  int64_t stage_rows = 0;
  cudaEvent_t ev_copied[2] = {nullptr, nullptr};
  cudaEvent_t ev_consumed[2] = {nullptr, nullptr};
  bool ev_consumed_valid[2] = {false, false};   // a kernel of an earlier call may still read stage buffer b
  float* yhat_stage[2] = {nullptr, nullptr};    // prediction staging blocks of the host-streamed b2_score
  void* bounce[2] = {nullptr, nullptr};         // pinned bounce blocks for pageable host rows (filled by host threads)
  cudaEvent_t ev_bounce[2] = {nullptr, nullptr};
  bool s_zero_pending = false;         // b2_gram_reset is lazy: S is cleared (or overwritten) by the first kernel that adds to it
  // NCCL
  void* comm = nullptr;
  int n_ranks = 1, rank = 0;
  // one-shot peer-memory all-reduce of S (p2p.cu): exchange buffer exported over CUDA IPC
  double* xchg = nullptr;              // [2 parities][kMaxRanks][kMaxS*kMaxS] slots, then flags / ticket words
  double* xchg_peer[8] = {nullptr};    // this rank's view of every rank's exchange buffer (own entry == xchg)
  bool p2p_ready = false;
  bool p2p_local = false;              // peers attached inside this process (b2_comm_p2p_attach_local): no IPC handles to close
  unsigned int xchg_epoch = 0;
  unsigned long long xchg_timeout_ns = 10000000000ull;   // bound of the wait for a peer's flag (b2_comm_set_timeout_ms)
  bool xchg_pending = false;           // an exchange was launched since the status word was last read
  unsigned int* xchg_status_host = nullptr;  // pinned mirror of the exchange status word
  // fused fit (b2_fit): in-kernel grid barrier / ticket words of the Gram kernel's reduce + fold tail
  unsigned int* tc_sync = nullptr;     // [0], [1] barrier arrivals, [2] ticket
  int fused_fits = 0;                  // fits that took the fused path (b2_ctx_stats)
  int sm_limit = 0;                    // > 0: persistent kernels use at most this many SMs (b2_ctx_set_sm_limit)
  bool sm_limit_auto = false;          // the limit was set by b2_comm_p2p_attach_local (contexts sharing a device)
};

namespace b2 {

// ---- kernel launchers (each enqueues on ctx->stream and bumps ctx->launches) -----------------
int launch_gram_simt(b2_ctx* ctx, const void* X, int x_dtype, const float* y, int64_t n, int d,
                     int64_t ldx, const uint8_t* mask, int keep);
bool gram_tc_supported(const void* X, int x_dtype, const float* y, int64_t n, int d, int64_t ldx);
int64_t gram_tc_main_rows(int64_t n, int d, int64_t ldx, int* pack_out);
// fuse != nullptr: the Gram kernel computes its own shift, reduces the per-CTA partials and folds them into S in the
// same launch (grid barriers), and -- with an attached peer exchange -- stores S into every peer's slot (b2_fit)
struct TcFuse {
  int assign;                 // S = value instead of S += value (fresh statistic, no memset needed)
  int scatter;                // 1: store the folded S into the exchange slots of all ranks and publish the flags
  unsigned int epoch;         // exchange number when scatter == 1
};
int launch_gram_tc(b2_ctx* ctx, const void* X, int x_dtype, const float* y, int64_t n, int d,
                   int64_t ldx, const uint8_t* mask, int keep, const TcFuse* fuse = nullptr);
bool gram_narrow_supported(const void* X, int x_dtype, const float* y, int64_t n, int d, int64_t ldx,
                           const uint8_t* mask);
int launch_gram_narrow(b2_ctx* ctx, const void* X, int x_dtype, const float* y, int64_t n, int d,
                       int64_t ldx, const uint8_t* mask, int keep);
// gather_epoch != 0: the solve kernel first waits for the peer exchange `gather_epoch` and sums the slots into S
int launch_solve_cholesky(b2_ctx* ctx, double alpha, int fit_intercept, unsigned int gather_epoch = 0);
int launch_solve_eigvals(b2_ctx* ctx, double cond, int fit_intercept);
int launch_metrics(b2_ctx* ctx, const void* y, const void* yhat, int dtype, int64_t n, bool first);
int launch_solve_spectral(b2_ctx* ctx, double cond, int fit_intercept);
int launch_score(b2_ctx* ctx, const void* X, int x_dtype, int64_t n, int d, int64_t ldx,
                 const float* y, const uint8_t* mask, int keep, float* yhat, bool first_block);
int launch_p2p_allreduce(b2_ctx* ctx);
int launch_synth(b2_ctx* ctx, uint64_t seed, int64_t row_offset, int64_t n, int d, int64_t ldx,
                 int x_dtype, double alpha, double beta, double sigma, void* X, float* y);
int launch_synth_tranche(b2_ctx* ctx, uint64_t seed, int64_t n, double alpha, double beta, double sigma, float* X, float* y,
                         int64_t* n_kept_dev);
int ensure_s_cleared(b2_ctx* ctx);   // honours a lazy b2_gram_reset before a kernel that does S += ...

}  // namespace b2
