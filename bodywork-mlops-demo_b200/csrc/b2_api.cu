// b2_api.cu -- the C-ABI of libb2gram.so (declared in include/b2gram.h): context, caller-buffer
// helpers, dispatch between the tcgen05 and CUDA-core Gram kernels, host-streamed accumulation
// (pinned ring -> HBM staging, copy/compute overlap), NCCL all-reduce of the statistic, timing.
#include <dlfcn.h>
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>

#include <new>
#include <thread>
#include <vector>

#include "b2_internal.cuh"
#include "b2_xchg.cuh"

namespace b2 {

static thread_local char g_err[768] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

namespace {

// ---- NCCL through dlopen: no link-time dependency, the library loads on CPU-only boxes ------------
struct NcclUid { char internal[128]; };
struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(NcclUid*) = nullptr;
  int (*CommInitRank)(void**, int, NcclUid, int) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
constexpr int kNcclFloat64 = 8, kNcclSum = 0, kNcclMax = 2;

NcclApi* nccl() {
  static NcclApi api;
  static bool tried = false;
  if (!tried) {
    tried = true;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
      api.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
      if (api.lib) break;
    }
    if (api.lib) {
      api.GetUniqueId = reinterpret_cast<int (*)(NcclUid*)>(dlsym(api.lib, "ncclGetUniqueId"));
      api.CommInitRank = reinterpret_cast<int (*)(void**, int, NcclUid, int)>(dlsym(api.lib, "ncclCommInitRank"));
      api.CommDestroy = reinterpret_cast<int (*)(void*)>(dlsym(api.lib, "ncclCommDestroy"));
      api.AllReduce = reinterpret_cast<int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t)>(
          dlsym(api.lib, "ncclAllReduce"));
      api.GetErrorString = reinterpret_cast<const char* (*)(int)>(dlsym(api.lib, "ncclGetErrorString"));
    }
  }
  if (!api.lib || !api.GetUniqueId || !api.CommInitRank || !api.AllReduce) return nullptr;
  return &api;
}

#define B2_NCCL(api, call)                                                                     \
  do {                                                                                         \
    int r_ = (call);                                                                           \
    if (r_ != 0) {                                                                             \
      set_error("%s failed: %s", #call, (api)->GetErrorString ? (api)->GetErrorString(r_) : "?"); \
      return B2_E_COMM;                                                                        \
    }                                                                                          \
  } while (0)

int use_device(b2_ctx* ctx) {
  if (ctx == nullptr) {
    set_error("null context");
    return B2_E_ARG;
  }
  B2_CUDA(cudaSetDevice(ctx->device));
  return B2_OK;
}

int check_shape(b2_ctx* ctx, int x_dtype, int64_t n, int d, int64_t ldx, int mem_kind) {
  if (x_dtype != B2_F32 && x_dtype != B2_BF16) { set_error("x_dtype must be B2_F32 or B2_BF16"); return B2_E_ARG; }
  if (d < 1 || d > kMaxD) { set_error("d=%d out of range [1,%d]", d, kMaxD); return B2_E_ARG; }
  if (n < 0) { set_error("n_rows < 0"); return B2_E_ARG; }
  if (ldx < d) { set_error("ldx=%lld < d=%d", (long long)ldx, d); return B2_E_ARG; }
  if (mem_kind != B2_MEM_DEVICE && mem_kind != B2_MEM_HOST) { set_error("bad mem_kind %d", mem_kind); return B2_E_ARG; }
  (void)ctx;
  return B2_OK;
}

constexpr int64_t kMaxRowsPerLaunch = (int64_t)1 << 30;   // TMA coordinates / tile counters are int32

// One device-resident block through the selected Gram kernel.
int gram_block(b2_ctx* ctx, const void* X, int x_dtype, const float* y, int64_t n, int d, int64_t ldx,
               const uint8_t* mask, int keep) {
  if (n == 0) return B2_OK;
  if (n > kMaxRowsPerLaunch) {   // more rows than one launch indexes: same kernel family, several launches
    const int es = x_dtype == B2_F32 ? 4 : 2;
    for (int64_t r0 = 0; r0 < n; r0 += kMaxRowsPerLaunch) {
      const int64_t rows = n - r0 < kMaxRowsPerLaunch ? n - r0 : kMaxRowsPerLaunch;
      if (int r = gram_block(ctx, static_cast<const char*>(X) + (size_t)r0 * ldx * es, x_dtype, y + r0, rows, d, ldx,
                             mask != nullptr ? mask + r0 : nullptr, keep))
        return r;
    }
    return B2_OK;
  }
  if (int r = ensure_s_cleared(ctx)) return r;
  const bool tc_ok = gram_tc_supported(X, x_dtype, y, n, d, ldx) &&
                     (mask == nullptr || (reinterpret_cast<uintptr_t>(mask) & 15) == 0);
  const bool nw_ok = gram_narrow_supported(X, x_dtype, y, n, d, ldx, mask);
  int mode = ctx->kernel_mode;
  if (mode == B2_KERNEL_TCGEN05 && !tc_ok) {
    set_error("tcgen05 path needs d%%4==0 (fp32) / d%%8==0 (bf16), 16-byte aligned X/y/mask/row pitch, n>=32");
    return B2_E_UNSUPPORTED;
  }
  if (mode == B2_KERNEL_NARROW && !nw_ok) {
    set_error("narrow path needs d<=16, contiguous rows (ldx==d) and 16-byte aligned X/y/mask");
    return B2_E_UNSUPPORTED;
  }
  if (mode == B2_KERNEL_AUTO) {
    // narrow rows stream through the CUDA-core pipeline (HBM-bound); wide rows go to the tensor core;
    // tiny tranches (the reference's 1 440-row day) and odd layouts stay on the exact fp64 kernel
    if (nw_ok && n >= 4096) mode = B2_KERNEL_NARROW;
    else mode = (tc_ok && n >= 2048) ? B2_KERNEL_TCGEN05 : B2_KERNEL_SIMT;
  }
  ctx->s_kernels |= 1 << mode;
  if (mode == B2_KERNEL_NARROW) return launch_gram_narrow(ctx, X, x_dtype, y, n, d, ldx, mask, keep);
  if (mode == B2_KERNEL_TCGEN05) return launch_gram_tc(ctx, X, x_dtype, y, n, d, ldx, mask, keep);
  return launch_gram_simt(ctx, X, x_dtype, y, n, d, ldx, mask, keep);
}

int ensure_staging(b2_ctx* ctx) {
  if (ctx->stage_x[0] != nullptr) return B2_OK;
  ctx->stage_rows = 1 << 18;                                  // 262 144 rows per block (134 MB at 128 x fp32)
  ctx->stage_bytes_x = (size_t)ctx->stage_rows * kMaxD * 4;
  for (int b = 0; b < 2; ++b) {
    B2_CUDA(cudaMalloc(&ctx->stage_x[b], ctx->stage_bytes_x));
    B2_CUDA(cudaMalloc(reinterpret_cast<void**>(&ctx->stage_y[b]), (size_t)ctx->stage_rows * 4));
    B2_CUDA(cudaMalloc(reinterpret_cast<void**>(&ctx->stage_m[b]), (size_t)ctx->stage_rows));
    B2_CUDA(cudaEventCreateWithFlags(&ctx->ev_copied[b], cudaEventDisableTiming));
    B2_CUDA(cudaEventCreateWithFlags(&ctx->ev_consumed[b], cudaEventDisableTiming));
  }
  return B2_OK;
}

// Is a host pointer page-locked (cudaHostAlloc / cudaHostRegister)?  Pageable rows -- what numpy / pandas hand over --
// cannot be DMA'ed directly: the driver bounces them through one internal staging buffer on one thread (~11 GB/s
// measured here).  They take the library's own bounce ring instead: several host threads copy the next block into a
// pinned buffer while the previous block is on the wire.
bool host_pointer_is_pinned(const void* p) {
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return attr.type == cudaMemoryTypeHost || attr.type == cudaMemoryTypeManaged;
}

int ensure_bounce(b2_ctx* ctx) {
  if (ctx->bounce[0] != nullptr) return B2_OK;
  for (int b = 0; b < 2; ++b) {
    B2_CUDA(cudaHostAlloc(&ctx->bounce[b], ctx->stage_bytes_x, cudaHostAllocDefault));
    B2_CUDA(cudaEventCreateWithFlags(&ctx->ev_bounce[b], cudaEventDisableTiming));
  }
  return B2_OK;
}

static int copy_threads() {
  static const int nt_cfg = []() {
    const char* e = getenv("B2_COPY_THREADS");
    if (e != nullptr && atoi(e) > 0) return atoi(e) > 64 ? 64 : atoi(e);
    const unsigned hw = std::thread::hardware_concurrency();
    const int half = (int)(hw / 2);
    return half < 4 ? 4 : (half > 16 ? 16 : half);
  }();
  return nt_cfg;
}

void parallel_copy_rows(char* dst, const char* src, int64_t rows, size_t row_bytes, size_t src_pitch) {
  // copy threads: half the hardware threads, at most 16 (measured on the 64-thread GPU box, tools/perf_pageable.py);
  // B2_COPY_THREADS overrides
  int nt = copy_threads();
  if ((size_t)rows * row_bytes < ((size_t)8 << 20)) nt = 1;
  auto work = [=](int t) {
    const int64_t lo = rows * t / nt, hi = rows * (t + 1) / nt;
    if (src_pitch == row_bytes) {
      memcpy(dst + (size_t)lo * row_bytes, src + (size_t)lo * src_pitch, (size_t)(hi - lo) * row_bytes);
    } else {
      for (int64_t r = lo; r < hi; ++r) memcpy(dst + (size_t)r * row_bytes, src + (size_t)r * src_pitch, row_bytes);
    }
  };
  if (nt == 1) { work(0); return; }
  std::vector<std::thread> pool;
  pool.reserve(nt - 1);
  for (int t = 1; t < nt; ++t) pool.emplace_back(work, t);
  work(0);
  for (auto& th : pool) th.join();
}

// gather + convert `rows` rows of d strided host columns into a row-major fp32 block (b2_upload_columns)
template <typename T>
static void pack_rows(float* dst, const void* const* cols, const int64_t* strides, int64_t r0, int64_t rows, int d) {
  constexpr int kRowsPerTile = 64, kColsPerPass = 16;
  for (int64_t t0 = 0; t0 < rows; t0 += kRowsPerTile) {
    const int64_t tr = rows - t0 < kRowsPerTile ? rows - t0 : kRowsPerTile;
    for (int j0 = 0; j0 < d; j0 += kColsPerPass) {
      const int jc = d - j0 < kColsPerPass ? d - j0 : kColsPerPass;
      const char* src[kColsPerPass];
      int64_t st[kColsPerPass];
      for (int j = 0; j < jc; ++j) { st[j] = strides[j0 + j]; src[j] = static_cast<const char*>(cols[j0 + j]) + (r0 + t0) * st[j]; }
      for (int64_t r = 0; r < tr; ++r) {
        float* out = dst + (size_t)(t0 + r) * d + j0;
        for (int j = 0; j < jc; ++j) out[j] = (float)*reinterpret_cast<const T*>(src[j] + r * st[j]);
      }
    }
  }
}

// copy rows [r0, r0+rows) of a host matrix into a compact (ldx == d) staging block
int stage_rows_h2d(b2_ctx* ctx, int buf, const void* X, int es, const float* y, const uint8_t* mask, int64_t r0,
                   int64_t rows, int d, int64_t ldx, bool pinned) {
  const char* src = static_cast<const char*>(X) + (size_t)r0 * ldx * es;
  if (!pinned) {
    if (int r = ensure_bounce(ctx)) return r;
    B2_CUDA(cudaEventSynchronize(ctx->ev_bounce[buf]));                 // the H2D that last read this bounce block is done
    parallel_copy_rows(static_cast<char*>(ctx->bounce[buf]), src, rows, (size_t)d * es, (size_t)ldx * es);
    B2_CUDA(cudaMemcpyAsync(ctx->stage_x[buf], ctx->bounce[buf], (size_t)rows * d * es, cudaMemcpyHostToDevice, ctx->copy_stream));
    B2_CUDA(cudaEventRecord(ctx->ev_bounce[buf], ctx->copy_stream));
  } else if (ldx == d) {
    B2_CUDA(cudaMemcpyAsync(ctx->stage_x[buf], src, (size_t)rows * d * es, cudaMemcpyHostToDevice, ctx->copy_stream));
  } else {
    B2_CUDA(cudaMemcpy2DAsync(ctx->stage_x[buf], (size_t)d * es, src, (size_t)ldx * es, (size_t)d * es, rows,
                              cudaMemcpyHostToDevice, ctx->copy_stream));
  }
  if (y != nullptr)
    B2_CUDA(cudaMemcpyAsync(ctx->stage_y[buf], y + r0, (size_t)rows * 4, cudaMemcpyHostToDevice, ctx->copy_stream));
  if (mask != nullptr)
    B2_CUDA(cudaMemcpyAsync(ctx->stage_m[buf], mask + r0, (size_t)rows, cudaMemcpyHostToDevice, ctx->copy_stream));
  return B2_OK;
}

}  // namespace

int ensure_s_cleared(b2_ctx* ctx) {
  if (ctx->s_zero_pending) {
    B2_CUDA(cudaMemsetAsync(ctx->S, 0, sizeof(double) * kMaxS * kMaxS, ctx->stream));
    ctx->s_zero_pending = false;
  }
  return B2_OK;
}

}  // namespace b2

using namespace b2;

extern "C" {

int b2_abi_version(void) { return B2_ABI_VERSION; }
const char* b2_last_error(void) { return g_err; }

int b2_device_count(int* n_out) {
  if (n_out == nullptr) { set_error("n_out is null"); return B2_E_ARG; }
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) {
    cudaGetLastError();
    *n_out = 0;
    set_error("cudaGetDeviceCount: %s", cudaGetErrorString(e));
    return B2_E_CUDA;
  }
  *n_out = n;
  return B2_OK;
}

// streams, events and device scratch of a fresh context (b2_ctx_create destroys the context if this fails)
static int ctx_allocate(b2_ctx* ctx) {
  B2_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  B2_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  B2_CUDA(cudaEventCreate(&ctx->ev_t0));
  B2_CUDA(cudaEventCreate(&ctx->ev_t1));
  for (int i = 0; i < kKernelEventPairs; ++i) {
    B2_CUDA(cudaEventCreate(&ctx->ev_k[i][0]));
    B2_CUDA(cudaEventCreate(&ctx->ev_k[i][1]));
  }
  ctx->simt_ctas = ctx->sm_count;
  ctx->score_ctas = ctx->sm_count * 8;
  B2_CUDA(cudaMalloc(reinterpret_cast<void**>(&ctx->S), sizeof(double) * kMaxS * kMaxS));
  B2_CUDA(cudaMalloc(reinterpret_cast<void**>(&ctx->tc_part), sizeof(double) * (size_t)ctx->sm_count * kTcAccElems));
  B2_CUDA(cudaMalloc(reinterpret_cast<void**>(&ctx->tc_side), sizeof(double) * (size_t)ctx->sm_count * kTcSideDoubles));
  B2_CUDA(cudaMalloc(reinterpret_cast<void**>(&ctx->tc_red), sizeof(double) * (kTcAccElems + 16 + kMaxD + 8)));
  B2_CUDA(cudaMalloc(reinterpret_cast<void**>(&ctx->shift), sizeof(float) * kShiftFloats));
  B2_CUDA(cudaMalloc(reinterpret_cast<void**>(&ctx->simt_part), sizeof(double) * (size_t)ctx->simt_ctas * kMaxS * kMaxS));
  B2_CUDA(cudaMalloc(reinterpret_cast<void**>(&ctx->score_part), sizeof(double) * ((size_t)ctx->score_ctas + 2) * 10));
  B2_CUDA(cudaMalloc(reinterpret_cast<void**>(&ctx->coef_dev), sizeof(double) * (kMaxD + 1)));
  B2_CUDA(cudaMalloc(reinterpret_cast<void**>(&ctx->solve_out), sizeof(double) * (2 * kMaxD + 8)));
  B2_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&ctx->solve_host), sizeof(double) * (2 * kMaxD + 8), cudaHostAllocDefault));
  B2_CUDA(cudaMalloc(reinterpret_cast<void**>(&ctx->tc_sync), 64));
  B2_CUDA(cudaMemset(ctx->tc_sync, 0, 64));
  B2_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&ctx->xchg_status_host), 64, cudaHostAllocDefault));
  ctx->xchg_status_host[0] = 0u;
  B2_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&ctx->coef_host), 2 * sizeof(double) * (kMaxD + 1), cudaHostAllocDefault));
  for (int b = 0; b < 2; ++b) B2_CUDA(cudaEventCreateWithFlags(&ctx->ev_coef[b], cudaEventDisableTiming));
  B2_CUDA(cudaMemset(ctx->shift, 0, sizeof(float) * kShiftFloats));
  B2_CUDA(cudaMemset(ctx->S, 0, sizeof(double) * kMaxS * kMaxS));
  B2_CUDA(cudaMemset(ctx->tc_side, 0, sizeof(double) * (size_t)ctx->sm_count * kTcSideDoubles));
  B2_CUDA(cudaMemset(ctx->tc_red, 0, sizeof(double) * (kTcAccElems + 16 + kMaxD + 8)));
  return B2_OK;
}

int b2_ctx_create(int device, b2_ctx** out) {
  if (out == nullptr) { set_error("out is null"); return B2_E_ARG; }
  *out = nullptr;
  int n = 0;
  if (b2_device_count(&n) != B2_OK || n == 0) {
    set_error("no usable CUDA device (libb2gram has no CPU fallback)");
    return B2_E_CUDA;
  }
  if (device < 0 || device >= n) { set_error("device %d out of range (0..%d)", device, n - 1); return B2_E_ARG; }
  B2_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  B2_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_error("device %d is sm_%d%d; libb2gram is built for sm_100a only", device, prop.major, prop.minor);
    return B2_E_UNSUPPORTED;
  }
  b2_ctx* ctx = new (std::nothrow) b2_ctx();
  if (ctx == nullptr) { set_error("out of host memory"); return B2_E_STATE; }
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  ctx->hbm_bytes = prop.totalGlobalMem;
  snprintf(ctx->name, sizeof(ctx->name), "%s", prop.name);
  if (int r = ctx_allocate(ctx)) {   // streams, events, scratch: release whatever was created before the failure
    b2_ctx_destroy(ctx);
    return r;
  }
  *out = ctx;
  return B2_OK;
}

int b2_ctx_destroy(b2_ctx* ctx) {
  if (ctx == nullptr) return B2_OK;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  if (ctx->comm != nullptr) b2_comm_destroy(ctx);
  b2_comm_p2p_detach(ctx);
  if (ctx->xchg != nullptr) cudaFree(ctx->xchg);
  void* bufs[] = {ctx->S, ctx->tc_part, ctx->tc_side, ctx->tc_red, ctx->shift, ctx->simt_part, ctx->score_part,
                  ctx->coef_dev, ctx->solve_out, ctx->stage_x[0], ctx->stage_x[1], ctx->stage_y[0], ctx->stage_y[1],
                  ctx->stage_m[0], ctx->stage_m[1], ctx->yhat_stage[0], ctx->yhat_stage[1], ctx->tc_sync, ctx->synth_count};
  for (void* p : bufs) if (p != nullptr) cudaFree(p);
  if (ctx->solve_host != nullptr) cudaFreeHost(ctx->solve_host);
  if (ctx->xchg_status_host != nullptr) cudaFreeHost(ctx->xchg_status_host);
  if (ctx->coef_host != nullptr) cudaFreeHost(ctx->coef_host);
  for (int b = 0; b < 2; ++b) {
    if (ctx->bounce[b] != nullptr) cudaFreeHost(ctx->bounce[b]);
    if (ctx->ev_bounce[b] != nullptr) cudaEventDestroy(ctx->ev_bounce[b]);
  }
  for (int b = 0; b < 2; ++b) if (ctx->ev_coef[b]) cudaEventDestroy(ctx->ev_coef[b]);
  for (int b = 0; b < 2; ++b) {
    if (ctx->ev_copied[b]) cudaEventDestroy(ctx->ev_copied[b]);
    if (ctx->ev_consumed[b]) cudaEventDestroy(ctx->ev_consumed[b]);
  }
  for (int i = 0; i < kKernelEventPairs; ++i)
    for (int e = 0; e < 2; ++e)
      if (ctx->ev_k[i][e] != nullptr) cudaEventDestroy(ctx->ev_k[i][e]);
  if (ctx->ev_t0 != nullptr) cudaEventDestroy(ctx->ev_t0);
  if (ctx->ev_t1 != nullptr) cudaEventDestroy(ctx->ev_t1);
  if (ctx->stream != nullptr) cudaStreamDestroy(ctx->stream);
  if (ctx->copy_stream != nullptr) cudaStreamDestroy(ctx->copy_stream);
  cudaGetLastError();   // a half-built context may have left a sticky-free error code behind
  delete ctx;
  return B2_OK;
}

int b2_ctx_sync(b2_ctx* ctx) {
  if (int r = use_device(ctx)) return r;
  B2_CUDA(cudaStreamSynchronize(ctx->copy_stream));
  B2_CUDA(cudaStreamSynchronize(ctx->stream));
  return B2_OK;
}

int b2_ctx_info(b2_ctx* ctx, char* name, int name_cap, int* sm_count, size_t* hbm_bytes) {
  if (ctx == nullptr) { set_error("null context"); return B2_E_ARG; }
  if (name != nullptr && name_cap > 0) snprintf(name, (size_t)name_cap, "%s", ctx->name);
  if (sm_count != nullptr) *sm_count = ctx->sm_count;
  if (hbm_bytes != nullptr) *hbm_bytes = ctx->hbm_bytes;
  return B2_OK;
}

int b2_ctx_set_kernel(b2_ctx* ctx, int kernel) {
  if (ctx == nullptr || kernel < B2_KERNEL_AUTO || kernel > B2_KERNEL_NARROW) { set_error("bad kernel id"); return B2_E_ARG; }
  ctx->kernel_mode = kernel;
  return B2_OK;
}

int b2_ctx_set_drain_rows(b2_ctx* ctx, int rows) {
  if (ctx == nullptr || rows < kTcRows || rows % kTcRows != 0) { set_error("drain_rows must be a positive multiple of %d", kTcRows); return B2_E_ARG; }
  ctx->drain_rows = rows;
  return B2_OK;
}

int b2_ctx_set_sm_limit(b2_ctx* ctx, int n_sms) {
  if (ctx == nullptr || n_sms < 0) { set_error("n_sms must be >= 0 (0 = all SMs)"); return B2_E_ARG; }
  ctx->sm_limit = n_sms;
  ctx->sm_limit_auto = false;
  return B2_OK;
}

int b2_ctx_set_precision(b2_ctx* ctx, int precision) {
  if (ctx == nullptr || (precision != B2_PRECISION_SPLIT && precision != B2_PRECISION_BF16)) {
    set_error("precision must be B2_PRECISION_SPLIT or B2_PRECISION_BF16");
    return B2_E_ARG;
  }
  ctx->precision = precision;
  return B2_OK;
}

// ---- buffers ------------------------------------------------------------------------------------
int b2_dev_alloc(b2_ctx* ctx, size_t bytes, void** out) {
  if (int r = use_device(ctx)) return r;
  if (out == nullptr) { set_error("out is null"); return B2_E_ARG; }
  B2_CUDA(cudaMalloc(out, bytes ? bytes : 1));
  return B2_OK;
}
int b2_dev_free(b2_ctx* ctx, void* p) {
  if (int r = use_device(ctx)) return r;
  B2_CUDA(cudaFree(p));
  return B2_OK;
}
int b2_host_alloc(b2_ctx* ctx, size_t bytes, void** out) {
  if (int r = use_device(ctx)) return r;
  if (out == nullptr) { set_error("out is null"); return B2_E_ARG; }
  B2_CUDA(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault));
  return B2_OK;
}
int b2_host_free(b2_ctx* ctx, void* p) {
  if (int r = use_device(ctx)) return r;
  B2_CUDA(cudaFreeHost(p));
  return B2_OK;
}
int b2_copy_h2d(b2_ctx* ctx, void* dst, const void* src, size_t bytes) {
  if (int r = use_device(ctx)) return r;
  B2_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
  B2_CUDA(cudaStreamSynchronize(ctx->stream));
  return B2_OK;
}
// ---- DataFrame columns -> row-major fp32 rows in HBM --------------------------------------------------------------------
// pandas keeps every column of `data` as its own strided array; `data[cols].to_numpy(dtype=float32)` + ascontiguousarray
// is two single-threaded passes (a transposing copy and a conversion) and then a pageable H2D copy -- 90 % of train_model's
// time once the fit takes a millisecond.  Here the host threads of the bounce ring gather 16 columns at a time into the
// pinned bounce block (full 64-byte lines written, every column read as its own sequential stream), converting on the fly,
// while the previous block is on the wire.
// the gather + conversion alone, host to host (no device needed): rows [0, n_rows) of d strided columns -> out[n_rows][d]
static int pack_columns_threads(float* dst, const void* const* cols, const int64_t* strides, int dtype, int64_t r0, int64_t rows,
                                int d) {
  const int nt = copy_threads();
  auto work = [=](int t) {
    const int64_t lo = rows * t / nt / 64 * 64, hi = (t == nt - 1) ? rows : rows * (t + 1) / nt / 64 * 64;
    if (hi <= lo) return;
    if (dtype == B2_F64) pack_rows<double>(dst + (size_t)lo * d, cols, strides, r0 + lo, hi - lo, d);
    else pack_rows<float>(dst + (size_t)lo * d, cols, strides, r0 + lo, hi - lo, d);
  };
  if (rows < 4096 || nt == 1) {
    if (dtype == B2_F64) pack_rows<double>(dst, cols, strides, r0, rows, d); else pack_rows<float>(dst, cols, strides, r0, rows, d);
    return B2_OK;
  }
  std::vector<std::thread> pool;
  pool.reserve(nt - 1);
  for (int t = 1; t < nt; ++t) pool.emplace_back(work, t);
  work(0);
  for (auto& th : pool) th.join();
  return B2_OK;
}

int b2_pack_columns(const void* const* cols, const int64_t* strides, int dtype, int64_t n_rows, int d, float* out) {
  if (cols == nullptr || strides == nullptr || out == nullptr || n_rows < 0 || d < 1 || d > kMaxD ||
      (dtype != B2_F32 && dtype != B2_F64)) {
    set_error("b2_pack_columns: bad arguments (1 <= d <= %d, dtype B2_F32 or B2_F64)", kMaxD);
    return B2_E_ARG;
  }
  for (int j = 0; j < d; ++j)
    if (cols[j] == nullptr) { set_error("b2_pack_columns: column %d is null", j); return B2_E_ARG; }
  return pack_columns_threads(out, cols, strides, dtype, 0, n_rows, d);
}

int b2_upload_columns(b2_ctx* ctx, const void* const* cols, const int64_t* strides, int dtype, int64_t n_rows, int d,
                      float* X_dev) {
  if (int r = use_device(ctx)) return r;
  if (cols == nullptr || strides == nullptr || X_dev == nullptr || n_rows < 0 || d < 1 || d > kMaxD ||
      (dtype != B2_F32 && dtype != B2_F64)) {
    set_error("b2_upload_columns: bad arguments (1 <= d <= %d, dtype B2_F32 or B2_F64)", kMaxD);
    return B2_E_ARG;
  }
  for (int j = 0; j < d; ++j)
    if (cols[j] == nullptr) { set_error("b2_upload_columns: column %d is null", j); return B2_E_ARG; }
  if (int r = ensure_staging(ctx)) return r;
  if (int r = ensure_bounce(ctx)) return r;
  int buf = 0;
  for (int64_t r0 = 0; r0 < n_rows; r0 += ctx->stage_rows, buf ^= 1) {
    const int64_t rows = n_rows - r0 < ctx->stage_rows ? n_rows - r0 : ctx->stage_rows;
    B2_CUDA(cudaEventSynchronize(ctx->ev_bounce[buf]));               // the H2D that last read this bounce block is done
    float* dst = static_cast<float*>(ctx->bounce[buf]);
    pack_columns_threads(dst, cols, strides, dtype, r0, rows, d);
    B2_CUDA(cudaMemcpyAsync(X_dev + (size_t)r0 * d, dst, (size_t)rows * d * sizeof(float), cudaMemcpyHostToDevice, ctx->copy_stream));
    B2_CUDA(cudaEventRecord(ctx->ev_bounce[buf], ctx->copy_stream));
  }
  B2_CUDA(cudaStreamSynchronize(ctx->copy_stream));
  return B2_OK;
}

int b2_copy_d2h(b2_ctx* ctx, void* dst, const void* src, size_t bytes) {
  if (int r = use_device(ctx)) return r;
  B2_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  B2_CUDA(cudaStreamSynchronize(ctx->stream));
  return B2_OK;
}
int b2_copy_d2d(b2_ctx* ctx, void* dst, const void* src, size_t bytes) {
  if (int r = use_device(ctx)) return r;
  B2_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, ctx->stream));   // asynchronous: ordered on the stream
  return B2_OK;
}
int b2_dev_memset(b2_ctx* ctx, void* dst, int value, size_t bytes) {
  if (int r = use_device(ctx)) return r;
  B2_CUDA(cudaMemsetAsync(dst, value, bytes, ctx->stream));
  return B2_OK;
}

// ---- Gram -----------------------------------------------------------------------------------------
int b2_gram_reset(b2_ctx* ctx, int d) {
  if (int r = use_device(ctx)) return r;
  if (d < 1 || d > kMaxD) { set_error("d=%d out of range [1,%d]", d, kMaxD); return B2_E_ARG; }
  ctx->d = d;
  ctx->s_kernels = 0;
  ctx->s_zero_pending = true;   // cleared (or overwritten) by the first kernel that adds to S: one launch less per fit
  return B2_OK;
}

int b2_gram_kernels(b2_ctx* ctx, int* kernels_out) {
  if (ctx == nullptr || kernels_out == nullptr) { set_error("bad arguments to b2_gram_kernels"); return B2_E_ARG; }
  *kernels_out = ctx->s_kernels;
  return B2_OK;
}

int b2_gram_accumulate(b2_ctx* ctx, const void* X, int x_dtype, const float* y, int64_t n_rows, int d, int64_t ldx,
                       int mem_kind, const uint8_t* row_mask, int mask_keep) {
  if (int r = use_device(ctx)) return r;
  if (int r = check_shape(ctx, x_dtype, n_rows, d, ldx, mem_kind)) return r;
  if (ctx->d == 0) { set_error("b2_gram_reset has not been called"); return B2_E_STATE; }
  if (d != ctx->d) { set_error("d=%d differs from the statistic's d=%d", d, ctx->d); return B2_E_ARG; }
  if (n_rows > 0 && (X == nullptr || y == nullptr)) { set_error("X / y is null"); return B2_E_ARG; }
  ctx->k_launches = 0;
  if (mem_kind == B2_MEM_DEVICE) return gram_block(ctx, X, x_dtype, y, n_rows, d, ldx, row_mask, mask_keep);

  // host rows: stream blocks through a 2-deep HBM staging ring, copies overlapping the kernels
  if (int r = ensure_staging(ctx)) return r;
  const int es = x_dtype == B2_F32 ? 4 : 2;
  const bool x_pinned = host_pointer_is_pinned(X);
  int64_t blk = 0;
  int rc = B2_OK;
  auto step = [&](int64_t r0, int buf, int64_t rows) -> int {
    // a kernel of this call -- or of an EARLIER call that returned without a stream sync -- may still read this block
    if (ctx->ev_consumed_valid[buf]) B2_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_consumed[buf], 0));
    if (int r = stage_rows_h2d(ctx, buf, X, es, y, row_mask, r0, rows, d, ldx, x_pinned)) return r;
    B2_CUDA(cudaEventRecord(ctx->ev_copied[buf], ctx->copy_stream));
    B2_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_copied[buf], 0));
    if (int r = gram_block(ctx, ctx->stage_x[buf], x_dtype, ctx->stage_y[buf], rows, d, d,
                           row_mask ? ctx->stage_m[buf] : nullptr, mask_keep))
      return r;
    B2_CUDA(cudaEventRecord(ctx->ev_consumed[buf], ctx->stream));
    ctx->ev_consumed_valid[buf] = true;
    return B2_OK;
  };
  for (int64_t r0 = 0; r0 < n_rows && rc == B2_OK; r0 += ctx->stage_rows, ++blk) {
    const int64_t rows = (n_rows - r0 < ctx->stage_rows) ? n_rows - r0 : ctx->stage_rows;
    rc = step(r0, (int)(blk & 1), rows);
  }
  // the caller may reuse its host buffers on return -- also when a block failed
  const cudaError_t drained = cudaStreamSynchronize(ctx->copy_stream);
  if (rc != B2_OK) return rc;
  B2_CUDA(drained);
  return B2_OK;
}

// The peer-memory exchange reports a peer that did not deliver within the timeout through a status word in the
// exchange buffer; it is read together with the next result the host fetches, so a late or dead rank turns into
// B2_E_COMM instead of a fit on a partial statistic.  Call after the stream has been synchronised.
static int queue_exchange_status_read(b2_ctx* ctx) {
  if (!ctx->xchg_pending || ctx->xchg == nullptr) return B2_OK;
  B2_CUDA(cudaMemcpyAsync(ctx->xchg_status_host, xchg_flags(ctx->xchg) + kXchgStatusWord, sizeof(unsigned int),
                          cudaMemcpyDeviceToHost, ctx->stream));
  return B2_OK;
}
static int check_exchange_status(b2_ctx* ctx) {
  if (!ctx->xchg_pending || ctx->xchg == nullptr) return B2_OK;
  ctx->xchg_pending = false;
  const unsigned int st = ctx->xchg_status_host[0];
  if (st != 0u) {
    ctx->xchg_status_host[0] = 0u;
    cudaMemsetAsync(xchg_flags(ctx->xchg) + kXchgStatusWord, 0, sizeof(unsigned int), ctx->stream);
    set_error("peer-memory exchange %u timed out after %.1f s: a rank did not deliver its partial statistic "
              "(S on this rank is incomplete)", st, (double)ctx->xchg_timeout_ns * 1e-9);
    return B2_E_COMM;
  }
  return B2_OK;
}

int b2_gram_allreduce(b2_ctx* ctx) {
  if (int r = use_device(ctx)) return r;
  if (ctx->d == 0) { set_error("b2_gram_reset has not been called"); return B2_E_STATE; }
  if (int r = ensure_s_cleared(ctx)) return r;
  if (ctx->n_ranks > 1 && ctx->p2p_ready) return launch_p2p_allreduce(ctx);   // peer-memory one-shot exchange
  if (ctx->comm == nullptr) return B2_OK;
  NcclApi* api = nccl();
  if (api == nullptr) { set_error("libnccl.so.2 could not be loaded"); return B2_E_COMM; }
  const size_t count = (size_t)(ctx->d + 2) * (ctx->d + 2);
  B2_NCCL(api, api->AllReduce(ctx->S, ctx->S, count, kNcclFloat64, kNcclSum, ctx->comm, ctx->stream));
  return B2_OK;
}

int b2_gram_export(b2_ctx* ctx, double* S_out, int64_t* n_rows_out) {
  if (int r = use_device(ctx)) return r;
  if (ctx->d == 0) { set_error("b2_gram_reset has not been called"); return B2_E_STATE; }
  const int dp = ctx->d + 2;
  if (S_out == nullptr) { set_error("S_out is null"); return B2_E_ARG; }
  if (int r = ensure_s_cleared(ctx)) return r;
  B2_CUDA(cudaMemcpyAsync(S_out, ctx->S, sizeof(double) * dp * dp, cudaMemcpyDeviceToHost, ctx->stream));
  if (int r = queue_exchange_status_read(ctx)) return r;
  B2_CUDA(cudaStreamSynchronize(ctx->stream));
  if (int r = check_exchange_status(ctx)) return r;
  if (n_rows_out != nullptr) *n_rows_out = (int64_t)(S_out[ctx->d * dp + ctx->d] + 0.5);
  return B2_OK;
}

int b2_gram_import(b2_ctx* ctx, const double* S_in, int d) {
  if (int r = use_device(ctx)) return r;
  if (d < 1 || d > kMaxD || S_in == nullptr) { set_error("bad arguments to b2_gram_import"); return B2_E_ARG; }
  ctx->d = d;
  ctx->s_kernels = 0;
  ctx->s_zero_pending = false;
  B2_CUDA(cudaMemsetAsync(ctx->S, 0, sizeof(double) * kMaxS * kMaxS, ctx->stream));
  B2_CUDA(cudaMemcpyAsync(ctx->S, S_in, sizeof(double) * (d + 2) * (d + 2), cudaMemcpyHostToDevice, ctx->stream));
  B2_CUDA(cudaStreamSynchronize(ctx->stream));
  return B2_OK;
}

// ---- solve ------------------------------------------------------------------------------------------
// from_pinned: the Cholesky kernel has written its result into ctx->solve_host itself (no copy node to wait for)
static int fetch_solution(b2_ctx* ctx, bool from_pinned, double* coef, double* intercept, double* singular, int* rank,
                          double* info) {
  double* host = ctx->solve_host;
  if (!from_pinned)
    B2_CUDA(cudaMemcpyAsync(host, ctx->solve_out, sizeof(double) * (2 * kMaxD + 8), cudaMemcpyDeviceToHost, ctx->stream));
  if (int r = queue_exchange_status_read(ctx)) return r;
  B2_CUDA(cudaStreamSynchronize(ctx->stream));
  if (int r = check_exchange_status(ctx)) return r;
  if (coef != nullptr) memcpy(coef, host, sizeof(double) * ctx->d);
  if (intercept != nullptr) *intercept = host[kMaxD];
  *info = host[kMaxD + 1];
  if (rank != nullptr) *rank = (int)host[kMaxD + 2];
  if (singular != nullptr) memcpy(singular, host + kMaxD + 3, sizeof(double) * ctx->d);
  return B2_OK;
}

static int finish_cholesky(b2_ctx* ctx, double* coef, double* intercept) {
  double info = 0.0;
#ifdef B2_DEV_KNOBS
  double phase[kMaxD];
  if (int r = fetch_solution(ctx, true, coef, intercept, getenv("B2_SOLVE_TIMING") ? phase : nullptr, nullptr, &info)) return r;
  if (getenv("B2_SOLVE_TIMING"))
    fprintf(stderr, "[b2_solve] cycles: build %.0f diag %.0f panel %.0f update %.0f backward %.0f\n", phase[0], phase[1],
            phase[2], phase[3], phase[4]);
#else
  if (int r = fetch_solution(ctx, true, coef, intercept, nullptr, nullptr, &info)) return r;
#endif
  if (info < 0.0) {
    ctx->xchg_pending = false;
    set_error("peer-memory exchange timed out after %.1f s inside the solve: a rank did not deliver its partial "
              "statistic", (double)ctx->xchg_timeout_ns * 1e-9);
    cudaMemsetAsync(xchg_flags(ctx->xchg) + kXchgStatusWord, 0, sizeof(unsigned int), ctx->stream);
    return B2_E_COMM;
  }
  if (info != 0.0) {
    set_error("pivot %d of the LDL^T factorisation is not positive: the centred Gram matrix is rank deficient "
              "(use alpha > 0 or b2_solve_spectral)", (int)info);
    return B2_E_SINGULAR;
  }
  return B2_OK;
}

int b2_solve(b2_ctx* ctx, double alpha, int fit_intercept, double* coef, double* intercept) {
  if (int r = use_device(ctx)) return r;
  if (ctx->d == 0) { set_error("b2_gram_reset has not been called"); return B2_E_STATE; }
  if (!(alpha >= 0.0)) { set_error("alpha must be >= 0"); return B2_E_ARG; }
  if (int r = ensure_s_cleared(ctx)) return r;
  if (int r = launch_solve_cholesky(ctx, alpha, fit_intercept)) return r;
  return finish_cholesky(ctx, coef, intercept);
}

int b2_solve_spectral(b2_ctx* ctx, double cond, int fit_intercept, double* coef, double* intercept, double* singular,
                      int* rank) {
  if (int r = use_device(ctx)) return r;
  if (ctx->d == 0) { set_error("b2_gram_reset has not been called"); return B2_E_STATE; }
  if (int r = ensure_s_cleared(ctx)) return r;
  if (int r = launch_solve_spectral(ctx, cond, fit_intercept)) return r;
  double info = 0.0;
  return fetch_solution(ctx, false, coef, intercept, singular, rank, &info);
}

int b2_solve_eigvals(b2_ctx* ctx, double cond, int fit_intercept, double* singular, int* rank, int64_t* n_rows_out) {
  if (int r = use_device(ctx)) return r;
  if (ctx->d == 0) { set_error("b2_gram_reset has not been called"); return B2_E_STATE; }
  if (int r = ensure_s_cleared(ctx)) return r;
  if (int r = launch_solve_eigvals(ctx, cond, fit_intercept)) return r;
  double info = 0.0;
  if (int r = fetch_solution(ctx, false, nullptr, nullptr, singular, rank, &info)) return r;
  if (n_rows_out != nullptr) *n_rows_out = (int64_t)(ctx->solve_host[kMaxD + 3 + kMaxD] + 0.5);
#ifdef B2_DEV_KNOBS
  if (getenv("B2_SOLVE_TIMING")) {
    const double* t = ctx->solve_host + kMaxD + 3 + kMaxD + 1;
    fprintf(stderr, "[b2_solve_eigvals] cycles: build %.0f tridiagonalise %.0f scale %.0f multisection %.0f\n", t[0], t[1], t[2], t[3]);
  }
#endif
  return B2_OK;
}

// ---- the whole fit in one call ----------------------------------------------------------------------------
// reset + accumulate + all-reduce + solve.  Device-resident rows that take the tensor-core kernel run as four launches
// with no memset, no separate scatter / gather kernels and no D2H copy node: shift sample, Gram kernel, finalize kernel
// (reduces and folds the per-CTA partials, overwrites S, stores it straight into the peers' exchange slots) and the
// solve kernel (waits for the peers' slots, sums them, factors, writes the coefficients into pinned host memory).
// Everything else is the plain sequence of the four calls.
int b2_fit(b2_ctx* ctx, const void* X, int x_dtype, const float* y, int64_t n_rows, int d, int64_t ldx, int mem_kind,
           const uint8_t* row_mask, int mask_keep, double alpha, int fit_intercept, double* coef, double* intercept) {
  if (int r = use_device(ctx)) return r;
  if (int r = check_shape(ctx, x_dtype, n_rows, d, ldx, mem_kind)) return r;
  if (!(alpha >= 0.0)) { set_error("alpha must be >= 0"); return B2_E_ARG; }
  if (n_rows > 0 && (X == nullptr || y == nullptr)) { set_error("X / y is null"); return B2_E_ARG; }
  static const bool no_fused = getenv("B2_NO_FUSED") != nullptr;      // diagnostic switch: the four-call sequence
  bool fused = !no_fused && mem_kind == B2_MEM_DEVICE && n_rows <= kMaxRowsPerLaunch &&
               gram_tc_supported(X, x_dtype, y, n_rows, d, ldx) &&
               (row_mask == nullptr || (reinterpret_cast<uintptr_t>(row_mask) & 15) == 0);
  if (fused) {
    const bool nw_ok = gram_narrow_supported(X, x_dtype, y, n_rows, d, ldx, row_mask);
    if (ctx->kernel_mode == B2_KERNEL_AUTO) fused = !(nw_ok && n_rows >= 4096) && n_rows >= 2048;
    else fused = ctx->kernel_mode == B2_KERNEL_TCGEN05;
  }
  if (!fused) {
    if (int r = b2_gram_reset(ctx, d)) return r;
    if (int r = b2_gram_accumulate(ctx, X, x_dtype, y, n_rows, d, ldx, mem_kind, row_mask, mask_keep)) return r;
    if (int r = b2_gram_allreduce(ctx)) return r;
    return b2_solve(ctx, alpha, fit_intercept, coef, intercept);
  }
  ctx->d = d;
  ctx->k_launches = 0;
  ctx->s_kernels = 1 << B2_KERNEL_TCGEN05;
  const int es = x_dtype == B2_F32 ? 4 : 2;
  const int64_t n_main = gram_tc_main_rows(n_rows, d, ldx, nullptr);
  if (n_main < n_rows) ctx->s_kernels |= 1 << B2_KERNEL_SIMT;
  TcFuse fuse;
  fuse.assign = 1; fuse.scatter = 0; fuse.epoch = 0;
  if (n_main < n_rows) {   // the few rows the packed layout leaves over go in first; the fused fold then adds to S
    ctx->s_zero_pending = true;
    if (int r = ensure_s_cleared(ctx)) return r;
    if (int r = launch_gram_simt(ctx, static_cast<const char*>(X) + (size_t)n_main * ldx * es, x_dtype, y + n_main,
                                 n_rows - n_main, d, ldx, row_mask != nullptr ? row_mask + n_main : nullptr, mask_keep))
      return r;
    fuse.assign = 0;
  }
  const bool p2p = ctx->n_ranks > 1 && ctx->p2p_ready;
  if (p2p) { fuse.scatter = 1; fuse.epoch = ++ctx->xchg_epoch; }
  if (int r = launch_gram_tc(ctx, X, x_dtype, y, n_rows, d, ldx, row_mask, mask_keep, &fuse)) return r;
  ctx->fused_fits += 1;
  if (!p2p && ctx->comm != nullptr) {
    if (int r = b2_gram_allreduce(ctx)) return r;
  }
  if (int r = launch_solve_cholesky(ctx, alpha, fit_intercept, p2p ? fuse.epoch : 0u)) return r;
  return finish_cholesky(ctx, coef, intercept);
}

// ---- scoring ---------------------------------------------------------------------------------------
int b2_score(b2_ctx* ctx, const void* X, int x_dtype, int64_t n_rows, int d, int64_t ldx, int mem_kind,
             const double* coef, double intercept, const float* y, const uint8_t* row_mask, int mask_keep,
             float* yhat, double* stats_out) {
  if (int r = use_device(ctx)) return r;
  if (int r = check_shape(ctx, x_dtype, n_rows, d, ldx, mem_kind)) return r;
  if (coef == nullptr || (n_rows > 0 && X == nullptr)) { set_error("coef / X is null"); return B2_E_ARG; }
  // coefficients go up through one of two pinned slots (no stream sync per call: the slot is only waited for when it
  // is reused, two calls later)
  {
    const int slot = ctx->coef_slot;
    ctx->coef_slot ^= 1;
    B2_CUDA(cudaEventSynchronize(ctx->ev_coef[slot]));
    double* cbuf = ctx->coef_host + (size_t)slot * (kMaxD + 1);
    memset(cbuf, 0, sizeof(double) * (kMaxD + 1));
    memcpy(cbuf, coef, sizeof(double) * d);
    cbuf[kMaxD] = intercept;
    B2_CUDA(cudaMemcpyAsync(ctx->coef_dev, cbuf, sizeof(double) * (kMaxD + 1), cudaMemcpyHostToDevice, ctx->stream));
    B2_CUDA(cudaEventRecord(ctx->ev_coef[slot], ctx->stream));
  }
  double* acc = ctx->score_part + (size_t)ctx->score_ctas * 10;
  if (n_rows == 0) {
    B2_CUDA(cudaMemsetAsync(acc, 0, sizeof(double) * 10, ctx->stream));
  } else if (mem_kind == B2_MEM_DEVICE) {
    if (int r = launch_score(ctx, X, x_dtype, n_rows, d, ldx, y, row_mask, mask_keep, yhat, true)) return r;
  } else {
    if (int r = ensure_staging(ctx)) return r;
    const int es = x_dtype == B2_F32 ? 4 : 2;
    const bool x_pinned = host_pointer_is_pinned(X);
    // predictions of a staged block land in a device block of their own (allocated once per context) and are copied
    // back behind the kernel
    float* yhat_dev[2] = {nullptr, nullptr};
    if (yhat != nullptr) {
      for (int b = 0; b < 2; ++b) {
        if (ctx->yhat_stage[b] == nullptr &&
            cudaMalloc(reinterpret_cast<void**>(&ctx->yhat_stage[b]), (size_t)ctx->stage_rows * 4) != cudaSuccess) {
          cudaGetLastError();
          set_error("out of device memory for the prediction staging blocks");
          return B2_E_CUDA;
        }
        yhat_dev[b] = ctx->yhat_stage[b];
      }
    }
    int64_t blk = 0;
    int rc = B2_OK;
    for (int64_t r0 = 0; r0 < n_rows && rc == B2_OK; r0 += ctx->stage_rows, ++blk) {
      const int buf = (int)(blk & 1);
      const int64_t rows = (n_rows - r0 < ctx->stage_rows) ? n_rows - r0 : ctx->stage_rows;
      if (ctx->ev_consumed_valid[buf]) cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_consumed[buf], 0);
      rc = stage_rows_h2d(ctx, buf, X, es, y, row_mask, r0, rows, d, ldx, x_pinned);
      if (rc != B2_OK) break;
      cudaEventRecord(ctx->ev_copied[buf], ctx->copy_stream);
      cudaStreamWaitEvent(ctx->stream, ctx->ev_copied[buf], 0);
      rc = launch_score(ctx, ctx->stage_x[buf], x_dtype, rows, d, d, y ? ctx->stage_y[buf] : nullptr,
                        row_mask ? ctx->stage_m[buf] : nullptr, mask_keep, yhat ? yhat_dev[buf] : nullptr, blk == 0);
      if (rc != B2_OK) break;
      if (yhat != nullptr)
        cudaMemcpyAsync(yhat + r0, yhat_dev[buf], (size_t)rows * 4, cudaMemcpyDeviceToHost, ctx->stream);
      cudaEventRecord(ctx->ev_consumed[buf], ctx->stream);
      ctx->ev_consumed_valid[buf] = true;
    }
    cudaStreamSynchronize(ctx->copy_stream);
    cudaStreamSynchronize(ctx->stream);
    if (rc != B2_OK) return rc;
    B2_CUDA(cudaGetLastError());
  }
  if (stats_out != nullptr && y != nullptr) {
    B2_CUDA(cudaMemcpyAsync(stats_out, acc, sizeof(double) * 10, cudaMemcpyDeviceToHost, ctx->stream));
    B2_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  return B2_OK;
}

int b2_score_allreduce(b2_ctx* ctx, double* stats) {
  if (int r = use_device(ctx)) return r;
  if (stats == nullptr) { set_error("stats is null"); return B2_E_ARG; }
  if (ctx->comm == nullptr) {
    if (ctx->n_ranks > 1) { set_error("b2_score_allreduce needs the NCCL communicator (b2_comm_init)"); return B2_E_STATE; }
    return B2_OK;
  }
  NcclApi* api = nccl();
  if (api == nullptr) { set_error("libnccl.so.2 could not be loaded"); return B2_E_COMM; }
  double* acc = ctx->score_part + (size_t)ctx->score_ctas * 10;   // 10 sums
  double* mx = acc + 10;                                          // 2 maxima
  B2_CUDA(cudaStreamSynchronize(ctx->stream));   // the previous b2_score may still be reading its totals
  double host[10], hmax[2];
  memcpy(host, stats, sizeof(host));
  hmax[0] = host[4]; hmax[1] = host[9];
  host[4] = 0.0; host[9] = 0.0;
  B2_CUDA(cudaMemcpyAsync(acc, host, sizeof(host), cudaMemcpyHostToDevice, ctx->stream));
  B2_CUDA(cudaMemcpyAsync(mx, hmax, sizeof(hmax), cudaMemcpyHostToDevice, ctx->stream));
  B2_CUDA(cudaStreamSynchronize(ctx->stream));   // host / hmax live on this stack frame
  B2_NCCL(api, api->AllReduce(acc, acc, 10, kNcclFloat64, kNcclSum, ctx->comm, ctx->stream));
  B2_NCCL(api, api->AllReduce(mx, mx, 2, kNcclFloat64, kNcclMax, ctx->comm, ctx->stream));
  B2_CUDA(cudaMemcpyAsync(host, acc, sizeof(host), cudaMemcpyDeviceToHost, ctx->stream));
  B2_CUDA(cudaMemcpyAsync(hmax, mx, sizeof(hmax), cudaMemcpyDeviceToHost, ctx->stream));
  B2_CUDA(cudaStreamSynchronize(ctx->stream));
  host[4] = hmax[0]; host[9] = hmax[1];
  memcpy(stats, host, sizeof(host));
  return B2_OK;
}

// ---- synthetic rows -------------------------------------------------------------------------------------
int b2_synth(b2_ctx* ctx, uint64_t seed, int64_t row_offset, int64_t n_rows, int d, int64_t ldx, int x_dtype,
             double alpha, double beta, double sigma, void* X_dev, float* y_dev) {
  if (int r = use_device(ctx)) return r;
  if (int r = check_shape(ctx, x_dtype, n_rows, d, ldx, B2_MEM_DEVICE)) return r;
  if (n_rows > 0 && (X_dev == nullptr || y_dev == nullptr)) { set_error("X / y is null"); return B2_E_ARG; }
  return launch_synth(ctx, seed, row_offset, n_rows, d, ldx, x_dtype, alpha, beta, sigma, X_dev, y_dev);
}

// y >= 0 filtered one-feature tranche of day `day` (stage_3_synthetic_data_generation.py:28-43)
int b2_synth_tranche(b2_ctx* ctx, uint64_t seed, int64_t n_rows, int day, double beta, double sigma, float* X_dev,
                     float* y_dev, int64_t* n_kept_out) {
  if (int r = use_device(ctx)) return r;
  if (n_rows < 0 || day < 1 || n_kept_out == nullptr || (n_rows > 0 && (X_dev == nullptr || y_dev == nullptr))) {
    set_error("bad arguments to b2_synth_tranche");
    return B2_E_ARG;
  }
  if (ctx->synth_count == nullptr) B2_CUDA(cudaMalloc(reinterpret_cast<void**>(&ctx->synth_count), 16));
  // alpha(d) = kappa + amplitude * sin(2 pi f (d - 1) / 364), kappa = 1, amplitude = 0.5, f = 6  (stage_3...:31-33,38)
  const double alpha = 1.0 + 0.5 * sin(2.0 * 3.14159265358979323846 * 6.0 * (double)(day - 1) / 364.0);
  if (int r = launch_synth_tranche(ctx, seed, n_rows, alpha, beta, sigma, X_dev, y_dev,
                                   reinterpret_cast<int64_t*>(ctx->synth_count)))
    return r;
  long long kept = 0;
  B2_CUDA(cudaMemcpyAsync(&kept, ctx->synth_count, sizeof(kept), cudaMemcpyDeviceToHost, ctx->stream));
  B2_CUDA(cudaStreamSynchronize(ctx->stream));
  *n_kept_out = (int64_t)kept;
  return B2_OK;
}

// ---- model_metrics on two vectors (stage_1_train_model.py:79-90), fp32 or fp64 inputs -------------------------
int b2_metrics(b2_ctx* ctx, const void* y_actual, const void* y_predicted, int dtype, int64_t n_rows, int mem_kind,
               double* stats_out) {
  if (int r = use_device(ctx)) return r;
  if (dtype != B2_F32 && dtype != B2_F64) { set_error("dtype must be B2_F32 or B2_F64"); return B2_E_ARG; }
  if (n_rows < 0 || stats_out == nullptr || (n_rows > 0 && (y_actual == nullptr || y_predicted == nullptr))) {
    set_error("bad arguments to b2_metrics");
    return B2_E_ARG;
  }
  if (mem_kind != B2_MEM_DEVICE && mem_kind != B2_MEM_HOST) { set_error("bad mem_kind %d", mem_kind); return B2_E_ARG; }
  double* acc = ctx->score_part + (size_t)ctx->score_ctas * 10;
  const size_t es = dtype == B2_F32 ? 4 : 8;
  if (n_rows == 0) {
    B2_CUDA(cudaMemsetAsync(acc, 0, sizeof(double) * 10, ctx->stream));
  } else if (mem_kind == B2_MEM_DEVICE) {
    if (int r = launch_metrics(ctx, y_actual, y_predicted, dtype, n_rows, true)) return r;
  } else {
    // host vectors: blocks through the two staging buffers of the streamed paths (x block = y_actual, y block region
    // is too small for fp64, so both vectors share the X block: [rows] actual then [rows] predicted)
    if (int r = ensure_staging(ctx)) return r;
    const int64_t blk_rows = (int64_t)(ctx->stage_bytes_x / (2 * es));
    int64_t blk = 0;
    for (int64_t r0 = 0; r0 < n_rows; r0 += blk_rows, ++blk) {
      const int buf = (int)(blk & 1);
      const int64_t rows = n_rows - r0 < blk_rows ? n_rows - r0 : blk_rows;
      if (ctx->ev_consumed_valid[buf]) B2_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_consumed[buf], 0));
      char* dst = static_cast<char*>(ctx->stage_x[buf]);
      B2_CUDA(cudaMemcpyAsync(dst, static_cast<const char*>(y_actual) + (size_t)r0 * es, (size_t)rows * es,
                              cudaMemcpyHostToDevice, ctx->copy_stream));
      B2_CUDA(cudaMemcpyAsync(dst + (size_t)blk_rows * es, static_cast<const char*>(y_predicted) + (size_t)r0 * es,
                              (size_t)rows * es, cudaMemcpyHostToDevice, ctx->copy_stream));
      B2_CUDA(cudaEventRecord(ctx->ev_copied[buf], ctx->copy_stream));
      B2_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_copied[buf], 0));
      if (int r = launch_metrics(ctx, dst, dst + (size_t)blk_rows * es, dtype, rows, blk == 0)) return r;
      B2_CUDA(cudaEventRecord(ctx->ev_consumed[buf], ctx->stream));
      ctx->ev_consumed_valid[buf] = true;
    }
    B2_CUDA(cudaStreamSynchronize(ctx->copy_stream));
  }
  B2_CUDA(cudaMemcpyAsync(stats_out, acc, sizeof(double) * 10, cudaMemcpyDeviceToHost, ctx->stream));
  B2_CUDA(cudaStreamSynchronize(ctx->stream));
  return B2_OK;
}

// counters of the context: [0] fits that took the fused path of b2_fit, [1] exchanges started, [2] kernels launched
int b2_ctx_stats(b2_ctx* ctx, int64_t* out3) {
  if (ctx == nullptr || out3 == nullptr) { set_error("null argument"); return B2_E_ARG; }
  out3[0] = ctx->fused_fits;
  out3[1] = (int64_t)ctx->xchg_epoch;
  out3[2] = ctx->launches;
  return B2_OK;
}

// ---- multi-GPU --------------------------------------------------------------------------------------------
int b2_comm_unique_id(char* id_out) {
  if (id_out == nullptr) { set_error("id_out is null"); return B2_E_ARG; }
  NcclApi* api = nccl();
  if (api == nullptr) { set_error("libnccl.so.2 could not be loaded"); return B2_E_COMM; }
  NcclUid uid;
  B2_NCCL(api, api->GetUniqueId(&uid));
  memcpy(id_out, uid.internal, 128);
  return B2_OK;
}

int b2_comm_init(b2_ctx* ctx, int n_ranks, int rank, const char* id) {
  if (int r = use_device(ctx)) return r;
  if (n_ranks < 1 || rank < 0 || rank >= n_ranks || id == nullptr) { set_error("bad communicator arguments"); return B2_E_ARG; }
  if (ctx->comm != nullptr) { set_error("communicator already initialised"); return B2_E_STATE; }
  NcclApi* api = nccl();
  if (api == nullptr) { set_error("libnccl.so.2 could not be loaded"); return B2_E_COMM; }
  NcclUid uid;
  memcpy(uid.internal, id, 128);
  B2_NCCL(api, api->CommInitRank(&ctx->comm, n_ranks, uid, rank));
  ctx->n_ranks = n_ranks;
  ctx->rank = rank;
  return B2_OK;
}

int b2_comm_destroy(b2_ctx* ctx) {
  if (ctx == nullptr || ctx->comm == nullptr) return B2_OK;
  NcclApi* api = nccl();
  if (api != nullptr && api->CommDestroy != nullptr) api->CommDestroy(ctx->comm);
  ctx->comm = nullptr;
  ctx->n_ranks = 1;
  ctx->rank = 0;
  return B2_OK;
}

static int ensure_xchg(b2_ctx* ctx) {
  if (ctx->xchg == nullptr) {
    B2_CUDA(cudaMalloc(reinterpret_cast<void**>(&ctx->xchg), kXchgBytes));
    B2_CUDA(cudaMemset(ctx->xchg, 0, kXchgBytes));
    B2_CUDA(cudaDeviceSynchronize());
  }
  return B2_OK;
}

int b2_comm_p2p_export(b2_ctx* ctx, char* handle_out) {
  if (int r = use_device(ctx)) return r;
  if (handle_out == nullptr) { set_error("handle_out is null"); return B2_E_ARG; }
  if (int r = ensure_xchg(ctx)) return r;
  cudaIpcMemHandle_t h;
  B2_CUDA(cudaIpcGetMemHandle(&h, ctx->xchg));
  static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
  memcpy(handle_out, &h, 64);
  return B2_OK;
}

// A (re-)attached exchange starts at exchange number 0 on every rank: clear this rank's flags, ticket and status
// (stale numbers from an earlier attachment would satisfy the first wait at once).  The caller's rendezvous must put
// a barrier between the attach of all ranks and the first exchange -- peers write into this buffer.
static int reset_exchange_words(b2_ctx* ctx) {
  B2_CUDA(cudaStreamSynchronize(ctx->stream));
  B2_CUDA(cudaMemset(xchg_flags(ctx->xchg), 0, 256));
  B2_CUDA(cudaDeviceSynchronize());
  ctx->xchg_epoch = 0;
  ctx->xchg_pending = false;
  ctx->xchg_status_host[0] = 0u;
  return B2_OK;
}

int b2_comm_p2p_attach(b2_ctx* ctx, int n_ranks, int rank, const char* handles) {
  if (int r = use_device(ctx)) return r;
  if (n_ranks < 2 || n_ranks > kMaxRanks || rank < 0 || rank >= n_ranks || handles == nullptr || ctx->xchg == nullptr) {
    set_error("b2_comm_p2p_attach: bad arguments (2..%d ranks; call b2_comm_p2p_export first)", kMaxRanks);
    return B2_E_ARG;
  }
  if (ctx->p2p_ready) { set_error("peer exchange already attached"); return B2_E_STATE; }
  if (int r = reset_exchange_words(ctx)) return r;
  for (int r = 0; r < n_ranks; ++r) {
    if (r == rank) { ctx->xchg_peer[r] = ctx->xchg; continue; }
    cudaIpcMemHandle_t h;
    memcpy(&h, handles + (size_t)r * 64, 64);
    void* p = nullptr;
    B2_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    ctx->xchg_peer[r] = static_cast<double*>(p);
  }
  ctx->n_ranks = n_ranks;
  ctx->rank = rank;
  ctx->p2p_ready = true;
  ctx->p2p_local = false;
  return B2_OK;
}

// Same exchange between contexts of ONE process (a C client driving several GPUs, or two contexts on one GPU): the
// peers' buffers are ordinary device pointers, reached through cudaDeviceEnablePeerAccess when the devices differ.
int b2_comm_p2p_attach_local(b2_ctx* ctx, int n_ranks, int rank, b2_ctx* const* peers) {
  if (int r = use_device(ctx)) return r;
  if (n_ranks < 2 || n_ranks > kMaxRanks || rank < 0 || rank >= n_ranks || peers == nullptr || peers[rank] != ctx) {
    set_error("b2_comm_p2p_attach_local: bad arguments (2..%d contexts, peers[rank] == ctx)", kMaxRanks);
    return B2_E_ARG;
  }
  if (ctx->p2p_ready) { set_error("peer exchange already attached"); return B2_E_STATE; }
  for (int r = 0; r < n_ranks; ++r) {
    if (peers[r] == nullptr) { set_error("peers[%d] is null", r); return B2_E_ARG; }
    B2_CUDA(cudaSetDevice(peers[r]->device));
    if (int rc = ensure_xchg(peers[r])) return rc;
  }
  B2_CUDA(cudaSetDevice(ctx->device));
  if (int r = reset_exchange_words(ctx)) return r;
  for (int r = 0; r < n_ranks; ++r) {
    if (peers[r]->device != ctx->device) {
      int can = 0;
      B2_CUDA(cudaDeviceCanAccessPeer(&can, ctx->device, peers[r]->device));
      if (!can) { set_error("device %d cannot map the memory of device %d", ctx->device, peers[r]->device); return B2_E_UNSUPPORTED; }
      const cudaError_t e = cudaDeviceEnablePeerAccess(peers[r]->device, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) B2_CUDA(e);
      cudaGetLastError();
    }
    ctx->xchg_peer[r] = peers[r]->xchg;
  }
  // contexts that share ONE device: a peer's kernel waiting for this rank's flags holds an SM, and the cooperative Gram
  // launch needs all of its CTAs resident at once -- leave those SMs free (a test / single-GPU configuration)
  int same_device = 0;
  for (int r = 0; r < n_ranks; ++r) same_device += (r != rank && peers[r]->device == ctx->device) ? 1 : 0;
  if (same_device > 0 && ctx->sm_limit == 0) { ctx->sm_limit = ctx->sm_count - 9 * same_device; ctx->sm_limit_auto = true; }
  ctx->n_ranks = n_ranks;
  ctx->rank = rank;
  ctx->p2p_ready = true;
  ctx->p2p_local = true;
  return B2_OK;
}

int b2_comm_p2p_detach(b2_ctx* ctx) {
  if (ctx == nullptr) { set_error("null context"); return B2_E_ARG; }
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->p2p_ready && !ctx->p2p_local)
    for (int r = 0; r < ctx->n_ranks; ++r)
      if (r != ctx->rank && ctx->xchg_peer[r] != nullptr) cudaIpcCloseMemHandle(ctx->xchg_peer[r]);
  for (int r = 0; r < kMaxRanks; ++r) ctx->xchg_peer[r] = nullptr;
  if (ctx->p2p_ready && ctx->comm == nullptr) { ctx->n_ranks = 1; ctx->rank = 0; }
  if (ctx->sm_limit_auto) { ctx->sm_limit = 0; ctx->sm_limit_auto = false; }
  ctx->p2p_ready = false;
  ctx->p2p_local = false;
  cudaGetLastError();
  return B2_OK;
}

int b2_comm_set_timeout_ms(b2_ctx* ctx, int64_t ms) {
  if (ctx == nullptr || ms < 1) { set_error("timeout must be >= 1 ms"); return B2_E_ARG; }
  ctx->xchg_timeout_ns = (unsigned long long)ms * 1000000ull;
  return B2_OK;
}

int b2_comm_info(b2_ctx* ctx, int* n_ranks_out, int* rank_out, int* exchange_out) {
  if (ctx == nullptr) { set_error("null context"); return B2_E_ARG; }
  if (n_ranks_out != nullptr) *n_ranks_out = ctx->n_ranks;
  if (rank_out != nullptr) *rank_out = ctx->rank;
  if (exchange_out != nullptr)
    *exchange_out = (ctx->n_ranks > 1 && ctx->p2p_ready) ? B2_EXCHANGE_PEER : (ctx->comm != nullptr ? B2_EXCHANGE_NCCL : B2_EXCHANGE_NONE);
  return B2_OK;
}

int b2_comm_barrier(b2_ctx* ctx) {
  if (int r = use_device(ctx)) return r;
  if (ctx->comm == nullptr) return b2_ctx_sync(ctx);
  NcclApi* api = nccl();
  if (api == nullptr) { set_error("libnccl.so.2 could not be loaded"); return B2_E_COMM; }
  double* slot = ctx->tc_red + kTcAccElems + 8;  // spare scratch
  B2_NCCL(api, api->AllReduce(slot, slot, 1, kNcclFloat64, kNcclSum, ctx->comm, ctx->stream));
  B2_CUDA(cudaStreamSynchronize(ctx->stream));
  return B2_OK;
}

// ---- timing ---------------------------------------------------------------------------------------------------
int b2_timer_start(b2_ctx* ctx) {
  if (int r = use_device(ctx)) return r;
  B2_CUDA(cudaEventRecord(ctx->ev_t0, ctx->stream));
  return B2_OK;
}
int b2_timer_stop(b2_ctx* ctx, double* ms_out) {
  if (int r = use_device(ctx)) return r;
  B2_CUDA(cudaEventRecord(ctx->ev_t1, ctx->stream));
  B2_CUDA(cudaEventSynchronize(ctx->ev_t1));
  float ms = 0.f;
  B2_CUDA(cudaEventElapsedTime(&ms, ctx->ev_t0, ctx->ev_t1));
  if (ms_out != nullptr) *ms_out = (double)ms;
  return B2_OK;
}
int b2_last_kernel_ms(b2_ctx* ctx, double* gram_ms_out, int* launches_out) {
  if (int r = use_device(ctx)) return r;
  double total = 0.0;
  const int n = ctx->k_pairs < kKernelEventPairs ? ctx->k_pairs : kKernelEventPairs;
  for (int i = 0; i < n; ++i) {
    B2_CUDA(cudaEventSynchronize(ctx->ev_k[i][1]));
    float ms = 0.f;
    B2_CUDA(cudaEventElapsedTime(&ms, ctx->ev_k[i][0], ctx->ev_k[i][1]));
    total += ms;
  }
  if (gram_ms_out != nullptr) *gram_ms_out = total;
  if (launches_out != nullptr) *launches_out = n;
  ctx->k_pairs = 0;
  return B2_OK;
}
int b2_launch_count(b2_ctx* ctx, int64_t* n_out) {
  if (ctx == nullptr || n_out == nullptr) { set_error("null argument"); return B2_E_ARG; }
  *n_out = ctx->launches;
  return B2_OK;
}

}  // extern "C"
