// common.cuh -- context, error plumbing and small device helpers shared by the
// translation units of libmcmcgpu.so.
#pragma once
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/mcmc_gpu.h"
#include "rng.cuh"

struct mg_ctx {
  int device = 0;
  uint64_t seed = 0;
  uint64_t epoch = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  cudaStream_t aux = nullptr;      // second stream: Stats passes overlapped with sampling segments
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  bool ev_pending = false;
  double last_kernel_ms = 0.0;
  int64_t launches = 0;
  int64_t naccept = 0, nreject = 0;  // Mcmc.get_counters (mcmc.ml:27-35)
  int64_t rj_cross[2] = {0, 0};      // last mg_rjmcmc_array: cross-model proposals, of which accepted
  int sm_count = 148;
  // per-launch timing of the dominant kernel of the last call (bench.py roofline): event pairs on the context's
  // stream around EVERY launch of that kernel, collected lazily by mg_ctx_last_kernel_stats
  std::vector<cudaEvent_t> kt_ev;
  int kt_used = 0;
  const void *kt_func = nullptr;
  std::string kt_name;
  double kt_mean_ms = 0.0;
  int64_t kt_launches = 0;
  mg_nested_observer nest_observer = nullptr;   // Nested ?observer (nested.ml:123-125)
  void *nest_observer_user = nullptr;
  int *d_devflag = nullptr;        // device word set by a kernel whose bounded spin-wait ran out (MG_DEVERR_*)
  int sticky = MG_OK;              // a device-side failure that every later call reports until mg_ctx_clear_error
  std::string err;
};

// codes a kernel leaves in mg_ctx::d_devflag instead of trapping (a trap poisons the CUDA context of the process)
enum { MG_DEVERR_NONE = 0, MG_DEVERR_MH_QUEUE = 1, MG_DEVERR_KD_LOOKBACK = 2 };

namespace mg {

inline int set_err(mg_ctx *ctx, int code, const char *fmt, ...) {
  char buf[2048];
  va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
  if (ctx) ctx->err = buf;
  return code;
}

#define MG_CUDA(ctx, call)                                                          \
  do {                                                                              \
    cudaError_t e_ = (call);                                                        \
    if (e_ != cudaSuccess)                                                          \
      return mg::set_err((ctx), e_ == cudaErrorMemoryAllocation ? MG_ENOMEM : MG_ECUDA, \
                         "cuda: %s at %s:%d", cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

#define MG_CHECK_LAUNCH(ctx)                                                        \
  do {                                                                              \
    (ctx)->launches++;                                                              \
    MG_CUDA(ctx, cudaGetLastError());                                               \
  } while (0)

#define MG_REQUIRE(ctx, cond, ...)                                                  \
  do { if (!(cond)) return mg::set_err((ctx), MG_EINVAL, __VA_ARGS__); } while (0)

// RAII device buffer freed on scope exit (stream-ordered).
template <class T>
struct DevBuf {
  T *p = nullptr; size_t n = 0; cudaStream_t s = nullptr;
  DevBuf() {}
  DevBuf(const DevBuf &) = delete;
  DevBuf &operator=(const DevBuf &) = delete;
  cudaError_t alloc(size_t count, cudaStream_t stream) {
    release(); n = count; s = stream;
    if (count == 0) { p = nullptr; return cudaSuccess; }
    return cudaMallocAsync((void **)&p, count * sizeof(T), stream);
  }
  void release() { if (p) { cudaFreeAsync(p, s); p = nullptr; } n = 0; }
  ~DevBuf() { release(); }
  T *get() const { return p; }
};

// Read (and clear) the device error word after a synchronisation point.  A timed-out wait means the launch's
// results are invalid; the CUDA context itself stays healthy, so the error is reported by the call that observes it.
inline int poll_device_error(mg_ctx *ctx) {
  if (!ctx->d_devflag) return MG_OK;
  int h = 0;
  if (cudaMemcpyAsync(&h, ctx->d_devflag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
      cudaStreamSynchronize(ctx->stream) != cudaSuccess)
    return set_err(ctx, MG_ECUDA, "cuda: %s (reading the device error word)", cudaGetErrorString(cudaGetLastError()));
  if (h == MG_DEVERR_NONE) return MG_OK;
  cudaMemsetAsync(ctx->d_devflag, 0, sizeof(int), ctx->stream);
  return set_err(ctx, MG_ECUDA, "cuda: device-side wait timed out (%s); the results of that launch are invalid, the context remains usable",
                 h == MG_DEVERR_MH_QUEUE ? "Metropolis-Hastings task queue" : "kd-tree partition look-back");
}

// kernel-timer helpers: kt_reset names the kernel (host address of the __global__ function), kt_start / kt_stop
// bracket one launch
inline void kt_reset(mg_ctx *ctx, const void *func) { ctx->kt_used = 0; ctx->kt_func = func; ctx->kt_launches = -1; }
inline void kt_start(mg_ctx *ctx) {
  if ((size_t)(2 * ctx->kt_used + 2) > ctx->kt_ev.size()) {
    const size_t want = ctx->kt_ev.size() + 64;
    while (ctx->kt_ev.size() < want) { cudaEvent_t e = nullptr; cudaEventCreate(&e); ctx->kt_ev.push_back(e); }
  }
  cudaEventRecord(ctx->kt_ev[2 * ctx->kt_used], ctx->stream);
}
inline void kt_stop(mg_ctx *ctx) { cudaEventRecord(ctx->kt_ev[2 * ctx->kt_used + 1], ctx->stream); ctx->kt_used++; ctx->kt_launches = -1; }

inline void time_begin(mg_ctx *ctx) { cudaEventRecord(ctx->ev0, ctx->stream); }
inline void time_end(mg_ctx *ctx) { cudaEventRecord(ctx->ev1, ctx->stream); ctx->ev_pending = true; }

inline CallKey next_key(mg_ctx *ctx) { CallKey k = derive_key(ctx->seed, ctx->epoch); ctx->epoch++; return k; }

// upload a host parameter blob; empty blobs give a valid dummy pointer
template <class T>
inline cudaError_t upload(DevBuf<T> &buf, const T *host, size_t n, cudaStream_t s) {
  cudaError_t e = buf.alloc(n ? n : 1, s);
  if (e != cudaSuccess) return e;
  if (n) e = cudaMemcpyAsync(buf.get(), host, n * sizeof(T), cudaMemcpyHostToDevice, s);
  return e;
}

}  // namespace mg
