// mcmc.cu -- Mcmc.mcmc_array (mcmc.ml:37-72) as a batched ensemble of
// independent Metropolis-Hastings chains: one thread per chain, chain state
// in registers for the whole run, one fused kernel for propose / log-density /
// accept-reject / record-sample.
//
// HBM layout.  state: [D+2][C] (coordinates, ll, lp), samples: [n][D+2][C].
// Thread c of a warp owns chain c, so every store of a field is one fully
// coalesced 256-byte warp transaction; the sample block is written once --
// through the TMA ([4 steps][D+2][32 chains] tiles, mcmc_balanced.cuh) by the
// balanced sampler, with streaming stores by the static-mapping kernel -- and
// never read by this kernel.
// Roofline: the only mandatory traffic is the recorded sample,
// 8 (D+2) / nskip bytes per chain-step (SURVEY.md 8d); at nskip = 1 and D = 10
// that is 96 B/step against ~100 FP64 instructions + 5 Philox blocks per step
// (474 warp instructions in all: the step is bound by instruction issue).
#include "mcmc_kernel.cuh"

#include <cstdlib>

namespace mg {

// instantiations live in mcmc_static.cu / mcmc_dyn.cu (one object per dimension)
#define MG_STATIC_DIMS(X) X(2) X(4) X(8) X(10) X(16) X(20) X(32)
#define MG_DYN_DIMS(X) X(2) X(4) X(8) X(16) X(32) X(64)
#define MG_DECL_STATIC(DD) int mh_static_gauss_##DD(mg_ctx *, const mg_logfn *, const mg_proposal *, const MhLaunch &, bool *);
#define MG_DECL_DYN(DD)                                                                                          \
  int mh_dyn_##DD(mg_ctx *, const DynFnParams &, const DynFnParams &, const DynPropParams &, const MhLaunch &, bool *);
MG_STATIC_DIMS(MG_DECL_STATIC)
MG_DYN_DIMS(MG_DECL_DYN)

__global__ void init_state_kernel(const double *__restrict__ x0, int shared, int D, int64_t C,
                                  double *__restrict__ state) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  for (int i = 0; i < D; ++i) state[(int64_t)i * C + c] = shared ? x0[i] : x0[c * D + i];
  state[(int64_t)D * C + c] = 0.0;
  state[(int64_t)(D + 1) * C + c] = 0.0;
}

// [n][F][C] -> [C][n][F] through a shared-memory tile (C is the contiguous
// axis of the source, F*n the contiguous axis of the destination).
__global__ void to_chain_major_kernel(const double *__restrict__ src, int64_t rows /* n*F */, int64_t C,
                                      double *__restrict__ dst) {
  __shared__ double tile[32][33];
  const int64_t c0 = (int64_t)blockIdx.x * 32, r0 = (int64_t)blockIdx.y * 32;
  for (int k = threadIdx.y; k < 32; k += blockDim.y) {
    const int64_t r = r0 + k, c = c0 + threadIdx.x;
    if (r < rows && c < C) tile[k][threadIdx.x] = src[r * C + c];
  }
  __syncthreads();
  for (int k = threadIdx.y; k < 32; k += blockDim.y) {
    const int64_t c = c0 + k, r = r0 + threadIdx.x;
    if (r < rows && c < C) dst[c * rows + r] = tile[threadIdx.x][k];
  }
}

int jit_launch_mh(mg_ctx *ctx, const DynFnParams &like, const DynFnParams &prior, const DynPropParams &prop,
                  const MhLaunch &L);  // jit.cu
int sample_block_stats(mg_ctx *ctx, const double *d_blk, int64_t n, int F, int64_t C, double *d_out);  // stats.cu
int chain_moments_finish(mg_ctx *ctx, cudaStream_t st, const double *mom, int F, int64_t C, int64_t n, double *d_out);

static int validate_cfg(mg_ctx *ctx, const mg_mcmc_cfg *cfg) {
  MG_REQUIRE(ctx, cfg != nullptr, "mcmc_array: null cfg");
  MG_REQUIRE(ctx, cfg->nchains >= 1, "mcmc_array: nchains must be >= 1");
  MG_REQUIRE(ctx, cfg->dim >= 1 && cfg->dim <= 64, "mcmc_array: dim must be in 1..64");
  MG_REQUIRE(ctx, cfg->nbin >= 0 && cfg->nskip >= 1 && cfg->n >= 0, "mcmc_array: bad nbin/nskip/n");
  MG_REQUIRE(ctx, cfg->nchains / MH_BLOCK < 2147483647LL, "mcmc_array: too many chains for one launch");
  // the Philox counter addresses (chain, step) with 48 + 40 bits (rng.cuh); accept counters are int32 per chain
  MG_REQUIRE(ctx, cfg->chain_offset < (1ull << 48) && (uint64_t)cfg->nchains <= (1ull << 48) - cfg->chain_offset,
             "mcmc_array: global chain ids must stay below 2^48");
  {
    const long double steps = (long double)cfg->nbin + (cfg->n > 0 ? (long double)(cfg->n - 1) * (long double)cfg->nskip : 0.0L);
    MG_REQUIRE(ctx, steps < 2147483647.0L, "mcmc_array: more than 2^31 - 1 steps per chain in one call (cut the run into calls)");
  }
  return MG_OK;
}

}  // namespace mg

using namespace mg;

// One launch of the ensemble kernel.  *mom_done (mom_done may be null where L.mom is): it kept the running moments.
static int mcmc_launch_segment(mg_ctx *ctx, const mg_logfn *like, const mg_logfn *prior, const mg_proposal *prop,
                               const MhLaunch &L, bool *mom_done) {
  const mg_mcmc_cfg *cfg = L.cfg;
  int rc;
  if (mom_done) *mom_done = false;
  if ((rc = validate_cfg(ctx, cfg))) return rc;
  if ((rc = validate_logfn(ctx, like, cfg->dim, "log_likelihood"))) return rc;
  if ((rc = validate_logfn(ctx, prior, cfg->dim, "log_prior"))) return rc;
  if ((rc = validate_proposal(ctx, prop, cfg->dim))) return rc;
  MG_REQUIRE(ctx, L.state != nullptr, "mcmc_array: null state");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  const int D = cfg->dim;

  if (like->kind == MG_FN_GAUSS_CORR && like->scale == 1.0 && prior->kind == MG_FN_ZERO &&
      prop->kind == MG_PROP_BOX) {
    switch (D) {
#define MG_CASE(DD) case DD: return mh_static_gauss_##DD(ctx, like, prop, L, mom_done);
      MG_STATIC_DIMS(MG_CASE)
#undef MG_CASE
      default: break;
    }
  }
  DevLogFn dl, dp; DevProposal dj;
  MG_CUDA(ctx, dl.upload_from(like, ctx->stream));
  MG_CUDA(ctx, dp.upload_from(prior, ctx->stream));
  MG_CUDA(ctx, dj.upload_from(prop, ctx->stream));
  if (like->kind >= MG_FN_USER || prior->kind >= MG_FN_USER)  // user plugins: kernel compiled at run time
    return jit_launch_mh(ctx, dl.params, dp.params, dj.params, L);
#define MG_TRY(DD) if (D <= DD) rc = mh_dyn_##DD(ctx, dl.params, dp.params, dj.params, L, mom_done); else
  MG_DYN_DIMS(MG_TRY) rc = set_err(ctx, MG_EINVAL, "mcmc_array: dim too large");
#undef MG_TRY
  return rc;  // parameter blobs are freed stream-ordered after the kernel
}

extern "C" int mg_mcmc_array_dev(mg_ctx *ctx, const mg_logfn *like, const mg_logfn *prior,
                                 const mg_proposal *prop, const mg_mcmc_cfg *cfg, double *d_state,
                                 double *d_samples, int32_t *d_accept) {
  if (!ctx) return MG_EINVAL;
  int rc;
  if ((rc = validate_cfg(ctx, cfg))) return rc;
  return mcmc_launch_segment(ctx, like, prior, prop, MhLaunch{cfg, next_key(ctx), 0, 1, d_state, d_samples, d_accept, nullptr},
                             nullptr);
}

extern "C" int mg_mcmc_array(mg_ctx *ctx, const mg_logfn *like, const mg_logfn *prior, const mg_proposal *prop,
                             const mg_mcmc_cfg *cfg, const double *x0, double *out_samples, int64_t *out_accept,
                             int64_t *out_reject) {
  if (!ctx) return MG_EINVAL;
  int rc;
  if ((rc = validate_cfg(ctx, cfg))) return rc;
  MG_REQUIRE(ctx, x0 != nullptr, "mcmc_array: null start point");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  const int D = cfg->dim, F = D + 2;
  const int64_t C = cfg->nchains, n = cfg->n;
  cudaStream_t s = ctx->stream;
  DevBuf<double> d_x0, d_state, d_samples, d_t;
  DevBuf<int32_t> d_acc;
  const size_t nx0 = cfg->x0_shared ? (size_t)D : (size_t)C * D;
  MG_CUDA(ctx, upload(d_x0, x0, nx0, s));
  MG_CUDA(ctx, d_state.alloc((size_t)F * C, s));
  MG_CUDA(ctx, d_acc.alloc((size_t)C, s));
  MG_CUDA(ctx, cudaMemsetAsync(d_acc.get(), 0, sizeof(int32_t) * C, s));
  if (out_samples && n > 0) MG_CUDA(ctx, d_samples.alloc((size_t)n * F * C, s));
  init_state_kernel<<<(unsigned)((C + 255) / 256), 256, 0, s>>>(d_x0.get(), cfg->x0_shared, D, C, d_state.get());
  MG_CHECK_LAUNCH(ctx);
  // Samples to the host while the sampler runs: the run is cut into segments (same chains: the step index of a launch
  // is an argument, the state carries over) and segment k's slice of the [n][D+2][C] block leaves on the second stream
  // while segment k + 1 computes.  Each launch is issued before the copy of the previous slice, so a pageable
  // destination (whose copy blocks the host) does not hold the sampler back.  MCMC_GPU_D2H_SEGMENTS (default 8; 1 = off).  Measured (config 2 at nskip = 100,
  // 636 MB to pinned host memory): 1 segment 24.8 ms, 2: 19.6, 4: 17.3, 8: 16.4 ms per call (the sampler alone: 13.3 ms).
  int nseg = 1;
  {
    const char *e_min = getenv("MCMC_GPU_D2H_MIN_MB");   // blocks below this size go out in one piece (default 64 MB)
    const double min_bytes = (e_min ? atof(e_min) : 64.0) * 1024.0 * 1024.0;
    if (out_samples && n > 16 && cfg->layout != MG_LAYOUT_CHAIN_MAJOR && ctx->aux && sizeof(double) * (double)n * F * C >= min_bytes) {
      const char *e = getenv("MCMC_GPU_D2H_SEGMENTS");
      const int want = e ? atoi(e) : 8;
      nseg = want < 1 ? 1 : (want > 64 ? 64 : want);
      // a segment keeps at least 1,024 steps (the balanced sampler wants >= 512 per launch), unless the tests ask
      const int64_t by_steps = (n - 1) * cfg->nskip / 1024;
      if (!getenv("MCMC_GPU_D2H_MIN_MB") && nseg > by_steps) nseg = by_steps < 1 ? 1 : (int)by_steps;
      if (nseg > n - 1) nseg = (int)(n - 1);
    }
  }
  if (nseg > 1) {
    const CallKey key = next_key(ctx);
    const int64_t nrec = n - 1;
    std::vector<cudaEvent_t> evs((size_t)nseg, nullptr);
    int64_t done = 0, first[65], count[65];
    auto launch = [&](int k) -> int {
      const int64_t m = nrec / nseg + (k < nrec % nseg ? 1 : 0);
      mg_mcmc_cfg seg = *cfg;
      seg.nbin = (k == 0) ? cfg->nbin : 0;
      seg.n = m + 1;
      const uint64_t t0 = (k == 0) ? 0 : (uint64_t)(cfg->nbin + done * cfg->nskip);
      first[k] = (k == 0) ? 0 : 1 + done; count[k] = (k == 0) ? m + 1 : m;
      double *dst = d_samples.get() + (size_t)first[k] * F * C;
      int r = mcmc_launch_segment(ctx, like, prior, prop, MhLaunch{&seg, key, t0, k == 0 ? 1 : 0, d_state.get(), dst, d_acc.get(), nullptr},
                                  nullptr);
      if (r) return r;
      MG_CUDA(ctx, cudaEventCreateWithFlags(&evs[k], cudaEventDisableTiming));
      MG_CUDA(ctx, cudaEventRecord(evs[k], s));
      done += m;
      return MG_OK;
    };
    rc = launch(0);
    for (int k = 0; k < nseg && rc == MG_OK; ++k) {
      if (k + 1 < nseg) rc = launch(k + 1);
      if (rc) break;
      cudaError_t e = cudaStreamWaitEvent(ctx->aux, evs[k], 0);
      if (e == cudaSuccess)
        e = cudaMemcpyAsync(out_samples + (size_t)first[k] * F * C, d_samples.get() + (size_t)first[k] * F * C,
                            sizeof(double) * (size_t)count[k] * F * C, cudaMemcpyDeviceToHost, ctx->aux);
      if (e != cudaSuccess) rc = set_err(ctx, MG_ECUDA, "cuda: %s (samples to host)", cudaGetErrorString(e));
    }
    cudaError_t e2 = cudaStreamSynchronize(ctx->aux);
    for (cudaEvent_t e : evs) if (e) cudaEventDestroy(e);
    if (rc) return rc;
    if (e2 != cudaSuccess) return set_err(ctx, MG_ECUDA, "cuda: %s (samples to host)", cudaGetErrorString(e2));
  } else if ((rc = mg_mcmc_array_dev(ctx, like, prior, prop, cfg, d_state.get(), d_samples.get(), d_acc.get()))) return rc;
  if (out_samples && n > 0 && nseg == 1) {
    const double *src = d_samples.get();
    if (cfg->layout == MG_LAYOUT_CHAIN_MAJOR) {
      MG_CUDA(ctx, d_t.alloc((size_t)n * F * C, s));
      dim3 grid((unsigned)((C + 31) / 32), (unsigned)((n * F + 31) / 32)), block(32, 8);
      to_chain_major_kernel<<<grid, block, 0, s>>>(d_samples.get(), n * F, C, d_t.get());
      MG_CHECK_LAUNCH(ctx);
      src = d_t.get();
    }
    MG_CUDA(ctx, cudaMemcpyAsync(out_samples, src, sizeof(double) * (size_t)n * F * C, cudaMemcpyDeviceToHost, s));
  }
  std::vector<int32_t> acc((size_t)C);
  MG_CUDA(ctx, cudaMemcpyAsync(acc.data(), d_acc.get(), sizeof(int32_t) * C, cudaMemcpyDeviceToHost, s));
  MG_CUDA(ctx, cudaStreamSynchronize(s));
  if ((rc = poll_device_error(ctx))) return rc;
  const int64_t steps = cfg->nbin + (n > 0 ? (n - 1) * cfg->nskip : 0);
  for (int64_t c = 0; c < C; ++c) {
    ctx->naccept += acc[c]; ctx->nreject += steps - acc[c];
    if (out_accept) out_accept[c] = acc[c];
    if (out_reject) out_reject[c] = steps - acc[c];
  }
  return MG_OK;
}

extern "C" int mg_mcmc_array_resident(mg_ctx *ctx, const mg_logfn *like, const mg_logfn *prior,
                                      const mg_proposal *prop, const mg_mcmc_cfg *cfg, const double *x0,
                                      double *d_samples, double *out_final, int64_t *out_accept,
                                      int64_t *out_reject, double *out_mean, double *out_std) {
  if (!ctx) return MG_EINVAL;
  int rc;
  if ((rc = validate_cfg(ctx, cfg))) return rc;
  MG_REQUIRE(ctx, x0 != nullptr, "mcmc_array: null start point");
  MG_REQUIRE(ctx, d_samples != nullptr || (!out_mean && !out_std), "mcmc_array: statistics need a sample block");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  const int D = cfg->dim, F = D + 2;
  const int64_t C = cfg->nchains, n = cfg->n;
  cudaStream_t s = ctx->stream;
  DevBuf<double> d_x0, d_state, d_final, d_stats;
  DevBuf<int32_t> d_acc;
  const size_t nx0 = cfg->x0_shared ? (size_t)D : (size_t)C * D;
  MG_CUDA(ctx, upload(d_x0, x0, nx0, s));
  MG_CUDA(ctx, d_state.alloc((size_t)F * C, s));
  MG_CUDA(ctx, d_acc.alloc((size_t)C, s));
  MG_CUDA(ctx, cudaMemsetAsync(d_acc.get(), 0, sizeof(int32_t) * C, s));
  init_state_kernel<<<(unsigned)((C + 255) / 256), 256, 0, s>>>(d_x0.get(), cfg->x0_shared, D, C, d_state.get());
  MG_CHECK_LAUNCH(ctx);
  // Statistics: the balanced sampler can keep per-chain running moments of the samples it records (d_mom); where the
  // launch reports that it did not, the block is read back once.  Overlapping that read with the sampler on a second
  // stream gave no gain on B200 (profiles/r01_mh_ncu_summary.md): the sampler's 4 warps x 122 registers fill every
  // scheduler's 16K-register slice, so the Stats CTAs find no room until it ends.
  const bool want_stats = (out_mean || out_std) && n > 0;
  std::vector<double> stats(2 * F);
  DevBuf<double> d_mom;
  if (want_stats) {
    MG_CUDA(ctx, d_stats.alloc(2 * F, s));
    MG_CUDA(ctx, d_mom.alloc((size_t)3 * F * C, s));
    MG_CUDA(ctx, cudaMemsetAsync(d_mom.get(), 0, sizeof(double) * 3 * F * C, s));
  }
  bool mom_done = false;
  rc = mcmc_launch_segment(ctx, like, prior, prop,
                           MhLaunch{cfg, next_key(ctx), 0, 1, d_state.get(), d_samples, d_acc.get(), d_mom.get()}, &mom_done);
  if (rc) return rc;
  if (want_stats) {
    if (mom_done) rc = chain_moments_finish(ctx, s, d_mom.get(), F, C, n, d_stats.get());
    else rc = sample_block_stats(ctx, d_samples, n, F, C, d_stats.get());
    if (rc) return rc;
    MG_CUDA(ctx, cudaMemcpyAsync(stats.data(), d_stats.get(), sizeof(double) * 2 * F, cudaMemcpyDeviceToHost, s));
  }
  if (out_final) {
    MG_CUDA(ctx, d_final.alloc((size_t)F * C, s));
    dim3 grid((unsigned)((C + 31) / 32), (unsigned)((F + 31) / 32)), block(32, 8);
    to_chain_major_kernel<<<grid, block, 0, s>>>(d_state.get(), F, C, d_final.get());
    MG_CHECK_LAUNCH(ctx);
    MG_CUDA(ctx, cudaMemcpyAsync(out_final, d_final.get(), sizeof(double) * F * C, cudaMemcpyDeviceToHost, s));
  }
  std::vector<int32_t> acc((size_t)C);
  MG_CUDA(ctx, cudaMemcpyAsync(acc.data(), d_acc.get(), sizeof(int32_t) * C, cudaMemcpyDeviceToHost, s));
  MG_CUDA(ctx, cudaStreamSynchronize(s));
  if ((rc = poll_device_error(ctx))) return rc;
  const int64_t steps = cfg->nbin + (n > 0 ? (n - 1) * cfg->nskip : 0);
  for (int64_t c = 0; c < C; ++c) {
    ctx->naccept += acc[c]; ctx->nreject += steps - acc[c];
    if (out_accept) out_accept[c] = acc[c];
    if (out_reject) out_reject[c] = steps - acc[c];
  }
  if (out_mean) memcpy(out_mean, stats.data(), sizeof(double) * F);
  if (out_std) memcpy(out_std, stats.data() + F, sizeof(double) * F);
  return MG_OK;
}
