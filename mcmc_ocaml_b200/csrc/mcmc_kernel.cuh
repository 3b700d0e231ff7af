// mcmc_kernel.cuh -- host side (launch) of the fused Metropolis-Hastings
// ensemble kernel; the kernel itself is in mcmc_kernel_dev.cuh.
// Instantiated per plugin combination in mcmc_static.cu (compile-time D,
// parameters staged in shared memory) and mcmc_dyn.cu (registered kinds).
#pragma once
#include "common.cuh"
#include "host_plugins.hpp"
#include "mcmc_kernel_dev.cuh"
#include "mcmc_balanced.cuh"

#include <algorithm>
#include <cstdlib>
#include <cstdio>
#include <vector>

namespace mg {

// Steps per task of the balanced kernel: long enough that the state round trip
// (2 x (D+2) doubles per chain) and the queue traffic vanish, short enough that
// a run has many tasks per group to even out.
constexpr int64_t kSegSteps = 128;
static_assert(kDevErrMhQueue == MG_DEVERR_MH_QUEUE, "device error codes out of sync");

// cuTensorMapEncodeTiled, fetched from the driver (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static inline EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = [] {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) != cudaSuccess || qr != cudaDriverEntryPointSuccess) p = nullptr;
    return (EncodeTiledFn)p;
  }();
  return fn;
}
// the [slots][F][C] float64 sample block as a 3-D tensor, box = [kTmaSteps][F][32 chains]
static inline bool make_sample_tensor_map(CUtensorMap *tm, double *samples, int64_t slots, int F, int64_t C) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc || !samples || slots < 1 || (C & 1) || ((uintptr_t)samples & 15) || C >= (1ll << 32) || slots >= (1ll << 31)) return false;
  const cuuint64_t gdim[3] = {(cuuint64_t)C, (cuuint64_t)F, (cuuint64_t)slots};
  const cuuint64_t gstride[2] = {(cuuint64_t)C * 8, (cuuint64_t)C * 8 * (cuuint64_t)F};
  const cuuint32_t box[3] = {(cuuint32_t)MH_BLOCK, (cuuint32_t)F, (cuuint32_t)kTmaSteps};
  const cuuint32_t estr[3] = {1, 1, 1};
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, samples, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// One launch of the ensemble kernel: steps t0 .. of the run keyed by `key`.
struct MhLaunch {
  const mg_mcmc_cfg *cfg;
  CallKey key;
  uint64_t t0;
  int record_first;
  double *state, *samples;
  int32_t *accept;
  double *mom;   // [3][D+2][C], zeroed: per-chain running moments of the recorded samples are wanted; or null
};

// mom (may be null): where to keep the running moments of the recorded samples.  Only the balanced kernel keeps
// them, over a run that records from slot 0; *mom_done (non-null where mom is) tells whether this launch did.
template <class Like, class Prior, class Prop, int D>
static int launch_mh(mg_ctx *ctx, const MhArgs<Like, Prior, Prop, D> &a, double *mom, bool *mom_done) {
  const int64_t ngroups = (a.C + MH_BLOCK - 1) / MH_BLOCK;
  const int64_t total_steps = a.nbin + (a.n > 0 ? (a.n - 1) * a.nskip : 0);
  // Dynamic hand-out pays when the warps do not divide evenly over the schedulers.  The persistent grid holds the
  // largest whole number of warps per scheduler that the ensemble can keep busy all the time (no warp ever waits for
  // work until the tail: a polling warp on a saturated scheduler is starved by the arbiter and picks its group up late).
  const int64_t nsched = (int64_t)ctx->sm_count * 4;
  if (total_steps >= 4 * kSegSteps && ngroups > nsched && ngroups < (1ll << 30)) {
    // running moments requested: that instantiation holds more registers per warp, so its own occupancy sizes the
    // persistent grid
    const bool with_mom = mom != nullptr && a.t0 == 0 && a.record_first && a.samples != nullptr;
    int occ = 0;
    if (with_mom) MG_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, mh_balanced_kernel<Like, Prior, Prop, D, true, false>, MH_BLOCK, 0));
    else MG_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, mh_balanced_kernel<Like, Prior, Prop, D, false, false>, MH_BLOCK, 0));
    int64_t grid = std::min<int64_t>((int64_t)std::max(occ, 1) * ctx->sm_count, (ngroups / nsched) * nsched);
    if (const char *e = getenv("MCMC_GPU_MH_GRID")) grid = std::max(1, atoi(e));
    if (grid != ngroups) {
    MhQueue q;
    q.seg_steps = kSegSteps;
    const int64_t nrec = a.n > 1 ? a.n - 1 : 0;   // slots 1 .. n-1
    int64_t nseg;
    for (;; q.seg_steps *= 2) {
      q.seg_slots = std::max<int64_t>(1, q.seg_steps / a.nskip);
      q.nseg_burn = (int32_t)((a.nbin + q.seg_steps - 1) / q.seg_steps);
      nseg = q.nseg_burn + (nrec + q.seg_slots - 1) / q.seg_slots;
      if (ngroups * nseg + grid < 0xFFFFFFF0ll) break;
    }
    q.nseg = (int32_t)nseg;
    q.ngroups = (uint32_t)ngroups;
    q.total = (uint32_t)(ngroups * nseg);
    if (getenv("MCMC_GPU_DEBUG")) fprintf(stderr, "mh_balanced: occ %d grid %lld groups %lld seg %lld nseg %d\n", occ, (long long)grid, (long long)ngroups, (long long)q.seg_steps, q.nseg);
    q.cap = 1u;
    while (q.cap < 2u * q.ngroups) q.cap <<= 1;
    DevBuf<unsigned long long> ring;
    DevBuf<unsigned int> ctr;
    DevBuf<int32_t> seg_next;
    MG_CUDA(ctx, ring.alloc(q.cap, ctx->stream));
    MG_CUDA(ctx, ctr.alloc(2, ctx->stream));
    MG_CUDA(ctx, seg_next.alloc(q.ngroups, ctx->stream));
    q.ring = ring.get(); q.ctr = ctr.get(); q.seg_next = seg_next.get();
    q.err = ctx->d_devflag;
    q.wait_cycles = kQueueWaitCycles;
    if (const char *e = getenv("MCMC_GPU_WAIT_CYCLES")) q.wait_cycles = std::max(1ll, atoll(e));
    mh_queue_init_kernel<<<(q.cap + 255u) / 256u, 256, 0, ctx->stream>>>(q);
    MG_CHECK_LAUNCH(ctx);
    // running moments of the recorded samples: the variant with the accumulators is a separate instantiation, the
    // plain kernel does not pay for them
    // Recorded samples leave through the TMA (one bulk tensor store per kTmaSteps samples of a warp) when the block's
    // shape allows a tensor map (even C, compile-time dimension, a tile of at most 16 KB); plain stores otherwise.
    CUtensorMap tmap;
    memset(&tmap, 0, sizeof tmap);
    const int F = (Prop::kStaticDim ? D : a.d) + 2;
    const int64_t slots = a.n - (a.record_first ? 0 : 1);
    const bool use_tma = Prop::kStaticDim && (D + 2) * kTmaSteps * MH_BLOCK * 8 <= 16 * 1024 && a.samples != nullptr &&
                         make_sample_tensor_map(&tmap, a.samples, slots, F, a.C);
    time_begin(ctx);
    MhArgs<Like, Prior, Prop, D> am = a;
    if (with_mom) { am.mom = mom; *mom_done = true; }
    const void *fn;
#define MG_MHB_LAUNCH(MOM, TMA)                                                                         \
    do {                                                                                                \
      fn = (const void *)mh_balanced_kernel<Like, Prior, Prop, D, MOM, TMA>;                            \
      kt_reset(ctx, fn); kt_start(ctx);                                                                 \
      mh_balanced_kernel<Like, Prior, Prop, D, MOM, TMA><<<(unsigned)grid, MH_BLOCK, 0, ctx->stream>>>(am, q, tmap); \
    } while (0)
    if constexpr (Prop::kStaticDim && (D + 2) * kTmaSteps * MH_BLOCK * 8 <= 16 * 1024) {
      if (with_mom && use_tma) MG_MHB_LAUNCH(true, true);
      else if (with_mom) MG_MHB_LAUNCH(true, false);
      else if (use_tma) MG_MHB_LAUNCH(false, true);
      else MG_MHB_LAUNCH(false, false);
    } else {
      if (with_mom) MG_MHB_LAUNCH(true, false);
      else MG_MHB_LAUNCH(false, false);
    }
#undef MG_MHB_LAUNCH
    kt_stop(ctx);
    MG_CHECK_LAUNCH(ctx);
    time_end(ctx);
    return MG_OK;  // queue buffers are freed stream-ordered after the kernel
    }
  }
  const int64_t grid = ngroups;
  time_begin(ctx);
  kt_reset(ctx, (const void *)mh_ensemble_kernel<Like, Prior, Prop, D>);
  kt_start(ctx);
  mh_ensemble_kernel<Like, Prior, Prop, D><<<(unsigned)grid, MH_BLOCK, 0, ctx->stream>>>(a);
  kt_stop(ctx);
  MG_CHECK_LAUNCH(ctx);
  time_end(ctx);
  return MG_OK;
}

// everything but the plugin parameters; a.mom is set by launch_mh for the kernel that keeps the moments
template <class A>
static void fill_common(A &a, const MhLaunch &L) {
  const mg_mcmc_cfg *cfg = L.cfg;
  a.d = cfg->dim; a.pad = 0; a.C = cfg->nchains; a.chain_offset = cfg->chain_offset;
  a.nbin = cfg->nbin; a.nskip = cfg->nskip; a.n = cfg->n; a.key = L.key;
  a.t0 = L.t0; a.record_first = L.record_first; a.pad2 = 0;
  a.rk = make_round_keys(L.key);
  a.state = L.state; a.samples = L.samples; a.accept = L.accept; a.mom = nullptr;
}

}  // namespace mg
