// rj.cu -- Mcmc.make_rjmcmc_sampler / rjmcmc_array (mcmc.ml:83-153): ensembles
// of independent two-model reversible-jump chains, one thread per chain.
//
// A chain's state is (model, x[Dmax], ll, lp) in registers.  Cross-model
// proposals are Interpolate_pdf draws.  The reference descends a kd-tree three
// times per cross-model step (draw into the target model, density of the drawn
// point, density of the current point for the reverse jump,
// test/mcmc_test.ml:175-178); here the drawn point's density comes with its
// draw and the current point's is kept until the point changes, so most
// cross-model steps descend once.  The descent keeps its box in shared memory
// (kdtree.cuh).  Traffic per step: 1 byte (model) or
// 8 (Dmax+2) bytes (full sample) per recorded chain-step plus ~16 B per tree
// level gathered through L2 -- latency-bound pointer chasing, not HBM-bound.
#include "common.cuh"
#include "host_plugins.hpp"

#include "rj_kernel_dev.cuh"

namespace mg {

template <int DMAX>
__global__ void __maxnreg__(MG_RJ_MAXNREG(DMAX))
rj_ensemble_kernel(const __grid_constant__ RjArgs a) {
  rj_ensemble_body<DMAX>(a);
}

// the k-model kernel (mg_rjmcmc_array_k): same body over a table of up to MG_RJ_MAX_MODELS models
template <int DMAX>
__global__ void __maxnreg__(MG_RJ_MAXNREG(DMAX))
rj_ensemble_k_kernel(const __grid_constant__ RjArgsT<MG_RJ_MAX_MODELS> a) {
  rj_ensemble_body<DMAX, MG_RJ_MAX_MODELS>(a);
}

int jit_launch_rj(mg_ctx *ctx, const RjArgs &a, int Dm, unsigned grid, unsigned block, size_t smem);   // jit.cu

// largest tree dimension for which a run enables the per-point draw cache by itself (include/mcmc_gpu.h)
constexpr int kDrawCacheMaxDim = 8;

template <int NM> static int rj_launch(mg_ctx *, const RjArgsT<NM> &, bool, int, unsigned, int, size_t, cudaStream_t);
template <> int rj_launch<2>(mg_ctx *ctx, const RjArgsT<2> &a, bool any_user, int Dm, unsigned grid, int block, size_t smem,
                             cudaStream_t s) {
  if (any_user) return jit_launch_rj(ctx, a, Dm, grid, (unsigned)block, smem);
#define MG_RJ_LAUNCH(DD)                                                                              \
  do {                                                                                                \
    if (smem > 48 * 1024)                                                                             \
      MG_CUDA(ctx, cudaFuncSetAttribute(rj_ensemble_kernel<DD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    rj_ensemble_kernel<DD><<<grid, block, smem, s>>>(a);                                              \
  } while (0)
  if (Dm <= 2) MG_RJ_LAUNCH(2);
  else if (Dm <= 4) MG_RJ_LAUNCH(4);
  else if (Dm <= 8) MG_RJ_LAUNCH(8);
  else if (Dm <= 16) MG_RJ_LAUNCH(16);
  else if (Dm <= 32) MG_RJ_LAUNCH(32);
  else MG_RJ_LAUNCH(64);
#undef MG_RJ_LAUNCH
  return MG_OK;
}
template <> int rj_launch<MG_RJ_MAX_MODELS>(mg_ctx *ctx, const RjArgsT<MG_RJ_MAX_MODELS> &a, bool any_user, int Dm, unsigned grid,
                                            int block, size_t smem, cudaStream_t s) {
  if (any_user) return set_err(ctx, MG_EINVAL, "rjmcmc_array_k: user-registered log-densities are supported by the two-model call only");
#define MG_RJ_LAUNCH(DD)                                                                              \
  do {                                                                                                \
    if (smem > 48 * 1024)                                                                             \
      MG_CUDA(ctx, cudaFuncSetAttribute(rj_ensemble_k_kernel<DD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    rj_ensemble_k_kernel<DD><<<grid, block, smem, s>>>(a);                                            \
  } while (0)
  if (Dm <= 4) MG_RJ_LAUNCH(4);
  else if (Dm <= 8) MG_RJ_LAUNCH(8);
  else if (Dm <= 16) MG_RJ_LAUNCH(16);
  else if (Dm <= 32) MG_RJ_LAUNCH(32);
  else MG_RJ_LAUNCH(64);
#undef MG_RJ_LAUNCH
  return MG_OK;
}

// Mcmc.rjmcmc_array for K models; NM = 2 is the reference's two-model call, NM = MG_RJ_MAX_MODELS the extension.
template <int NM>
static int rj_run(mg_ctx *ctx, const mg_rj_model *const *M, int K, const mg_rjmcmc_cfg *cfg, const double *const *starts,
                  uint8_t *out_model, double *out_samples, int64_t *out_counts) {
  int rc;
  int DT = 0, Dm = 0;
  bool any_user = false;      // a user-registered log-density: the kernel is compiled at run time with it inlined
  for (int k = 0; k < K; ++k) {
    const int D = M[k]->like.dim;
    MG_REQUIRE(ctx, D >= 1 && D <= 64, "rjmcmc_array: dim must be in 1..64");
    if ((rc = validate_logfn(ctx, &M[k]->like, D, "log_likelihood"))) return rc;
    if ((rc = validate_logfn(ctx, &M[k]->prior, D, "log_prior"))) return rc;
    if (M[k]->like.kind >= MG_FN_USER || M[k]->prior.kind >= MG_FN_USER) any_user = true;
    if ((rc = validate_proposal(ctx, &M[k]->prop, D))) return rc;
    if (M[k]->into.kind == MG_INTO_INTERP) {
      MG_REQUIRE(ctx, M[k]->into.tree != nullptr, "rjmcmc_array: interpolated jump without a tree");
      MG_REQUIRE(ctx, M[k]->into.tree->h.D == D, "rjmcmc_array: tree dimension != model dimension");
      DT = DT > D ? DT : D;
    } else if (M[k]->into.kind == MG_INTO_INDEP_GAUSS) {
      MG_REQUIRE(ctx, M[k]->into.params && M[k]->into.nparams == 2 * D, "rjmcmc_array: into-gaussian needs mu[D], sigma[D]");
    } else return set_err(ctx, MG_EINVAL, "rjmcmc_array: unknown into-proposal kind %d", M[k]->into.kind);
    Dm = Dm > D ? Dm : D;
  }
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  const int64_t C = cfg->nchains, n = cfg->n;
  const int F = Dm + 2;
  DevLogFn dl[NM], dp[NM]; DevProposal dj[NM];
  DevBuf<double> dinto[NM], d_samples, d_t;
  DevBuf<uint8_t> d_model;
  DevBuf<unsigned long long> d_counts;
  DevBuf<double> d_start;
  DevBuf<int> d_fail;
  RjArgsT<NM> a{};
  std::vector<double> h_start((size_t)64 * NM, 0.0);
  for (int k = 0; k < K; ++k)
    for (int i = 0; i < M[k]->like.dim; ++i) h_start[(size_t)64 * k + i] = starts[k][i];
  MG_CUDA(ctx, upload(d_start, h_start.data(), h_start.size(), s));
  MG_CUDA(ctx, d_counts.alloc(NM + 3, s));
  MG_CUDA(ctx, cudaMemsetAsync(d_counts.get(), 0, (NM + 3) * sizeof(unsigned long long), s));
  MG_CUDA(ctx, d_fail.alloc(1, s));
  MG_CUDA(ctx, cudaMemsetAsync(d_fail.get(), 0, sizeof(int), s));
  for (int k = 0; k < K; ++k) {
    MG_CUDA(ctx, dl[k].upload_from(&M[k]->like, s));
    MG_CUDA(ctx, dp[k].upload_from(&M[k]->prior, s));
    MG_CUDA(ctx, dj[k].upload_from(&M[k]->prop, s));
    RjModelDev &m = a.m[k];
    m.like = dl[k].params; m.prior = dp[k].params; m.prop = dj[k].params;
    m.into_kind = M[k]->into.kind; m.nstop = M[k]->into.nstop; m.D = M[k]->like.dim;
    m.p = M[k]->p; m.log_p = log(M[k]->p);   // mcmc.ml:91, host libm like the reference
    m.into_p = nullptr;
    memset(&m.tree, 0, sizeof m.tree);
    if (m.into_kind == MG_INTO_INTERP) {
      // leaf-level Interp.draw through the per-point cell records (kdtree.cu: mg_kdtree_enable_draw_cache)
      mg_kdtree *tr = const_cast<mg_kdtree *>(M[k]->into.tree);
      if (m.nstop == 0 && tr->h.D <= kDrawCacheMaxDim && !tr->d_draw_cache && tr->ctx == ctx && C * (cfg->nbin + n * cfg->nskip) >= tr->h.N) {
        if ((rc = mg_kdtree_enable_draw_cache(tr)) == MG_ENOMEM) rc = MG_OK;   // no room: descend as before
        if (rc) return rc;
      }
      m.tree = M[k]->into.tree->view();
    }
    else {
      MG_CUDA(ctx, upload(dinto[k], M[k]->into.params, (size_t)M[k]->into.nparams, s));
      m.into_p = dinto[k].get();
    }
  }
  if (out_model && n > 0) MG_CUDA(ctx, d_model.alloc((size_t)n * C, s));
  if (out_samples && n > 0) MG_CUDA(ctx, d_samples.alloc((size_t)n * F * C, s));
  a.C = C; a.nbin = cfg->nbin; a.nskip = cfg->nskip; a.n = n; a.chain_offset = cfg->chain_offset;
  a.key = next_key(ctx);
  a.Dm = Dm; a.DT = DT; a.K = K;
  a.out_model = d_model.get(); a.out_samples = d_samples.get();
  a.counts = d_counts.get(); a.start = d_start.get(); a.fail = d_fail.get();
  const int block = DT <= 32 ? 64 : 32;
  const size_t smem = kd_scratch_bytes(DT > 0 ? DT : 1, block);
  const unsigned grid = (unsigned)((C + block - 1) / block);
  time_begin(ctx);
  if ((rc = rj_launch<NM>(ctx, a, any_user, Dm, grid, block, smem, s))) return rc;
  MG_CHECK_LAUNCH(ctx);
  time_end(ctx);
  if (out_model && n > 0) MG_CUDA(ctx, cudaMemcpyAsync(out_model, d_model.get(), (size_t)n * C, cudaMemcpyDeviceToHost, s));
  if (out_samples && n > 0)
    MG_CUDA(ctx, cudaMemcpyAsync(out_samples, d_samples.get(), sizeof(double) * (size_t)n * F * C, cudaMemcpyDeviceToHost, s));
  unsigned long long cnt[NM + 3];
  int h_fail = 0;
  MG_CUDA(ctx, cudaMemcpyAsync(cnt, d_counts.get(), sizeof cnt, cudaMemcpyDeviceToHost, s));
  MG_CUDA(ctx, cudaMemcpyAsync(&h_fail, d_fail.get(), sizeof(int), cudaMemcpyDeviceToHost, s));
  MG_CUDA(ctx, cudaStreamSynchronize(s));
  if (h_fail) return set_err(ctx, MG_EFAIL, "draw: empty tree");   // interpolate_pdf.ml:117,124
  for (int k = 0; k < K; ++k) out_counts[k] = (int64_t)cnt[k];
  const int64_t steps = C * (cfg->nbin + (n > 0 ? (n - 1) * cfg->nskip : 0));
  ctx->naccept += (int64_t)cnt[NM]; ctx->nreject += steps - (int64_t)cnt[NM];
  ctx->rj_cross[0] = (int64_t)cnt[NM + 1]; ctx->rj_cross[1] = (int64_t)cnt[NM + 2];
  return MG_OK;
}

}  // namespace mg

using namespace mg;

extern "C" int mg_rjmcmc_array(mg_ctx *ctx, const mg_rj_model *A, const mg_rj_model *B, const mg_rjmcmc_cfg *cfg,
                               const double *a0, const double *b0, uint8_t *out_model, double *out_samples,
                               int64_t out_counts[2]) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, A && B && cfg && a0 && b0 && out_counts, "rjmcmc_array: null argument");
  MG_REQUIRE(ctx, cfg->nchains >= 1 && cfg->nbin >= 0 && cfg->nskip >= 1 && cfg->n >= 0, "rjmcmc_array: bad nbin/nskip/n");
  // mcmc.ml:90 assert(pa +. pb -. 1.0 < sqrt epsilon_float)  -- one-sided, as coded
  if (!(A->p + B->p - 1.0 < sqrt(2.220446049250313e-16))) return set_err(ctx, MG_EFAIL, "Assert_failure mcmc.ml:90");
  const mg_rj_model *M[2] = {A, B};
  const double *starts[2] = {a0, b0};
  return rj_run<2>(ctx, M, 2, cfg, starts, out_model, out_samples, out_counts);
}

// k-model reversible jump (SURVEY 8f rank 3).  The reference's sampler is strictly two-model (rjmcmc_value = A | B,
// mcmc.ml:83-87); this keeps its structure -- model prior p_k inside the log prior (:116-118, :128), jump densities
// log p_target + log q_into_target (:103-112), the one-sided assertion on the priors' sum (:90) -- and lets a step
// choose its target among K models (rj_kernel_dev.cuh: rj_pick_model).  With K = 2 the chains are those of
// mg_rjmcmc_array, draw for draw.
extern "C" int mg_rjmcmc_array_k(mg_ctx *ctx, const mg_rj_model *models, int32_t nmodels, const mg_rjmcmc_cfg *cfg,
                                 const double *const *starts, uint8_t *out_model, double *out_samples, int64_t *out_counts) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, models && cfg && starts && out_counts, "rjmcmc_array_k: null argument");
  MG_REQUIRE(ctx, nmodels >= 2 && nmodels <= MG_RJ_MAX_MODELS, "rjmcmc_array_k: 2..MG_RJ_MAX_MODELS models");
  MG_REQUIRE(ctx, cfg->nchains >= 1 && cfg->nbin >= 0 && cfg->nskip >= 1 && cfg->n >= 0, "rjmcmc_array_k: bad nbin/nskip/n");
  double psum = 0.0;
  const mg_rj_model *M[MG_RJ_MAX_MODELS];
  for (int k = 0; k < nmodels; ++k) {
    MG_REQUIRE(ctx, starts[k] != nullptr, "rjmcmc_array_k: null start point");
    MG_REQUIRE(ctx, models[k].p > 0.0, "rjmcmc_array_k: model priors must be positive");
    psum = psum + models[k].p; M[k] = models + k;
  }
  if (!(psum - 1.0 < sqrt(2.220446049250313e-16))) return set_err(ctx, MG_EFAIL, "Assert_failure mcmc.ml:90 (sum of the model priors)");
  return rj_run<MG_RJ_MAX_MODELS>(ctx, M, nmodels, cfg, starts, out_model, out_samples, out_counts);
}

extern "C" int mg_rjmcmc_jump_counters(const mg_ctx *ctx, int64_t *proposed, int64_t *accepted) {
  if (!ctx) return MG_EINVAL;
  if (proposed) *proposed = ctx->rj_cross[0];
  if (accepted) *accepted = ctx->rj_cross[1];
  return MG_OK;
}
