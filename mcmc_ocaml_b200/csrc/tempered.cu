// tempered.cu -- evidence by parallel tempering (include/mcmc_gpu.h, "Evidence by parallel tempering"): M ladders of
// T tempered Metropolis-Hastings chains, swaps between neighbouring rungs as warp shuffles, thermodynamic-integration
// and stepping-stone estimates of log Z.
//
// Work and bytes: one replica-step is one dynamic-plugin MH step (the work of mg_mcmc_array_dev's step) plus a few
// FP64 adds for the running sums; a swap round adds one Philox block and 2 + (D + 2) shuffles per lane.  The kernel
// reads the plugin parameters (L1/L2 resident) and writes 3 doubles + 2 ints per replica at the end: it is bound by
// instruction issue and FP64, not by HBM.  The reduction over ladders is a second, tiny kernel: one thread per rung in
// ladder order, so the record does not depend on the launch shape and needs no atomics.
#include <algorithm>
#include <cmath>

#include "comm.cuh"
#include "host_plugins.hpp"
#include "tempered_kernel_dev.cuh"

namespace mg {

template <int DMAX>
__global__ void __maxnreg__(MG_TP_MAXNREG(DMAX))
tempered_kernel(const __grid_constant__ TpArgs a) {
  tempered_body<DMAX>(a);
}

// Per-rank record: thread k < T folds rung k over the ladders in ladder order, thread T folds TI_m and SS_m.
__global__ void tempered_reduce_kernel(const __grid_constant__ TpArgs a, TpRankRec *out) {
  const int k = threadIdx.x, T = a.T;
  if (k < T) {
    double n = 0.0, mean = 0.0, m2 = 0.0, nf = 0.0, A = neg_inf(), S = 0.0;
    long long acc = 0, sacc = 0;
    for (int64_t m = 0; m < a.M; ++m) {
      const int64_t i = m * T + k;
      tp_welford(n, mean, m2, nf, a.lmean[i]);
      if (k + 1 < T) tp_lse_add(A, S, a.lse_a[i] + log(a.lse_s[i]));
      acc += a.acc[i];
      sacc += a.sacc[i];
    }
    out->n[k] = n; out->mean[k] = mean; out->m2[k] = m2; out->nf[k] = nf;
    out->lse_a[k] = A; out->lse_s[k] = S;
    out->acc[k] = acc; out->sacc[k] = sacc;
  } else if (k == T) {
    double ti[4] = {0.0, 0.0, 0.0, 0.0}, ss[4] = {0.0, 0.0, 0.0, 0.0};
    const double ns = (double)a.nsteps;
    for (int64_t m = 0; m < a.M; ++m) {
      const double *L = a.lmean + m * T;
      double tim = 0.0, ssm = 0.0;
      for (int q = 0; q + 1 < T; ++q) {
        tim = tim + (a.betas[q + 1] - a.betas[q]) * (L[q] + L[q + 1]) / 2.0;
        ssm = ssm + (a.lse_a[m * T + q] + log(a.lse_s[m * T + q] / ns));
      }
      tp_welford(ti[0], ti[1], ti[2], ti[3], tim);
      tp_welford(ss[0], ss[1], ss[2], ss[3], ssm);
    }
    for (int q = 0; q < 4; ++q) { out->ti[q] = ti[q]; out->ss[q] = ss[q]; }
  }
}

int jit_launch_tempered(mg_ctx *ctx, const TpArgs &a, int D, unsigned grid, unsigned block);   // jit.cu

// What every rank contributes to the sharded call: the arguments that must agree, its ladder count, its record.
struct TpRecord {
  int32_t T, D;
  int64_t nbin, nsteps, swap_every, M;
  double betas[TP_MAXT];
  TpRankRec r;
};

static int tp_validate(mg_ctx *ctx, const mg_logfn *like, const mg_logfn *prior, const mg_proposal *props,
                       const double *betas, const mg_tempered_cfg *cfg, const double *x0, const mg_tempered_out *out) {
  MG_REQUIRE(ctx, like && prior && props && betas && cfg && x0 && out, "evidence_tempered: null argument");
  const int T = cfg->ntemps, D = cfg->dim;
  MG_REQUIRE(ctx, cfg->nladders >= 1, "evidence_tempered: nladders must be >= 1");
  MG_REQUIRE(ctx, T >= 2 && T <= TP_MAXT, "evidence_tempered: ntemps must be in 2..32");
  MG_REQUIRE(ctx, D >= 1 && D <= 64, "evidence_tempered: dim must be in 1..64");
  MG_REQUIRE(ctx, cfg->nsteps >= 1 && cfg->nbin >= 0 && cfg->swap_every >= 0, "evidence_tempered: bad nbin/nsteps/swap_every");
  MG_REQUIRE(ctx, cfg->nbin < 2147483647LL - cfg->nsteps, "evidence_tempered: nbin + nsteps must stay below 2^31");
  for (int k = 0; k < T; ++k)
    MG_REQUIRE(ctx, std::isfinite(betas[k]) && (k == 0 ? betas[0] >= 0.0 : betas[k] > betas[k - 1]),
               "evidence_tempered: betas must be finite, >= 0 and strictly increasing");
  MG_REQUIRE(ctx, betas[T - 1] == 1.0, "evidence_tempered: the last beta must be 1");
  // the swap draws address ladder m's pair k as chain (ladder_offset + m) * 32 + k of the 48-bit chain id (rng.cuh)
  MG_REQUIRE(ctx, cfg->ladder_offset < (1ull << 43) && (uint64_t)cfg->nladders <= (1ull << 43) - cfg->ladder_offset,
             "evidence_tempered: global ladder ids must stay below 2^43");
  int rc;
  if ((rc = validate_logfn(ctx, like, D, "log_likelihood"))) return rc;
  if ((rc = validate_logfn(ctx, prior, D, "log_prior"))) return rc;
  for (int k = 0; k < T; ++k)
    if ((rc = validate_proposal(ctx, props + k, D))) return rc;
  return MG_OK;
}

// Runs this rank's ladders and reduces them to rec.r; writes out->final and out->ladder_mean_ll.
static int tp_run(mg_ctx *ctx, const mg_logfn *like, const mg_logfn *prior, const mg_proposal *props,
                  const double *betas, const mg_tempered_cfg *cfg, const double *x0, mg_tempered_out *out,
                  TpRecord &rec) {
  const int T = cfg->ntemps, D = cfg->dim;
  const int64_t M = cfg->nladders, MT = M * T;
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  DevLogFn dl, dp;
  DevProposal dj[TP_MAXT];
  DevBuf<double> d_x0, d_lmean, d_la, d_ls, d_final;
  DevBuf<int32_t> d_acc, d_sacc;
  DevBuf<TpRankRec> d_rec;
  MG_CUDA(ctx, dl.upload_from(like, s));
  MG_CUDA(ctx, dp.upload_from(prior, s));
  TpArgs a;
  memset(&a, 0, sizeof a);
  for (int k = 0; k < T; ++k) {
    MG_CUDA(ctx, dj[k].upload_from(props + k, s));
    a.props[k] = dj[k].params;
    a.betas[k] = betas[k];
  }
  MG_CUDA(ctx, upload(d_x0, x0, cfg->x0_shared ? (size_t)D : (size_t)M * D, s));
  MG_CUDA(ctx, d_lmean.alloc((size_t)MT, s));
  MG_CUDA(ctx, d_la.alloc((size_t)MT, s));
  MG_CUDA(ctx, d_ls.alloc((size_t)MT, s));
  MG_CUDA(ctx, d_acc.alloc((size_t)MT, s));
  MG_CUDA(ctx, d_sacc.alloc((size_t)MT, s));
  MG_CUDA(ctx, d_rec.alloc(1, s));
  if (out->final) MG_CUDA(ctx, d_final.alloc((size_t)MT * (D + 2), s));
  a.like = dl.params; a.prior = dp.params;
  a.d = D; a.T = T; a.M = M; a.ladder_offset = cfg->ladder_offset;
  a.nbin = cfg->nbin; a.nsteps = cfg->nsteps; a.swap_every = cfg->swap_every;
  a.x0_shared = cfg->x0_shared ? 1 : 0;
  a.key = next_key(ctx);
  a.rk = make_round_keys(a.key);
  a.x0 = d_x0.get(); a.lmean = d_lmean.get(); a.lse_a = d_la.get(); a.lse_s = d_ls.get();
  a.acc = d_acc.get(); a.sacc = d_sacc.get(); a.final = d_final.get();
  const int64_t per_warp = 32 / T, warps = (M + per_warp - 1) / per_warp;
  const unsigned grid = (unsigned)((warps * 32 + TP_BLOCK - 1) / TP_BLOCK);
  int rc;
  time_begin(ctx);
  if (like->kind >= MG_FN_USER || prior->kind >= MG_FN_USER) {   // user plugins: kernel compiled at run time
    if ((rc = jit_launch_tempered(ctx, a, D, grid, TP_BLOCK))) return rc;
  } else {
    const void *fn;
#define MG_TP_LAUNCH(DD)                                                   \
    do {                                                                   \
      fn = (const void *)tempered_kernel<DD>;                              \
      kt_reset(ctx, fn); kt_start(ctx);                                    \
      tempered_kernel<DD><<<grid, TP_BLOCK, 0, s>>>(a);                    \
      kt_stop(ctx);                                                        \
    } while (0)
    if (D <= 2) MG_TP_LAUNCH(2);
    else if (D <= 4) MG_TP_LAUNCH(4);
    else if (D <= 8) MG_TP_LAUNCH(8);
    else if (D <= 16) MG_TP_LAUNCH(16);
    else if (D <= 32) MG_TP_LAUNCH(32);
    else MG_TP_LAUNCH(64);
#undef MG_TP_LAUNCH
  }
  MG_CHECK_LAUNCH(ctx);
  time_end(ctx);
  tempered_reduce_kernel<<<1, 64, 0, s>>>(a, d_rec.get());
  MG_CHECK_LAUNCH(ctx);
  MG_CUDA(ctx, cudaMemcpyAsync(&rec.r, d_rec.get(), sizeof(TpRankRec), cudaMemcpyDeviceToHost, s));
  if (out->final)
    MG_CUDA(ctx, cudaMemcpyAsync(out->final, d_final.get(), sizeof(double) * (size_t)MT * (D + 2), cudaMemcpyDeviceToHost, s));
  if (out->ladder_mean_ll)
    MG_CUDA(ctx, cudaMemcpyAsync(out->ladder_mean_ll, d_lmean.get(), sizeof(double) * (size_t)MT, cudaMemcpyDeviceToHost, s));
  MG_CUDA(ctx, cudaStreamSynchronize(s));
  return MG_OK;
}

// Swap rounds of the measured phase (rounds that follow steps nbin .. nbin + nsteps - 1) that try pair (k, k+1).
static int64_t tp_swaps_tried(int64_t nbin, int64_t nsteps, int64_t every, int k) {
  if (every <= 0) return 0;
  const int64_t lo = (nbin + every) / every - 1;        // first round after a step t >= nbin: ceil((nbin+1)/every) - 1
  const int64_t hi = (nbin + nsteps) / every - 1;       // last round
  if (hi < lo) return 0;
  auto upto = [&](int64_t r) { return r < 0 ? 0 : (r - (k & 1)) / 2 + (r >= (k & 1) ? 1 : 0); };   // #{0 <= q <= r, q = k mod 2}
  return upto(hi) - upto(lo - 1);
}

// The records of the ranks, pooled in rank order (Chan's update, log-sum-exp), and the outputs: the finish of the
// single-GPU and the sharded call alike.
static void tp_finish(const std::vector<TpRecord> &recs, mg_tempered_out *out) {
  const TpRecord &h = recs[0];
  const int T = h.T;
  int64_t M = 0;
  for (const TpRecord &r : recs) M += r.M;
  auto chan = [](double &n, double &mean, double &m2, double &nf, double nb, double mb, double m2b, double nfb) {
    nf = nf + nfb;
    if (nb == 0.0) return;
    if (n == 0.0) { n = nb; mean = mb; m2 = m2b; return; }
    const double nn = n + nb, delta = mb - mean;
    mean = mean + delta * (nb / nn);
    m2 = m2 + m2b + delta * delta * (n * nb / nn);
    n = nn;
  };
  const double sqM = std::sqrt((double)M);
  auto sd_err = [&](double n, double m2, double nf) {   // sd over ladders / sqrt(M); NaN if M = 1 or a value is not finite
    return nf == 0.0 ? std::sqrt(m2 / (n - 1.0)) / sqM : std::nan("");
  };
  std::vector<double> mean_ll((size_t)T);
  double log_z_ss = 0.0;
  for (int k = 0; k < T; ++k) {
    double n = 0.0, mean = 0.0, m2 = 0.0, nf = 0.0, A = -HUGE_VAL, S = 0.0;
    int64_t acc = 0, sacc = 0;
    for (const TpRecord &r : recs) {
      chan(n, mean, m2, nf, r.r.n[k], r.r.mean[k], r.r.m2[k], r.r.nf[k]);
      tp_lse_add(A, S, r.r.lse_a[k] + std::log(r.r.lse_s[k]));
      acc += r.r.acc[k]; sacc += r.r.sacc[k];
    }
    mean_ll[k] = nf == 0.0 ? mean : nf;
    if (out->mean_ll) out->mean_ll[k] = mean_ll[k];
    if (out->mean_ll_err) out->mean_ll_err[k] = sd_err(n, m2, nf);
    if (out->accept) out->accept[k] = acc;
    if (k + 1 < T) {
      log_z_ss = log_z_ss + ((A + std::log(S)) - std::log((double)M * (double)h.nsteps));
      if (out->swaps_accepted) out->swaps_accepted[k] = sacc;
      if (out->swaps_tried) out->swaps_tried[k] = M * tp_swaps_tried(h.nbin, h.nsteps, h.swap_every, k);
    }
  }
  double log_z_ti = 0.0;
  for (int k = 0; k + 1 < T; ++k) log_z_ti = log_z_ti + (h.betas[k + 1] - h.betas[k]) * (mean_ll[k] + mean_ll[k + 1]) / 2.0;
  double ti[4] = {0.0, 0.0, 0.0, 0.0}, ss[4] = {0.0, 0.0, 0.0, 0.0};
  for (const TpRecord &r : recs) {
    chan(ti[0], ti[1], ti[2], ti[3], r.r.ti[0], r.r.ti[1], r.r.ti[2], r.r.ti[3]);
    chan(ss[0], ss[1], ss[2], ss[3], r.r.ss[0], r.r.ss[1], r.r.ss[2], r.r.ss[3]);
  }
  out->log_z_ss = log_z_ss;
  out->log_z_ss_err = sd_err(ss[0], ss[2], ss[3]);
  out->log_z_ti = log_z_ti;
  out->log_z_ti_err = sd_err(ti[0], ti[2], ti[3]);
}

static void tp_header(const mg_tempered_cfg *cfg, const double *betas, TpRecord &rec) {
  memset(&rec, 0, sizeof rec);
  rec.T = cfg->ntemps; rec.D = cfg->dim; rec.nbin = cfg->nbin; rec.nsteps = cfg->nsteps;
  rec.swap_every = cfg->swap_every; rec.M = cfg->nladders;
  for (int k = 0; k < cfg->ntemps; ++k) rec.betas[k] = betas[k];
}

}  // namespace mg

using namespace mg;

extern "C" int mg_evidence_tempered(mg_ctx *ctx, const mg_logfn *like, const mg_logfn *prior, const mg_proposal *props,
                                    const double *betas, const mg_tempered_cfg *cfg, const double *x0,
                                    mg_tempered_out *out) {
  if (!ctx) return MG_EINVAL;
  int rc;
  if ((rc = tp_validate(ctx, like, prior, props, betas, cfg, x0, out))) return rc;
  std::vector<TpRecord> recs(1);
  tp_header(cfg, betas, recs[0]);
  if ((rc = tp_run(ctx, like, prior, props, betas, cfg, x0, out, recs[0]))) return rc;
  tp_finish(recs, out);
  return MG_OK;
}

extern "C" int mg_evidence_tempered_sharded(mg_comm *c, const mg_logfn *like, const mg_logfn *prior,
                                            const mg_proposal *props, const double *betas, const mg_tempered_cfg *cfg,
                                            const double *x0, mg_tempered_out *out) {
  if (!c) return MG_EINVAL;
  mg_ctx *ctx = mg_comm_ctx(c);
  std::vector<TpRecord> mine(1), all;
  int rc = tp_validate(ctx, like, prior, props, betas, cfg, x0, out);
  if (rc == MG_OK) {
    tp_header(cfg, betas, mine[0]);
    rc = tp_run(ctx, like, prior, props, betas, cfg, x0, out, mine[0]);
  } else {
    ctx->epoch++;   // every rank consumes the same epoch of its context's key
  }
  if ((rc = comm_gather(c, rc, mine, all, "evidence_tempered (sharded)"))) return rc;
  const TpRecord &h = all[0];
  for (size_t r = 1; r < all.size(); ++r) {
    const TpRecord &o = all[r];
    bool same = o.T == h.T && o.D == h.D && o.nbin == h.nbin && o.nsteps == h.nsteps && o.swap_every == h.swap_every;
    for (int k = 0; same && k < h.T; ++k) same = memcmp(&o.betas[k], &h.betas[k], sizeof(double)) == 0;
    MG_REQUIRE(ctx, same, "evidence_tempered (sharded): rank %d has another ntemps, betas, dim, nbin, nsteps or swap_every", (int)r);
  }
  tp_finish(all, out);
  return MG_OK;
}
