// tempered_oracle.cpp -- TEST INFRASTRUCTURE (oracle).  Not part of the product.  The CPU restatement of
// mg_evidence_tempered (include/mcmc_gpu.h, "Evidence by parallel tempering"): ladders run replica by replica with the
// same plugin objects (og_models.hpp) and the same counter-based stream (og_rng.hpp) as the Metropolis-Hastings oracle
// in oracle.cpp, std::exp / std::log for the transcendentals.  Built on demand by oracle/tempered.py with the flags of
// oracle/Makefile.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "og_models.hpp"
#include "og_rng.hpp"

using namespace og;

// The swap draws' purpose, an addition to the stream layout of og_rng.hpp (P_PT_SWAP in the library's rng.cuh)
static constexpr uint32_t P_PT_SWAP = 10;

static thread_local std::string g_err;
static int fail(int code, const std::string &m) { g_err = m; return code; }

// the smallest |log u - log_accept_prob| since the last reset (the near-tie diagnostic of oracle.cpp)
static thread_local double tl_margin = HUGE_VAL;
static inline void note_margin(double log_u, double log_accept_prob) {
  const double m = std::fabs(log_u - log_accept_prob);
  if (m < tl_margin) tl_margin = m;
}

// mcmc.ml:37-56, as oracle.cpp's mh_step
template <class LL, class LP, class JP, class LJP>
static inline bool mh_step(Rng &r, int D, double *x, double &ll, double &lp, double *prop,
                           LL &&log_likelihood, LP &&log_prior, JP &&jump_proposal,
                           LJP &&log_jump_prob) {
  double start_log_post = ll + lp;
  jump_proposal(r, x, prop);
  double proposed_like = log_likelihood(prop), proposed_prior = log_prior(prop);
  double proposed_log_posterior = proposed_like + proposed_prior;
  double log_forward_jump = log_jump_prob(x, prop), log_backward_jump = log_jump_prob(prop, x);
  double log_accept_prob =
      proposed_log_posterior - start_log_post + log_backward_jump - log_forward_jump;
  const double log_u = std::log(r.uniform());
  note_margin(log_u, log_accept_prob);
  if (log_u < log_accept_prob) {  // strict <, :47
    for (int i = 0; i < D; ++i) x[i] = prop[i];
    ll = proposed_like; lp = proposed_prior;
    return true;
  }
  return false;
}

template <class F>
static void parallel_for(int64_t n, int nthreads, F &&f) {
  if (nthreads <= 1 || n <= 1) { for (int64_t i = 0; i < n; ++i) f(i); return; }
  std::vector<std::thread> th;
  int T = (int)std::min<int64_t>(nthreads, n);
  for (int t = 0; t < T; ++t)
    th.emplace_back([&, t]() { for (int64_t i = t; i < n; i += T) f(i); });
  for (auto &x : th) x.join();
}

// log-sum-exp accumulation: a the running maximum, s = sum exp(w - a); w = -inf adds nothing, NaN poisons s
static inline void pt_lse_add(double &a, double &s, double w) {
  if (w > a) { s = s * std::exp(a - w) + 1.0; a = w; }
  else if (!(w < -1.7976931348623157e308)) s = s + std::exp(w - a);
}
// Welford over the finite values; the non-finite ones are summed apart
static inline void pt_welford(double &n, double &mean, double &m2, double &nf, double x) {
  if (std::isfinite(x)) {
    n = n + 1.0;
    const double delta = x - mean;
    mean = mean + delta / n;
    m2 = m2 + delta * (x - mean);
  } else {
    nf = nf + x;
  }
}

// One ladder (global id gl) of T rungs, run replica by replica with the swap rounds between steps.
// Per rung: Lm = p + S1 / nsteps, (la, ls), accepted MH steps, accepted swaps of pair (k, k+1); final [T][D+2];
// margin [T]: the smallest |log u - log_accept| over the MH tests of the rung and the swap tests it takes part in.
static void pt_ladder(const CallKey &ck, const LogFn &like, const LogFn &prior, const std::vector<Proposal> &props,
                      const double *betas, const mg_tempered_cfg &cfg, const double *start, uint64_t gl, double *Lm,
                      double *la, double *ls, int64_t *acc, int64_t *sacc, int64_t *stried, double *fin, double *margin) {
  const int T = cfg.ntemps, D = cfg.dim;
  std::vector<std::vector<double>> x(T, std::vector<double>(start, start + D));
  std::vector<double> ll(T), lp(T), p(T, 0.0), sum(T, 0.0), comp(T, 0.0), nf(T, 0.0), y(D);
  for (int k = 0; k < T; ++k) {
    ll[k] = like(x[k].data()); lp[k] = prior(x[k].data());   // mcmc.ml:59-61
    la[k] = -HUGE_VAL; ls[k] = 0.0; acc[k] = 0; sacc[k] = 0; stried[k] = 0; margin[k] = HUGE_VAL;
  }
  for (int64_t t = 0; t < cfg.nbin + cfg.nsteps; ++t) {
    for (int k = 0; k < T; ++k) {   // tempered mh_step: tl(x) = (beta == 0 ? 0 : beta * ll) + lp
      const double b = betas[k];
      const uint64_t g = gl * (uint64_t)T + (uint64_t)k;
      tl_margin = HUGE_VAL;
      Rng r(ck, P_MH, g, (uint64_t)t);
      auto L = [&](const double *v) { return like(v); };
      auto P = [&](const double *v) { return prior(v); };
      auto J = [&](Rng &rr, const double *a, double *bb) { props[k].propose(rr, a, bb); };
      auto Q = [&](const double *a, const double *bb) { return props[k].log_q(a, bb); };
      double tll = b == 0.0 ? 0.0 : b * ll[k];
      // mh_step on (tempered ll, lp): the accepted proposal's plain ll is kept alongside
      double pl = 0.0;
      auto TL = [&](const double *v) { pl = L(v); return b == 0.0 ? 0.0 : b * pl; };
      double tll_new = tll;
      const bool a = mh_step(r, D, x[k].data(), tll_new, lp[k], y.data(), TL, P, J, Q);
      if (a) ll[k] = pl;
      margin[k] = std::min(margin[k], tl_margin);
      if (a && t >= cfg.nbin) acc[k]++;
    }
    if (cfg.swap_every > 0 && (t + 1) % cfg.swap_every == 0) {
      const int64_t r = (t + 1) / cfg.swap_every - 1;
      for (int k = (int)(r & 1); k + 1 < T; k += 2) {
        Rng rr(ck, P_PT_SWAP, gl * 32u + (uint64_t)k, (uint64_t)r);
        const double log_u = std::log(rr.uniform());
        const double delta = (betas[k + 1] - betas[k]) * (ll[k] - ll[k + 1]);
        const double mg = std::fabs(log_u - delta);
        if (mg < margin[k]) margin[k] = mg;
        if (mg < margin[k + 1]) margin[k + 1] = mg;
        if (t >= cfg.nbin) stried[k]++;
        if (log_u < delta) {
          std::swap(x[k], x[k + 1]); std::swap(ll[k], ll[k + 1]); std::swap(lp[k], lp[k + 1]);
          if (t >= cfg.nbin) sacc[k]++;
        }
      }
    }
    if (t >= cfg.nbin) {
      for (int k = 0; k < T; ++k) {
        if (t == cfg.nbin) p[k] = std::isfinite(ll[k]) ? ll[k] : 0.0;
        const double v = ll[k] - p[k];
        if (std::isfinite(v)) {   // Neumaier
          const double s2 = sum[k] + v;
          if (std::fabs(sum[k]) >= std::fabs(v)) comp[k] = comp[k] + ((sum[k] - s2) + v);
          else comp[k] = comp[k] + ((v - s2) + sum[k]);
          sum[k] = s2;
        } else {
          nf[k] = nf[k] + v;
        }
        if (k + 1 < T) pt_lse_add(la[k], ls[k], (betas[k + 1] - betas[k]) * ll[k]);
      }
    }
  }
  for (int k = 0; k < T; ++k) {
    Lm[k] = p[k] + ((sum[k] + comp[k]) + nf[k]) / (double)cfg.nsteps;
    if (fin) {
      for (int i = 0; i < D; ++i) fin[k * (D + 2) + i] = x[k][i];
      fin[k * (D + 2) + D] = ll[k]; fin[k * (D + 2) + D + 1] = lp[k];
    }
  }
}


#define OG_TRY try {
#define OG_CATCH                                                             \
  }                                                                          \
  catch (const std::invalid_argument &e) { return fail(MG_EINVAL, e.what()); } \
  catch (const std::exception &e) { return fail(MG_EFAIL, e.what()); }

extern "C" {

const char *og_tempered_last_error() { return g_err.c_str(); }

// mg_evidence_tempered.  margin: [M][T] or null (near-tie diagnostic, see pt_ladder); swaps_tried: counted, not
// computed from a formula
int og_evidence_tempered(uint64_t seed, uint64_t epoch, const mg_logfn *like, const mg_logfn *prior,
                         const mg_proposal *props, const double *betas, const mg_tempered_cfg *cfg, const double *x0,
                         mg_tempered_out *out, double *margin, int nthreads) {
  OG_TRY
  const int T = cfg->ntemps, D = cfg->dim;
  const int64_t M = cfg->nladders;
  if (M < 1 || T < 2 || T > 32 || cfg->nsteps < 1 || cfg->nbin < 0 || cfg->swap_every < 0)
    return fail(MG_EINVAL, "evidence_tempered: bad arguments");
  for (int k = 0; k < T; ++k)
    if (!std::isfinite(betas[k]) || (k == 0 ? betas[0] < 0.0 : !(betas[k] > betas[k - 1])))
      return fail(MG_EINVAL, "evidence_tempered: bad betas");
  if (betas[T - 1] != 1.0) return fail(MG_EINVAL, "evidence_tempered: the last beta must be 1");
  LogFn L(like), P(prior);
  std::vector<Proposal> J;
  for (int k = 0; k < T; ++k) J.emplace_back(props + k);
  const CallKey ck = derive_key(seed, epoch);
  const size_t MT = (size_t)M * T;
  std::vector<double> Lm(MT), la(MT), ls(MT), mg(MT);
  std::vector<int64_t> acc(MT), sacc(MT), stried(MT);
  parallel_for(M, nthreads, [&](int64_t m) {
    const double *s = cfg->x0_shared ? x0 : x0 + m * D;
    pt_ladder(ck, L, P, J, betas, *cfg, s, cfg->ladder_offset + (uint64_t)m, &Lm[m * T], &la[m * T], &ls[m * T],
              &acc[m * T], &sacc[m * T], &stried[m * T], out->final ? out->final + (size_t)m * T * (D + 2) : nullptr,
              &mg[m * T]);
  });
  if (margin) std::copy(mg.begin(), mg.end(), margin);
  if (out->ladder_mean_ll) std::copy(Lm.begin(), Lm.end(), out->ladder_mean_ll);
  // pooled over the ladders in ladder order
  const double ns = (double)cfg->nsteps, sqM = std::sqrt((double)M);
  auto err = [&](double n, double m2, double nf) { return nf == 0.0 ? std::sqrt(m2 / (n - 1.0)) / sqM : std::nan(""); };
  std::vector<double> mean_ll(T);
  double log_z_ss = 0.0;
  for (int k = 0; k < T; ++k) {
    double n = 0.0, mean = 0.0, m2 = 0.0, nf = 0.0, A = -HUGE_VAL, S = 0.0;
    int64_t a = 0, sa = 0, st = 0;
    for (int64_t m = 0; m < M; ++m) {
      pt_welford(n, mean, m2, nf, Lm[m * T + k]);
      if (k + 1 < T) pt_lse_add(A, S, la[m * T + k] + std::log(ls[m * T + k]));
      a += acc[m * T + k]; sa += sacc[m * T + k]; st += stried[m * T + k];
    }
    mean_ll[k] = nf == 0.0 ? mean : nf;
    if (out->mean_ll) out->mean_ll[k] = mean_ll[k];
    if (out->mean_ll_err) out->mean_ll_err[k] = err(n, m2, nf);
    if (out->accept) out->accept[k] = a;
    if (k + 1 < T) {
      double A1 = -HUGE_VAL, S1 = 0.0;        // the rank pooling of the library, with one rank
      pt_lse_add(A1, S1, A + std::log(S));
      log_z_ss = log_z_ss + ((A1 + std::log(S1)) - std::log((double)M * ns));
      if (out->swaps_accepted) out->swaps_accepted[k] = sa;
      if (out->swaps_tried) out->swaps_tried[k] = st;
    }
  }
  double log_z_ti = 0.0;
  for (int k = 0; k + 1 < T; ++k) log_z_ti = log_z_ti + (betas[k + 1] - betas[k]) * (mean_ll[k] + mean_ll[k + 1]) / 2.0;
  double ti[4] = {0, 0, 0, 0}, ss[4] = {0, 0, 0, 0};
  for (int64_t m = 0; m < M; ++m) {
    double tim = 0.0, ssm = 0.0;
    for (int q = 0; q + 1 < T; ++q) {
      tim = tim + (betas[q + 1] - betas[q]) * (Lm[m * T + q] + Lm[m * T + q + 1]) / 2.0;
      ssm = ssm + (la[m * T + q] + std::log(ls[m * T + q] / ns));
    }
    pt_welford(ti[0], ti[1], ti[2], ti[3], tim);
    pt_welford(ss[0], ss[1], ss[2], ss[3], ssm);
  }
  out->log_z_ss = log_z_ss; out->log_z_ss_err = err(ss[0], ss[2], ss[3]);
  out->log_z_ti = log_z_ti; out->log_z_ti_err = err(ti[0], ti[2], ti[3]);
  return MG_OK;
  OG_CATCH
}

}  // extern "C"
