// tempered_kernel_dev.cuh -- device side of the parallel-tempering evidence kernel (include/mcmc_gpu.h, "Evidence by
// parallel tempering", has the definition).  No host includes: this header is also compiled at run time by NVRTC for
// user-registered plugins (jit.cu).
//
// Mapping: one replica (ladder m, rung k) per lane; ladder j of a warp takes lanes [jT, jT + T), so a warp holds
// floor(32 / T) ladders.  Lanes past the last whole ladder, and the ladders past M, run no steps but take part in the
// shuffles of the swap rounds.  State, pivot, compensated sum, log-sum-exp pair and counters stay in registers for the
// whole run; the only global stores are each replica's record at the end.
#pragma once
#include "models.cuh"
#include "rng.cuh"

namespace mg {

#ifndef MG_TP_MAXNREG
#define MG_TP_MAXNREG(D) ((D) <= 10 ? 128 : 255)
#endif
constexpr int TP_BLOCK = 64;
constexpr int TP_MAXT = 32;

struct TpArgs {
  DynFnParams like, prior;
  DynPropParams props[TP_MAXT];
  double betas[TP_MAXT];
  int32_t d, T;
  int64_t M;
  uint64_t ladder_offset;
  int64_t nbin, nsteps, swap_every;
  int32_t x0_shared, pad;
  CallKey key;
  RoundKeys rk;
  const double *x0;       // [M][D] or [D]
  double *lmean;          // [M][T] p + S1 / nsteps
  double *lse_a, *lse_s;  // [M][T] (a, s); rung T-1 unused
  int32_t *acc;           // [M][T] accepted MH steps (measured phase)
  int32_t *sacc;          // [M][T] accepted swaps of pair (k, k+1), recorded by rung k
  double *final;          // [M][T][D+2] or null
};

// The per-rank record of the ladders of one call: what the sharded call exchanges.  Per rung k: the Welford mean and
// M2 of the finite L_mk and their count, the sum of the non-finite ones, the log-sum-exp of a_mk + log s_mk; the same
// moments for TI_m and SS_m (n, mean, M2, non-finite sum); the int64 counts.
struct TpRankRec {
  double n[TP_MAXT], mean[TP_MAXT], m2[TP_MAXT], nf[TP_MAXT];
  double lse_a[TP_MAXT], lse_s[TP_MAXT];
  double ti[4], ss[4];
  long long acc[TP_MAXT], sacc[TP_MAXT];
};

// log-sum-exp accumulation from (a, s) = (-inf, 0): a is the running maximum, s = sum exp(w - a).  w = -inf adds
// nothing (w < -DBL_MAX); a NaN makes s NaN.
__host__ __device__ __forceinline__ void tp_lse_add(double &a, double &s, double w) {
  if (w > a) { s = s * exp(a - w) + 1.0; a = w; }
  else if (!(w < -1.7976931348623157e308)) s = s + exp(w - a);
}
// Welford's update over the finite values; the non-finite ones are summed apart (nf) and take the result over
__host__ __device__ __forceinline__ void tp_welford(double &n, double &mean, double &m2, double &nf, double x) {
  if (isfinite(x)) {
    n = n + 1.0;
    const double delta = x - mean;
    mean = mean + delta / n;
    m2 = m2 + delta * (x - mean);
  } else {
    nf = nf + x;
  }
}

// mh_step (mcmc_kernel_dev.cuh) with the log posterior tl(x) = (beta == 0 ? 0 : beta * ll(x)) + lp(x); the shared
// step is not given a beta branch so that the plain sampler's code does not change.
template <int D, class RNG>
__device__ __forceinline__ int tp_mh_step(const TpArgs &a, const DynPropParams &prop, double beta, RNG &r,
                                          double (&x)[D], double &ll, double &lp) {
  const int dd = a.d;
  const double start_log_post = (beta == 0.0 ? 0.0 : beta * ll) + lp;
  double y[D];
  DynProp::template propose<D, RNG>(prop, nullptr, r, x, y, dd);
  const double proposed_like = DynFn::template eval<D>(a.like, nullptr, y, dd);
  const double proposed_prior = DynFn::template eval<D>(a.prior, nullptr, y, dd);
  const double proposed_log_posterior = (beta == 0.0 ? 0.0 : beta * proposed_like) + proposed_prior;
  double log_accept_prob = proposed_log_posterior - start_log_post;
  const double log_forward_jump = DynProp::template log_q<D>(prop, nullptr, x, y, dd);
  const double log_backward_jump = DynProp::template log_q<D>(prop, nullptr, y, x, dd);
  log_accept_prob = log_accept_prob + log_backward_jump - log_forward_jump;
  const bool acc = log_u_less_than(r.uniform(), log_accept_prob);
#pragma unroll
  for (int i = 0; i < D; ++i) x[i] = acc ? y[i] : x[i];
  ll = acc ? proposed_like : ll;
  lp = acc ? proposed_prior : lp;
  return acc ? 1 : 0;
}

template <int D>
__device__ __forceinline__ void tempered_body(const TpArgs &a) {
  const unsigned FULL = 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31;
  const int T = a.T, dd = a.d;
  const int per_warp = 32 / T;
  const int j = lane / T, k = lane - j * T;
  const int64_t warp = ((int64_t)blockIdx.x * TP_BLOCK + threadIdx.x) >> 5;
  const int64_t m = warp * per_warp + j;
  const bool live = j < per_warp && m < a.M;
  const int kk = live ? k : 0;
  const int64_t mm = live ? m : 0;
  const uint64_t gl = a.ladder_offset + (uint64_t)mm;
  const uint64_t g = gl * (uint64_t)T + (uint64_t)kk;
  const DynPropParams prop = a.props[kk];
  const double beta = a.betas[kk];
  const double dlo = kk + 1 < T ? a.betas[kk + 1] - beta : 0.0;   // beta_k+1 - beta_k (pair k, k+1)
  const double dhi = kk > 0 ? beta - a.betas[kk - 1] : 0.0;        // beta_k - beta_k-1 (pair k-1, k)
  double x[D];
  const double *x0 = a.x0_shared ? a.x0 : a.x0 + mm * dd;
#pragma unroll
  for (int i = 0; i < D; ++i) x[i] = (i < dd) ? x0[i] : 0.0;
  double ll = DynFn::template eval<D>(a.like, nullptr, x, dd);   // mcmc.ml:59-61
  double lp = DynFn::template eval<D>(a.prior, nullptr, x, dd);
  double p = 0.0, sum = 0.0, comp = 0.0, nf = 0.0;
  double la = neg_inf(), ls = 0.0;
  int nacc = 0, nsw = 0;
  const int64_t nt = a.nbin + a.nsteps;
  int64_t until_swap = a.swap_every, rr = 0;   // steps to the next swap round, its number
  for (int64_t t = 0; t < nt; ++t) {
    int acc = 0;
    if (live) {
      Rng r(a.key, P_MH, g, (uint64_t)t, &a.rk);
      acc = tp_mh_step<D>(a, prop, beta, r, x, ll, lp);
    }
    if (a.swap_every > 0 && --until_swap == 0) {
      until_swap = a.swap_every;
      const int par = (int)(rr & 1);
      const bool low = ((k & 1) == par) && k + 1 < T;     // this lane is rung k of pair (k, k+1)
      const bool high = ((k & 1) != par) && k > 0;        // this lane is rung k+1 of pair (k, k+1)
      const int src = low ? lane + 1 : high ? lane - 1 : lane;
      const double llo = __shfl_sync(FULL, ll, src);
      bool sw = false;
      if (live && (low || high)) {
        const int kl = low ? k : k - 1;
        const double ll_lo = low ? ll : llo, ll_hi = low ? llo : ll;
        Rng r(a.key, P_PT_SWAP, gl * (uint64_t)TP_MAXT + (uint64_t)kl, (uint64_t)rr);
        sw = log_u_less_than(r.uniform(), (low ? dlo : dhi) * (ll_lo - ll_hi));
      }
      if (__any_sync(FULL, sw)) {
#pragma unroll
        for (int i = 0; i < D; ++i) {
          if (i < dd) { const double o = __shfl_sync(FULL, x[i], src); x[i] = sw ? o : x[i]; }
        }
        const double lpo = __shfl_sync(FULL, lp, src);
        ll = sw ? llo : ll;
        lp = sw ? lpo : lp;
      }
      if (t >= a.nbin && sw && low) ++nsw;
      ++rr;
    }
    if (t >= a.nbin) {
      nacc += acc;
      if (t == a.nbin) p = isfinite(ll) ? ll : 0.0;
      const double v = ll - p;
      if (isfinite(v)) {   // Neumaier
        const double s2 = sum + v;
        if (fabs(sum) >= fabs(v)) comp = comp + ((sum - s2) + v);
        else comp = comp + ((v - s2) + sum);
        sum = s2;
      } else {
        nf = nf + v;
      }
      if (kk + 1 < T) tp_lse_add(la, ls, dlo * ll);
    }
  }
  if (!live) return;
  const int64_t idx = m * T + k;
  a.lmean[idx] = p + ((sum + comp) + nf) / (double)a.nsteps;
  a.lse_a[idx] = la;
  a.lse_s[idx] = ls;
  a.acc[idx] = nacc;
  a.sacc[idx] = nsw;
  if (a.final) {
    double *f = a.final + idx * (dd + 2);
#pragma unroll
    for (int i = 0; i < D; ++i)
      if (i < dd) f[i] = x[i];
    f[dd] = ll;
    f[dd + 1] = lp;
  }
}

}  // namespace mg
