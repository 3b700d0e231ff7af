// nested.cu -- Nested.nested_evidence (nested.ml:122-146) with batched
// constrained live-point replacement.
//
// The reference retires ONE live point per iteration and replaces it with the
// end point of an nmcmc-step constrained Metropolis-Hastings chain whose
// proposal is differential evolution over the current live set
// (nested.ml:50-74, mcmc.ml:198-218): nmcmc sequential likelihood calls per
// retired point.  Here the K lowest points are retired together
// (cfg.batch = K; K = 1 is the reference's schedule): K independent
// replacement chains run as one kernel, one thread per chain, all constrained
// to ll >= the K-th lowest log-likelihood; the j-th point of a batch leaves
// nlive - j points above it, so its shrinkage factor is 1 - 1/(nlive - j)
// (with j = 0 always, K = 1 reproduces nested.ml:131,139 operation for
// operation).  The live set ([nlive][D] rows, 12.8 MB at BASELINE config 4)
// stays L2-resident; the DE proposal gathers two rows per step.
#include "common.cuh"
#include "host_plugins.hpp"
#include "nested_kernel_dev.cuh"
#include "radix_sort.cuh"
#include "reduce_sum.cuh"

#include <cuda_pipeline.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>

namespace mg {

template <int DMAX>
__global__ void nest_init_kernel(NestArgs a, double *__restrict__ x_out, double *__restrict__ ll_out,
                                 double *__restrict__ lp_out) {
  nest_init_body<DMAX>(a, x_out, ll_out, lp_out);
}
template <int DMAX>
__global__ void nest_replace_simple_kernel(NestArgs a, NestProp p, int s0, int s1, int first, int last, double *chain_x,
                                           double *chain_cl) {
  nest_replace_simple_body<DMAX>(a, p, s0, s1, first, last, chain_x, chain_cl);
}
// user plugins: the two kernels above compiled at run time with the registered functions inlined (jit.cu)
int jit_launch_nest_init(mg_ctx *ctx, int D, const NestArgs &a, double *x_out, double *ll_out, double *lp_out);
int jit_launch_nest_replace(mg_ctx *ctx, int D, const NestArgs &a, const NestProp &p, int s0, int s1, int first, int last,
                            double *chain_x, double *chain_cl);

// draw_new_live_point (nested.ml:50-74) in two kernels.
//
// A step of the constrained chain is: a differential-evolution proposal (two
// live-point indices, a scale that is 1 or a Gaussian draw -- mcmc.ml:198-218),
// the likelihood of the proposed point, and the accept test.  Only the last
// two depend on the chain's state; the proposal's random part does not.  With
// one batch of K chains the kernel is latency-bound (K = 8,192 is 256 warps
// on 592 schedulers, nmcmc strictly sequential steps), so what counts is the
// length of the dependent path per step.  nest_propose_kernel therefore draws
// the random part of every (chain, step) up front, one thread each, at full
// occupancy; nest_replace_kernel then walks the steps with the two live rows
// of step s+1 already in flight while step s computes, leaving
// y = x + delta, the log-likelihood and the comparison on the critical path.
// Same Philox stream, same draw order per (chain, step), same arithmetic:
// output identical to the single-kernel form.
constexpr int NEST_BLOCK = 32;   // threads per CTA of nest_replace_kernel
constexpr int kSR = 4;           // stages of the proposal-scalar ring (step s reads s and s+1, writes s+2)
// doubles per staged live row: 16-byte aligned and an odd number of 16-byte units when D % 4 == 0 (conflict-free
// 128-bit reads by the row's owner); odd D: an odd number of doubles
__host__ __device__ constexpr int nest_row_stride(int D) { return (D % 2 == 0) ? D + 2 : (D | 1); }

__global__ void nest_propose_kernel(NestArgs a, NestProp p, int s0, int S) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)S * a.K) return;
  const int s = (int)(idx / a.K), j = (int)(idx % a.K);
  Rng r(a.key, P_NEST_MCMC, (uint64_t)(a.R + j), (uint64_t)(s0 + s));
  const uint64_t n = (uint64_t)a.nlive;
  const uint64_t i0 = r.below(n);
  uint64_t j0;
  do { j0 = r.below(n); } while (j0 == i0);
  double dscale;
  if (a.mode_hop != 0.0 && r.uniform() < a.mode_hop) dscale = 1.0;
  else dscale = draw_gaussian(r, 0.0, a.de_sigma);
  p.i0[idx] = (int32_t)i0; p.j0[idx] = (int32_t)j0; p.ds[idx] = dscale; p.u[idx] = r.uniform();
}

// chain_x [DMAX][K], chain_cl [K]: chain state between launches when nmcmc is walked in several chunks.
// kFull: the run-time dimension equals DMAX, every `d < D` guard folds away.
//
// One warp per CTA, one thread per chain.  The two live rows a step needs are gathered by the WARP, not by the
// thread: consecutive lanes copy consecutive 16-byte (8-byte when D is odd) pieces of a row straight into shared
// memory with cp.async, so a 128-byte row costs one line request instead of sixteen 8-byte requests from one lane
// (thread-per-row loads kept the L1 tag stage busy for ~1,000 cycles per step and every later load queued behind
// them).  Rows of step s+1 and scalars of step s+2 are in flight while step s computes.
// FAST (only with kFull): the plugin pair is known at compile time -- 1: Gaussian shell under a closed box, 2: under
// an open box (BASELINE.json config 4 and the reference's nested tests) -- and its parameters live in registers: no
// switch on the kind, no parameter loads in the step.  Same expressions as the SHELL / BOX cases of DynFn
// (models.cuh), so the chains are the same.  FAST = 0: any registered plugin pair through DynFn.
template <int DMAX, bool kFull, int FAST = 0>
__global__ void nest_replace_kernel(NestArgs a, NestProp p, int s0, int s1, int first, int last, double *chain_x,
                                    double *chain_cl) {
  static_assert(FAST == 0 || kFull, "the register-resident plugin pair needs D == DMAX");
  extern __shared__ __align__(16) double s_rows[];            // [2 stages][2 * NEST_BLOCK rows][RS]
  __shared__ int32_t s_i0[kSR][NEST_BLOCK], s_j0[kSR][NEST_BLOCK];
  __shared__ double s_ds[kSR][NEST_BLOCK], s_u[kSR][NEST_BLOCK];
  const int tx = threadIdx.x;
  const int K = a.K;
  const int jr = blockIdx.x * NEST_BLOCK + tx;
  const bool live = jr < K;
  const int j = live ? jr : K - 1;     // the whole warp takes part in the row copies; spare lanes shadow the last chain
  const int D = kFull ? DMAX : a.D;
  const bool vec = (D % 2) == 0;       // 16-byte pieces need even D (row starts are then 16-byte aligned)
  const int RS = nest_row_stride(D);   // doubles per staged row
  const double thr = a.threshold;
  // FAST: centre, (mu, sigma, log sigma) of the shell and the box in registers
  double f_c[FAST ? DMAX : 1], f_lo[FAST ? DMAX : 1], f_hi[FAST ? DMAX : 1];
  double f_mu = 0.0, f_sigma = 1.0, f_ls = 0.0, f_inside = 0.0;
  if (FAST) {
#pragma unroll
    for (int d = 0; d < DMAX; ++d) {
      f_c[d] = __ldg(a.like.p + d); f_lo[d] = __ldg(a.prior.p + d); f_hi[d] = __ldg(a.prior.p + DMAX + d);
    }
    f_mu = __ldg(a.like.p + DMAX); f_sigma = __ldg(a.like.p + DMAX + 1); f_ls = __ldg(a.like.p + a.like.np);
    f_inside = __ldg(a.prior.p + 2 * DMAX);
  }
  auto like_of = [&](const double (&pt)[DMAX]) -> double {
    if (FAST) {            // MG_FN_SHELL (models.cuh)
      double s = 0.0;
#pragma unroll
      for (int i = 0; i < DMAX; ++i) { const double dx = pt[i] - f_c[i]; s = s + dx * dx; }
      return log_gaussian_ls(f_mu, f_sigma, f_ls, sqrt(s));
    }
    return DynFn::eval<DMAX>(a.like, nullptr, pt, D);
  };
  auto prior_of = [&](const double (&pt)[DMAX]) -> double {
    if (FAST == 1) {       // MG_FN_BOX_CLOSED
      int out = 0;
#pragma unroll
      for (int i = 0; i < DMAX; ++i) out |= (int)(pt[i] < f_lo[i]) | (int)(pt[i] > f_hi[i]);
      return out ? neg_inf() : f_inside;
    }
    if (FAST == 2) {       // MG_FN_BOX_OPEN
      int in = 1;
#pragma unroll
      for (int i = 0; i < DMAX; ++i) in &= (int)(pt[i] > f_lo[i]) & (int)(pt[i] < f_hi[i]);
      return in ? f_inside : neg_inf();
    }
    return DynFn::eval<DMAX>(a.prior, nullptr, pt, D);
  };
  auto mcmc_logl = [&](const double (&pt)[DMAX]) {           // :54-59
    // both evaluated (they are pure and independent), then selected: nothing waits behind a branch
    const double l = like_of(pt);
    const double pr = prior_of(pt);
    return (l >= thr) ? pr : neg_inf();
  };
  double x[DMAX], y[DMAX], delta[DMAX];
  double cl;
  if (first) {
    Rng rs(a.key, P_NEST_START, (uint64_t)(a.R + j), 0);
    // livepts.(Random.int nlive) (:63); with K > 1 the start must satisfy the common threshold
    const int start = (a.K - 1) + (int)rs.below((uint64_t)(a.nlive - a.K + 1));
#pragma unroll (DMAX <= 16 ? DMAX : 1)
    for (int d = 0; d < DMAX; ++d) x[d] = (d < D) ? a.live_x[(int64_t)start * D + d] : 0.0;
    cl = mcmc_logl(x);
  } else {
#pragma unroll (DMAX <= 16 ? DMAX : 1)
    for (int d = 0; d < DMAX; ++d) x[d] = (d < D) ? chain_x[(int64_t)d * K + j] : 0.0;
    cl = chain_cl[j];
  }
  const double cp = 0.0;                                     // mcmc_logp, :60
  const int S = s1 - s0;
  auto fetch_scalars = [&](int t) {    // own column of the scalar ring
    if (t < S) {
      const int64_t q = (int64_t)t * K + j;
      const int st = t % kSR;
      __pipeline_memcpy_async(&s_i0[st][tx], p.i0 + q, 4);
      __pipeline_memcpy_async(&s_j0[st][tx], p.j0 + q, 4);
      __pipeline_memcpy_async(&s_ds[st][tx], p.ds + q, 8);
      __pipeline_memcpy_async(&s_u[st][tx], p.u + q, 8);
    }
  };
  auto fetch_rows = [&](int t) {       // rows x (0..31) and y (32..63) of all the warp's chains for step t
    if (t < S) {
      const int st = t % kSR;
      double *dst = s_rows + (size_t)(t & 1) * (2 * NEST_BLOCK) * RS;
      if (vec) {
        const int cpr = D / 2;         // 16-byte pieces per row
#pragma unroll (kFull && DMAX <= 16 ? DMAX : 1)
        for (int it = 0; it < 2 * cpr; ++it) {
          const int c = tx + it * NEST_BLOCK;
          const int row = c / cpr, k = c - row * cpr;
          const int idx = (row < NEST_BLOCK) ? s_i0[st][row] : s_j0[st][row - NEST_BLOCK];
          __pipeline_memcpy_async(dst + (size_t)row * RS + 2 * k, a.live_x + (int64_t)idx * D + 2 * k, 16);
        }
      } else {
        for (int c = tx; c < 2 * NEST_BLOCK * D; c += NEST_BLOCK) {
          const int row = c / D, k = c - row * D;
          const int idx = (row < NEST_BLOCK) ? s_i0[st][row] : s_j0[st][row - NEST_BLOCK];
          __pipeline_memcpy_async(dst + (size_t)row * RS + k, a.live_x + (int64_t)idx * D + k, 8);
        }
      }
    }
  };
  // prologue: scalars of steps 0 and 1, then rows of step 0
  fetch_scalars(0); fetch_scalars(1);
  __pipeline_commit();
  __pipeline_wait_prior(0);
  __syncwarp();
  fetch_rows(0);
  __pipeline_commit();
  for (int s = 0; s < S; ++s) {                              // :65-67
    __pipeline_wait_prior(0);          // rows of step s, scalars of step s+1
    __syncwarp();
    // delta = d * (y_row - x_row), mcmc.ml:214-216; own rows out of the staging buffer
    const int st = s % kSR;
    const double ds = s_ds[st][tx], u_cur = s_u[st][tx];
    {
      const double *rx = s_rows + (size_t)(s & 1) * (2 * NEST_BLOCK) * RS + (size_t)tx * RS;
      const double *ry = rx + (size_t)NEST_BLOCK * RS;
      if (kFull) {
        const double2 *rx2 = reinterpret_cast<const double2 *>(rx), *ry2 = reinterpret_cast<const double2 *>(ry);
#pragma unroll (DMAX <= 16 ? DMAX / 2 : 1)
        for (int d = 0; d < DMAX / 2; ++d) {
          const double2 vx = rx2[d], vy = ry2[d];
          delta[2 * d] = ds * (vy.x - vx.x); delta[2 * d + 1] = ds * (vy.y - vx.y);
        }
      } else {
#pragma unroll (DMAX <= 16 ? DMAX : 1)
        for (int d = 0; d < DMAX; ++d) delta[d] = (d < D) ? ds * (ry[d] - rx[d]) : 0.0;
      }
    }
    fetch_rows(s + 1);                 // into the other stage: its last readers passed the barrier above
    fetch_scalars(s + 2);
    __pipeline_commit();
    // make_mcmc_sampler (mcmc.ml:37-56) with the closures of :54-61
#pragma unroll (DMAX <= 16 ? DMAX : 1)
    for (int d = 0; d < DMAX; ++d) y[d] = (d < D) ? x[d] + delta[d] : 0.0;
    const double start_log_post = cl + cp;
    const double proposed_like = mcmc_logl(y);
    const double proposed_log_posterior = proposed_like + 0.0;
    const double log_accept_prob = proposed_log_posterior - start_log_post + 0.0 - 0.0;
    if (log_u_less_than(u_cur, log_accept_prob)) {
#pragma unroll (DMAX <= 16 ? DMAX : 1)
      for (int d = 0; d < DMAX; ++d) x[d] = y[d];
      cl = proposed_like;
    }
  }
  __pipeline_wait_prior(0);
  if (!live) return;
  if (!last) {
#pragma unroll (DMAX <= 16 ? DMAX : 1)
    for (int d = 0; d < DMAX; ++d)
      if (d < D) chain_x[(int64_t)d * K + j] = x[d];
    chain_cl[j] = cl;
    return;
  }
  const double nl = like_of(x);                                    // :68-69
  const double np = prior_of(x);
  if (!(nl >= thr)) *a.fail = 1;                                   // :70-72
#pragma unroll (DMAX <= 16 ? DMAX : 1)
  for (int d = 0; d < DMAX; ++d)
    if (d < D) a.fresh_x[(int64_t)j * D + d] = x[d];
  a.fresh_ll[j] = nl; a.fresh_lp[j] = np;
}

// ---- replace_live_point for a batch (nested.ml:26-43) without re-sorting the whole live set -------------------
// The survivors [K, nlive) are already ascending; the K new points are sorted by one CTA (bitonic network on
// (ordered ll, j): stable) and merged by rank: a new point lands before survivors of equal ll (the reference's
// bubble-up stops at `>` not `>=`, :36), new points of equal ll keep their order j.  Two launches per batch
// instead of the ~40 of a full radix sort.
constexpr int NEST_SORT_MAX = 8192;

__global__ void __launch_bounds__(1024)
nest_sort_fresh_kernel(const double *__restrict__ fll, int K, int P /* pow2 >= K */, uint64_t *__restrict__ skey,
                       int32_t *__restrict__ sidx) {
  extern __shared__ __align__(16) unsigned char nsf_smem[];
  uint64_t *key = reinterpret_cast<uint64_t *>(nsf_smem);
  int32_t *idx = reinterpret_cast<int32_t *>(key + P);
  for (int i = threadIdx.x; i < P; i += blockDim.x) {
    key[i] = (i < K) ? f64_to_ordered(fll[i]) : ~0ull;
    idx[i] = (i < K) ? i : 0x7FFFFFFF;
  }
  __syncthreads();
  for (int k = 2; k <= P; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < P; i += blockDim.x) {
        const int l = i ^ j;
        if (l > i) {
          const bool up = (i & k) == 0;
          const uint64_t ka = key[i], kb = key[l];
          const int32_t ia = idx[i], ib = idx[l];
          const bool a_gt_b = (ka > kb) || (ka == kb && ia > ib);
          if (a_gt_b == up) { key[i] = kb; key[l] = ka; idx[i] = ib; idx[l] = ia; }
        }
      }
      __syncthreads();
    }
  }
  for (int i = threadIdx.x; i < K; i += blockDim.x) { skey[i] = key[i]; sidx[i] = idx[i]; }
}

__global__ void nest_merge_kernel(const double *__restrict__ ox, const double *__restrict__ oll,
                                  const double *__restrict__ olp,            // old live set: [0,K) retired, [K,nlive) survivors
                                  const double *__restrict__ fx, const double *__restrict__ fll,
                                  const double *__restrict__ flp,            // the K new points
                                  const uint64_t *__restrict__ skey, const int32_t *__restrict__ sidx, int nlive, int K,
                                  int D, double *__restrict__ nx, double *__restrict__ nll, double *__restrict__ nlp) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nlive) return;
  const int ns = nlive - K;
  const double *srow; double ll, lp; int rank;
  if (e < K) {                       // new point at sorted position e: survivors strictly below it come first
    const uint64_t k = skey[e];
    int lo = 0, hi = ns;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (f64_to_ordered(oll[K + mid]) < k) lo = mid + 1; else hi = mid; }
    const int j = sidx[e];
    rank = e + lo; srow = fx + (int64_t)j * D; ll = fll[j]; lp = flp[j];
  } else {                           // survivor a: new points with ll <= its own come first
    const int a = e - K;
    const uint64_t k = f64_to_ordered(oll[e]);
    int lo = 0, hi = K;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (skey[mid] <= k) lo = mid + 1; else hi = mid; }
    rank = a + lo; srow = ox + (int64_t)e * D; ll = oll[e]; lp = olp[e];
  }
  nll[rank] = ll; nlp[rank] = lp;
  double *drow = nx + (int64_t)rank * D;
  for (int d = 0; d < D; ++d) drow[d] = srow[d];
}

__global__ void nest_keys_kernel(const double *__restrict__ ll, int n, uint64_t *__restrict__ keys, int32_t *__restrict__ vals) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { keys[i] = f64_to_ordered(ll[i]); vals[i] = i; }
}
__global__ void nest_gather_kernel(const double *__restrict__ x, const double *__restrict__ ll,
                                   const double *__restrict__ lp, const int32_t *__restrict__ order, int n, int D,
                                   double *__restrict__ xo, double *__restrict__ llo, double *__restrict__ lpo) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int s = order[i];
  for (int d = 0; d < D; ++d) xo[(int64_t)i * D + d] = x[(int64_t)s * D + d];
  llo[i] = ll[s]; lpo[i] = lp[s];
}

// Shrinkage schedule shared with the oracle (oracle.cpp `Shrink`): host libm.
struct Shrink {
  int nlive, K;
  std::vector<double> s, lvf;  // partial sums of log1p(-1/(nlive-j)); log(1/(nlive-j))
  double S;
  Shrink(int nlive_, int K_) : nlive(nlive_), K(K_), s(K_ + 1, 0.0), lvf(K_, 0.0) {
    for (int j = 0; j < K; ++j) {
      s[j + 1] = s[j] + std::log1p(-(1.0 / (double)(nlive - j)));
      lvf[j] = std::log(1.0 / (double)(nlive - j));
    }
    S = s[K];
  }
};

// stats.ml:240-248 on the host (glibc), used by the running tracker
static inline double h_log_sum_logs(double a, double b) {
  if (a == -INFINITY && b == -INFINITY) return -INFINITY;
  if (b > a) std::swap(a, b);
  return a + std::log1p(std::exp(b - a));
}

// evidence_error_and_weights (nested.ml:81-120), one thread per point.
// tab: [0..K) s_j, [K..2K) log vol_fraction_j, [2K] S
__global__ void nest_weights_kernel(const double *__restrict__ ll, int64_t n, int64_t ilive, int K,
                                    const double *__restrict__ tab, double log_dv_live, double *__restrict__ wts,
                                    double *__restrict__ dlow, double *__restrict__ dhigh) {
  const double log_half = -0.69314718055994530942;
  const double S = tab[2 * K];
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
    auto log_dv = [&](int64_t i) { return tab[K + (int)(i % K)] + ((double)(i / K) * S + tab[(int)(i % K)]); };
    double w = neg_inf();
    if (k < ilive) {
      if (k >= 1) w = log_sum_logs(w, log_half + (log_dv(k - 1) + ll[k]));      // dhigh of iteration k-1
      const double dl = log_dv(k) + ll[k];
      w = log_sum_logs(w, log_half + dl);                                       // dlow of iteration k
      dlow[k] = dl; dhigh[k] = log_dv(k) + ll[k + 1];
      if (k == ilive - 1) w = log_sum_logs(w, log_half + (log_dv_live + ll[k])); // tail iteration i = ilive
    } else {
      if (k == ilive && ilive >= 1) w = log_sum_logs(w, log_half + (log_dv(ilive - 1) + ll[k]));
      const double t = log_half + (log_dv_live + ll[k]);
      if (k >= 1) w = log_sum_logs(w, t);                 // tail iteration i = k   (skipped for i = 0)
      if (k + 1 <= n - 1) w = log_sum_logs(w, t);         // tail iteration i = k+1
      // tail iteration i = k contributes dlow = dv + ll[k-1], dhigh = dv + ll[k]
      if (k >= 1) { dlow[k] = log_dv_live + ll[k - 1]; dhigh[k] = log_dv_live + ll[k]; }
      else { dlow[k] = neg_inf(); dhigh[k] = neg_inf(); }
    }
    wts[k] = w;
  }
}

__global__ void nest_normalise_kernel(double *__restrict__ wts, int64_t n, double log_ev) {
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x)
    wts[k] = wts[k] - log_ev;
}

__global__ void max_kernel(const double *__restrict__ x, int64_t n, unsigned long long *__restrict__ out) {
  unsigned long long m = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const unsigned long long k = f64_to_ordered(x[i]);
    m = k > m ? k : m;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) { const unsigned long long o = __shfl_xor_sync(0xffffffffu, m, off); m = o > m ? o : m; }
  if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}

static inline double ordered_to_f64(unsigned long long k) {
  unsigned long long b = (k >> 63) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k;
  double d; memcpy(&d, &b, 8); return d;
}

// log sum_i exp(x_i) over a device array (max + compensated sum)
static int device_logsumexp(mg_ctx *ctx, const double *d_x, int64_t n, double *out) {
  cudaStream_t s = ctx->stream;
  DevBuf<unsigned long long> d_m;
  MG_CUDA(ctx, d_m.alloc(1, s));
  MG_CUDA(ctx, cudaMemsetAsync(d_m.get(), 0, 8, s));
  max_kernel<<<egrid(ctx, n), EB, 0, s>>>(d_x, n, d_m.get());
  MG_CHECK_LAUNCH(ctx);
  unsigned long long hm = 0;
  MG_CUDA(ctx, cudaMemcpyAsync(&hm, d_m.get(), 8, cudaMemcpyDeviceToHost, s));
  MG_CUDA(ctx, cudaStreamSynchronize(s));
  const double m = ordered_to_f64(hm);
  if (m == -INFINITY) { *out = -INFINITY; return MG_OK; }
  double sum = 0.0;
  int rc = reduce_sum(ctx, n, [d_x, m] __device__(int64_t i) { return exp(d_x[i] - m); }, &sum);
  if (rc) return rc;
  *out = m + std::log(sum);
  return MG_OK;
}

static int weights_dev(mg_ctx *ctx, const double *d_ll, int64_t n, int nlive, int K, double ll_last_retired_unused,
                       double *log_ev, double *log_dev, double *d_wts) {
  (void)ll_last_retired_unused;
  cudaStream_t s = ctx->stream;
  Shrink sh(nlive, K);
  std::vector<double> tab(2 * K + 1);
  for (int j = 0; j < K; ++j) { tab[j] = sh.s[j]; tab[K + j] = sh.lvf[j]; }
  tab[2 * K] = sh.S;
  const int64_t ilive = n - nlive;
  // nested.ml:97: log_vol_fraction + (ilive-1) * log_reduction_frac
  const int64_t il1 = ilive - 1;
  double log_x_il1;
  if (il1 >= 0) log_x_il1 = (double)(il1 / K) * sh.S + sh.s[il1 % K];
  else log_x_il1 = (double)il1 * sh.S;  // ilive = 0: (float_of_int (-1)) *. log_reduction_frac (K = 1 form)
  const double log_dv_live = std::log(1.0 / (double)nlive) + log_x_il1;
  DevBuf<double> d_tab, d_dlow, d_dhigh;
  MG_CUDA(ctx, upload(d_tab, tab.data(), tab.size(), s));
  MG_CUDA(ctx, d_dlow.alloc(n, s));
  MG_CUDA(ctx, d_dhigh.alloc(n, s));
  nest_weights_kernel<<<egrid(ctx, n), EB, 0, s>>>(d_ll, n, ilive, K, d_tab.get(), log_dv_live, d_wts, d_dlow.get(), d_dhigh.get());
  MG_CHECK_LAUNCH(ctx);
  double low, high;
  int rc;
  if ((rc = device_logsumexp(ctx, d_dlow.get(), n, &low))) return rc;
  if ((rc = device_logsumexp(ctx, d_dhigh.get(), n, &high))) return rc;
  const double log_half = -0.69314718055994530942;
  *log_ev = log_half + h_log_sum_logs(low, high);                 // :114
  *log_dev = high + std::log1p(-std::exp(low - high));            // :115
  nest_normalise_kernel<<<egrid(ctx, n), EB, 0, s>>>(d_wts, n, *log_ev);
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

}  // namespace mg

using namespace mg;

// nested.ml:152-178 on the host: n is small (the reference asks for ~100 draws) and the running sums are a
// sequential float64 scan in the reference's order.
extern "C" int mg_nested_posterior_indices(mg_ctx *ctx, const double *logw, int64_t npts, int64_t n, int64_t *out_idx) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, logw && out_idx && npts >= 1 && n >= 0, "posterior_samples: bad arguments");
  const CallKey key = next_key(ctx);
  std::vector<double> sw((size_t)npts);
  sw[0] = std::exp(logw[0]);
  for (int64_t i = 1; i < npts; ++i) sw[i] = std::exp(logw[i]) + sw[i - 1];      // :171-173
  for (int64_t k = 0; k < n; ++k) {
    uint32_t w[4];
    const uint64_t g = (uint64_t)k;
    philox4x32_10(0u, 0u, (uint32_t)g, (uint32_t)((g >> 32) & 0xFFFFu) | ((uint32_t)P_POST << 16), key.k0, key.k1, w);
    uint64_t bits = (0x3FFull << 52) | ((((uint64_t)w[0] << 32) | w[1]) & 0xFFFFFFFFFFFFFull);
    double m; memcpy(&m, &bits, 8);
    const double x = m - 1.0;                                                     // Random.float 1.0
    int64_t idx;
    if (x <= sw[0]) idx = 0;                                                      // weight_binary_search_index :152-165
    else { int64_t lo = 0, hi = npts - 1; while (hi - lo > 1) { const int64_t mid = (lo + hi) / 2; if (x <= sw[mid]) hi = mid; else lo = mid; } idx = hi; }
    out_idx[k] = idx;
  }
  return MG_OK;
}

extern "C" double mg_nested_log_total_error(double log_ev, double log_dev, int32_t nlive) {
  const double log_rel_error2 = -std::log((double)nlive);          // nested.ml:148-150
  return 0.5 * h_log_sum_logs(2.0 * log_dev, log_rel_error2 + 2.0 * log_ev);
}

extern "C" int mg_nested_weights(mg_ctx *ctx, const double *ll, int64_t n, int32_t nlive, int32_t batch,
                                 double *log_ev, double *log_dev, double *logw) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, ll && log_ev && log_dev && logw, "nested_weights: null argument");
  MG_REQUIRE(ctx, nlive >= 2 && n >= nlive && batch >= 1 && batch < nlive, "nested_weights: bad sizes");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  DevBuf<double> d_ll, d_w;
  MG_CUDA(ctx, upload(d_ll, ll, (size_t)n, ctx->stream));
  MG_CUDA(ctx, d_w.alloc(n, ctx->stream));
  int rc = weights_dev(ctx, d_ll.get(), n, nlive, batch, 0.0, log_ev, log_dev, d_w.get());
  if (rc) return rc;
  MG_CUDA(ctx, cudaMemcpyAsync(logw, d_w.get(), sizeof(double) * n, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MG_OK;
}

extern "C" int mg_nested_set_observer(mg_ctx *ctx, mg_nested_observer fn, void *user) {
  if (!ctx) return MG_EINVAL;
  ctx->nest_observer = fn; ctx->nest_observer_user = user;
  return MG_OK;
}

extern "C" int mg_nested_evidence(mg_ctx *ctx, const mg_logfn *like, const mg_logfn *prior, const double *prior_lo,
                                  const double *prior_hi, const mg_nested_cfg *cfg, double *log_ev, double *log_dev,
                                  int64_t *npts, double *pts, double *ll, double *lp, double *logw) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, like && prior && prior_lo && prior_hi && cfg && log_ev && log_dev && npts && ll && logw,
             "nested_evidence: null argument");
  const int D = cfg->dim, nlive = cfg->nlive, K = cfg->batch;
  MG_REQUIRE(ctx, D >= 1 && D <= 64, "nested_evidence: dim must be in 1..64");
  MG_REQUIRE(ctx, nlive >= 2 && cfg->nmcmc >= 0, "nested_evidence: bad nlive / nmcmc");
  MG_REQUIRE(ctx, K >= 1 && K < nlive, "nested_evidence: need 1 <= batch < nlive");
  MG_REQUIRE(ctx, cfg->max_points >= nlive + K, "nested_evidence: max_points too small");
  int rc;
  if ((rc = validate_logfn(ctx, like, D, "log_likelihood"))) return rc;
  if ((rc = validate_logfn(ctx, prior, D, "log_prior"))) return rc;
  const bool user = like->kind >= MG_FN_USER || prior->kind >= MG_FN_USER;   // kernels compiled at run time (jit.cu)
  const bool simple = user || getenv("MCMC_GPU_NEST_SIMPLE") != nullptr;       // plain-load chain kernel (same chains)
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  const double t_entry = std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
  DevLogFn dl, dp;
  MG_CUDA(ctx, dl.upload_from(like, s));
  MG_CUDA(ctx, dp.upload_from(prior, s));
  DevBuf<double> d_plo, d_phi, lx[2], lll[2], llp[2], fx, fll, flp, rx, rll, rlp;
  DevBuf<uint64_t> keys;
  DevBuf<int32_t> order;
  DevBuf<int> d_fail;
  MG_CUDA(ctx, upload(d_plo, prior_lo, D, s));
  MG_CUDA(ctx, upload(d_phi, prior_hi, D, s));
  for (int b = 0; b < 2; ++b) {
    MG_CUDA(ctx, lx[b].alloc((size_t)nlive * D, s));
    MG_CUDA(ctx, lll[b].alloc(nlive, s));
    MG_CUDA(ctx, llp[b].alloc(nlive, s));
  }
  MG_CUDA(ctx, fx.alloc((size_t)K * D, s)); MG_CUDA(ctx, fll.alloc(K, s)); MG_CUDA(ctx, flp.alloc(K, s));
  const int64_t cap = cfg->max_points;
  MG_CUDA(ctx, rx.alloc((size_t)cap * D, s)); MG_CUDA(ctx, rll.alloc(cap, s)); MG_CUDA(ctx, rlp.alloc(cap, s));
  MG_CUDA(ctx, keys.alloc(nlive, s)); MG_CUDA(ctx, order.alloc(nlive, s));
  DevBuf<uint64_t> skey; DevBuf<int32_t> sidx;
  MG_CUDA(ctx, skey.alloc(K, s)); MG_CUDA(ctx, sidx.alloc(K, s));
  if (K <= NEST_SORT_MAX && K > 4096)
    MG_CUDA(ctx, cudaFuncSetAttribute(nest_sort_fresh_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, NEST_SORT_MAX * 12));
  MG_CUDA(ctx, d_fail.alloc(1, s));
  MG_CUDA(ctx, cudaMemsetAsync(d_fail.get(), 0, sizeof(int), s));
  // proposals of one chunk of steps for all K chains (24 B each): at most ~200 MB
  int chunk = std::max(1, std::min(std::max(cfg->nmcmc, 1), std::max(16, (1 << 23) / K)));
  if (const char *e = getenv("MCMC_GPU_NEST_CHUNK")) chunk = std::max(1, std::min(chunk, atoi(e)));   // tests: force the multi-chunk path
  // two sets: when a batch is one chunk, the draws of batch b+1 are made on the second stream while the chains of
  // batch b run (the draws do not depend on the live set; the chain kernel leaves most of the machine idle)
  const bool overlap = chunk >= cfg->nmcmc && cfg->nmcmc > 0;
  DevBuf<int32_t> pi0[2], pj0[2];
  DevBuf<double> pds[2], pu[2], chain_x, chain_cl;
  NestProp prop2[2];
  for (int b = 0; b < (overlap ? 2 : 1); ++b) {
    MG_CUDA(ctx, pi0[b].alloc((size_t)chunk * K, s)); MG_CUDA(ctx, pj0[b].alloc((size_t)chunk * K, s));
    MG_CUDA(ctx, pds[b].alloc((size_t)chunk * K, s)); MG_CUDA(ctx, pu[b].alloc((size_t)chunk * K, s));
    prop2[b] = NestProp{pi0[b].get(), pj0[b].get(), pds[b].get(), pu[b].get()};
  }
  MG_CUDA(ctx, chain_x.alloc((size_t)64 * K, s)); MG_CUDA(ctx, chain_cl.alloc(K, s));
  cudaEvent_t ev_drawn[2] = {nullptr, nullptr}, ev_used[2] = {nullptr, nullptr};
  // declared after the buffers: runs first on any exit and drains the second stream before they are released
  struct EvGuard { cudaEvent_t *a, *b; cudaStream_t aux; ~EvGuard() { cudaStreamSynchronize(aux); for (int i = 0; i < 2; ++i) { if (a[i]) cudaEventDestroy(a[i]); if (b[i]) cudaEventDestroy(b[i]); } } } ev_guard{ev_drawn, ev_used, ctx->aux};
  if (overlap)
    for (int b = 0; b < 2; ++b) {
      MG_CUDA(ctx, cudaEventCreateWithFlags(&ev_drawn[b], cudaEventDisableTiming));
      MG_CUDA(ctx, cudaEventCreateWithFlags(&ev_used[b], cudaEventDisableTiming));
    }

  NestArgs a{};
  a.like = dl.params; a.prior = dp.params; a.plo = d_plo.get(); a.phi = d_phi.get();
  a.key = next_key(ctx);
  a.D = D; a.nlive = nlive; a.K = K; a.nmcmc = cfg->nmcmc;
  a.mode_hop = cfg->mode_hopping_frac;
  a.de_sigma = 2.38 / std::sqrt(2.0 * (double)D);   // mcmc.ml:212
  a.fresh_x = fx.get(); a.fresh_ll = fll.get(); a.fresh_lp = flp.get(); a.fail = d_fail.get();

#define MG_NEST_DISPATCH(KERNEL, GRID, BLOCK, ...)                                   \
  do {                                                                               \
    if (D <= 2) KERNEL<2><<<GRID, BLOCK, 0, s>>>(__VA_ARGS__);                       \
    else if (D <= 4) KERNEL<4><<<GRID, BLOCK, 0, s>>>(__VA_ARGS__);                  \
    else if (D <= 8) KERNEL<8><<<GRID, BLOCK, 0, s>>>(__VA_ARGS__);                  \
    else if (D <= 16) KERNEL<16><<<GRID, BLOCK, 0, s>>>(__VA_ARGS__);                \
    else if (D <= 32) KERNEL<32><<<GRID, BLOCK, 0, s>>>(__VA_ARGS__);                \
    else KERNEL<64><<<GRID, BLOCK, 0, s>>>(__VA_ARGS__);                             \
  } while (0)

  const size_t row_smem = (size_t)2 * 2 * NEST_BLOCK * nest_row_stride(D) * sizeof(double);
  // the shell-in-a-box pair with its parameters in registers (see nest_replace_kernel, FAST)
  const int fast = (like->kind == MG_FN_SHELL && like->scale == 1.0 && prior->scale == 1.0)
                       ? (prior->kind == MG_FN_BOX_CLOSED ? 1 : (prior->kind == MG_FN_BOX_OPEN ? 2 : 0)) : 0;
#define MG_NEST_CASE2(KERNEL, DM, GRID, BLOCK, ...)                                  \
  do {                                                                               \
    if (D == DM && DM <= 16 && fast == 1) {                                          \
      KERNEL<(DM <= 16 ? DM : 2), true, 1><<<GRID, BLOCK, row_smem, s>>>(__VA_ARGS__); \
    } else if (D == DM && DM <= 16 && fast == 2) {                                   \
      KERNEL<(DM <= 16 ? DM : 2), true, 2><<<GRID, BLOCK, row_smem, s>>>(__VA_ARGS__); \
    } else if (D == DM) {                                                            \
      if (row_smem > 48 * 1024) MG_CUDA(ctx, cudaFuncSetAttribute(KERNEL<DM, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)row_smem)); \
      KERNEL<DM, true><<<GRID, BLOCK, row_smem, s>>>(__VA_ARGS__);                   \
    } else {                                                                         \
      if (row_smem > 48 * 1024) MG_CUDA(ctx, cudaFuncSetAttribute(KERNEL<DM, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)row_smem)); \
      KERNEL<DM, false><<<GRID, BLOCK, row_smem, s>>>(__VA_ARGS__);                  \
    }                                                                                \
  } while (0)
#define MG_NEST_DISPATCH2(KERNEL, GRID, BLOCK, ...)                                  \
  do {                                                                               \
    if (D <= 2) MG_NEST_CASE2(KERNEL, 2, GRID, BLOCK, __VA_ARGS__);                  \
    else if (D <= 4) MG_NEST_CASE2(KERNEL, 4, GRID, BLOCK, __VA_ARGS__);             \
    else if (D <= 8) MG_NEST_CASE2(KERNEL, 8, GRID, BLOCK, __VA_ARGS__);             \
    else if (D <= 16) MG_NEST_CASE2(KERNEL, 16, GRID, BLOCK, __VA_ARGS__);           \
    else if (D <= 32) MG_NEST_CASE2(KERNEL, 32, GRID, BLOCK, __VA_ARGS__);           \
    else MG_NEST_CASE2(KERNEL, 64, GRID, BLOCK, __VA_ARGS__);                        \
  } while (0)

  int cur = 0;
  if (user) { if ((rc = jit_launch_nest_init(ctx, D, a, lx[1].get(), lll[1].get(), llp[1].get()))) return rc; }
  else MG_NEST_DISPATCH(nest_init_kernel, (nlive + 127) / 128, 128, a, lx[1].get(), lll[1].get(), llp[1].get());
  MG_CHECK_LAUNCH(ctx);
  // the chain kernel of one chunk of steps: pipelined (built-in plugins), plain loads, or compiled at run time
  auto launch_replace = [&](const NestProp &pp, int s0, int s1, int first, int last) -> int {
    if (user) return jit_launch_nest_replace(ctx, D, a, pp, s0, s1, first, last, chain_x.get(), chain_cl.get());
    if (simple) {
      MG_NEST_DISPATCH(nest_replace_simple_kernel, (K + 63) / 64, 64, a, pp, s0, s1, first, last, chain_x.get(), chain_cl.get());
      return MG_OK;
    }
    MG_NEST_DISPATCH2(nest_replace_kernel, (K + NEST_BLOCK - 1) / NEST_BLOCK, NEST_BLOCK, a, pp, s0, s1, first, last,
                      chain_x.get(), chain_cl.get());
    return MG_OK;
  };
  // Array.fast_sort by log_likelihood (:132): stable radix sort + gather
  auto sort_live = [&](int from, int to) -> int {
    nest_keys_kernel<<<(nlive + 255) / 256, 256, 0, s>>>(lll[from].get(), nlive, keys.get(), order.get());
    MG_CHECK_LAUNCH(ctx);
    int r = radix_sort_pairs(ctx, keys.get(), order.get(), nlive, 1);
    if (r) return r;
    nest_gather_kernel<<<(nlive + 255) / 256, 256, 0, s>>>(lx[from].get(), lll[from].get(), llp[from].get(), order.get(),
                                                          nlive, D, lx[to].get(), lll[to].get(), llp[to].get());
    MG_CHECK_LAUNCH(ctx);
    return MG_OK;
  };
  if ((rc = sort_live(1, 0))) return rc;
  cur = 0;

  Shrink sh(nlive, K);
  double log_vol = 0.0, log_int = -INFINITY;
  int64_t R = 0;
  std::vector<double> h_low(K);
  double h_edge[2];
  time_begin(ctx);
  const bool dbg = getenv("MCMC_GPU_DEBUG") != nullptr;
  double t_chain = 0, t_sort = 0, t_rest = 0; int nb = 0;
  auto now = [&]() { cudaStreamSynchronize(s); return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t_loop0 = dbg ? now() : 0;
  for (;;) {
    double tA = dbg ? now() : 0;
    if (R + K + nlive > cap) return set_err(ctx, MG_EFAIL, "nested_evidence: max_points too small");
    // threshold = ll of the K-th lowest live point; the K lowest are retired
    MG_CUDA(ctx, cudaMemcpyAsync(h_low.data(), lll[cur].get(), sizeof(double) * K, cudaMemcpyDeviceToHost, s));
    MG_CUDA(ctx, cudaStreamSynchronize(s));
    a.live_x = lx[cur].get(); a.live_ll = lll[cur].get(); a.live_lp = llp[cur].get();
    a.R = R; a.threshold = h_low[K - 1];
    if (overlap) {
      const int64_t np_ = (int64_t)cfg->nmcmc * K;
      const int b = (int)((R / K) & 1);
      if (R == 0) {   // first batch: its draws on the main stream
        nest_propose_kernel<<<(unsigned)((np_ + 255) / 256), 256, 0, s>>>(a, prop2[0], 0, cfg->nmcmc);
        MG_CHECK_LAUNCH(ctx);
      } else {
        MG_CUDA(ctx, cudaStreamWaitEvent(s, ev_drawn[b], 0));
      }
      if ((rc = launch_replace(prop2[b], 0, cfg->nmcmc, 1, 1))) return rc;
      MG_CHECK_LAUNCH(ctx);
      MG_CUDA(ctx, cudaEventRecord(ev_used[b], s));
      // draws of the next batch (ids R+K ..) into the other set, once the chains that read it have finished
      NestArgs an = a; an.R = R + K;
      if (R > 0) MG_CUDA(ctx, cudaStreamWaitEvent(ctx->aux, ev_used[1 - b], 0));
      else { cudaEvent_t e0; MG_CUDA(ctx, cudaEventCreateWithFlags(&e0, cudaEventDisableTiming)); MG_CUDA(ctx, cudaEventRecord(e0, s)); MG_CUDA(ctx, cudaStreamWaitEvent(ctx->aux, e0, 0)); cudaEventDestroy(e0); }
      nest_propose_kernel<<<(unsigned)((np_ + 255) / 256), 256, 0, ctx->aux>>>(an, prop2[1 - b], 0, cfg->nmcmc);
      MG_CHECK_LAUNCH(ctx);
      MG_CUDA(ctx, cudaEventRecord(ev_drawn[1 - b], ctx->aux));
    } else
    for (int s0 = 0;;) {
      const NestProp &prop = prop2[0];
      const int s1 = std::min(cfg->nmcmc, s0 + chunk);
      if (s1 > s0) {
        const int64_t np_ = (int64_t)(s1 - s0) * K;
        nest_propose_kernel<<<(unsigned)((np_ + 255) / 256), 256, 0, s>>>(a, prop, s0, s1 - s0);
        MG_CHECK_LAUNCH(ctx);
      }
      if ((rc = launch_replace(prop, s0, s1, s0 == 0 ? 1 : 0, s1 >= cfg->nmcmc ? 1 : 0))) return rc;
      MG_CHECK_LAUNCH(ctx);
      if (s1 >= cfg->nmcmc) break;
      s0 = s1;
    }
    double tB = dbg ? now() : 0;
    // retired_pt :: retired_pts (:137)
    MG_CUDA(ctx, cudaMemcpyAsync(rx.get() + R * D, lx[cur].get(), sizeof(double) * K * D, cudaMemcpyDeviceToDevice, s));
    MG_CUDA(ctx, cudaMemcpyAsync(rll.get() + R, lll[cur].get(), sizeof(double) * K, cudaMemcpyDeviceToDevice, s));
    MG_CUDA(ctx, cudaMemcpyAsync(rlp.get() + R, llp[cur].get(), sizeof(double) * K, cudaMemcpyDeviceToDevice, s));
    if (ctx->nest_observer) {   // ?observer (nested.ml:123-125,136): called with every retired point, in retirement order
      std::vector<double> ox((size_t)K * D), oll(K), olp(K);
      MG_CUDA(ctx, cudaMemcpyAsync(ox.data(), lx[cur].get(), sizeof(double) * K * D, cudaMemcpyDeviceToHost, s));
      MG_CUDA(ctx, cudaMemcpyAsync(oll.data(), lll[cur].get(), sizeof(double) * K, cudaMemcpyDeviceToHost, s));
      MG_CUDA(ctx, cudaMemcpyAsync(olp.data(), llp[cur].get(), sizeof(double) * K, cudaMemcpyDeviceToHost, s));
      MG_CUDA(ctx, cudaStreamSynchronize(s));
      for (int j = 0; j < K; ++j) ctx->nest_observer(ctx->nest_observer_user, ox.data() + (size_t)j * D, D, oll[j], olp[j]);
    }
    double tC = dbg ? now() : 0;
    if (K <= NEST_SORT_MAX) {
      // replace_live_point (:26-43): sort the K new points, merge them into the (sorted) survivors
      int P = 1; while (P < K) P <<= 1;
      nest_sort_fresh_kernel<<<1, 1024, (size_t)P * 12, s>>>(fll.get(), K, P, skey.get(), sidx.get());
      MG_CHECK_LAUNCH(ctx);
      nest_merge_kernel<<<(nlive + 255) / 256, 256, 0, s>>>(lx[cur].get(), lll[cur].get(), llp[cur].get(), fx.get(), fll.get(),
                                                           flp.get(), skey.get(), sidx.get(), nlive, K, D, lx[1 - cur].get(),
                                                           lll[1 - cur].get(), llp[1 - cur].get());
      MG_CHECK_LAUNCH(ctx);
    } else {
      // new points take the vacated front slots, then a stable sort of the whole set
      MG_CUDA(ctx, cudaMemcpyAsync(lx[cur].get(), fx.get(), sizeof(double) * K * D, cudaMemcpyDeviceToDevice, s));
      MG_CUDA(ctx, cudaMemcpyAsync(lll[cur].get(), fll.get(), sizeof(double) * K, cudaMemcpyDeviceToDevice, s));
      MG_CUDA(ctx, cudaMemcpyAsync(llp[cur].get(), flp.get(), sizeof(double) * K, cudaMemcpyDeviceToDevice, s));
      if ((rc = sort_live(cur, 1 - cur))) return rc;
    }
    cur = 1 - cur;
    double tD = dbg ? now() : 0;
    if (dbg) { t_chain += tB - tA; t_rest += tC - tB; t_sort += tD - tC; ++nb; }
    // running tracker (:138-141), quirk F5d kept: log_dv = log_vol +. vol_fraction
    for (int j = 0; j < K; ++j) {
      const double vol_fraction = 1.0 / (double)(nlive - j);
      const double log_new_vol = log_vol + std::log1p(-vol_fraction);
      const double log_dv = log_vol + vol_fraction;
      log_int = h_log_sum_logs(log_int, h_low[j] + log_dv);
      log_vol = log_new_vol;
    }
    R += K;
    int h_fail = 0;
    MG_CUDA(ctx, cudaMemcpyAsync(h_edge, lll[cur].get() + (nlive - 1), sizeof(double), cudaMemcpyDeviceToHost, s));
    MG_CUDA(ctx, cudaMemcpyAsync(&h_fail, d_fail.get(), sizeof(int), cudaMemcpyDeviceToHost, s));
    MG_CUDA(ctx, cudaStreamSynchronize(s));
    if (h_fail) return set_err(ctx, MG_EFAIL, "Error in draw_new_live_point: new log(L) below the threshold");  // :70-72
    // remaining_integral_negligable (:45-48)
    const double log_live_estimate = log_vol + h_edge[0];
    if (log_live_estimate - h_log_sum_logs(log_int, log_live_estimate) <= std::log(cfg->epsrel)) break;
  }
  if (overlap) { MG_CUDA(ctx, cudaStreamWaitEvent(s, ev_drawn[(int)((R / K) & 1)], 0)); }   // the draws made ahead for a batch that never ran
  time_end(ctx);
  const double t_loop1 = dbg ? now() : 0;
  if (dbg) fprintf(stderr, "nested: %d batches; per batch: chains %.3f ms, copies %.3f ms, sort %.3f ms\n", nb, 1e3 * t_chain / nb, 1e3 * t_rest / nb, 1e3 * t_sort / nb);
  const int64_t n = R + nlive;
  if (n > cap) return set_err(ctx, MG_EFAIL, "nested_evidence: max_points too small");
  // all points ascending in ll: retired (in order) followed by the sorted live set (:143)
  MG_CUDA(ctx, cudaMemcpyAsync(rx.get() + R * D, lx[cur].get(), sizeof(double) * nlive * D, cudaMemcpyDeviceToDevice, s));
  MG_CUDA(ctx, cudaMemcpyAsync(rll.get() + R, lll[cur].get(), sizeof(double) * nlive, cudaMemcpyDeviceToDevice, s));
  MG_CUDA(ctx, cudaMemcpyAsync(rlp.get() + R, llp[cur].get(), sizeof(double) * nlive, cudaMemcpyDeviceToDevice, s));
  DevBuf<double> d_w;
  MG_CUDA(ctx, d_w.alloc(n, s));
  if ((rc = weights_dev(ctx, rll.get(), n, nlive, K, 0.0, log_ev, log_dev, d_w.get()))) return rc;
  if (pts) MG_CUDA(ctx, cudaMemcpyAsync(pts, rx.get(), sizeof(double) * n * D, cudaMemcpyDeviceToHost, s));
  MG_CUDA(ctx, cudaMemcpyAsync(ll, rll.get(), sizeof(double) * n, cudaMemcpyDeviceToHost, s));
  if (lp) MG_CUDA(ctx, cudaMemcpyAsync(lp, rlp.get(), sizeof(double) * n, cudaMemcpyDeviceToHost, s));
  MG_CUDA(ctx, cudaMemcpyAsync(logw, d_w.get(), sizeof(double) * n, cudaMemcpyDeviceToHost, s));
  MG_CUDA(ctx, cudaStreamSynchronize(s));
  if (dbg) fprintf(stderr, "nested: setup %.3f s, loop %.3f s, weights + copy-out %.3f s\n", t_loop0 - t_entry, t_loop1 - t_loop0, now() - t_loop1);
  *npts = n;
  return MG_OK;
}
