// diagnostics.cu -- ensemble convergence diagnostics of a sample block [n][D+2][C]: split-Rhat (Gelman et al., BDA3),
// the ensemble autocorrelation and Geyer's (1992) initial-monotone-sequence estimate of the integrated autocorrelation
// time and effective sample size, plus the same time per sequence.  An addition beyond the reference, in the standing
// of mg_stats_autocorrelation's integrated length (SURVEY F6); definitions in include/mcmc_gpu.h and DESIGN.md 4b,
// transcribed line by line in oracle/diagnostics_np.py.
//
// Decomposition.  One CTA per (group of 32 chains, half, field); lanes are chains, so a step row of the group is one
// coalesced 256-byte load.  Each tile of DG_TS steps is staged in shared memory with a halo of the padded lag range
// (zeros past the sequence's end), as values about a per-sequence pivot (its first value).  Warps split the lag range
// in blocks of 16 lags (and, when there are fewer than eight blocks, the tile's steps); a thread keeps its 16 (or 32)
// raw lag sums R(t) = sum_s z_s z_{s+t} in registers for the whole sequence, with a sliding window of 16 partner
// values: per step one shared load of z_s and one of the next partner feed 16 explicit fma() (the library builds with
// -fmad=false).  The block is read from HBM once; the halo rows are re-read from L2.
//
// Epilogue (per CTA): the centred autocovariances follow from the raw sums, the pivot-relative sum S1 and the head
// and tail sums H(t) = sum_{s<t} z_s, T(t) = sum_{s>=N-t} z_s:
//   N gamma(t) = R(t) - d (2 S1 - H(t) - T(t)) + (N - t) d^2,   d = S1 / N
// then tau_m per sequence (Geyer), and one record per CTA: (count, mean and M2 of the sequence means, sum s_m^2,
// sum_m gamma_m(t)).  A pool kernel folds the records of a field in a fixed order (Chan's update for the means,
// compensated sums for the rest); the host turns the pooled record into Rhat, rho, tau, ESS.  The same host step pools
// the records of several ranks (mg_comm_chain_diagnostics), so one rank and one GPU give the same bits.
#include <math_constants.h>

#include <algorithm>
#include <cmath>

#include "comm.cuh"
#include "reduce.cuh"

namespace mg {

constexpr int DG_THREADS = 256, DG_WARPS = DG_THREADS / 32;
constexpr int DG_TS = 128;          // steps per tile
constexpr int DG_LB = 16;           // lags per register block
static_assert(MG_DIAG_MAXLAG == 2 * DG_WARPS * DG_LB, "two register blocks of 16 lags per warp");

struct DgArgs {
  const double *x;
  int64_t n, C, ngroups;      // rows, chains, groups of 32 chains
  int F, L, nblk;             // fields, lags, lag blocks of 16
  int64_t N;                  // steps per sequence
  int64_t M;                  // sequences (split: 2 C)
  double *rec;                // [F][nct][L + 4] per-CTA records
  double *seq_tau;            // [F][M] or null
};

// R(t) += sum_{s in [a0, a0 + len)} z_s z_{s+t} for the 16 lags t = 16 b + j; p = tile + lane, row stride 32
__device__ __forceinline__ void lag_block(const double *__restrict__ p, int a0, int len, int b, double (&acc)[DG_LB]) {
  double win[DG_LB];
  const int off = b * DG_LB;
#pragma unroll
  for (int j = 0; j < DG_LB; ++j) win[j] = p[(a0 + off + j) * 32];
  for (int s = a0; s < a0 + len; s += DG_LB) {
#pragma unroll
    for (int i = 0; i < DG_LB; ++i) {
      const double xv = p[(s + i) * 32];
#pragma unroll
      for (int j = 0; j < DG_LB; ++j) acc[j] = fma(xv, win[(i + j) & (DG_LB - 1)], acc[j]);
      win[i] = p[(s + i + off + DG_LB) * 32];   // win[(i' + j) % 16] = z_{s + i' + off + j} for the steps i' > i
    }
  }
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Geyer's initial monotone sequence on rho(t) = g(t) / g(0), t < L; g in shared memory with row stride 32
__device__ __forceinline__ double seq_geyer(const double *__restrict__ g, int L) {
  const double g0 = g[0];
  if (!(g0 > 0.0) || !isfinite(g0)) return CUDART_NAN;
  double total = 0.0, prev = 0.0;
  for (int k = 0; k < L / 2; ++k) {
    const double P = g[(2 * k) * 32] / g0 + g[(2 * k + 1) * 32] / g0;
    if (P <= 0.0) break;
    const double cur = (k == 0 || P < prev) ? P : prev;
    total += cur;
    prev = cur;
  }
  return -1.0 + 2.0 * total;
}

template <int NBW>
__global__ void __launch_bounds__(DG_THREADS, 2) diag_seq_kernel(const DgArgs a) {
  extern __shared__ double tile[];                   // [rows][32]
  __shared__ double s_part[DG_WARPS][32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int f = blockIdx.y;
  const int64_t half = blockIdx.x / a.ngroups, g = blockIdx.x - half * a.ngroups;
  const int64_t c = g * 32 + lane;
  const bool valid = c < a.C;
  const int64_t N = a.N;
  const int64_t rstride = (int64_t)a.F * a.C;
  const int64_t r0 = half ? a.n - N : 0;
  const double *col = a.x + r0 * rstride + (int64_t)f * a.C + (valid ? c : 0);   // sample s of this lane's sequence
  const double piv = valid ? __ldg(col) : 0.0;
  const int nblk = a.nblk;
  const int rows = DG_TS + DG_LB * nblk;
  // warp roles: NG lag groups x NS step slices (NBW = 1), or eight warps with two lag blocks each (NBW = 2)
  int NG = 8;
  if (NBW == 1) { NG = 1; while (NG < nblk) NG <<= 1; }
  const int NS = DG_WARPS / NG, sl = w / NG, len = DG_TS / NS;
  double acc[NBW][DG_LB];
#pragma unroll
  for (int k = 0; k < NBW; ++k)
#pragma unroll
    for (int j = 0; j < DG_LB; ++j) acc[k][j] = 0.0;
  double s1 = 0.0;
  for (int64_t s0 = 0; s0 < N; s0 += DG_TS) {
    __syncthreads();
#pragma unroll 4
    for (int r = w; r < rows; r += DG_WARPS) {
      const int64_t s = s0 + r;
      const double z = (valid && s < N) ? __ldg(col + s * rstride) - piv : 0.0;
      tile[r * 32 + lane] = z;
      if (r < DG_TS) s1 += z;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < NBW; ++k) {
      const int b = NBW == 1 ? w % NG : w + DG_WARPS * k;
      if (b < nblk) lag_block(tile + lane, sl * len, len, b, acc[k]);
    }
  }
  s_part[w][lane] = s1;
  __syncthreads();
  // raw lag sums per slice -> shared, then summed over the slices in slice order
  const int L = a.L;
  const int pstride = DG_LB * NG * NBW;              // rows per slice
#pragma unroll
  for (int k = 0; k < NBW; ++k) {
    const int b = NBW == 1 ? w % NG : w + DG_WARPS * k;
    if (b < nblk)
#pragma unroll
      for (int j = 0; j < DG_LB; ++j) tile[(sl * pstride + b * DG_LB + j) * 32 + lane] = acc[k][j];
  }
  __syncthreads();
  double *Q = tile;                                  // [L][32]: R(t), then gamma(t)
  if (NS > 1) {
    Q = tile + (size_t)NS * pstride * 32;            // NS * pstride = DG_TS rows; DG_TS + L <= rows
    for (int t = w; t < L; t += DG_WARPS) {
      double r = 0.0;
      for (int q = 0; q < NS; ++q) r += tile[(q * pstride + t) * 32 + lane];
      Q[t * 32 + lane] = r;
    }
    __syncthreads();
  }
  const double Nd = (double)N;
  double *rec = a.rec + ((int64_t)f * gridDim.x + blockIdx.x) * (L + 4);
  if (w == 0) {
    double S1 = 0.0;
    for (int q = 0; q < DG_WARPS; ++q) S1 += s_part[q][lane];
    const double d = S1 / Nd;
    double h = 0.0, tl = 0.0;                        // H(t), T(t)
    for (int t = 0; t < L; ++t) {
      const double R = Q[t * 32 + lane];
      const double gam = (R - d * (2.0 * S1 - h - tl) + (Nd - (double)t) * (d * d)) / Nd;
      Q[t * 32 + lane] = valid ? gam : 0.0;
      if (valid) {
        h += __ldg(col + (int64_t)t * rstride) - piv;
        tl += __ldg(col + (N - 1 - t) * rstride) - piv;
      }
    }
    __syncwarp();
    const double tau_m = seq_geyer(Q + lane, L);
    if (valid && a.seq_tau) a.seq_tau[(int64_t)f * a.M + half * a.C + c] = tau_m;
    // the CTA's record: count, mean and M2 of its sequence means, sum of s_m^2
    const double cnt = warp_sum(valid ? 1.0 : 0.0);
    const double xb = piv + d;
    const double mean = warp_sum(valid ? xb : 0.0) / cnt;
    const double dv = valid ? xb - mean : 0.0;
    const double M2 = warp_sum(dv * dv);
    const double s2 = warp_sum(valid ? Nd / (Nd - 1.0) * Q[lane] : 0.0);
    if (lane == 0) { rec[0] = cnt; rec[1] = mean; rec[2] = M2; rec[3] = s2; }
  }
  __syncthreads();
  for (int t = w; t < L; t += DG_WARPS) {
    const double sg = warp_sum(Q[t * 32 + lane]);
    if (lane == 0) rec[4 + t] = sg;
  }
}

// Fold the per-CTA records of field blockIdx.x, in CTA order, into one record [L + 4] of the same layout.
constexpr int DG_POOL = 256;
__global__ void __launch_bounds__(DG_POOL) diag_pool_kernel(const double *__restrict__ rec, int64_t nct, int L,
                                                            double *__restrict__ out) {
  const int f = blockIdx.x;
  const int W = L + 4;
  const double *r = rec + (int64_t)f * nct * W;
  // columns 3 .. L + 3: compensated sums, one thread per column
  for (int k = 3 + threadIdx.x; k < W; k += DG_POOL) {
    Comp acc;
    for (int64_t i = 0; i < nct; ++i) acc.add(r[i * W + k]);
    out[(int64_t)f * W + k] = acc.value();
  }
  // (count, mean, M2): Chan's update over a contiguous range per thread, then over the threads in order
  __shared__ double sn[DG_POOL], sm[DG_POOL], sM[DG_POOL];
  const int64_t per = (nct + DG_POOL - 1) / DG_POOL;
  double n = 0.0, m = 0.0, M2 = 0.0;
  for (int64_t i = threadIdx.x * per; i < nct && i < (threadIdx.x + 1) * per; ++i) {
    const double nb = r[i * W], mb = r[i * W + 1], Mb = r[i * W + 2], tot = n + nb, dl = mb - m;
    m = m + dl * (nb / tot);
    M2 = M2 + Mb + dl * dl * (n * nb / tot);
    n = tot;
  }
  sn[threadIdx.x] = n; sm[threadIdx.x] = m; sM[threadIdx.x] = M2;
  __syncthreads();
  if (threadIdx.x == 0) {
    double tn = 0.0, tm = 0.0, tM = 0.0;
    for (int q = 0; q < DG_POOL; ++q) {
      const double nb = sn[q];
      if (nb == 0.0) continue;
      const double tot = tn + nb, dl = sm[q] - tm;
      tm = tm + dl * (nb / tot);
      tM = tM + sM[q] + dl * dl * (tn * nb / tot);
      tn = tot;
    }
    out[(int64_t)f * W] = tn; out[(int64_t)f * W + 1] = tm; out[(int64_t)f * W + 2] = tM;
  }
}

static int diag_check_cfg(mg_ctx *ctx, const mg_diag_cfg *cfg) {
  MG_REQUIRE(ctx, cfg, "chain_diagnostics: null configuration");
  MG_REQUIRE(ctx, cfg->n >= 1 && cfg->nchains >= 1 && cfg->dim >= 1, "chain_diagnostics: bad block shape");
  MG_REQUIRE(ctx, cfg->split == 0 || cfg->split == 1, "chain_diagnostics: split is 0 or 1");
  MG_REQUIRE(ctx, !cfg->split || cfg->n >= 4, "chain_diagnostics: split needs n >= 4");
  const int64_t N = cfg->split ? cfg->n / 2 : cfg->n;
  MG_REQUIRE(ctx, cfg->maxlag >= 2 && (int64_t)cfg->maxlag < N, "chain_diagnostics: need 2 <= maxlag <= N - 1 (N = %lld)",
             (long long)N);
  MG_REQUIRE(ctx, cfg->maxlag <= MG_DIAG_MAXLAG, "chain_diagnostics: maxlag above %d", MG_DIAG_MAXLAG);
  MG_REQUIRE(ctx, (cfg->nchains + 31) / 32 * (cfg->split ? 2 : 1) < (1LL << 31), "chain_diagnostics: too many chains");
  return MG_OK;
}

// The local pass: d_pooled [F][L + 4] = this block's pooled record of every field; d_seq_tau [F][M] or null.
static int diag_local(mg_ctx *ctx, const double *d_x, const mg_diag_cfg *cfg, double *d_pooled, double *d_seq_tau) {
  cudaStream_t st = ctx->stream;
  const int F = cfg->dim + 2, L = cfg->maxlag, nblk = (L + DG_LB - 1) / DG_LB;
  DgArgs a;
  a.x = d_x; a.n = cfg->n; a.C = cfg->nchains; a.ngroups = (cfg->nchains + 31) / 32;
  a.F = F; a.L = L; a.nblk = nblk;
  a.N = cfg->split ? cfg->n / 2 : cfg->n;
  a.M = cfg->split ? 2 * cfg->nchains : cfg->nchains;
  a.seq_tau = d_seq_tau;
  const int64_t nct = a.ngroups * (cfg->split ? 2 : 1);
  DevBuf<double> recs;
  MG_CUDA(ctx, recs.alloc((size_t)F * nct * (L + 4), st));
  a.rec = recs.get();
  const size_t smem = sizeof(double) * 32 * (DG_TS + DG_LB * nblk);
  const dim3 grid((unsigned)nct, F);
  time_begin(ctx);
  if (nblk <= DG_WARPS) {
    MG_CUDA(ctx, cudaFuncSetAttribute(diag_seq_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    diag_seq_kernel<1><<<grid, DG_THREADS, smem, st>>>(a);
  } else {
    MG_CUDA(ctx, cudaFuncSetAttribute(diag_seq_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    diag_seq_kernel<2><<<grid, DG_THREADS, smem, st>>>(a);
  }
  MG_CHECK_LAUNCH(ctx);
  time_end(ctx);
  diag_pool_kernel<<<F, DG_POOL, 0, st>>>(recs.get(), nct, L, d_pooled);
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

// Pooled records of R ranks (host [R][F][L + 4], rank order) -> the outputs; the same arithmetic on every rank.
static void diag_finish(const double *recs, int R, int F, int L, int64_t N, double *rhat, double *ess, double *tau,
                        int32_t *closed, double *rho) {
  const int W = L + 4;
  const double nan = std::nan(""), Nd = (double)N;
  std::vector<double> gbar(L);
  for (int f = 0; f < F; ++f) {
    double M = 0.0, mean = 0.0, M2 = 0.0;
    Comp s2;
    std::vector<Comp> gs(L);
    bool finite = true;
    for (int r = 0; r < R; ++r) {
      const double *q = recs + ((size_t)r * F + f) * W;
      for (int k = 0; k < W; ++k) finite = finite && std::isfinite(q[k]);
      if (q[0] == 0.0) continue;
      const double tot = M + q[0], dl = q[1] - mean;
      mean = mean + dl * (q[0] / tot);
      M2 = M2 + q[2] + dl * dl * (M * q[0] / tot);
      M = tot;
      s2.add(q[3]);
      for (int t = 0; t < L; ++t) gs[t].add(q[4 + t]);
    }
    const double Wv = s2.value() / M;
    const double B = M > 1.0 ? Nd / (M - 1.0) * M2 : 0.0;
    const double vp = (Nd - 1.0) / Nd * Wv + B / Nd;
    if (!finite || !(vp > 0.0) || !std::isfinite(vp)) {
      if (rhat) rhat[f] = nan;
      if (ess) ess[f] = nan;
      if (tau) tau[f] = nan;
      if (closed) closed[f] = 0;
      if (rho) for (int t = 0; t < L; ++t) rho[(size_t)f * L + t] = nan;
      continue;
    }
    if (rhat) rhat[f] = M == 1.0 ? nan : (Wv > 0.0 ? std::sqrt(vp / Wv) : INFINITY);
    gbar[0] = 1.0;
    for (int t = 1; t < L; ++t) gbar[t] = 1.0 - (Wv - gs[t].value() / M) / vp;
    double total = 0.0, prev = 0.0;
    int cl = 0;
    for (int k = 0; k < L / 2; ++k) {
      const double P = gbar[2 * k] + gbar[2 * k + 1];
      if (P <= 0.0) { cl = 1; break; }
      const double cur = (k == 0 || P < prev) ? P : prev;
      total += cur;
      prev = cur;
    }
    const double tv = -1.0 + 2.0 * total;
    if (tau) tau[f] = tv;
    if (ess) ess[f] = M * Nd / tv;
    if (closed) closed[f] = cl;
    if (rho) for (int t = 0; t < L; ++t) rho[(size_t)f * L + t] = gbar[t];
  }
}

// local pass + pooled record to the host
static int diag_local_record(mg_ctx *ctx, const double *d_x, const mg_diag_cfg *cfg, double *d_seq_tau,
                             std::vector<double> &rec) {
  const int F = cfg->dim + 2, W = cfg->maxlag + 4;
  DevBuf<double> pooled;
  MG_CUDA(ctx, pooled.alloc((size_t)F * W, ctx->stream));
  int rc = diag_local(ctx, d_x, cfg, pooled.get(), d_seq_tau);
  if (rc) return rc;
  rec.resize((size_t)F * W);
  MG_CUDA(ctx, cudaMemcpyAsync(rec.data(), pooled.get(), sizeof(double) * rec.size(), cudaMemcpyDeviceToHost, ctx->stream));
  MG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MG_OK;
}

}  // namespace mg

using namespace mg;

extern "C" int mg_stats_chain_diagnostics_dev(mg_ctx *ctx, const double *d_samples, const mg_diag_cfg *cfg,
                                              double *out_rhat, double *out_ess, double *out_tau,
                                              int32_t *out_window_closed, double *out_rho, double *d_seq_tau) {
  if (!ctx) return MG_EINVAL;
  int rc = diag_check_cfg(ctx, cfg);
  if (rc) return rc;
  MG_REQUIRE(ctx, d_samples && out_rhat && out_ess && out_tau && out_window_closed, "chain_diagnostics: null argument");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  std::vector<double> rec;
  if ((rc = diag_local_record(ctx, d_samples, cfg, d_seq_tau, rec))) return rc;
  const int64_t N = cfg->split ? cfg->n / 2 : cfg->n;
  diag_finish(rec.data(), 1, cfg->dim + 2, cfg->maxlag, N, out_rhat, out_ess, out_tau, out_window_closed, out_rho);
  return MG_OK;
}

extern "C" int mg_stats_chain_diagnostics(mg_ctx *ctx, const double *samples, const mg_diag_cfg *cfg, double *out_rhat,
                                          double *out_ess, double *out_tau, int32_t *out_window_closed, double *out_rho,
                                          double *seq_tau) {
  if (!ctx) return MG_EINVAL;
  int rc = diag_check_cfg(ctx, cfg);
  if (rc) return rc;
  MG_REQUIRE(ctx, samples, "chain_diagnostics: null samples");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  const int64_t F = cfg->dim + 2, M = cfg->split ? 2 * cfg->nchains : cfg->nchains;
  DevBuf<double> d_x, d_tau;
  MG_CUDA(ctx, upload(d_x, samples, (size_t)cfg->n * F * cfg->nchains, ctx->stream));
  if (seq_tau) MG_CUDA(ctx, d_tau.alloc((size_t)F * M, ctx->stream));
  rc = mg_stats_chain_diagnostics_dev(ctx, d_x.get(), cfg, out_rhat, out_ess, out_tau, out_window_closed, out_rho,
                                      seq_tau ? d_tau.get() : nullptr);
  if (rc) return rc;
  if (seq_tau) {
    MG_CUDA(ctx, cudaMemcpyAsync(seq_tau, d_tau.get(), sizeof(double) * F * M, cudaMemcpyDeviceToHost, ctx->stream));
    MG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return MG_OK;
}

// Chains sharded over the ranks: every rank runs the local pass on its own [n][D+2][C_r] block and pools it into one
// record per field, F (L + 4) doubles; the records are all-gathered and folded in rank order by the same host step as
// the single-GPU call, so every rank gets the same bytes and one rank gives the single-GPU bits.  A header exchange
// first checks that dim and maxlag, which size the records, and n and split agree.
extern "C" int mg_comm_chain_diagnostics(mg_comm *c, const double *d_samples_local, const mg_diag_cfg *cfg_local,
                                         double *out_rhat, double *out_ess, double *out_tau, int32_t *out_window_closed,
                                         double *out_rho, double *d_seq_tau) {
  if (!c) return MG_EINVAL;
  mg_ctx *ctx = mg_comm_ctx(c);
  int rc = diag_check_cfg(ctx, cfg_local);
  if (rc == MG_OK && !(d_samples_local && out_rhat && out_ess && out_tau && out_window_closed))
    rc = set_err(ctx, MG_EINVAL, "chain_diagnostics (comm): null argument");
  if (rc == MG_OK && cudaSetDevice(ctx->device) != cudaSuccess) rc = set_err(ctx, MG_ECUDA, "cuda: cannot select the device");
  std::vector<int64_t> hdr(4, 0), hdrs;
  if (rc == MG_OK) hdr = {cfg_local->dim, cfg_local->maxlag, cfg_local->n, cfg_local->split};
  if ((rc = comm_gather(c, rc, hdr, hdrs, "chain_diagnostics (comm)"))) return rc;
  for (int r = 0; r < mg_comm_size(c); ++r)
    if (!std::equal(hdr.begin(), hdr.end(), hdrs.begin() + 4 * r))
      return set_err(ctx, MG_EINVAL, "chain_diagnostics (comm): rank %d has another dim, maxlag, n or split", r);
  const int F = cfg_local->dim + 2, L = cfg_local->maxlag;
  std::vector<double> rec((size_t)F * (L + 4)), recs;
  rc = diag_local_record(ctx, d_samples_local, cfg_local, d_seq_tau, rec);
  if ((rc = comm_gather(c, rc, rec, recs, "chain_diagnostics (comm)"))) return rc;
  const int64_t N = cfg_local->split ? cfg_local->n / 2 : cfg_local->n;
  diag_finish(recs.data(), mg_comm_size(c), F, L, N, out_rhat, out_ess, out_tau, out_window_closed, out_rho);
  return MG_OK;
}
