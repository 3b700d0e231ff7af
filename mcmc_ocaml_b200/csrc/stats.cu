// stats.cu -- Stats.mean / std / multi_mean / multi_std / slow_autocorrelation
// (stats.ml:17-87,223-238) as coalesced grid-stride reductions.
//
// The reference sums left to right in float64 (stats.ml:19-22).  A parallel
// sum cannot reproduce that rounding sequence; instead every thread keeps a
// compensated (Neumaier) partial, partials are combined in a fixed order
// (warp shuffle tree, then one block-order pass), so the result is
// deterministic and within a few ulp of the exactly rounded sum -- closer to
// exact than the reference's own sequential sum.  The tested error model is in
// DESIGN.md section S (tests/test_stats_exact_gpu.py).
// All kernels are HBM-bound: 8 bytes read per element per pass.
#include "comm.cuh"
#include "models.cuh"
#include "rng.cuh"
#include "reduce.cuh"

namespace mg {

constexpr int RED_BLOCK = 256;

// IEEE sum of a compensated accumulator: once an infinity enters, the compensation term turns NaN (inf - inf)
// while the running sum holds the right +-inf (or NaN where both signs met), so the running sum is the answer.
__device__ __forceinline__ double comp_sum(const Comp &a) { return isfinite(a.s) ? a.value() : a.s; }

// sqrt of a variance: only a finite negative round-off is clamped to 0; NaN (a non-finite input, or 0/0 at N = 1)
// stays NaN as in the reference's fold
__device__ __forceinline__ double std_of_var(double var) { return sqrt(var < 0.0 ? 0.0 : var); }

// ---- sample block [n][F][C] ---------------------------------------------------
// One pass for both moments: sums of a = x - p_f and a^2 about a pivot p_f, so that
//   mean = p + S1/N,   var = (S2 - S1^2/N) / (N - 1)
// read the 62.9 GB sample block once instead of twice.  S1 and S2 are compensated, so the error of var is
// dominated by the cancellation in S2 - S1^2/N, about eps (mean - p)^2 / var relative.  The pivot is therefore
// taken from the data: the finite value nearest the mean of a fixed, evenly spaced subsample of up to PIV_SAMPLES
// values of the field (block_field_pivot_kernel), so |mean - p| is of order sigma / sqrt(PIV_SAMPLES) however far
// out any single sample (say an outlying start point in slot 0) lies.  Being a sample, p makes every deviation of a
// constant field exactly 0.
// A CTA whose partial sums come out non-finite reads its rows once more to classify the non-finite values, so the
// finish gives what the reference's fold gives: mean NaN with a NaN or with both infinities, else +-inf with one of them; std NaN with any non-finite
// value, and NaN for N = 1.
constexpr int MOM_BLOCK = RED_BLOCK;
constexpr int64_t PIV_SAMPLES = 4096;
constexpr unsigned NF_NAN = 1u, NF_PINF = 2u, NF_NINF = 4u;

constexpr int64_t PIV_ROWS = 16;

// Subsample value j < R * Q of field f: R = min(n, PIV_ROWS) evenly spaced rows (samples), Q evenly spaced chains in
// each.  Whole rows keep the reads on a few pages: values scattered over a block of tens of GB cost a page-table
// walk each.
__device__ __forceinline__ double pivot_sample(const double *__restrict__ blk, int64_t n, int F, int f, int64_t C,
                                               int64_t R, int64_t Q, int64_t j) {
  const int64_t s = (j / Q) * n / R, c = (j % Q) * C / Q;   // products < 2^12 * n, 2^12 * C: no overflow
  return blk[(s * F + f) * C + c];
}

// (d, j) lexicographic minimum; "none" is (inf, INT_MAX)
__device__ __forceinline__ void take_nearer(double &bd, int &bj, double od, int oj) {
  if (od < bd || (od == bd && oj < bj)) { bd = od; bj = oj; }
}

// One CTA per field (strided over grid x).  Reads at most 2 * PIV_SAMPLES values per field.
__global__ void __launch_bounds__(RED_BLOCK)
block_field_pivot_kernel(const double *__restrict__ blk, int64_t n, int F, int64_t C, double *__restrict__ pivot) {
  __shared__ double s_mean, s_bd[RED_BLOCK / 32];
  __shared__ int s_bj[RED_BLOCK / 32];
  const int64_t R = n < PIV_ROWS ? n : PIV_ROWS, Q = C < PIV_SAMPLES / R ? C : PIV_SAMPLES / R, K = R * Q;
  for (int f = blockIdx.x; f < F; f += gridDim.x) {
    Comp sum, cnt;
    for (int64_t j = threadIdx.x; j < K; j += RED_BLOCK) {
      const double v = pivot_sample(blk, n, F, f, C, R, Q, j);
      if (isfinite(v)) { sum.add(v); cnt.add(1.0); }
    }
    const double t = block_reduce_comp<RED_BLOCK>(sum);
    const double m = block_reduce_comp<RED_BLOCK>(cnt);
    if (threadIdx.x == 0) s_mean = (m > 0.0 && isfinite(t / m)) ? t / m : 0.0;
    __syncthreads();
    const double mean = s_mean;
    double bd = INFINITY;
    int bj = INT_MAX;
    for (int64_t j = threadIdx.x; j < K; j += RED_BLOCK) {
      const double v = pivot_sample(blk, n, F, f, C, R, Q, j);
      if (isfinite(v)) take_nearer(bd, bj, fabs(v - mean), (int)j);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1)
      take_nearer(bd, bj, __shfl_down_sync(0xffffffffu, bd, off), __shfl_down_sync(0xffffffffu, bj, off));
    if ((threadIdx.x & 31) == 0) { s_bd[threadIdx.x >> 5] = bd; s_bj[threadIdx.x >> 5] = bj; }
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int w = 1; w < RED_BLOCK / 32; ++w) take_nearer(bd, bj, s_bd[w], s_bj[w]);
      pivot[f] = bj == INT_MAX ? 0.0 : pivot_sample(blk, n, F, f, C, R, Q, bj);
    }
    __syncthreads();
  }
}

// Visit the values of field f in the rows a CTA at grid x position bx owns.  The double2 path needs an even C (rows
// then start on 16 bytes relative to the base) and a 16-byte aligned base: a caller may pass any device pointer.
template <class Fn>
__device__ __forceinline__ void for_each_owned_value(const double *__restrict__ blk, int64_t n, int F, int64_t C,
                                                     int f, Fn fn) {
  const int64_t nvec = C / 2;
  const bool vec_ok = (C % 2 == 0) && (reinterpret_cast<uintptr_t>(blk) % 16 == 0);
  for (int64_t s = blockIdx.x; s < n; s += gridDim.x) {
    const double *row = blk + (s * F + f) * C;
    if (vec_ok) {
      const double2 *row2 = reinterpret_cast<const double2 *>(row);
      for (int64_t c = threadIdx.x; c < nvec; c += MOM_BLOCK) {
        const double2 v = __ldcs(row2 + c);
        fn(v.x); fn(v.y);
      }
    } else {
      for (int64_t c = threadIdx.x; c < C; c += MOM_BLOCK) fn(__ldcs(row + c));
    }
  }
}

// Fields stride over grid y (F may exceed its 65535 limit).  A non-finite value makes the CTA's partials non-finite
// (an inf or NaN never leaves a compensated sum), which block_field_classify_kernel then looks into.
__global__ void __launch_bounds__(MOM_BLOCK)
block_field_moments_kernel(const double *__restrict__ blk, int64_t n, int F, int64_t C,
                           const double *__restrict__ pivot, double *__restrict__ partial /* [3][F][gridDim.x] */) {
  for (int f = blockIdx.y; f < F; f += gridDim.y) {
    const double sh = pivot[f];
    Comp a1, a2;
    for_each_owned_value(blk, n, F, C, f, [&](double v) {
      const double a = v - sh;
      a1.add(a); a2.add(a * a);
    });
    const double t1 = block_reduce_comp<MOM_BLOCK>(a1);
    const double t2 = block_reduce_comp<MOM_BLOCK>(a2);
    if (threadIdx.x == 0) {
      partial[(int64_t)f * gridDim.x + blockIdx.x] = t1;
      partial[((int64_t)F + f) * gridDim.x + blockIdx.x] = t2;
    }
  }
}

// Same grid as the moments kernel.  A CTA whose partials are finite saw only finite values and records class 0;
// otherwise it reads its rows again and records which of NaN / +inf / -inf they hold.  The moments pass thus spends
// nothing on the check, and the second read happens only for a field that holds a non-finite value.
__global__ void __launch_bounds__(MOM_BLOCK)
block_field_classify_kernel(const double *__restrict__ blk, int64_t n, int F, int64_t C,
                            double *__restrict__ partial /* [3][F][gridDim.x] */) {
  for (int f = blockIdx.y; f < F; f += gridDim.y) {
    const int64_t i = (int64_t)f * gridDim.x + blockIdx.x;
    unsigned cls = 0;
    if (!isfinite(partial[i]) || !isfinite(partial[(int64_t)F * gridDim.x + i])) {
      unsigned nf = 0;
      for_each_owned_value(blk, n, F, C, f, [&](double v) {
        if (!isfinite(v)) nf |= isnan(v) ? NF_NAN : (v > 0.0 ? NF_PINF : NF_NINF);
      });
      cls = (__syncthreads_or(nf & NF_NAN) ? NF_NAN : 0u) | (__syncthreads_or(nf & NF_PINF) ? NF_PINF : 0u) |
            (__syncthreads_or(nf & NF_NINF) ? NF_NINF : 0u);
    }
    if (threadIdx.x == 0) partial[(int64_t)2 * F * gridDim.x + i] = (double)cls;
  }
}

// partial: [3][F][nb]
__global__ void finish_moments_kernel(const double *__restrict__ partial, int nb, int F, double cnt,
                                      const double *__restrict__ pivot, double *__restrict__ out) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= F) return;
  Comp s1, s2;
  unsigned cls = 0;
  for (int b = 0; b < nb; ++b) {
    s1.add(partial[(int64_t)f * nb + b]);
    s2.add(partial[((int64_t)F + f) * nb + b]);
    cls |= (unsigned)partial[((int64_t)2 * F + f) * nb + b];
  }
  const double S1 = s1.value(), S2 = s2.value();
  if ((cls & NF_NAN) || (cls & (NF_PINF | NF_NINF)) == (NF_PINF | NF_NINF)) out[f] = NAN;
  else if (cls) out[f] = (cls & NF_PINF) ? INFINITY : -INFINITY;
  else out[f] = pivot[f] + S1 / cnt;
  out[F + f] = cls ? NAN : std_of_var(fma(-S1, S1 / cnt, S2) / (cnt - 1.0));
}

// ---- row-major table [n][D]: column sums ----------------------------------
// blockDim = D * floor(256 / D), so a thread always sees the same column and
// the block reads contiguous memory.
template <int POW>
__global__ void table_col_reduce_kernel(const double *__restrict__ xs, int64_t total /* n*D */, int D,
                                        const double *__restrict__ shift, double *__restrict__ partial /*[gridDim.x][D]*/) {
  extern __shared__ double sm[];  // [blockDim.x]
  const int d = threadIdx.x % D;
  const double sh = shift ? shift[d] : 0.0;
  Comp acc;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (int64_t)gridDim.x * blockDim.x) {
    const double a = xs[k] - sh;
    acc.add(POW == 1 ? a : a * a);
  }
  sm[threadIdx.x] = comp_sum(acc);
  __syncthreads();
  if ((int)threadIdx.x < D) {
    Comp t;
    for (int k = threadIdx.x; k < (int)blockDim.x; k += D) t.add(sm[k]);
    partial[(int64_t)blockIdx.x * D + threadIdx.x] = comp_sum(t);
  }
}
__global__ void finish_cols_kernel(const double *__restrict__ partial, int nb, int D, double denom, int do_sqrt,
                                   double *__restrict__ out) {
  const int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= D) return;
  Comp acc;
  for (int b = 0; b < nb; ++b) acc.add(partial[(int64_t)b * D + d]);
  const double v = comp_sum(acc) / denom;
  out[d] = do_sqrt ? sqrt(v) : v;
}

// ---- autocorrelation (stats.ml:223-238), lags strided over grid y (nslides may exceed its 65535 limit) ----
__global__ void __launch_bounds__(RED_BLOCK)
autocorr_kernel(const double *__restrict__ x, int64_t n, int nslides, double mu, double sigma2,
                double *__restrict__ partial) {
  for (int lag = blockIdx.y; lag < nslides; lag += gridDim.y) {
    Comp acc;
    const int64_t m = n - lag;
    for (int64_t j = (int64_t)blockIdx.x * RED_BLOCK + threadIdx.x; j < m; j += (int64_t)gridDim.x * RED_BLOCK) {
      const double dx = x[j] - mu, dxs = x[j + lag] - mu;
      acc.add(dx * dxs / sigma2);
    }
    const double tot = block_reduce_comp<RED_BLOCK>(acc);
    if (threadIdx.x == 0) partial[(int64_t)lag * gridDim.x + blockIdx.x] = tot;
  }
}
__global__ void finish_autocorr_kernel(const double *__restrict__ partial, int nb, int nslides, int64_t n,
                                       double *__restrict__ out) {
  const int lag = blockIdx.x * blockDim.x + threadIdx.x;
  if (lag >= nslides) return;
  Comp acc;
  for (int b = 0; b < nb; ++b) acc.add(partial[(int64_t)lag * nb + b]);
  out[lag] = acc.value() / (double)(n - lag);
}

constexpr int64_t GRID_Y_MAX = 65535;

static int grid_for(mg_ctx *ctx, int64_t work_items) {
  int64_t g = (int64_t)ctx->sm_count * 8;
  if (g > work_items) g = work_items;
  return (int)(g < 1 ? 1 : g);
}

// Pool the per-chain running moments of the balanced sampler (mcmc_balanced.cuh, kMom): chain c holds its pivot
// p_c, S1_c = sum (v - p_c), S2_c = sum (v - p_c)^2 over its n recorded samples.  Chain mean m_c = p_c + S1_c / n,
// chain M2_c = S2_c - S1_c^2 / n; pooled mean = sum_c m_c / C and M2 = sum_c M2_c + n sum_c (m_c - mean)^2
// (the parallel-variance combination).  One CTA per field, compensated sums in a fixed order.
__global__ void __launch_bounds__(RED_BLOCK)
chain_moments_finish_kernel(const double *__restrict__ mom, int F, int64_t C, double n, double *__restrict__ out /* [2][F] */) {
  const int f = blockIdx.x;
  const double *piv = mom + (int64_t)f * C, *s1 = mom + (int64_t)(F + f) * C, *s2 = mom + (int64_t)(2 * F + f) * C;
  Comp acc;
  for (int64_t c = threadIdx.x; c < C; c += RED_BLOCK) acc.add(piv[c] + s1[c] / n);
  const double mean = block_reduce_comp<RED_BLOCK>(acc) / (double)C;
  __shared__ double s_mean;
  if (threadIdx.x == 0) s_mean = mean;
  __syncthreads();
  const double mu = s_mean;
  Comp m2;
  for (int64_t c = threadIdx.x; c < C; c += RED_BLOCK) {
    const double a = s1[c], mc = piv[c] + a / n, d = mc - mu;
    m2.add(s2[c] - a * a / n);
    m2.add(n * d * d);
  }
  const double M2 = block_reduce_comp<RED_BLOCK>(m2);
  if (threadIdx.x == 0) { out[f] = mu; out[F + f] = std_of_var(M2 / (n * (double)C - 1.0)); }   // stats.ml:85 (n - 1)
}

int chain_moments_finish(mg_ctx *ctx, cudaStream_t st, const double *mom, int F, int64_t C, int64_t n, double *d_out) {
  chain_moments_finish_kernel<<<F, RED_BLOCK, 0, st>>>(mom, F, C, (double)n, d_out);
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

// per-field mean and std of a device sample block; results in d_out[0..F) (mean), d_out[F..2F) (std)
int sample_block_stats(mg_ctx *ctx, const double *d_blk, int64_t n, int F, int64_t C, double *d_out) {
  cudaStream_t s = ctx->stream;
  const int gx = grid_for(ctx, n);
  DevBuf<double> partial, pivot;
  MG_CUDA(ctx, partial.alloc((size_t)3 * F * gx, s));
  MG_CUDA(ctx, pivot.alloc((size_t)F, s));
  block_field_pivot_kernel<<<F, RED_BLOCK, 0, s>>>(d_blk, n, F, C, pivot.get());
  MG_CHECK_LAUNCH(ctx);
  const dim3 grid(gx, (unsigned)std::min<int64_t>(F, GRID_Y_MAX));
  block_field_moments_kernel<<<grid, MOM_BLOCK, 0, s>>>(d_blk, n, F, C, pivot.get(), partial.get());
  MG_CHECK_LAUNCH(ctx);
  block_field_classify_kernel<<<grid, MOM_BLOCK, 0, s>>>(d_blk, n, F, C, partial.get());
  MG_CHECK_LAUNCH(ctx);
  finish_moments_kernel<<<(F + 63) / 64, 64, 0, s>>>(partial.get(), gx, F, (double)n * (double)C, pivot.get(), d_out);
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

// column mean (pow 1) or std about `d_shift` (pow 2) of a device table [n][D]
static int table_cols(mg_ctx *ctx, const double *d_xs, int64_t n, int D, const double *d_shift, int pow,
                      double denom, int do_sqrt, double *d_out) {
  cudaStream_t s = ctx->stream;
  const int bs = D * (256 / D > 0 ? 256 / D : 1);
  const int64_t total = n * D;
  const int gx = grid_for(ctx, (total + bs - 1) / bs);
  DevBuf<double> partial;
  MG_CUDA(ctx, partial.alloc((size_t)gx * D, s));
  if (pow == 1) table_col_reduce_kernel<1><<<gx, bs, bs * sizeof(double), s>>>(d_xs, total, D, d_shift, partial.get());
  else table_col_reduce_kernel<2><<<gx, bs, bs * sizeof(double), s>>>(d_xs, total, D, d_shift, partial.get());
  MG_CHECK_LAUNCH(ctx);
  finish_cols_kernel<<<(D + 63) / 64, 64, 0, s>>>(partial.get(), gx, D, denom, do_sqrt, d_out);
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

}  // namespace mg

using namespace mg;

extern "C" int mg_stats_sample_block_dev(mg_ctx *ctx, const double *d_samples, int64_t n, int32_t D, int64_t C,
                                         double *out_mean, double *out_std) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, d_samples && n >= 1 && D >= 1 && C >= 1, "stats: bad sample block");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  const int F = D + 2;
  DevBuf<double> d_out;
  MG_CUDA(ctx, d_out.alloc((size_t)2 * F, ctx->stream));
  int rc = sample_block_stats(ctx, d_samples, n, F, C, d_out.get());
  if (rc) return rc;
  std::vector<double> h(2 * F);
  MG_CUDA(ctx, cudaMemcpyAsync(h.data(), d_out.get(), sizeof(double) * 2 * F, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (out_mean) memcpy(out_mean, h.data(), sizeof(double) * F);
  if (out_std) memcpy(out_std, h.data() + F, sizeof(double) * F);
  return MG_OK;
}

extern "C" int mg_stats_multi_mean(mg_ctx *ctx, const double *xs, int64_t n, int32_t D, double *out) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, xs && out && n >= 1 && D >= 1 && D <= 256, "multi_mean: bad arguments");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  DevBuf<double> d_xs, d_out;
  MG_CUDA(ctx, upload(d_xs, xs, (size_t)n * D, ctx->stream));
  MG_CUDA(ctx, d_out.alloc(D, ctx->stream));
  int rc = table_cols(ctx, d_xs.get(), n, D, nullptr, 1, (double)n, 0, d_out.get());
  if (rc) return rc;
  MG_CUDA(ctx, cudaMemcpyAsync(out, d_out.get(), sizeof(double) * D, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MG_OK;
}

extern "C" int mg_stats_multi_std(mg_ctx *ctx, const double *xs, int64_t n, int32_t D, const double *mean_or_null,
                                  double *out) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, xs && out && n >= 2 && D >= 1 && D <= 256, "multi_std: bad arguments");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  DevBuf<double> d_xs, d_mu, d_out;
  MG_CUDA(ctx, upload(d_xs, xs, (size_t)n * D, ctx->stream));
  MG_CUDA(ctx, d_mu.alloc(D, ctx->stream));
  MG_CUDA(ctx, d_out.alloc(D, ctx->stream));
  int rc;
  if (mean_or_null) MG_CUDA(ctx, cudaMemcpyAsync(d_mu.get(), mean_or_null, sizeof(double) * D, cudaMemcpyHostToDevice, ctx->stream));
  else if ((rc = table_cols(ctx, d_xs.get(), n, D, nullptr, 1, (double)n, 0, d_mu.get()))) return rc;
  if ((rc = table_cols(ctx, d_xs.get(), n, D, d_mu.get(), 2, (double)(n - 1), 1, d_out.get()))) return rc;
  MG_CUDA(ctx, cudaMemcpyAsync(out, d_out.get(), sizeof(double) * D, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MG_OK;
}

// Stats.multi_mean / multi_std (stats.ml:58-87) of samples held by several ranks, from each rank's own
// (count, mean[F], std[F]): a header exchange checks that F agrees, then the records are all-gathered and pooled in
// rank order with the parallel-variance update (Chan et al.), std with n - 1 as the reference.  Every rank receives
// the same values.
extern "C" int mg_comm_pool_moments(mg_comm *c, int64_t n_local, const double *mean_local, const double *std_local,
                                    int32_t F, int64_t *n_total, double *out_mean, double *out_std) {
  if (!c) return MG_EINVAL;
  mg_ctx *ctx = mg_comm_ctx(c);
  int rc = MG_OK;
  if (!(mean_local && std_local && F >= 1 && F <= 4096 && n_local >= 0)) rc = set_err(ctx, MG_EINVAL, "pool_moments: bad arguments");
  std::vector<int32_t> hdr = {F}, hdrs;
  if ((rc = comm_gather(c, rc, hdr, hdrs, "pool_moments"))) return rc;
  for (int r = 0; r < mg_comm_size(c); ++r)
    if (hdrs[r] != F) return set_err(ctx, MG_EINVAL, "pool_moments: rank %d has another F", r);
  std::vector<double> mine((size_t)1 + 2 * F), all;
  mine[0] = (double)n_local;
  for (int i = 0; i < F; ++i) {
    mine[1 + i] = mean_local[i];
    mine[1 + F + i] = n_local > 1 ? std_local[i] * std_local[i] * ((double)n_local - 1.0) : 0.0;   // sum of squared deviations
  }
  if ((rc = comm_gather(c, MG_OK, mine, all, "pool_moments"))) return rc;
  double n = 0.0;
  std::vector<double> mean(F, 0.0), m2(F, 0.0);
  for (int r = 0; r < mg_comm_size(c); ++r) {
    const double *rec = all.data() + (size_t)r * mine.size();
    const double cnt = rec[0];
    if (cnt == 0.0) continue;
    const double tot = n + cnt;
    for (int i = 0; i < F; ++i) {
      const double delta = rec[1 + i] - mean[i];
      mean[i] = mean[i] + delta * (cnt / tot);
      m2[i] = m2[i] + rec[1 + F + i] + delta * delta * (n * cnt / tot);
    }
    n = tot;
  }
  if (n_total) *n_total = (int64_t)n;
  for (int i = 0; i < F; ++i) {
    if (out_mean) out_mean[i] = mean[i];
    if (out_std) out_std[i] = n > 1.0 ? sqrt(m2[i] / (n - 1.0)) : 0.0;
  }
  return MG_OK;
}

extern "C" int mg_stats_mean(mg_ctx *ctx, const double *x, int64_t n, double *out) {
  return mg_stats_multi_mean(ctx, x, n, 1, out);
}

extern "C" int mg_stats_std(mg_ctx *ctx, const double *x, int64_t n, int have_mean, double mean, double *out) {
  return mg_stats_multi_std(ctx, x, n, 1, have_mean ? &mean : nullptr, out);
}

extern "C" int mg_stats_autocorrelation(mg_ctx *ctx, const double *x, int64_t n, int32_t nslides, double *out_r,
                                        double *out_length) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, x && out_r && n >= 2 && nslides >= 1, "slow_autocorrelation: bad arguments");
  if (!(nslides < n)) return set_err(ctx, MG_EFAIL, "Assert_failure stats.ml:229 (nslides < n)");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  DevBuf<double> d_x, d_ms, d_partial, d_out;
  MG_CUDA(ctx, upload(d_x, x, (size_t)n, s));
  MG_CUDA(ctx, d_ms.alloc(2, s));
  int rc;
  if ((rc = table_cols(ctx, d_x.get(), n, 1, nullptr, 1, (double)n, 0, d_ms.get()))) return rc;
  if ((rc = table_cols(ctx, d_x.get(), n, 1, d_ms.get(), 2, (double)(n - 1), 1, d_ms.get() + 1))) return rc;
  double ms[2];
  MG_CUDA(ctx, cudaMemcpyAsync(ms, d_ms.get(), sizeof ms, cudaMemcpyDeviceToHost, s));
  MG_CUDA(ctx, cudaStreamSynchronize(s));
  const double sigma2 = ms[1] * ms[1];  // stats.ml:228
  const int gx = grid_for(ctx, (n + RED_BLOCK - 1) / RED_BLOCK);
  MG_CUDA(ctx, d_partial.alloc((size_t)gx * nslides, s));
  MG_CUDA(ctx, d_out.alloc(nslides, s));
  autocorr_kernel<<<dim3(gx, (unsigned)std::min<int64_t>(nslides, GRID_Y_MAX)), RED_BLOCK, 0, s>>>(
      d_x.get(), n, nslides, ms[0], sigma2, d_partial.get());
  MG_CHECK_LAUNCH(ctx);
  finish_autocorr_kernel<<<(nslides + 63) / 64, 64, 0, s>>>(d_partial.get(), gx, nslides, n, d_out.get());
  MG_CHECK_LAUNCH(ctx);
  MG_CUDA(ctx, cudaMemcpyAsync(out_r, d_out.get(), sizeof(double) * nslides, cudaMemcpyDeviceToHost, s));
  MG_CUDA(ctx, cudaStreamSynchronize(s));
  if (out_length) {  // integrated autocorrelation length (an addition, SURVEY F6)
    double L = 1.0;
    for (int i = 1; i < nslides && out_r[i] > 0.0; ++i) L += 2.0 * out_r[i];
    *out_length = L;
  }
  return MG_OK;
}

// ---------------------------------------------------------------------------
// Stats.draw_uniform / draw_gaussian / draw_cauchy (stats.ml:89-91,113-128) in bulk: draw i of a call uses the
// Philox stream (P_DRAW, i, 1) -- the reference's global Random stream is not reproduced (SURVEY section 8 S3).
// ---------------------------------------------------------------------------
namespace mg {
__global__ void stats_draw_kernel(CallKey key, int kind, double a, double b, int64_t n, double *__restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    Rng r(key, P_DRAW, (uint64_t)i, 1);
    double v;
    if (kind == MG_DRAW_UNIFORM) v = draw_uniform(r, a, b);
    else if (kind == MG_DRAW_GAUSSIAN) v = draw_gaussian(r, a, b);
    else v = draw_cauchy(r, a, b);
    out[i] = v;
  }
}
}  // namespace mg

extern "C" int mg_stats_draw_dev(mg_ctx *ctx, int32_t kind, double a, double b, int64_t n, double *d_out) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, kind >= MG_DRAW_UNIFORM && kind <= MG_DRAW_CAUCHY, "stats_draw: unknown distribution %d", kind);
  MG_REQUIRE(ctx, n >= 0 && (d_out || n == 0), "stats_draw: bad arguments");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  const CallKey key = next_key(ctx);
  if (n == 0) return MG_OK;
  const int64_t blocks = std::min<int64_t>((n + 255) / 256, (int64_t)ctx->sm_count * 16);
  stats_draw_kernel<<<(unsigned)blocks, 256, 0, ctx->stream>>>(key, kind, a, b, n, d_out);
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

extern "C" int mg_stats_draw(mg_ctx *ctx, int32_t kind, double a, double b, int64_t n, double *out) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, n >= 0 && (out || n == 0), "stats_draw: bad arguments");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  DevBuf<double> d;
  MG_CUDA(ctx, d.alloc((size_t)n, ctx->stream));
  int rc = mg_stats_draw_dev(ctx, kind, a, b, n, d.get());
  if (rc) return rc;
  if (n) MG_CUDA(ctx, cudaMemcpyAsync(out, d.get(), sizeof(double) * n, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MG_OK;
}
