// stats.cu -- Stats.mean / std / multi_mean / multi_std / slow_autocorrelation
// (stats.ml:17-87,223-238) as coalesced grid-stride reductions.
//
// The reference sums left to right in float64 (stats.ml:19-22).  A parallel
// sum cannot reproduce that rounding sequence; instead every thread keeps a
// compensated (Neumaier) partial, partials are combined in a fixed order
// (warp shuffle tree, then one block-order pass), so the result is
// deterministic and within a few ulp of the exactly rounded sum -- closer to
// exact than the reference's own sequential sum.  Parity tolerance: 1e-12 rel.
// All kernels are HBM-bound: 8 bytes read per element per pass.
#include "common.cuh"
#include "models.cuh"
#include "rng.cuh"
#include "reduce.cuh"

namespace mg {

constexpr int RED_BLOCK = 256;

// ---- sample block [n][F][C] ---------------------------------------------------
// One pass for both moments: sums of (x - s_f) and (x - s_f)^2 about a pivot
// s_f (the field's first sample), so that
//   mean = s + S1/N,   var = (S2 - S1^2/N) / (N - 1)
// read the 62.9 GB sample block once instead of twice.  With the pivot inside
// the distribution the subtraction loses less than a digit, and both sums are
// compensated; agreement with Stats.multi_mean / multi_std stays within 1e-12
// (tests/test_mcmc_gpu.py::test_resident_call_and_block_stats).
constexpr int MOM_BLOCK = RED_BLOCK;
__global__ void __launch_bounds__(MOM_BLOCK)
block_field_moments_kernel(const double *__restrict__ blk, int64_t n, int F, int64_t C,
                           double *__restrict__ partial /* [2][F][gridDim.x] */) {
  const int f = blockIdx.y;
  const double sh = blk[(int64_t)f * C];   // pivot: sample 0, chain 0 of the block
  Comp a1, a2;
  const int64_t nvec = C / 2;
  const bool vec_ok = (C % 2 == 0);
  for (int64_t s = blockIdx.x; s < n; s += gridDim.x) {
    const double *row = blk + (s * F + f) * C;
    if (vec_ok) {
      const double2 *row2 = reinterpret_cast<const double2 *>(row);
      for (int64_t c = threadIdx.x; c < nvec; c += MOM_BLOCK) {
        const double2 v = __ldcs(row2 + c);
        const double a = v.x - sh, b = v.y - sh;
        a1.add(a); a1.add(b); a2.add(a * a); a2.add(b * b);
      }
    } else {
      for (int64_t c = threadIdx.x; c < C; c += MOM_BLOCK) {
        const double a = __ldcs(row + c) - sh;
        a1.add(a); a2.add(a * a);
      }
    }
  }
  const double t1 = block_reduce_comp<MOM_BLOCK>(a1);
  const double t2 = block_reduce_comp<MOM_BLOCK>(a2);
  if (threadIdx.x == 0) {
    partial[(int64_t)f * gridDim.x + blockIdx.x] = t1;
    partial[((int64_t)F + f) * gridDim.x + blockIdx.x] = t2;
  }
}

// partial: [2][F][nb]
__global__ void finish_moments_kernel(const double *__restrict__ partial, int nb, int F, double cnt,
                                      const double *__restrict__ blk, int64_t C, double *__restrict__ out) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= F) return;
  Comp s1, s2;
  for (int b = 0; b < nb; ++b) {
    s1.add(partial[(int64_t)f * nb + b]);
    s2.add(partial[((int64_t)F + f) * nb + b]);
  }
  const double sh = blk[(int64_t)f * C];
  const double S1 = s1.value(), S2 = s2.value();
  out[f] = sh + S1 / cnt;
  const double var = (S2 - S1 * (S1 / cnt)) / (cnt - 1.0);
  out[F + f] = sqrt(var > 0.0 ? var : 0.0);
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
  sm[threadIdx.x] = acc.value();
  __syncthreads();
  if ((int)threadIdx.x < D) {
    Comp t;
    for (int k = threadIdx.x; k < (int)blockDim.x; k += D) t.add(sm[k]);
    partial[(int64_t)blockIdx.x * D + threadIdx.x] = t.value();
  }
}
__global__ void finish_cols_kernel(const double *__restrict__ partial, int nb, int D, double denom, int do_sqrt,
                                   double *__restrict__ out) {
  const int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= D) return;
  Comp acc;
  for (int b = 0; b < nb; ++b) acc.add(partial[(int64_t)b * D + d]);
  const double v = acc.value() / denom;
  out[d] = do_sqrt ? sqrt(v) : v;
}

// ---- autocorrelation (stats.ml:223-238), one block row per lag -------------
__global__ void __launch_bounds__(RED_BLOCK)
autocorr_kernel(const double *__restrict__ x, int64_t n, double mu, double sigma2, double *__restrict__ partial) {
  const int lag = blockIdx.y;
  Comp acc;
  const int64_t m = n - lag;
  for (int64_t j = (int64_t)blockIdx.x * RED_BLOCK + threadIdx.x; j < m; j += (int64_t)gridDim.x * RED_BLOCK) {
    const double dx = x[j] - mu, dxs = x[j + lag] - mu;
    acc.add(dx * dxs / sigma2);
  }
  const double tot = block_reduce_comp<RED_BLOCK>(acc);
  if (threadIdx.x == 0) partial[(int64_t)lag * gridDim.x + blockIdx.x] = tot;
}
__global__ void finish_autocorr_kernel(const double *__restrict__ partial, int nb, int nslides, int64_t n,
                                       double *__restrict__ out) {
  const int lag = blockIdx.x * blockDim.x + threadIdx.x;
  if (lag >= nslides) return;
  Comp acc;
  for (int b = 0; b < nb; ++b) acc.add(partial[(int64_t)lag * nb + b]);
  out[lag] = acc.value() / (double)(n - lag);
}

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
  if (threadIdx.x == 0) { out[f] = mu; out[F + f] = sqrt(M2 / (n * (double)C - 1.0)); }   // stats.ml:85 (n - 1)
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
  DevBuf<double> partial;
  MG_CUDA(ctx, partial.alloc((size_t)2 * F * gx, s));
  block_field_moments_kernel<<<dim3(gx, F), MOM_BLOCK, 0, s>>>(d_blk, n, F, C, partial.get());
  MG_CHECK_LAUNCH(ctx);
  finish_moments_kernel<<<(F + 63) / 64, 64, 0, s>>>(partial.get(), gx, F, (double)n * (double)C, d_blk, C, d_out);
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
  autocorr_kernel<<<dim3(gx, nslides), RED_BLOCK, 0, s>>>(d_x.get(), n, ms[0], sigma2, d_partial.get());
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
