// quantiles.cu -- exact per-field order statistics and quantiles of a sample block [n][D+2][C], on one GPU and pooled
// over ranks.  Definitions in include/mcmc_gpu.h and DESIGN.md 4c, transcribed line by line in oracle/quantiles_np.py.
//
// Every answer is an order statistic of a field's pool (the n C values of the field, chains pooled) in the order of
// f64_to_ordered; a quantile needs ranks lo and lo + 1, and the ranks of one call are de-duplicated (at most
// QT_MAXT = 2 MG_QUANT_MAX).  All work is on the 64-bit ordered keys, so the answers are exact.
//
// 1. Sample: an evenly strided subsample of each field (S keys, S = N when the pool is small), sorted with
//    radix_sort.cuh.  Target rank k sits near sample rank k (S-1)/(N-1); its bracket is the pair of sample keys a
//    margin of 4 sigma of the sample rank (plus 16) either side, the open ends of the sample widened to the whole key
//    range.  A full sample (S = N) gives the exact bracket [x_(k), x_(k)].  Overlapping brackets of a field merge.
// 2. One read of the block (qt_pass_kernel): each key is counted in its region (below the first bracket, inside
//    bracket b, between two brackets, above the last) and, inside a bracket whose ends differ, appended to the field's
//    candidate buffer (warp-aggregated atomics); past the buffer's budget it is still counted but not written.  NaN is
//    flagged per field.  Loads are 8-byte and coalesced along a row's C chains; the block base may be any 8-byte
//    address.
// 3. Resolve (host): rank k hits its bracket when (keys below the bracket) <= k < (below + inside).  A bracket with
//    lo = hi answers with lo; otherwise, if the field's candidates fit the budget, the answer is the candidate of rank
//    k - below (+ the candidates of the field's earlier brackets), found by the radix select of step 4 over the
//    candidate buffer (8 passes over at most budget keys, not over the block).
// 4. Radix select (qt_select_kernel, and the fallback for ranks that miss or fields that overflow): MSB-first, 8-bit
//    digits; a pass histograms the next digit of the keys whose higher digits equal a target's prefix found so far
//    (up to QT_MAXT distinct prefixes x 256 int32 bins in shared memory) and the host walks the histogram.  Over the
//    block it is 8 more full reads of the field, exact, only slower.
// Sharded (mg_comm_quantiles): every rank runs the same steps on its own block; the brackets are the widest of the
// ranks' brackets (min of lo, max of hi), and the region counts, NaN and overflow flags and every select histogram
// are summed over the ranks in rank order.  Every decision is taken from those exchanged integers, so every rank
// takes the same path, and the answers, being exact order statistics of the union, are the single-GPU bits.
#include <algorithm>
#include <cmath>
#include <cstdlib>

#include "common.cuh"
#include "radix_sort.cuh"

namespace mg {

constexpr int QT_THREADS = 256;
constexpr int QT_UNROLL = 4;                    // loads in flight per thread
constexpr int QT_MAXT = 2 * MG_QUANT_MAX;       // target ranks per call
constexpr int QT_NREG = 2 * QT_MAXT + 1;        // regions of a field: below, inside / between the brackets, above
constexpr int64_t QT_CHUNK_MAX = 1LL << 30;     // keys per CTA: its int32 counters cannot overflow

__host__ __device__ __forceinline__ double ordered_to_f64(uint64_t k) {
  const uint64_t b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
#ifdef __CUDA_ARCH__
  return __longlong_as_double((long long)b);
#else
  double x; memcpy(&x, &b, 8); return x;
#endif
}

// Visit the keys of pool positions [j0, j1) of one field, j = s C + c at element s * rstride + c of the field's
// base, QT_UNROLL loads in flight per thread.  The trip count is the same for every thread of the CTA, so warp
// collectives inside visit() see full warps; visit(ok, value) is called with ok = false past j1.
template <class T, class Visit>
__device__ __forceinline__ void qt_walk(const T *__restrict__ base, int64_t C, int64_t rstride, int64_t j0, int64_t j1,
                                        Visit visit) {
  const int64_t ds = QT_THREADS / C, dc = QT_THREADS - ds * C;
  int64_t j = j0 + threadIdx.x, s = j / C, c = j - s * C;
  for (int64_t b0 = j0; b0 < j1; b0 += (int64_t)QT_THREADS * QT_UNROLL) {
    T v[QT_UNROLL];
    bool ok[QT_UNROLL];
#pragma unroll
    for (int u = 0; u < QT_UNROLL; ++u) {
      ok[u] = j < j1;
      v[u] = ok[u] ? __ldg(base + s * rstride + c) : (T)0;
      j += QT_THREADS; s += ds; c += dc;
      if (c >= C) { c -= C; ++s; }
    }
#pragma unroll
    for (int u = 0; u < QT_UNROLL; ++u) visit(ok[u], v[u]);
  }
}

__global__ void qt_sample_kernel(const double *__restrict__ x, int64_t C, int64_t rstride, int F, int64_t N, int64_t S,
                                 uint64_t *__restrict__ keys, int32_t *__restrict__ vals) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)F * S) return;
  const int64_t f = t / S, i = t - f * S;
  const int64_t j = (int64_t)((unsigned __int128)i * (uint64_t)N / (uint64_t)S);
  const int64_t s = j / C;
  keys[t] = f64_to_ordered(__ldg(x + s * rstride + f * C + (j - s * C)));
  vals[t] = 0;
}

// out [F][K][2] = the sorted sample's keys at ilo / ihi (-1: the open end of the key range)
__global__ void qt_bracket_kernel(const uint64_t *__restrict__ sorted, int64_t S, int F, int K,
                                  const int64_t *__restrict__ ilo, const int64_t *__restrict__ ihi,
                                  uint64_t *__restrict__ out) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)F * K) return;
  const int64_t f = t / K, j = t - f * K;
  out[2 * t] = ilo[j] < 0 ? 0ull : sorted[f * S + ilo[j]];
  out[2 * t + 1] = ihi[j] < 0 ? ~0ull : sorted[f * S + ihi[j]];
}

struct QtPassArgs {
  const double *x;
  int64_t C, rstride, len, per;   // chains, row stride (F C), keys per field, keys per CTA
  int chunks;                     // CTAs per field
  const uint64_t *lo, *hi;        // [F][QT_MAXT] merged brackets, ascending and disjoint
  const int *nb;                  // [F] brackets per field
  unsigned long long *cnt;        // [F][QT_NREG] keys per region
  unsigned long long *ccnt;       // [F] keys inside the brackets with lo != hi (written or not)
  uint64_t *cand;                 // [F][budget]
  int64_t budget;
  int *nan;                       // [F]
};

__global__ void __launch_bounds__(QT_THREADS) qt_pass_kernel(const QtPassArgs a) {
  __shared__ uint64_t slo[QT_MAXT], shi[QT_MAXT];
  __shared__ int scnt[QT_NREG];
  __shared__ int snan;
  const int64_t f = blockIdx.x / a.chunks, ch = blockIdx.x - f * a.chunks;
  const int nb = a.nb[f];
  for (int i = threadIdx.x; i < nb; i += QT_THREADS) { slo[i] = a.lo[f * QT_MAXT + i]; shi[i] = a.hi[f * QT_MAXT + i]; }
  for (int i = threadIdx.x; i < QT_NREG; i += QT_THREADS) scnt[i] = 0;
  if (threadIdx.x == 0) snan = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const unsigned below_me = (1u << lane) - 1u;
  const int64_t j0 = ch * a.per, j1 = min(a.len, j0 + a.per);
  uint64_t *cf = a.cand + f * a.budget;
  unsigned long long *ccnt = a.ccnt + f;
  const unsigned long long budget = (unsigned long long)a.budget;
  bool nan = false;
  qt_walk(a.x + f * a.C, a.C, a.rstride, j0, j1, [&](bool ok, double v) {
    nan = nan || (ok && isnan(v));
    const uint64_t k = f64_to_ordered(v);
    int t = 0, h = nb;                                 // t = brackets with lo <= k
    while (t < h) { const int m = (t + h) >> 1; if (slo[m] <= k) t = m + 1; else h = m; }
    const bool in = t > 0 && k <= shi[t - 1];
    const int reg = in ? 2 * t - 1 : 2 * t;
    const unsigned peers = __match_any_sync(0xffffffffu, ok ? reg : -1);
    if (ok && (peers & below_me) == 0) atomicAdd(&scnt[reg], __popc(peers));
    const bool put = ok && in && slo[t - 1] != shi[t - 1];
    const unsigned m = __ballot_sync(0xffffffffu, put);
    if (m) {
      const int leader = __ffs(m) - 1;
      unsigned long long base = 0;
      if (lane == leader) base = atomicAdd(ccnt, (unsigned long long)__popc(m));
      base = __shfl_sync(0xffffffffu, base, leader);
      const unsigned long long pos = base + __popc(m & below_me);
      if (put && pos < budget) cf[pos] = k;
    }
  });
  if (nan) snan = 1;
  __syncthreads();
  for (int r = threadIdx.x; r < 2 * nb + 1; r += QT_THREADS)
    if (scnt[r]) atomicAdd(a.cnt + f * QT_NREG + r, (unsigned long long)scnt[r]);
  if (threadIdx.x == 0 && snan) a.nan[f] = 1;
}

struct QtSelArgs {
  const void *base;               // the block (doubles) or the candidate buffer (keys)
  int64_t C, rstride, per;
  int chunks;                     // CTAs per slot
  const int *fld;                 // [nslot] field of the slot
  const int64_t *len;             // [nslot] keys of the slot
  const uint64_t *pref;           // [nslot][QT_MAXT] distinct prefixes (the key's top pbits bits), ascending
  const int *np;                  // [nslot]
  const int64_t *hoff;            // [nslot] offset of the slot's [np][256] histogram
  int pbits;                      // bits fixed so far: 8 * pass
  unsigned long long *hist;
};

// one MSB-first radix-select pass: histogram of digit 7 - pass of the keys that share a target's prefix
template <bool KEYS>
__global__ void __launch_bounds__(QT_THREADS) qt_select_kernel(const QtSelArgs a) {
  extern __shared__ int sh[];                          // [np][256]
  __shared__ uint64_t sp[QT_MAXT];
  const int64_t g = blockIdx.x / a.chunks, ch = blockIdx.x - g * a.chunks;
  const int np = a.np[g];
  for (int i = threadIdx.x; i < np; i += QT_THREADS) sp[i] = a.pref[g * QT_MAXT + i];
  for (int i = threadIdx.x; i < np * 256; i += QT_THREADS) sh[i] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const unsigned below_me = (1u << lane) - 1u;
  const int64_t j0 = ch * a.per, j1 = min(a.len[g], j0 + a.per);
  const int pbits = a.pbits, shift = 56 - pbits;
  auto visit = [&](bool ok, uint64_t k) {
    int idx = 0;
    if (pbits) {
      const uint64_t p = k >> (64 - pbits);
      int h = np;
      while (idx < h) { const int m = (idx + h) >> 1; if (sp[m] < p) idx = m + 1; else h = m; }
      ok = ok && idx < np && sp[idx] == p;
    }
    const int bin = idx * 256 + (int)((k >> shift) & 0xFF);
    const unsigned peers = __match_any_sync(0xffffffffu, ok ? bin : -1);
    if (ok && (peers & below_me) == 0) atomicAdd(&sh[bin], __popc(peers));
  };
  const int64_t f = a.fld[g];
  if (KEYS)
    qt_walk((const unsigned long long *)a.base + f * a.C, a.C, a.rstride, j0, j1,
            [&](bool ok, unsigned long long k) { visit(ok, (uint64_t)k); });
  else
    qt_walk((const double *)a.base + f * a.C, a.C, a.rstride, j0, j1,
            [&](bool ok, double v) { visit(ok, f64_to_ordered(v)); });
  __syncthreads();
  unsigned long long *hg = a.hist + a.hoff[g];
  for (int i = threadIdx.x; i < np * 256; i += QT_THREADS)
    if (sh[i]) atomicAdd(hg + i, (unsigned long long)sh[i]);
}

// ---- host --------------------------------------------------------------------------------------------------------

// Combine a host vector of integers over the ranks in rank order (op(i, acc, x)), carrying every rank's status: a
// failure on any rank is returned on every rank.  Without a communicator only the local status is returned.
template <class Op>
static int qt_exchange(mg_ctx *ctx, mg_comm *comm, int rc, std::vector<uint64_t> &v, Op op) {
  if (!comm) return rc;
  const int R = mg_comm_size(comm);
  const size_t W = v.size() + 1;
  std::vector<uint64_t> mine(W, 0), all(W * R);
  mine[0] = (uint64_t)rc;
  if (rc == MG_OK) std::copy(v.begin(), v.end(), mine.begin() + 1);
  const int rc2 = mg_comm_allgather(comm, mine.data(), all.data(), (int64_t)(sizeof(uint64_t) * W));
  if (rc) return rc;
  if (rc2) return rc2;
  for (int r = 0; r < R; ++r)
    if (all[W * r] != 0) return set_err(ctx, (int)all[W * r], "quantiles (comm): rank %d failed", r);
  for (size_t i = 0; i < v.size(); ++i) {
    uint64_t acc = all[1 + i];
    for (int r = 1; r < R; ++r) acc = op(i, acc, all[W * r + 1 + i]);
    v[i] = acc;
  }
  return MG_OK;
}
static uint64_t qt_sum(size_t, uint64_t a, uint64_t b) { return a + b; }

static int64_t qt_chunks(mg_ctx *ctx, int64_t nslot, int64_t maxlen) {
  int64_t ch = std::max<int64_t>(1, ((int64_t)ctx->sm_count * 32 + nslot - 1) / nslot);
  ch = std::max(ch, (maxlen + QT_CHUNK_MAX - 1) / QT_CHUNK_MAX);
  return std::max<int64_t>(1, std::min(ch, std::max<int64_t>(1, (maxlen + QT_THREADS - 1) / QT_THREADS)));
}

// Exact order statistics of several slots by radix select.  Slot g: field fld[g] of `base` (the block when !keys,
// the candidate buffer [F][C] when keys), len[g] local keys, ascending target ranks rank[g] (global when pooled);
// keys are returned in out[g].  8 passes, each one histogram exchange.
struct QtSlots {
  std::vector<int> fld;
  std::vector<int64_t> len;
  std::vector<std::vector<int64_t>> rank;
  std::vector<std::vector<uint64_t>> out;
};

static int qt_select(mg_ctx *ctx, mg_comm *comm, bool keys, const void *base, int64_t C, int64_t rstride, QtSlots &sl) {
  cudaStream_t st = ctx->stream;
  const int64_t ns = (int64_t)sl.fld.size();
  std::vector<std::vector<int64_t>> rem = sl.rank;
  std::vector<std::vector<uint64_t>> pre(ns);
  for (int64_t g = 0; g < ns; ++g) pre[g].assign(sl.rank[g].size(), 0);
  int64_t maxlen = 0;
  for (int64_t v : sl.len) maxlen = std::max(maxlen, v);
  const int64_t chunks = qt_chunks(ctx, ns, maxlen), per = (maxlen + chunks - 1) / chunks;
  DevBuf<int> d_fld, d_np;
  DevBuf<int64_t> d_len, d_hoff;
  DevBuf<uint64_t> d_pref;
  DevBuf<unsigned long long> d_hist;
  std::vector<int> np(ns);
  std::vector<int64_t> hoff(ns + 1);
  std::vector<uint64_t> pref((size_t)ns * QT_MAXT), hist;
  std::vector<std::vector<int>> tp(ns);            // target -> its prefix's index
  int rc = MG_OK;
  auto local = [&](int pass) -> int {
    if (pass == 0) {
      MG_CUDA(ctx, upload(d_fld, sl.fld.data(), (size_t)ns, st));
      MG_CUDA(ctx, upload(d_len, sl.len.data(), (size_t)ns, st));
    }
    MG_CUDA(ctx, upload(d_pref, pref.data(), pref.size(), st));
    MG_CUDA(ctx, upload(d_np, np.data(), (size_t)ns, st));
    MG_CUDA(ctx, upload(d_hoff, hoff.data(), (size_t)ns, st));
    MG_CUDA(ctx, d_hist.alloc((size_t)hoff[ns], st));
    MG_CUDA(ctx, cudaMemsetAsync(d_hist.get(), 0, sizeof(unsigned long long) * hoff[ns], st));
    int npmax = 1;
    for (int v : np) npmax = std::max(npmax, v);
    const size_t smem = sizeof(int) * 256 * npmax;
    QtSelArgs a;
    a.base = base; a.C = C; a.rstride = rstride; a.per = per; a.chunks = (int)chunks;
    a.fld = d_fld.get(); a.len = d_len.get(); a.pref = d_pref.get(); a.np = d_np.get(); a.hoff = d_hoff.get();
    a.pbits = 8 * pass; a.hist = d_hist.get();
    const dim3 grid((unsigned)(ns * chunks));
    if (keys) {
      MG_CUDA(ctx, cudaFuncSetAttribute(qt_select_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      qt_select_kernel<true><<<grid, QT_THREADS, smem, st>>>(a);
    } else {
      MG_CUDA(ctx, cudaFuncSetAttribute(qt_select_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      qt_select_kernel<false><<<grid, QT_THREADS, smem, st>>>(a);
    }
    MG_CHECK_LAUNCH(ctx);
    hist.resize((size_t)hoff[ns]);
    MG_CUDA(ctx, cudaMemcpyAsync(hist.data(), d_hist.get(), sizeof(uint64_t) * hist.size(), cudaMemcpyDeviceToHost, st));
    MG_CUDA(ctx, cudaStreamSynchronize(st));
    return MG_OK;
  };
  for (int pass = 0; pass < 8; ++pass) {
    // the distinct prefixes of each slot's targets: ascending, as the targets' ranks are
    hoff[0] = 0;
    for (int64_t g = 0; g < ns; ++g) {
      const size_t T = sl.rank[g].size();
      tp[g].assign(T, 0);
      int P = 0;
      for (size_t t = 0; t < T; ++t) {
        if (P == 0 || pref[(size_t)g * QT_MAXT + P - 1] != pre[g][t]) pref[(size_t)g * QT_MAXT + P++] = pre[g][t];
        tp[g][t] = P - 1;
      }
      np[g] = P;
      hoff[g + 1] = hoff[g] + 256LL * P;
    }
    if (rc == MG_OK) rc = local(pass);
    hist.resize((size_t)hoff[ns]);
    if ((rc = qt_exchange(ctx, comm, rc, hist, qt_sum))) return rc;
    for (int64_t g = 0; g < ns; ++g)
      for (size_t t = 0; t < sl.rank[g].size(); ++t) {
        const uint64_t *h = hist.data() + hoff[g] + 256LL * tp[g][t];
        int64_t r = rem[g][t];
        int d = 0;
        while (d < 256 && r >= (int64_t)h[d]) r -= (int64_t)h[d++];
        if (d == 256) return set_err(ctx, MG_EFAIL, "quantiles: radix select lost rank %lld", (long long)sl.rank[g][t]);
        rem[g][t] = r;
        pre[g][t] = (pre[g][t] << 8) | (uint64_t)d;
      }
  }
  sl.out = pre;
  return MG_OK;
}

// Order statistics of ascending, distinct global ranks (N = the pooled size over the ranks, C_local this rank's
// chains) for every field: keys [F][K]; nan [F] = 1 where the field holds a NaN.
int qt_order_keys(mg_ctx *ctx, mg_comm *comm, const double *d_x, int64_t n, int32_t D, int64_t C, int64_t N,
                  const std::vector<int64_t> &ranks, std::vector<uint64_t> &keys, std::vector<int> &nan_f) {
  cudaStream_t st = ctx->stream;
  const int F = D + 2, K = (int)ranks.size();
  const int64_t Nl = n * C, rstride = (int64_t)F * C;
  const int64_t S = std::min<int64_t>(Nl, std::min<int64_t>(1 << 20, std::max<int64_t>(1 << 12, (1LL << 26) / F)));
  const bool exact = S == N;                        // the sample is the whole pool (one rank)
  // 1. sample and brackets
  std::vector<int64_t> ilo(K), ihi(K);
  for (int j = 0; j < K; ++j) {
    const int64_t k = ranks[j];
    const int64_t pos = N > 1 ? (int64_t)((unsigned __int128)k * (uint64_t)(S - 1) / (uint64_t)(N - 1)) : 0;
    if (exact) { ilo[j] = ihi[j] = pos; continue; }
    const double q = N > 1 ? (double)k / (double)(N - 1) : 0.5;
    const int64_t M = (int64_t)std::ceil(4.0 * std::sqrt((double)S * q * (1.0 - q))) + 16;
    ilo[j] = pos - M > 0 ? pos - M : -1;
    ihi[j] = pos + M < S - 1 ? pos + M : -1;
  }
  std::vector<uint64_t> br((size_t)F * K * 2);
  int rc = [&]() -> int {
    DevBuf<uint64_t> sk;
    DevBuf<int32_t> sv;
    DevBuf<int64_t> d_ilo, d_ihi;
    DevBuf<uint64_t> d_br;
    MG_CUDA(ctx, sk.alloc((size_t)F * S, st));
    MG_CUDA(ctx, sv.alloc((size_t)F * S, st));
    const int64_t ns = (int64_t)F * S;
    qt_sample_kernel<<<(unsigned)((ns + 255) / 256), 256, 0, st>>>(d_x, C, rstride, F, Nl, S, sk.get(), sv.get());
    MG_CHECK_LAUNCH(ctx);
    int r = radix_sort_pairs(ctx, sk.get(), sv.get(), S, F);
    if (r) return r;
    MG_CUDA(ctx, upload(d_ilo, ilo.data(), (size_t)K, st));
    MG_CUDA(ctx, upload(d_ihi, ihi.data(), (size_t)K, st));
    MG_CUDA(ctx, d_br.alloc(br.size(), st));
    qt_bracket_kernel<<<(unsigned)(((int64_t)F * K + 255) / 256), 256, 0, st>>>(sk.get(), S, F, K, d_ilo.get(),
                                                                                 d_ihi.get(), d_br.get());
    MG_CHECK_LAUNCH(ctx);
    MG_CUDA(ctx, cudaMemcpyAsync(br.data(), d_br.get(), sizeof(uint64_t) * br.size(), cudaMemcpyDeviceToHost, st));
    MG_CUDA(ctx, cudaStreamSynchronize(st));
    return MG_OK;
  }();
  if ((rc = qt_exchange(ctx, comm, rc, br, [](size_t i, uint64_t a, uint64_t b) {
         return (i & 1) ? std::max(a, b) : std::min(a, b);
       })))
    return rc;
  // merge each field's overlapping brackets; tb[f][j] = bracket of target j
  std::vector<int> nb(F, 0);
  std::vector<uint64_t> blo((size_t)F * QT_MAXT), bhi((size_t)F * QT_MAXT);
  std::vector<int> tb((size_t)F * K);
  bool any_open = false;                            // a bracket with lo != hi: candidates are kept
  for (int f = 0; f < F; ++f) {
    uint64_t *lo = blo.data() + (size_t)f * QT_MAXT, *hi = bhi.data() + (size_t)f * QT_MAXT;
    int m = 0;
    for (int j = 0; j < K; ++j) {
      const uint64_t l = br[((size_t)f * K + j) * 2], h = br[((size_t)f * K + j) * 2 + 1];
      if (m > 0 && l <= hi[m - 1]) { lo[m - 1] = std::min(lo[m - 1], l); hi[m - 1] = std::max(hi[m - 1], h); }
      else { lo[m] = l; hi[m] = h; ++m; }
      tb[(size_t)f * K + j] = m - 1;
    }
    nb[f] = m;
    for (int b = 0; b < m; ++b) any_open = any_open || lo[b] != hi[b];
  }
  // 2. one read of the block
  const int64_t budget = any_open ? std::min(Nl, std::max<int64_t>(Nl / 8, 1 << 16)) : 0;
  DevBuf<uint64_t> cand;
  std::vector<uint64_t> tally((size_t)F * QT_NREG + 2 * (size_t)F);   // counts, NaN flags, overflow flags
  std::vector<uint64_t> lcc(F, 0);                 // this rank's keys in the open brackets of each field
  rc = [&]() -> int {
    DevBuf<uint64_t> d_lo, d_hi;
    DevBuf<int> d_nb, d_nan;
    DevBuf<unsigned long long> d_cnt, d_ccnt;
    MG_CUDA(ctx, upload(d_lo, blo.data(), blo.size(), st));
    MG_CUDA(ctx, upload(d_hi, bhi.data(), bhi.size(), st));
    MG_CUDA(ctx, upload(d_nb, nb.data(), (size_t)F, st));
    MG_CUDA(ctx, d_cnt.alloc((size_t)F * QT_NREG, st));
    MG_CUDA(ctx, d_ccnt.alloc((size_t)F, st));
    MG_CUDA(ctx, d_nan.alloc((size_t)F, st));
    MG_CUDA(ctx, cand.alloc((size_t)F * budget, st));
    MG_CUDA(ctx, cudaMemsetAsync(d_cnt.get(), 0, sizeof(unsigned long long) * F * QT_NREG, st));
    MG_CUDA(ctx, cudaMemsetAsync(d_ccnt.get(), 0, sizeof(unsigned long long) * F, st));
    MG_CUDA(ctx, cudaMemsetAsync(d_nan.get(), 0, sizeof(int) * F, st));
    QtPassArgs a;
    const int64_t chunks = qt_chunks(ctx, F, Nl);
    a.x = d_x; a.C = C; a.rstride = rstride; a.len = Nl; a.per = (Nl + chunks - 1) / chunks; a.chunks = (int)chunks;
    a.lo = d_lo.get(); a.hi = d_hi.get(); a.nb = d_nb.get(); a.cnt = d_cnt.get(); a.ccnt = d_ccnt.get();
    a.cand = cand.get(); a.budget = budget; a.nan = d_nan.get();
    time_begin(ctx);
    qt_pass_kernel<<<(unsigned)(F * chunks), QT_THREADS, 0, st>>>(a);
    MG_CHECK_LAUNCH(ctx);
    time_end(ctx);
    std::vector<int> nn(F);
    MG_CUDA(ctx, cudaMemcpyAsync(tally.data(), d_cnt.get(), sizeof(uint64_t) * F * QT_NREG, cudaMemcpyDeviceToHost, st));
    MG_CUDA(ctx, cudaMemcpyAsync(lcc.data(), d_ccnt.get(), sizeof(uint64_t) * F, cudaMemcpyDeviceToHost, st));
    MG_CUDA(ctx, cudaMemcpyAsync(nn.data(), d_nan.get(), sizeof(int) * F, cudaMemcpyDeviceToHost, st));
    MG_CUDA(ctx, cudaStreamSynchronize(st));
    for (int f = 0; f < F; ++f) {
      tally[(size_t)F * QT_NREG + f] = nn[f] ? 1 : 0;
      tally[(size_t)F * QT_NREG + F + f] = lcc[f] > (uint64_t)budget ? 1 : 0;
    }
    return MG_OK;
  }();
  if ((rc = qt_exchange(ctx, comm, rc, tally, qt_sum))) return rc;
  // 3. resolve: bracket value, candidate rank, or fallback
  keys.assign((size_t)F * K, 0);
  nan_f.assign(F, 0);
  QtSlots cs, fs;                                   // candidate select, fallback select
  std::vector<std::vector<int>> cs_t, fs_t;         // their targets' indices j
  for (int f = 0; f < F; ++f) {
    if (tally[(size_t)F * QT_NREG + f]) { nan_f[f] = 1; continue; }
    const bool over = tally[(size_t)F * QT_NREG + F + f] != 0;
    const uint64_t *cnt = tally.data() + (size_t)f * QT_NREG;
    std::vector<int64_t> below(nb[f]), before(nb[f]);   // keys below bracket b; candidates of the brackets before b
    int64_t acc = 0, cacc = 0;
    for (int b = 0; b < nb[f]; ++b) {
      acc += (int64_t)cnt[2 * b];
      below[b] = acc;
      before[b] = cacc;
      acc += (int64_t)cnt[2 * b + 1];
      if (blo[(size_t)f * QT_MAXT + b] != bhi[(size_t)f * QT_MAXT + b]) cacc += (int64_t)cnt[2 * b + 1];
    }
    std::vector<int64_t> cr, fr;
    std::vector<int> cj, fj;
    for (int j = 0; j < K; ++j) {
      const int b = tb[(size_t)f * K + j];
      const int64_t k = ranks[j], in = (int64_t)cnt[2 * b + 1];
      const bool hit = k >= below[b] && k < below[b] + in;
      if (hit && blo[(size_t)f * QT_MAXT + b] == bhi[(size_t)f * QT_MAXT + b]) keys[(size_t)f * K + j] = blo[(size_t)f * QT_MAXT + b];
      else if (hit && !over) { cr.push_back(k - below[b] + before[b]); cj.push_back(j); }
      else { fr.push_back(k); fj.push_back(j); }
    }
    if (!cr.empty()) { cs.fld.push_back(f); cs.rank.push_back(cr); cs_t.push_back(cj); }
    if (!fr.empty()) { fs.fld.push_back(f); fs.rank.push_back(fr); fs_t.push_back(fj); }
  }
  // 4. radix select over the candidate buffers, then over the block for what missed
  if (!cs.fld.empty()) {
    for (int f : cs.fld) cs.len.push_back((int64_t)lcc[f]);
    if ((rc = qt_select(ctx, comm, true, cand.get(), budget, 0, cs))) return rc;
    for (size_t g = 0; g < cs.fld.size(); ++g)
      for (size_t t = 0; t < cs_t[g].size(); ++t) keys[(size_t)cs.fld[g] * K + cs_t[g][t]] = cs.out[g][t];
  }
  cand.release();
  if (!fs.fld.empty()) {
    fs.len.assign(fs.fld.size(), Nl);
    if ((rc = qt_select(ctx, comm, false, d_x, C, rstride, fs))) return rc;
    for (size_t g = 0; g < fs.fld.size(); ++g)
      for (size_t t = 0; t < fs_t[g].size(); ++t) keys[(size_t)fs.fld[g] * K + fs_t[g][t]] = fs.out[g][t];
  }
  if (getenv("MCMC_GPU_DEBUG")) {
    size_t g = 0;
    for (int f = 0; f < F; ++f) {
      const bool fb = g < fs.fld.size() && fs.fld[g] == f;
      if (fb) ++g;
      fprintf(stderr, "quantiles: field %d: %s, %d full read%s\n", f, nan_f[f] ? "nan" : fb ? "fallback" : "bracket",
              fb ? 9 : 1, fb ? "s" : "");
    }
  }
  return MG_OK;
}

}  // namespace mg

using namespace mg;

namespace mg {

int qt_check(mg_ctx *ctx, const void *x, int64_t n, int32_t D, int64_t C, const void *list, int32_t nq,
             const double *out) {
  MG_REQUIRE(ctx, x && list && out, "quantiles: null argument");
  MG_REQUIRE(ctx, n >= 1 && C >= 1 && D >= 1 && D <= INT32_MAX - 2, "quantiles: bad block shape");
  MG_REQUIRE(ctx, nq >= 1 && nq <= MG_QUANT_MAX, "quantiles: need 1 <= nq <= %d", MG_QUANT_MAX);
  MG_REQUIRE(ctx, n <= INT64_MAX / C && (int64_t)D + 2 <= INT64_MAX / (n * C), "quantiles: block too large");
  return MG_OK;
}

// the ranks probs need (ascending, distinct); N = the pooled size
int qt_prob_ranks(mg_ctx *ctx, const double *probs, int32_t nq, int64_t N, std::vector<int64_t> &ranks) {
  ranks.clear();
  for (int i = 0; i < nq; ++i) {
    const double p = probs[i];
    MG_REQUIRE(ctx, p >= 0.0 && p <= 1.0, "quantiles: p = %g is outside [0, 1]", p);
    const double h = (double)(N - 1) * p;
    const int64_t lo = (int64_t)std::floor(h);
    ranks.push_back(lo);
    if (h - (double)lo != 0.0) ranks.push_back(std::min(lo + 1, N - 1));
  }
  std::sort(ranks.begin(), ranks.end());
  ranks.erase(std::unique(ranks.begin(), ranks.end()), ranks.end());
  return MG_OK;
}

// the quantile rule of include/mcmc_gpu.h, one rounding; volatile keeps the host compiler from fusing it
static double qt_interp(double a, double b, double g) {
  if (g == 0.0 || a == b) return a;
  if (a == -INFINITY) return b == INFINITY ? NAN : -INFINITY;
  if (b == INFINITY) return INFINITY;
  volatile double t = g * (b - a);
  return a + t;
}

// keys [F][K] of ranks -> out [F][nq]
void qt_finish_quantiles(const double *probs, int32_t nq, int64_t N, int F, const std::vector<int64_t> &ranks,
                         const std::vector<uint64_t> &keys, const std::vector<int> &nan_f, double *out) {
  const int K = (int)ranks.size();
  auto x = [&](int f, int64_t k) {
    const int j = (int)(std::lower_bound(ranks.begin(), ranks.end(), k) - ranks.begin());
    return ordered_to_f64(keys[(size_t)f * K + j]);
  };
  for (int f = 0; f < F; ++f)
    for (int i = 0; i < nq; ++i) {
      if (nan_f[f]) { out[(size_t)f * nq + i] = NAN; continue; }
      const double h = (double)(N - 1) * probs[i];
      const int64_t lo = (int64_t)std::floor(h);
      const double g = h - (double)lo;
      const double a = x(f, lo);
      out[(size_t)f * nq + i] = g == 0.0 ? a : qt_interp(a, x(f, std::min(lo + 1, N - 1)), g);
    }
}

}  // namespace mg

extern "C" int mg_stats_quantiles_dev(mg_ctx *ctx, const double *d_samples, int64_t n, int32_t D, int64_t C,
                                      const double *probs, int32_t nq, double *out) {
  if (!ctx) return MG_EINVAL;
  int rc = qt_check(ctx, d_samples, n, D, C, probs, nq, out);
  if (rc) return rc;
  const int64_t N = n * C;
  std::vector<int64_t> ranks;
  if ((rc = qt_prob_ranks(ctx, probs, nq, N, ranks))) return rc;
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  std::vector<uint64_t> keys;
  std::vector<int> nan_f;
  if ((rc = qt_order_keys(ctx, nullptr, d_samples, n, D, C, N, ranks, keys, nan_f))) return rc;
  qt_finish_quantiles(probs, nq, N, D + 2, ranks, keys, nan_f, out);
  return MG_OK;
}

extern "C" int mg_stats_quantiles(mg_ctx *ctx, const double *samples, int64_t n, int32_t D, int64_t C,
                                  const double *probs, int32_t nq, double *out) {
  if (!ctx) return MG_EINVAL;
  int rc = qt_check(ctx, samples, n, D, C, probs, nq, out);
  if (rc) return rc;
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  DevBuf<double> d_x;
  MG_CUDA(ctx, upload(d_x, samples, (size_t)(n * (D + 2) * C), ctx->stream));
  return mg_stats_quantiles_dev(ctx, d_x.get(), n, D, C, probs, nq, out);
}

extern "C" int mg_stats_order_statistics_dev(mg_ctx *ctx, const double *d_samples, int64_t n, int32_t D, int64_t C,
                                             const int64_t *ranks, int32_t nk, double *out) {
  if (!ctx) return MG_EINVAL;
  int rc = qt_check(ctx, d_samples, n, D, C, ranks, nk, out);
  if (rc) return rc;
  const int64_t N = n * C;
  std::vector<int64_t> rk(ranks, ranks + nk);
  for (int64_t k : rk) MG_REQUIRE(ctx, k >= 0 && k < N, "order_statistics: rank %lld is outside [0, %lld)", (long long)k, (long long)N);
  std::sort(rk.begin(), rk.end());
  rk.erase(std::unique(rk.begin(), rk.end()), rk.end());
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  std::vector<uint64_t> keys;
  std::vector<int> nan_f;
  if ((rc = qt_order_keys(ctx, nullptr, d_samples, n, D, C, N, rk, keys, nan_f))) return rc;
  const int F = D + 2, K = (int)rk.size();
  for (int f = 0; f < F; ++f)
    for (int i = 0; i < nk; ++i) {
      const int j = (int)(std::lower_bound(rk.begin(), rk.end(), ranks[i]) - rk.begin());
      out[(size_t)f * nk + i] = nan_f[f] ? NAN : ordered_to_f64(keys[(size_t)f * K + j]);
    }
  return MG_OK;
}
