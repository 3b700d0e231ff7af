// evidence.cu -- Evidence.evidence_harmonic_mean / evidence_lebesgue /
// evidence_direct (evidence.ml:101-107, 202-221, 148-165) on the GPU.
//
// Pipeline (device resident; every stage HBM-bound):
//   harmonic  one pass over ll (8 B/sample), compensated block reduction.
//   lebesgue  stable radix sort of -ll (evidence.ml:180) -> first gap in 1/L
//             above eps (parallel min, :167-179) -> mean 1/L of the prefix
//             (:182-189) -> drop equal-ll runs keeping the last, reversed
//             (:191-200; flag + scan + gather) -> kd-tree of the survivors,
//             not split below n objects (collect_subvolumes never looks
//             further, :83-89) -> one warp per cell: tight bounds, volume in
//             the reference's product order, median log-prior (:109-120) ->
//             compensated sum over cells / mean 1/L.
//   direct    D stable radix sorts (last coordinate first) = List.sort by
//             coordinates (:143-146) -> drop equal rows keeping the last,
//             reversed (:126-141) -> tree -> per cell volume * mean
//             posterior, summed by lane 0 in the reference's list order
//             (:122-124,150-160).
// Per-cell terms are bit-exact up to exp(); the sum over cells is compensated,
// i.e. closer to the exact sum than the reference's left-to-right fold.
#include "comm.cuh"
#include "kdtree.cuh"
#include "radix_sort.cuh"
#include "reduce.cuh"
#include "reduce_sum.cuh"
#include "scan.cuh"

namespace mg {

__global__ void neg_ll_keys_kernel(const double *__restrict__ ll, int64_t n, uint64_t *__restrict__ keys,
                                   int32_t *__restrict__ vals) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    keys[i] = f64_to_ordered(-ll[i]);  // compare_inverse_like, evidence.ml:99
    vals[i] = (int32_t)i;
  }
}

__global__ void coord_keys_kernel(const double *__restrict__ pts, const int32_t *__restrict__ order, int64_t n, int D,
                                  int d, uint64_t *__restrict__ keys) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    keys[i] = f64_to_ordered(pts[(int64_t)order[i] * D + d]);
}

__global__ void iota_kernel(int32_t *__restrict__ v, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) v[i] = (int32_t)i;
}

// first i with exp(-ll[o[i+1]]) - exp(-ll[o[i]]) > eps (evidence.ml:170-177); also flags delta < 0 / NaN
__global__ void first_gap_kernel(const double *__restrict__ ll, const int32_t *__restrict__ order, int64_t n,
                                 double eps, unsigned long long *__restrict__ first, int *__restrict__ bad) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i + 1 < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double ilx = exp(-ll[order[i]]), ily = exp(-ll[order[i + 1]]);
    const double delta = ily - ilx;
    if (!(delta >= 0.0)) *bad = 1;   // assert(delta >= 0.0), :175
    if (delta > eps) atomicMin(first, (unsigned long long)i);
  }
}

// remove_dups_rev (evidence.ml:191-200): keep i iff it is the last of its equal-ll run
__global__ void keep_ll_kernel(const double *__restrict__ ll, const int32_t *__restrict__ order, int64_t m,
                               int32_t *__restrict__ keep) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x)
    keep[i] = (i == m - 1 || !(ll[order[i]] == ll[order[i + 1]])) ? 1 : 0;
}

// rev_remove_dups compare_samples (evidence.ml:126-141): keep the last of each run of equal rows
__global__ void keep_rows_kernel(const double *__restrict__ pts, const int32_t *__restrict__ order, int64_t m, int D,
                                 int32_t *__restrict__ keep) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    int k = 1;
    if (i < m - 1) {
      const double *a = pts + (int64_t)order[i] * D, *b = pts + (int64_t)order[i + 1] * D;
      bool eq = true;
      for (int d = 0; d < D && eq; ++d) eq = (a[d] == b[d]);   // compare = 0 on non-NaN floats (-0.0 = 0.0)
      k = eq ? 0 : 1;
    }
    keep[i] = k;
  }
}

// after a stable sort on coordinate 0 only: is the order already lexicographic?  It is unless two
// neighbours share coordinate 0 and are out of order in a later coordinate.
__global__ void lex_order_check_kernel(const double *__restrict__ pts, const int32_t *__restrict__ order, int64_t n,
                                       int D, int *__restrict__ bad) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i + 1 < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double *a = pts + (int64_t)order[i] * D, *b = pts + (int64_t)order[i + 1] * D;
    if (a[0] == b[0]) {
      for (int d = 1; d < D; ++d) {
        if (a[d] < b[d]) break;
        if (a[d] > b[d]) { *bad = 1; break; }
      }
      // equal rows keep their input order (the sort is stable), as List.sort does
    }
  }
}

// survivors in REVERSED order: dst = K-1-rank.  One warp per 32 candidate rows: the row ids are read coalesced and
// broadcast, each row is then copied by consecutive lanes (a row is D contiguous doubles on both sides).
__global__ void gather_kernel(const double *__restrict__ pts, const double *__restrict__ ll,
                              const double *__restrict__ lp, const int32_t *__restrict__ order,
                              const int32_t *__restrict__ keep, const int32_t *__restrict__ rank, int64_t m, int64_t K,
                              int D, double *__restrict__ spts, double *__restrict__ sll, double *__restrict__ slp) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i0 = warp * 32; i0 < m; i0 += nwarps * 32) {
    const int64_t i = i0 + lane;
    const bool k = (i < m) && keep[i] != 0;
    const int64_t dst = k ? K - 1 - rank[i] : 0, src = k ? order[i] : 0;
    if (k) { sll[dst] = ll[src]; slp[dst] = lp[src]; }
    const unsigned mask = __ballot_sync(0xffffffffu, k);
    for (unsigned rem = mask; rem; rem &= rem - 1) {
      const int r = __ffs(rem) - 1;
      const int64_t rs = __shfl_sync(0xffffffffu, src, r), rd = __shfl_sync(0xffffffffu, dst, r);
      for (int d = lane; d < D; d += 32) spts[rd * D + d] = pts[rs * D + d];
    }
  }
}

// One warp per node of a tree that was not split below nmax objects.
// collect_subvolumes (evidence.ml:83-89) emits exactly the leaves with < nmax
// objects; a leaf of >= nmax identical points contributes nothing.
// MODE 0: exp(median log_prior) * tight volume   (evidence_lebesgue :209-220)
// MODE 1: tight volume * mean exp(ll + lp)       (evidence_direct_tree :150-160)
template <int MODE>
__global__ void __launch_bounds__(EB)
cell_terms_kernel(const KdNode *__restrict__ nodes, const int32_t *__restrict__ count, const int32_t *__restrict__ begin,
                  const int32_t *__restrict__ perm, const double *__restrict__ pts, const double *__restrict__ ll,
                  const double *__restrict__ lp, int64_t node0, int64_t node1, int D, int nmax, double *__restrict__ terms,
                  unsigned long long *__restrict__ ncells) {
  extern __shared__ double sh[];  // [warps][nmax] scratch values
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = EB / 32;
  double *vals = sh + (size_t)w * nmax;
  unsigned cells = 0;
  // terms[id] for the nodes [node0, node1) (a rank's share of the tree): the cell's term, 0.0 for a node that is
  // not one of collect_subvolumes' cells.  The terms are summed afterwards in node order by ONE deterministic
  // reduction over the whole array, so the result does not depend on how the nodes were spread over ranks.
  for (int64_t id = node0 + (int64_t)blockIdx.x * nw + w; id < node1; id += (int64_t)gridDim.x * nw) {
    const int cnt = count[id];
    if (nodes[id].left >= 0 || cnt >= nmax) { if (lane == 0) terms[id] = 0.0; continue; }   // not (length_at_least nmax objs) -> [c]
    const int b = begin[id];
    // bounds_of_objects (kd_tree.ml:96-110) + bounds_volume (:177-182, product in dimension order)
    // Lane d owns dimension d (d + 32, ... beyond 32): every point is one coalesced row read, no reduction across
    // lanes; the extents are then multiplied in dimension order.
    double v = 1.0;
    for (int d0 = 0; d0 < D; d0 += 32) {
      const int d = d0 + lane;
      double lo = __longlong_as_double(0x7FF0000000000000ll), hi = -lo;
      for (int k = 0; k < cnt; ++k) {
        const int64_t row = (int64_t)__ldg(perm + b + k) * D;
        if (d < D) { const double c = pts[row + d]; lo = fmin(lo, c); hi = fmax(hi, c); }
      }
      const double ext = hi - lo;
      const int nd = (D - d0 < 32) ? D - d0 : 32;
      for (int i = 0; i < nd; ++i) v = v * __shfl_sync(0xffffffffu, ext, i);
    }
    v = v + 0.0;
    for (int k = lane; k < cnt; k += 32) {
      const int32_t p = perm[b + k];
      vals[k] = (MODE == 0) ? lp[p] : exp(ll[p] + lp[p]);   // posterior, evidence.ml:95-97
    }
    __syncwarp();
    double term = 0.0;
    if (MODE == 0) {
      // median_sample (:109-120): rank every value (ties by position = stable sort)
      double lo_mid = 0.0, hi_mid = 0.0;
      const int r_hi = cnt / 2, r_lo = cnt / 2 - 1;
      for (int k = lane; k < cnt; k += 32) {
        const double x = vals[k];
        int r = 0;
        for (int j = 0; j < cnt; ++j) { const double y = vals[j]; r += (y < x || (y == x && j < k)) ? 1 : 0; }
        if (r == r_hi) hi_mid = x;
        if (r == r_lo) lo_mid = x;
      }
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {   // exactly one lane holds each (others hold 0.0): OR the bits
        hi_mid = __longlong_as_double(__double_as_longlong(hi_mid) | __shfl_xor_sync(0xffffffffu, __double_as_longlong(hi_mid), off));
        lo_mid = __longlong_as_double(__double_as_longlong(lo_mid) | __shfl_xor_sync(0xffffffffu, __double_as_longlong(lo_mid), off));
      }
      const double med = (cnt % 2 == 0) ? 0.5 * (lo_mid + hi_mid) : hi_mid;
      const double prior = exp(med);
      term = prior * v;
    } else {
      // mean_sample posterior (:122-124): left-to-right fold in list order, by lane 0
      double sum = 0.0;
      if (lane == 0) for (int k = 0; k < cnt; ++k) sum = sum + vals[k];
      sum = __shfl_sync(0xffffffffu, sum, 0);
      const double post = sum / (double)cnt;
      term = v * post;
    }
    __syncwarp();
    if (lane == 0) { terms[id] = term; ++cells; }
  }
  if (lane == 0 && cells) atomicAdd(ncells, (unsigned long long)cells);
}

struct Survivors {
  DevBuf<double> pts, ll, lp;
  int64_t K = 0;
};

// flag -> scan -> gather (reversed) of the first m entries of `order`
static int compact_reversed(mg_ctx *ctx, const double *d_pts, const double *d_ll, const double *d_lp,
                            const int32_t *d_order, const int32_t *d_keep, int64_t m, int D, Survivors &sv) {
  cudaStream_t s = ctx->stream;
  DevBuf<int32_t> rank, tmp, total;
  MG_CUDA(ctx, rank.alloc(m, s));
  MG_CUDA(ctx, tmp.alloc((size_t)scan_tmp_elems(m, 1) + 1, s));
  MG_CUDA(ctx, total.alloc(1, s));
  int rc = exclusive_scan_i32(ctx, d_keep, rank.get(), m, 1, tmp.get(), total.get());
  if (rc) return rc;
  int32_t K = 0;
  MG_CUDA(ctx, cudaMemcpyAsync(&K, total.get(), 4, cudaMemcpyDeviceToHost, s));
  MG_CUDA(ctx, cudaStreamSynchronize(s));
  sv.K = K;
  MG_CUDA(ctx, sv.pts.alloc((size_t)K * D, s));
  MG_CUDA(ctx, sv.ll.alloc(K, s));
  MG_CUDA(ctx, sv.lp.alloc(K, s));
  gather_kernel<<<egrid(ctx, m), EB, 0, s>>>(d_pts, d_ll, d_lp, d_order, d_keep, rank.get(), m, K, D, sv.pts.get(),
                                            sv.ll.get(), sv.lp.get());
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

// per-cell terms of the nodes [node0, node1) of a tree that was not split below nmax objects
template <int MODE>
int cell_terms_range(mg_ctx *ctx, const mg_kdtree *t, const double *spts, const double *sll, const double *slp, int nmax, int64_t node0,
                     int64_t node1, double *d_terms, unsigned long long *d_ncells) {
  if (node1 <= node0) return MG_OK;
  cudaStream_t s = ctx->stream;
  const char *blob = (const char *)t->d_blob;
  const unsigned g = egrid(ctx, node1 - node0, EB / 32);
  const size_t smem = (size_t)(EB / 32) * (nmax > 0 ? nmax : 1) * sizeof(double);
  if (smem > 48 * 1024) MG_CUDA(ctx, cudaFuncSetAttribute(cell_terms_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cell_terms_kernel<MODE><<<g, EB, smem, s>>>((const KdNode *)(blob + t->h.off_nodes), (const int32_t *)(blob + t->h.off_count),
                                              (const int32_t *)(blob + t->h.off_begin), (const int32_t *)(blob + t->h.off_perm),
                                              spts, sll, slp, node0, node1, t->h.D, nmax, d_terms, d_ncells);
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}
template int cell_terms_range<0>(mg_ctx *, const mg_kdtree *, const double *, const double *, const double *, int, int64_t, int64_t, double *, unsigned long long *);
template int cell_terms_range<1>(mg_ctx *, const mg_kdtree *, const double *, const double *, const double *, int, int64_t, int64_t, double *, unsigned long long *);

// the sum of the terms of all nodes, in node order: one deterministic compensated reduction (fixed grid for a given
// node count), the same on every rank and for every way the terms were produced
int sum_terms(mg_ctx *ctx, const double *d_terms, int64_t nn, double *out) {
  return reduce_sum(ctx, nn, [d_terms] __device__(int64_t i) { return d_terms[i]; }, out);
}

// tree of the survivors and the sum of the per-cell terms
template <int MODE>
static int integrate_cells(mg_ctx *ctx, const Survivors &sv, int D, int nmax, double *out, int64_t *ncells_out) {
  cudaStream_t s = ctx->stream;
  // The root box (bounds_of_objects, evidence.ml:164,206) does not influence
  // any split nor the tight per-cell volumes, so it is not computed.
  // The tree is not split below nmax objects, and it is scaffolding: the cell terms read the survivors' own rows, so
  // its blob carries no copy of them.
  std::vector<double> zeros(D, 0.0);
  KdTreePtr t;
  int rc = build_tree(ctx, sv.pts.get(), sv.K, D, zeros.data(), zeros.data(), nmax < 2 ? 2 : nmax, false, &t);
  if (rc) return rc;
  const int64_t nn = t->h.nnodes;
  DevBuf<double> terms;
  DevBuf<unsigned long long> ncells;
  cudaError_t e = terms.alloc((size_t)nn, s);
  if (e == cudaSuccess) e = ncells.alloc(1, s);
  if (e == cudaSuccess) e = cudaMemsetAsync(ncells.get(), 0, 8, s);
  if (e != cudaSuccess) return set_err(ctx, MG_ECUDA, "cuda: %s", cudaGetErrorString(e));
  rc = cell_terms_range<MODE>(ctx, t.get(), sv.pts.get(), sv.ll.get(), sv.lp.get(), nmax, 0, nn, terms.get(), ncells.get());
  if (rc == MG_OK) rc = sum_terms(ctx, terms.get(), nn, out);
  unsigned long long nc = 0;
  if (rc == MG_OK && ncells_out) {
    e = cudaMemcpyAsync(&nc, ncells.get(), 8, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) rc = set_err(ctx, MG_ECUDA, "cuda: %s (evidence cells)", cudaGetErrorString(e));
    *ncells_out = (int64_t)nc;
  }
  return rc;
}

}  // namespace mg

using namespace mg;

extern "C" int mg_evidence_harmonic_mean_dev(mg_ctx *ctx, const double *d_ll, int64_t N, double *out) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, d_ll && out && N >= 1, "evidence_harmonic_mean: bad arguments");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  double linv = 0.0;
  time_begin(ctx);
  int rc = reduce_sum(ctx, N, [d_ll] __device__(int64_t i) { return 1.0 / exp(d_ll[i]); }, &linv);  // evidence.ml:105
  time_end(ctx);
  if (rc) return rc;
  *out = (double)N / linv;
  return MG_OK;
}

extern "C" int mg_evidence_harmonic_mean(mg_ctx *ctx, const double *ll, int64_t N, double *out) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, ll && out && N >= 1, "evidence_harmonic_mean: bad arguments");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  DevBuf<double> d_ll;
  MG_CUDA(ctx, upload(d_ll, ll, (size_t)N, ctx->stream));
  return mg_evidence_harmonic_mean_dev(ctx, d_ll.get(), N, out);
}

// The same over samples SHARDED across ranks: every rank reduces the 1/L of its own shard (compensated), the
// (count, sum) pairs are all-gathered and folded in rank order.  Agrees with the single-GPU value to the rounding of
// the compensated sums (<= 2 ulp); identical on every rank.
extern "C" int mg_evidence_harmonic_mean_sharded(mg_comm *c, const double *d_ll_shard, int64_t n_shard, double *out) {
  if (!c) return MG_EINVAL;
  mg_ctx *ctx = mg_comm_ctx(c);
  int rc = MG_OK;
  if (!(out && n_shard >= 0 && (d_ll_shard || n_shard == 0)))
    rc = set_err(ctx, MG_EINVAL, "evidence_harmonic_mean (sharded): bad arguments");
  if (rc == MG_OK && cudaSetDevice(ctx->device) != cudaSuccess) rc = set_err(ctx, MG_ECUDA, "cuda: cannot select the device");
  std::vector<double> mine = {(double)n_shard, 0.0}, all;
  if (rc == MG_OK && n_shard > 0)
    rc = reduce_sum(ctx, n_shard, [d_ll_shard] __device__(int64_t i) { return 1.0 / exp(d_ll_shard[i]); }, &mine[1]);
  if ((rc = comm_gather(c, rc, mine, all, "evidence_harmonic_mean (sharded)"))) return rc;
  Comp linv; double n = 0.0;
  for (int r = 0; r < mg_comm_size(c); ++r) { n += all[2 * r]; linv.add(all[2 * r + 1]); }
  MG_REQUIRE(ctx, n >= 1.0, "evidence_harmonic_mean (sharded): no samples on any rank");
  *out = n / linv.value();
  return MG_OK;
}

// evidence.ml:202-205: the kept prefix, its mean 1/L, and the survivors of remove_dups_rev (reversed)
static int lebesgue_prepare(mg_ctx *ctx, const double *d_pts, const double *d_ll, const double *d_lp, int64_t N, int32_t D,
                            int32_t n, double eps, Survivors &sv, double *mean_il_out) {
  MG_REQUIRE(ctx, d_pts && d_ll && d_lp, "evidence_lebesgue: null argument");
  MG_REQUIRE(ctx, N >= 1, "bounds_of_objects: no objects");
  MG_REQUIRE(ctx, D >= 1 && D <= 64 && n >= 1 && N < (1LL << 30), "evidence_lebesgue: bad sizes");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  // collect_samples_up_to_eps (:167-180)
  DevBuf<uint64_t> keys;
  DevBuf<int32_t> order, keep;
  MG_CUDA(ctx, keys.alloc(N, s));
  MG_CUDA(ctx, order.alloc(N, s));
  neg_ll_keys_kernel<<<egrid(ctx, N), EB, 0, s>>>(d_ll, N, keys.get(), order.get());
  MG_CHECK_LAUNCH(ctx);
  int rc = radix_sort_pairs(ctx, keys.get(), order.get(), N, 1);
  if (rc) return rc;
  keys.release();
  DevBuf<unsigned long long> first;
  DevBuf<int> bad;
  MG_CUDA(ctx, first.alloc(1, s));
  MG_CUDA(ctx, bad.alloc(1, s));
  const unsigned long long none = ~0ull;
  MG_CUDA(ctx, cudaMemcpyAsync(first.get(), &none, 8, cudaMemcpyHostToDevice, s));
  MG_CUDA(ctx, cudaMemsetAsync(bad.get(), 0, sizeof(int), s));
  first_gap_kernel<<<egrid(ctx, N), EB, 0, s>>>(d_ll, order.get(), N, eps, first.get(), bad.get());
  MG_CHECK_LAUNCH(ctx);
  unsigned long long h_first = 0;
  int h_bad = 0;
  MG_CUDA(ctx, cudaMemcpyAsync(&h_first, first.get(), 8, cudaMemcpyDeviceToHost, s));
  MG_CUDA(ctx, cudaMemcpyAsync(&h_bad, bad.get(), sizeof(int), cudaMemcpyDeviceToHost, s));
  MG_CUDA(ctx, cudaStreamSynchronize(s));
  const int64_t m = (h_first == none) ? N : (int64_t)h_first + 1;
  // the assertion only covers pairs up to the cut in the reference (it stops there)
  if (h_bad) {
    // re-check restricted to the kept prefix: delta >= 0 must hold for i < m
    // (NaN log-likelihoods sort last under the ordered-key transform)
    double chk = 0.0;
    const int32_t *o = order.get();
    rc = reduce_sum(ctx, m > 1 ? m - 1 : 0, [d_ll, o] __device__(int64_t i) {
      const double d = exp(-d_ll[o[i + 1]]) - exp(-d_ll[o[i]]);
      return (d >= 0.0) ? 0.0 : 1.0; }, &chk);
    if (rc) return rc;
    if (chk != 0.0) return set_err(ctx, MG_EFAIL, "Assert_failure evidence.ml:175");
  }
  // mean_inv_like (:182-189)
  double tot_il = 0.0;
  {
    const int32_t *o = order.get();
    rc = reduce_sum(ctx, m, [d_ll, o] __device__(int64_t i) { return exp(-d_ll[o[i]]); }, &tot_il);
    if (rc) return rc;
  }
  const double mean_il = tot_il / (double)m;
  // remove_dups_rev (:191-200)
  MG_CUDA(ctx, keep.alloc(m, s));
  keep_ll_kernel<<<egrid(ctx, m), EB, 0, s>>>(d_ll, order.get(), m, keep.get());
  MG_CHECK_LAUNCH(ctx);
  if ((rc = compact_reversed(ctx, d_pts, d_ll, d_lp, order.get(), keep.get(), m, D, sv))) return rc;
  *mean_il_out = mean_il;
  return MG_OK;
}

extern "C" int mg_evidence_lebesgue_dev(mg_ctx *ctx, const double *d_pts, const double *d_ll, const double *d_lp,
                                        int64_t N, int32_t D, int32_t n, double eps, double *out) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, out != nullptr, "evidence_lebesgue: null argument");
  Survivors sv;
  double mean_il = 0.0, pm = 0.0;
  int rc = lebesgue_prepare(ctx, d_pts, d_ll, d_lp, N, D, n, eps, sv, &mean_il);
  if (rc) return rc;
  if ((rc = integrate_cells<0>(ctx, sv, D, n, &pm, nullptr))) return rc;
  *out = pm / mean_il;  // :221
  return MG_OK;
}

// evidence.ml:143-146,162-163: the samples sorted by coordinates with duplicates dropped (reversed)
static int direct_prepare(mg_ctx *ctx, const double *d_pts, const double *d_ll, const double *d_lp, int64_t N, int32_t D,
                          int32_t n, Survivors &sv) {
  MG_REQUIRE(ctx, d_pts && d_ll && d_lp, "evidence_direct: null argument");
  MG_REQUIRE(ctx, N >= 1, "bounds_of_objects: no objects");
  MG_REQUIRE(ctx, D >= 1 && D <= 64 && n >= 1 && N < (1LL << 30), "evidence_direct: bad sizes");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  // array_to_list_remove_dups (:143-146): List.sort compare_samples = LSD radix over the coordinates
  DevBuf<uint64_t> keys;
  DevBuf<int32_t> order, keep;
  MG_CUDA(ctx, keys.alloc(N, s));
  MG_CUDA(ctx, order.alloc(N, s));
  iota_kernel<<<egrid(ctx, N), EB, 0, s>>>(order.get(), N);
  MG_CHECK_LAUNCH(ctx);
  int rc;
  // Fast path: sort on coordinate 0 alone.  Ties in coordinate 0 are almost always whole repeated rows
  // (Metropolis-Hastings rejections), for which the stable order already is the lexicographic one.
  bool need_full = (D > 1);
  if (D > 1) {
    coord_keys_kernel<<<egrid(ctx, N), EB, 0, s>>>(d_pts, order.get(), N, D, 0, keys.get());
    MG_CHECK_LAUNCH(ctx);
    if ((rc = radix_sort_pairs(ctx, keys.get(), order.get(), N, 1))) return rc;
    DevBuf<int> d_bad;
    MG_CUDA(ctx, d_bad.alloc(1, s));
    MG_CUDA(ctx, cudaMemsetAsync(d_bad.get(), 0, sizeof(int), s));
    lex_order_check_kernel<<<egrid(ctx, N), EB, 0, s>>>(d_pts, order.get(), N, D, d_bad.get());
    MG_CHECK_LAUNCH(ctx);
    int h_bad = 0;
    MG_CUDA(ctx, cudaMemcpyAsync(&h_bad, d_bad.get(), sizeof(int), cudaMemcpyDeviceToHost, s));
    MG_CUDA(ctx, cudaStreamSynchronize(s));
    need_full = (h_bad != 0);
    if (need_full) { iota_kernel<<<egrid(ctx, N), EB, 0, s>>>(order.get(), N); MG_CHECK_LAUNCH(ctx); }
  }
  if (need_full || D == 1)
    for (int d = D - 1; d >= 0; --d) {   // full LSD pass over the coordinates, last first
      coord_keys_kernel<<<egrid(ctx, N), EB, 0, s>>>(d_pts, order.get(), N, D, d, keys.get());
      MG_CHECK_LAUNCH(ctx);
      if ((rc = radix_sort_pairs(ctx, keys.get(), order.get(), N, 1))) return rc;
    }
  keys.release();
  MG_CUDA(ctx, keep.alloc(N, s));
  keep_rows_kernel<<<egrid(ctx, N), EB, 0, s>>>(d_pts, order.get(), N, D, keep.get());
  MG_CHECK_LAUNCH(ctx);
  return compact_reversed(ctx, d_pts, d_ll, d_lp, order.get(), keep.get(), N, D, sv);
}

extern "C" int mg_evidence_direct_dev(mg_ctx *ctx, const double *d_pts, const double *d_ll, const double *d_lp,
                                      int64_t N, int32_t D, int32_t n, double *out) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, out != nullptr, "evidence_direct: null argument");
  Survivors sv;
  int rc = direct_prepare(ctx, d_pts, d_ll, d_lp, N, D, n, sv);
  if (rc) return rc;
  return integrate_cells<1>(ctx, sv, D, n, out, nullptr);
}

// ---- the same over the GPUs of one box (SURVEY.md 8e; evidence.ml:148-221) -----------------------------------------
// The global steps (sort, prefix cut, de-duplication) run on `root`, which holds the samples; the survivors' rows and
// ll / lp are replicated with NCCL broadcasts; the tree over them is built by all ranks together
// (mg_kdtree_build_distributed, bit-identical to the single-GPU tree); the tree's nodes are cut into
// contiguous ranges, one per rank, each rank evaluates the cell terms of its range; the per-node terms are
// all-gathered (ncclAllGather, in place) and every rank runs the SAME deterministic reduction over the complete
// array -- the result is bit-identical on every rank and to the single-GPU call.
static int evidence_sharded(mg_comm *c, int which, int32_t root, const double *d_pts, const double *d_ll, const double *d_lp,
                            int64_t N, int32_t D, int32_t n, double eps, double *out) {
  if (!c) return MG_EINVAL;
  mg_ctx *ctx = mg_comm_ctx(c);
  const int R = mg_comm_size(c), rank = mg_comm_rank(c);
  int rc = MG_OK;
  if (!(out && root >= 0 && root < R && n >= 1)) rc = set_err(ctx, MG_EINVAL, "evidence (sharded): bad arguments");
  if (rc == MG_OK && cudaSetDevice(ctx->device) != cudaSuccess) rc = set_err(ctx, MG_ECUDA, "cuda: cannot select the device");
  cudaStream_t s = ctx->stream;
  Survivors sv;
  double mean_il = 1.0;                 // mean 1/L of the kept prefix (Lebesgue)
  if (rc == MG_OK && rank == root)
    rc = which == 0 ? lebesgue_prepare(ctx, d_pts, d_ll, d_lp, N, D, n, eps, sv, &mean_il)
                    : direct_prepare(ctx, d_pts, d_ll, d_lp, N, D, n, sv);
  // one exchange: every rank's status (a failure anywhere ends the call on every rank instead of a hang), the
  // arguments that must agree, and the root's mean 1/L and survivor count
  struct Head { int64_t root, D, n; uint64_t eps; int64_t K; double mean_il; };
  std::vector<Head> head(1), heads;
  head[0] = {root, D, n, 0, sv.K, mean_il};
  memcpy(&head[0].eps, &eps, sizeof eps);
  if ((rc = comm_gather(c, rc, head, heads, "evidence (sharded)"))) return rc;
  for (int r = 0; r < R; ++r)
    if (heads[r].root != root || heads[r].D != D || heads[r].n != n || heads[r].eps != head[0].eps)
      return set_err(ctx, MG_EINVAL, "evidence (sharded): rank %d has another root, D, n or eps", r);
  // the survivors (rows, lp, and ll for the direct estimator) go to every rank; the tree over them is then built by
  // all ranks together (build_tree_distributed: top levels everywhere, one subtree per rank, one all-gather)
  const int64_t K = heads[root].K;
  if (rank != root) {
    sv.K = K;
    cudaError_t e = sv.pts.alloc((size_t)K * D, s);
    if (e == cudaSuccess) e = sv.lp.alloc((size_t)K, s);
    if (e == cudaSuccess && which == 1) e = sv.ll.alloc((size_t)K, s);
    if (e != cudaSuccess) return set_err(ctx, MG_ENOMEM, "cuda: %s", cudaGetErrorString(e));
  }
  rc = comm_broadcast_dev(c, sv.pts.get(), sizeof(double) * (size_t)K * D, root);
  if (rc == MG_OK) rc = comm_broadcast_dev(c, sv.lp.get(), sizeof(double) * (size_t)K, root);
  if (rc == MG_OK && which == 1) rc = comm_broadcast_dev(c, sv.ll.get(), sizeof(double) * (size_t)K, root);
  if (rc) return rc;
  KdTreePtr t;
  {
    std::vector<double> zeros(D, 0.0);            // the root box takes no part in the evidence (see integrate_cells)
    // the cell terms read the survivors' rows, not a copy inside the blob
    if ((rc = build_tree_distributed(c, sv.pts.get(), K, D, zeros.data(), zeros.data(), n < 2 ? 2 : n, false, &t))) return rc;
  }
  const int64_t nn = t->h.nnodes;
  const double *sll = sv.ll.get(), *slp = sv.lp.get();
  // my range of nodes; slices of equal length so that the gathered slices ARE the node-ordered array
  const int64_t slice = (nn + R - 1) / R;
  const int64_t n0 = std::min<int64_t>(nn, (int64_t)rank * slice), n1 = std::min<int64_t>(nn, n0 + slice);
  DevBuf<double> terms;
  DevBuf<unsigned long long> ncells;
  if (rc == MG_OK) {
    cudaError_t e = terms.alloc((size_t)slice * R, s);
    if (e == cudaSuccess) e = ncells.alloc(1, s);
    if (e == cudaSuccess) e = cudaMemsetAsync(ncells.get(), 0, 8, s);
    if (e == cudaSuccess) e = cudaMemsetAsync(terms.get() + (size_t)rank * slice, 0, sizeof(double) * (size_t)slice, s);
    if (e != cudaSuccess) rc = set_err(ctx, MG_ENOMEM, "cuda: %s", cudaGetErrorString(e));
  }
  if (rc == MG_OK)
    rc = which == 0 ? cell_terms_range<0>(ctx, t.get(), sv.pts.get(), sll, slp, n, n0, n1, terms.get(), ncells.get())
                    : cell_terms_range<1>(ctx, t.get(), sv.pts.get(), sll, slp, n, n0, n1, terms.get(), ncells.get());
  if (rc == MG_OK) rc = comm_allgather_dev(c, terms.get() + (size_t)rank * slice, terms.get(), sizeof(double) * (size_t)slice);
  double total = 0.0;
  if (rc == MG_OK) rc = sum_terms(ctx, terms.get(), nn, &total);
  if (rc) return rc;
  *out = which == 0 ? total / heads[root].mean_il : total;
  return MG_OK;
}

extern "C" int mg_evidence_lebesgue_sharded(mg_comm *c, int32_t root, const double *d_pts, const double *d_ll,
                                            const double *d_lp, int64_t N, int32_t D, int32_t n, double eps, double *out) {
  return evidence_sharded(c, 0, root, d_pts, d_ll, d_lp, N, D, n, eps, out);
}
extern "C" int mg_evidence_direct_sharded(mg_comm *c, int32_t root, const double *d_pts, const double *d_ll,
                                          const double *d_lp, int64_t N, int32_t D, int32_t n, double *out) {
  return evidence_sharded(c, 1, root, d_pts, d_ll, d_lp, N, D, n, 0.0, out);
}

static int evidence_host(mg_ctx *ctx, int which, const double *pts, const double *ll, const double *lp, int64_t N,
                         int32_t D, int32_t n, double eps, double *out) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, pts && ll && lp && out, "evidence: null argument");
  MG_REQUIRE(ctx, N >= 1, "bounds_of_objects: no objects");
  MG_REQUIRE(ctx, D >= 1 && D <= 64, "evidence: dim must be in 1..64");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  DevBuf<double> d_pts, d_ll, d_lp;
  MG_CUDA(ctx, upload(d_pts, pts, (size_t)N * D, ctx->stream));
  MG_CUDA(ctx, upload(d_ll, ll, (size_t)N, ctx->stream));
  MG_CUDA(ctx, upload(d_lp, lp, (size_t)N, ctx->stream));
  return which == 0 ? mg_evidence_lebesgue_dev(ctx, d_pts.get(), d_ll.get(), d_lp.get(), N, D, n, eps, out)
                    : mg_evidence_direct_dev(ctx, d_pts.get(), d_ll.get(), d_lp.get(), N, D, n, out);
}

extern "C" int mg_evidence_lebesgue(mg_ctx *ctx, const double *pts, const double *ll, const double *lp, int64_t N,
                                    int32_t D, int32_t n, double eps, double *out) {
  return evidence_host(ctx, 0, pts, ll, lp, N, D, n, eps, out);
}
extern "C" int mg_evidence_direct(mg_ctx *ctx, const double *pts, const double *ll, const double *lp, int64_t N,
                                  int32_t D, int32_t n, double *out) {
  return evidence_host(ctx, 1, pts, ll, lp, N, D, n, 0.0, out);
}

// bin/harmonic_evidence.ml:41-52: one CTA per bootstrap replicate.  Draw j of replicate b is draw j of stream
// (P_BOOT, b, 0) -- the sequence a sequential Random.int loop would consume; a thread takes whole groups of 11 draws
// (5 Philox blocks, rng.cuh).
namespace mg {
__global__ void inv_like_kernel(const double *__restrict__ ll, int64_t n, double *__restrict__ il) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    il[i] = 1.0 / exp(ll[i]);     // evidence.ml:105
}
__global__ void __launch_bounds__(EB)
harmonic_bootstrap_kernel(const double *__restrict__ il, int64_t n, CallKey key, double *__restrict__ evs) {
  const uint64_t b = blockIdx.x;
  Comp acc;
  const int64_t ngroups = (n + 10) / 11;
  for (int64_t q = threadIdx.x; q < ngroups; q += EB) {
    Rng r(key, P_BOOT, b, 0);
    r.j = (uint32_t)(11 * q);                       // the cursor addresses draws: jump to this group
    const int cnt = (int)((n - 11 * q < 11) ? n - 11 * q : 11);
    for (int k = 0; k < cnt; ++k) acc.add(il[r.below((uint64_t)n)]);
  }
  const double t = block_reduce_comp<EB>(acc);
  if (threadIdx.x == 0) evs[b] = (double)n / t;
}
}  // namespace mg

extern "C" int mg_evidence_harmonic_bootstrap(mg_ctx *ctx, const double *ll, int64_t N, int32_t nbstrap, double *out_evs) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, ll && out_evs && N >= 1 && nbstrap >= 1, "harmonic bootstrap: bad arguments");
  MG_REQUIRE(ctx, N < (1LL << 31), "harmonic bootstrap: too many samples");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  DevBuf<double> d_ll, d_il, d_evs;
  MG_CUDA(ctx, upload(d_ll, ll, (size_t)N, s));
  MG_CUDA(ctx, d_il.alloc(N, s));
  MG_CUDA(ctx, d_evs.alloc(nbstrap, s));
  inv_like_kernel<<<egrid(ctx, N), EB, 0, s>>>(d_ll.get(), N, d_il.get());
  MG_CHECK_LAUNCH(ctx);
  const CallKey key = next_key(ctx);
  time_begin(ctx);
  harmonic_bootstrap_kernel<<<(unsigned)nbstrap, EB, 0, s>>>(d_il.get(), N, key, d_evs.get());
  MG_CHECK_LAUNCH(ctx);
  time_end(ctx);
  MG_CUDA(ctx, cudaMemcpyAsync(out_evs, d_evs.get(), sizeof(double) * nbstrap, cudaMemcpyDeviceToHost, s));
  MG_CUDA(ctx, cudaStreamSynchronize(s));
  return MG_OK;
}

// Diagnostic (tests only): stable-sort float64 keys on the device and count
// order violations / non-permutation entries of the result.
namespace mg {
__global__ void sort_check_kernel(const double *__restrict__ x, const int32_t *__restrict__ order, int64_t n,
                                  unsigned long long *__restrict__ bad) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i + 1 < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double a = x[order[i]], b = x[order[i + 1]];
    if (a > b || (a == b && order[i] > order[i + 1])) atomicAdd(bad, 1ull);   // sorted and stable
  }
}
}  // namespace mg
extern "C" int mg_debug_sort_check(mg_ctx *ctx, const double *d_x, int64_t n, int64_t *violations) {
  if (!ctx) return MG_EINVAL;
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  DevBuf<uint64_t> keys; DevBuf<int32_t> order; DevBuf<unsigned long long> bad;
  MG_CUDA(ctx, keys.alloc(n, s)); MG_CUDA(ctx, order.alloc(n, s)); MG_CUDA(ctx, bad.alloc(1, s));
  MG_CUDA(ctx, cudaMemsetAsync(bad.get(), 0, 8, s));
  // keys of +x: reuse the -ll key kernel on the negated ordering is not needed; build keys directly
  DevBuf<double> neg;
  MG_CUDA(ctx, neg.alloc(n, s));
  const double *xx = d_x; double *ng = neg.get();
  double dummy;
  int rc = reduce_sum(ctx, n, [xx, ng] __device__(int64_t i) { ng[i] = -xx[i]; return 0.0; }, &dummy);
  if (rc) return rc;
  neg_ll_keys_kernel<<<egrid(ctx, n), EB, 0, s>>>(neg.get(), n, keys.get(), order.get());   // keys of -(-x) = x
  MG_CHECK_LAUNCH(ctx);
  if ((rc = radix_sort_pairs(ctx, keys.get(), order.get(), n, 1))) return rc;
  sort_check_kernel<<<egrid(ctx, n), EB, 0, s>>>(d_x, order.get(), n, bad.get());
  MG_CHECK_LAUNCH(ctx);
  unsigned long long h = 0;
  MG_CUDA(ctx, cudaMemcpyAsync(&h, bad.get(), 8, cudaMemcpyDeviceToHost, s));
  MG_CUDA(ctx, cudaStreamSynchronize(s));
  *violations = (int64_t)h;
  return MG_OK;
}
