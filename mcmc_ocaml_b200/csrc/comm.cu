// comm.cu -- the multi-GPU side of the C ABI: one process per GPU, one NCCL communicator per context.
//
// What shards (SURVEY.md 8e): chains and queries are independent (no data-path collective, chain ids are global);
// a kd-tree is built on one rank and replicated with ONE ncclBroadcast of its contiguous device blob, straight from
// the builder's blob into the receivers' blobs (no staging copy); per-rank statistics and per-cell evidence terms are
// all-gathered and combined in a fixed order, so every rank holds the same bits and the result does not depend on the
// number of ranks.
//
// NCCL is bound at run time (dlopen "libnccl.so.2"): the library has no link-time dependency on it, a process that
// already carries an NCCL (torch) shares that copy, and without NCCL only these entry points fail (MG_EFAIL).
#include <dlfcn.h>
#include <time.h>
#include <nccl.h>

#include <algorithm>
#include <vector>

#include "common.cuh"
#include "kdtree.cuh"

static_assert(sizeof(ncclUniqueId) == MG_COMM_ID_BYTES, "ncclUniqueId is 128 bytes");

namespace mg {

struct NcclApi {
  void *h = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*Broadcast)(const void *, void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  const char *(*GetErrorString)(ncclResult_t) = nullptr;
  ncclResult_t (*GetVersion)(int *) = nullptr;
  std::string why;
};

static NcclApi *nccl_api() {
  static NcclApi api = [] {
    NcclApi a;
    const char *names[] = {getenv("MCMC_GPU_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    for (const char *n : names) {
      if (!n || !*n) continue;
      a.h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
      if (a.h) break;
    }
    if (!a.h) { a.why = std::string("cannot load libnccl.so.2: ") + (dlerror() ? dlerror() : "not found"); return a; }
#define MG_SYM(field, name)                                                    \
  a.field = reinterpret_cast<decltype(a.field)>(dlsym(a.h, name));              \
  if (!a.field) { a.why = std::string("libnccl lacks ") + name; a.h = nullptr; return a; }
    MG_SYM(GetUniqueId, "ncclGetUniqueId") MG_SYM(CommInitRank, "ncclCommInitRank") MG_SYM(CommDestroy, "ncclCommDestroy")
    MG_SYM(Broadcast, "ncclBroadcast") MG_SYM(AllGather, "ncclAllGather") MG_SYM(GetErrorString, "ncclGetErrorString")
    MG_SYM(GetVersion, "ncclGetVersion")
#undef MG_SYM
    return a;
  }();
  return &api;
}

}  // namespace mg

struct mg_comm {
  mg_ctx *ctx = nullptr;
  ncclComm_t comm = nullptr;
  int nranks = 1, rank = 0;
  double last_collective_ms = 0.0;
};

using namespace mg;

#define MG_NCCL(ctx, call)                                                                              \
  do {                                                                                                  \
    ncclResult_t r_ = (call);                                                                           \
    if (r_ != ncclSuccess)                                                                              \
      return mg::set_err((ctx), MG_EFAIL, "nccl: %s at %s:%d", nccl_api()->GetErrorString(r_), __FILE__, __LINE__); \
  } while (0)

extern "C" int mg_comm_get_unique_id(uint8_t id[MG_COMM_ID_BYTES]) {
  NcclApi *api = nccl_api();
  if (!api->h || !id) return MG_EFAIL;
  ncclUniqueId u;
  if (api->GetUniqueId(&u) != ncclSuccess) return MG_EFAIL;
  memcpy(id, &u, MG_COMM_ID_BYTES);
  return MG_OK;
}

extern "C" int mg_comm_create(mg_ctx *ctx, int32_t nranks, int32_t rank, const uint8_t id[MG_COMM_ID_BYTES], mg_comm **out) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, out && nranks >= 1 && rank >= 0 && rank < nranks, "comm_create: bad rank / size");
  *out = nullptr;
  mg_comm *c = new mg_comm;
  c->ctx = ctx; c->nranks = nranks; c->rank = rank;
  if (nranks > 1) {
    NcclApi *api = nccl_api();
    if (!api->h) { delete c; return set_err(ctx, MG_EFAIL, "nccl: %s", api->why.c_str()); }
    if (!id) { delete c; return set_err(ctx, MG_EINVAL, "comm_create: null unique id"); }
    if (cudaSetDevice(ctx->device) != cudaSuccess) { delete c; return set_err(ctx, MG_ECUDA, "cuda: cannot select the device"); }
    ncclUniqueId u;
    memcpy(&u, id, MG_COMM_ID_BYTES);
    ncclResult_t r = api->CommInitRank(&c->comm, nranks, u, rank);
    if (r != ncclSuccess) { delete c; return set_err(ctx, MG_EFAIL, "nccl: %s (ncclCommInitRank)", api->GetErrorString(r)); }
  }
  *out = c;
  return MG_OK;
}

extern "C" void mg_comm_destroy(mg_comm *c) {
  if (!c) return;
  if (c->comm) {
    cudaSetDevice(c->ctx->device);
    cudaStreamSynchronize(c->ctx->stream);
    nccl_api()->CommDestroy(c->comm);
  }
  delete c;
}
extern "C" int32_t mg_comm_rank(const mg_comm *c) { return c ? c->rank : -1; }
extern "C" int32_t mg_comm_size(const mg_comm *c) { return c ? c->nranks : 0; }
extern "C" double mg_comm_last_collective_ms(const mg_comm *c) { return c ? c->last_collective_ms : 0.0; }
extern "C" int mg_comm_nccl_version(int32_t *version) {
  NcclApi *api = nccl_api();
  if (!api->h || !version) return MG_EFAIL;
  int v = 0;
  if (api->GetVersion(&v) != ncclSuccess) return MG_EFAIL;
  *version = v;
  return MG_OK;
}

namespace mg {

// device-to-device collectives on the context's stream, timed with events (the time a rank spends inside the call)
struct CollTimer {
  mg_comm *c; cudaEvent_t e0 = nullptr, e1 = nullptr;
  explicit CollTimer(mg_comm *c_) : c(c_) {
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaEventRecord(e0, c->ctx->stream);
  }
  void stop() {
    cudaEventRecord(e1, c->ctx->stream);
    cudaEventSynchronize(e1);
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, e0, e1) == cudaSuccess) c->last_collective_ms = ms;
  }
  ~CollTimer() { if (e0) cudaEventDestroy(e0); if (e1) cudaEventDestroy(e1); }
};

int comm_broadcast_dev(mg_comm *c, void *d_buf, size_t nbytes, int root) {
  if (c->nranks == 1 || nbytes == 0) return MG_OK;
  MG_NCCL(c->ctx, nccl_api()->Broadcast(d_buf, d_buf, nbytes, ncclUint8, root, c->comm, c->ctx->stream));
  c->ctx->launches++;
  return MG_OK;
}

int comm_allgather_dev(mg_comm *c, const void *d_send, void *d_recv, size_t nbytes_per_rank) {
  mg_ctx *ctx = c->ctx;
  if (c->nranks == 1) {
    if (d_send != d_recv) MG_CUDA(ctx, cudaMemcpyAsync(d_recv, d_send, nbytes_per_rank, cudaMemcpyDeviceToDevice, ctx->stream));
    return MG_OK;
  }
  MG_NCCL(ctx, nccl_api()->AllGather(d_send, d_recv, nbytes_per_rank, ncclUint8, c->comm, ctx->stream));
  ctx->launches++;
  return MG_OK;
}

}  // namespace mg

// All-gather of a small host record from every rank (per-rank counts, sums, partial statistics): recv holds
// nranks * nbytes in rank order on every rank.
extern "C" int mg_comm_allgather(mg_comm *c, const void *send, void *recv, int64_t nbytes) {
  if (!c) return MG_EINVAL;
  mg_ctx *ctx = c->ctx;
  MG_REQUIRE(ctx, send && recv && nbytes >= 0, "allgather: bad arguments");
  if (nbytes == 0) return MG_OK;
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  if (c->nranks == 1) { memmove(recv, send, (size_t)nbytes); return MG_OK; }
  DevBuf<uint8_t> d_send, d_recv;
  MG_CUDA(ctx, d_send.alloc((size_t)nbytes, ctx->stream));
  MG_CUDA(ctx, d_recv.alloc((size_t)nbytes * c->nranks, ctx->stream));
  MG_CUDA(ctx, cudaMemcpyAsync(d_send.get(), send, (size_t)nbytes, cudaMemcpyHostToDevice, ctx->stream));
  CollTimer tm(c);
  int rc = comm_allgather_dev(c, d_send.get(), d_recv.get(), (size_t)nbytes);
  if (rc) return rc;
  tm.stop();
  MG_CUDA(ctx, cudaMemcpyAsync(recv, d_recv.get(), (size_t)nbytes * c->nranks, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MG_OK;
}

extern "C" int mg_comm_barrier(mg_comm *c) {
  if (!c) return MG_EINVAL;
  uint8_t one = 1;
  std::vector<uint8_t> all((size_t)c->nranks);
  return mg_comm_allgather(c, &one, all.data(), 1);
}

// Kd-tree built on `root`, replicated on every rank: the header first (sizes), then ONE broadcast of the blob from the
// builder's blob straight into each receiver's freshly allocated blob.  On the root *out is `tree` itself.
extern "C" int mg_kdtree_broadcast(mg_comm *c, mg_kdtree *tree, int32_t root, mg_kdtree **out) {
  if (!c) return MG_EINVAL;
  mg_ctx *ctx = c->ctx;
  MG_REQUIRE(ctx, out && root >= 0 && root < c->nranks, "kdtree_broadcast: bad arguments");
  MG_REQUIRE(ctx, c->rank != root || tree != nullptr, "kdtree_broadcast: the root has no tree");
  MG_REQUIRE(ctx, c->rank != root || tree->ctx == ctx, "kdtree_broadcast: the tree belongs to another context");
  *out = nullptr;
  if (c->nranks == 1) { *out = tree; return MG_OK; }
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  int rc;
  DevBuf<uint8_t> d_hdr;
  constexpr size_t HB = 256;                     // the header occupies the blob's first 256-byte section
  static_assert(sizeof(KdHeader) <= HB, "header section");
  void *hdr_buf = nullptr;
  if (c->rank == root) hdr_buf = tree->d_blob;
  else { MG_CUDA(ctx, d_hdr.alloc(HB, s)); hdr_buf = d_hdr.get(); }
  CollTimer tm(c);
  if ((rc = comm_broadcast_dev(c, hdr_buf, HB, root))) return rc;
  if (c->rank == root) {
    if ((rc = comm_broadcast_dev(c, tree->d_blob, (size_t)tree->h.nbytes, root))) return rc;
    tm.stop();
    *out = tree;
    return MG_OK;
  }
  KdHeader h;
  MG_CUDA(ctx, cudaMemcpyAsync(&h, hdr_buf, sizeof h, cudaMemcpyDeviceToHost, s));
  MG_CUDA(ctx, cudaStreamSynchronize(s));
  // a bad header must not leave this rank out of the collective the others have entered: receive into a blob of the
  // announced size if that is at all possible, then judge
  const bool sane = h.magic == KD_MAGIC && h.nbytes >= (int64_t)HB && h.nbytes < (1LL << 40);
  if (!sane) return set_err(ctx, MG_EFAIL, "kdtree_broadcast: the root sent no kd-tree header");
  KdTreePtr t;
  if ((rc = kd_alloc(ctx, h, &t))) return rc;
  rc = comm_broadcast_dev(c, t->d_blob, (size_t)h.nbytes, root);
  if (rc == MG_OK) { tm.stop(); rc = validate_blob_header(ctx, h); }
  if (rc) return rc;
  *out = t.release();
  return MG_OK;
}

mg_ctx *mg_comm_ctx(const mg_comm *c) { return c ? c->ctx : nullptr; }

#include "reduce_sum.cuh"

// Evidence.evidence_harmonic_mean (evidence.ml:101-107) over samples SHARDED across ranks: every rank reduces the
// 1/L of its own shard (compensated), the (count, sum) pairs are all-gathered and folded in rank order.  Agrees with
// the single-GPU value to the rounding of the compensated sums (<= 2 ulp); identical on every rank.
extern "C" int mg_evidence_harmonic_mean_sharded(mg_comm *c, const double *d_ll_shard, int64_t n_shard, double *out) {
  if (!c) return MG_EINVAL;
  mg_ctx *ctx = c->ctx;
  MG_REQUIRE(ctx, out && n_shard >= 0 && (d_ll_shard || n_shard == 0), "evidence_harmonic_mean (sharded): bad arguments");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  double mine[2] = {(double)n_shard, 0.0};
  if (n_shard > 0) {
    int rc = reduce_sum(ctx, n_shard, [d_ll_shard] __device__(int64_t i) { return 1.0 / exp(d_ll_shard[i]); }, &mine[1]);
    if (rc) return rc;
  }
  std::vector<double> all((size_t)2 * c->nranks);
  int rc = mg_comm_allgather(c, mine, all.data(), sizeof mine);
  if (rc) return rc;
  Comp linv; double n = 0.0;
  for (int r = 0; r < c->nranks; ++r) { n += all[2 * r]; linv.add(all[2 * r + 1]); }
  MG_REQUIRE(ctx, n >= 1.0, "evidence_harmonic_mean (sharded): no samples on any rank");
  *out = n / linv.value();
  return MG_OK;
}

// Mcmc.rjmcmc_array (mcmc.ml:121-139) with the ensemble's chains cut into contiguous ranges, one per rank: rank r runs
// the global chain ids cfg->chain_offset + [b_r, e_r) (the Philox stream is addressed by the global id, so the
// chains do not depend on the number of ranks), then rjmcmc_model_counts (mcmc.ml:141-149) and the accept / jump
// counters of all ranks are all-gathered and summed.  out_model / out_samples receive this rank's shard only
// ([n][C_r], [n][Dmax+2][C_r]); *shard_begin / *shard_count tell which chains those are.
extern "C" int mg_rjmcmc_array_sharded(mg_comm *c, const mg_rj_model *A, const mg_rj_model *B, const mg_rjmcmc_cfg *cfg,
                                       const double *a0, const double *b0, uint8_t *out_model, double *out_samples,
                                       int64_t out_counts[2], int64_t *shard_begin, int64_t *shard_count) {
  if (!c) return MG_EINVAL;
  mg_ctx *ctx = c->ctx;
  MG_REQUIRE(ctx, cfg && out_counts, "rjmcmc_array (sharded): null argument");
  const int64_t C = cfg->nchains, base = C / c->nranks, rem = C % c->nranks;
  const int64_t b = (int64_t)c->rank * base + std::min<int64_t>(c->rank, rem), cnt = base + (c->rank < rem ? 1 : 0);
  if (shard_begin) *shard_begin = b;
  if (shard_count) *shard_count = cnt;
  int64_t mine[5] = {0, 0, 0, 0, 0};          // #A, #B, accepted, cross-model proposed, cross-model accepted
  int rc = MG_OK;
  if (cnt > 0) {
    mg_rjmcmc_cfg local = *cfg;
    local.nchains = cnt; local.chain_offset = cfg->chain_offset + (uint64_t)b;
    const int64_t acc0 = ctx->naccept;
    rc = mg_rjmcmc_array(ctx, A, B, &local, a0, b0, out_model, out_samples, mine);
    mine[2] = ctx->naccept - acc0; mine[3] = ctx->rj_cross[0]; mine[4] = ctx->rj_cross[1];
  } else {
    ctx->epoch++;                              // every rank consumes the same epoch of its context's key
  }
  int64_t status = rc;
  std::vector<int64_t> all((size_t)6 * c->nranks);
  int64_t rec[6] = {mine[0], mine[1], mine[2], mine[3], mine[4], status};
  int rc2 = mg_comm_allgather(c, rec, all.data(), sizeof rec);
  if (rc) return rc;
  if (rc2) return rc2;
  int64_t tot[5] = {0, 0, 0, 0, 0};
  for (int r = 0; r < c->nranks; ++r) {
    if (all[6 * r + 5] != 0) return set_err(ctx, (int)all[6 * r + 5], "rjmcmc_array (sharded): rank %d failed", r);
    for (int k = 0; k < 5; ++k) tot[k] += all[6 * r + k];
  }
  out_counts[0] = tot[0]; out_counts[1] = tot[1];
  ctx->rj_cross[0] = tot[3]; ctx->rj_cross[1] = tot[4];
  return MG_OK;
}

// Stats.multi_mean / multi_std (stats.ml:58-87) of samples held by several ranks, from each rank's own
// (count, mean[F], std[F]): the pairs are all-gathered and pooled in rank order with the parallel-variance update
// (Chan et al.), std with n - 1 as the reference.  Every rank receives the same values.
extern "C" int mg_comm_pool_moments(mg_comm *c, int64_t n_local, const double *mean_local, const double *std_local,
                                    int32_t F, int64_t *n_total, double *out_mean, double *out_std) {
  if (!c) return MG_EINVAL;
  mg_ctx *ctx = c->ctx;
  MG_REQUIRE(ctx, mean_local && std_local && F >= 1 && F <= 4096 && n_local >= 0, "pool_moments: bad arguments");
  std::vector<double> mine((size_t)1 + 2 * F), all(((size_t)1 + 2 * F) * c->nranks);
  mine[0] = (double)n_local;
  for (int i = 0; i < F; ++i) {
    mine[1 + i] = mean_local[i];
    mine[1 + F + i] = n_local > 1 ? std_local[i] * std_local[i] * ((double)n_local - 1.0) : 0.0;   // sum of squared deviations
  }
  int rc = mg_comm_allgather(c, mine.data(), all.data(), (int64_t)(sizeof(double) * mine.size()));
  if (rc) return rc;
  double n = 0.0;
  std::vector<double> mean(F, 0.0), m2(F, 0.0);
  for (int r = 0; r < c->nranks; ++r) {
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

// =====================================================================================================================
// Distributed kd-tree build (SURVEY.md 8e / 8f rank 3): Kd_tree.tree_of_objects (kd_tree.ml:155-175) with the
// subtrees below level k = log2(ranks) built on different GPUs.
//
// Every rank holds the N points (replicated input: the posterior draws a model's interpolated jumps are made from).
//   1. every rank builds the TOP of the tree, truncated where nodes fall below ~N / ranks points: k levels, 2^k leaves;
//      the same arithmetic on the same data, so all ranks hold the same top and the same stable order of the points;
//   2. rank r gathers the rows of leaf r in that order and builds the complete tree of those N / ranks points with
//      the single-GPU builder -- the rule depends on a node's points and their order only, so this IS the subtree the
//      single-GPU build hangs under node r;
//   3. one ncclAllGather moves every rank's (nodes, count, begin, perm) sections; an unpack kernel gives the nodes
//      their breadth-first numbers in the whole tree (level L of the whole tree = the ranks' levels L - k side by
//      side, children adjacent) and maps the local point ids back through the top's order.
// The result is bit-identical to mg_kdtree_build_dev on one GPU (tools/multi_gpu_check.py compares every array).
// Inputs whose top does not come out as a complete k-level tree (ties that stop a node from splitting), fewer than
// 4096 points per rank or a rank count that is not a power of two are built by every rank for itself.
namespace mg {

constexpr int KDD_MAXL = 96;         // levels of a subtree
constexpr int KDD_MAXR = 64;         // ranks

__global__ void kdd_gather_rows_kernel(const double *__restrict__ pts, const int32_t *__restrict__ perm, int64_t n, int D,
                                       double *__restrict__ out) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n * D) return;
  const int64_t i = k / D; const int j = (int)(k - i * D);
  out[k] = pts[(int64_t)perm[i] * D + j];
}

struct KddTables {
  int32_t lb[KDD_MAXR][KDD_MAXL + 1];   // per rank: first local node of every local level
  int32_t goff[KDD_MAXR][KDD_MAXL + 1]; // per rank: nodes of lower ranks on the same level
  int32_t gbase[KDD_MAXL + 2];          // whole tree: first node of level k + l
  int32_t nl[KDD_MAXR], nn[KDD_MAXR], npts[KDD_MAXR], pbegin[KDD_MAXR];
  int64_t off_count[KDD_MAXR], off_begin[KDD_MAXR], off_perm[KDD_MAXR];   // byte offsets inside a rank's chunk
};

__global__ void kdd_unpack_nodes_kernel(const KddTables *__restrict__ T, int r, const uint8_t *__restrict__ chunk,
                                        KdNode *__restrict__ nodes, int32_t *__restrict__ count, int32_t *__restrict__ begin) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= T->nn[r]) return;
  const int32_t *lb = T->lb[r];
  int lo = 0, hi = T->nl[r];                     // level l with lb[l] <= i < lb[l + 1]
  while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (lb[mid] <= i) lo = mid; else hi = mid; }
  const int l = lo;
  const int gid = T->gbase[l] + T->goff[r][l] + (i - lb[l]);
  KdNode nd = reinterpret_cast<const KdNode *>(chunk)[i];
  if (nd.left >= 0) nd.left = T->gbase[l + 1] + T->goff[r][l + 1] + (nd.left - lb[l + 1]);
  nodes[gid] = nd;
  count[gid] = reinterpret_cast<const int32_t *>(chunk + T->off_count[r])[i];
  begin[gid] = T->pbegin[r] + reinterpret_cast<const int32_t *>(chunk + T->off_begin[r])[i];
}

__global__ void kdd_unpack_perm_kernel(const KddTables *__restrict__ T, int r, const uint8_t *__restrict__ chunk,
                                       const int32_t *__restrict__ top_perm, int32_t *__restrict__ perm) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= T->npts[r]) return;
  const int b = T->pbegin[r];
  perm[b + j] = top_perm[b + reinterpret_cast<const int32_t *>(chunk + T->off_perm[r])[j]];
}

int build_tree_distributed(mg_comm *c, const double *d_pts, int64_t N, int D, const double *low, const double *high,
                           int min_split, bool with_pts, KdTreePtr *out) {
  mg_ctx *ctx = c->ctx;
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  if (min_split < 2) min_split = 2;
  const int R = c->nranks;
  int k = 0;
  while ((1 << k) < R) ++k;
  const int64_t ms_top = (N >> k) + 3;           // no node of level k reaches it, every node above does (without ties)
  const bool shard = R > 1 && (1 << k) == R && R <= KDD_MAXR && N / R >= 4096 && (int64_t)min_split < ms_top && ms_top < (1LL << 31);
  if (!shard) return build_tree(ctx, d_pts, N, D, low, high, min_split, with_pts, out);
  cudaStream_t s = ctx->stream;
  int rc;
  static const bool dbg = getenv("MCMC_GPU_DEBUG") != nullptr;
  double t_prev = 0.0;
  auto phase = [&](const char *name) {           // MCMC_GPU_DEBUG: wall time of the phases (adds synchronisation)
    if (!dbg) return;
    cudaStreamSynchronize(s);
    timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts);
    const double now = ts.tv_sec + 1e-9 * ts.tv_nsec;
    uint64_t reserved = 0, used = 0;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, ctx->device) == cudaSuccess) {
      cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &reserved);
      cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemCurrent, &used);
    }
    if (name) fprintf(stderr, "[kd-dist rank %d] %-10s %8.3f ms   pool reserved %.2f GB used %.2f GB\n", c->rank, name, 1e3 * (now - t_prev),
                      1e-9 * reserved, 1e-9 * used);
    t_prev = now;
  };
  phase(nullptr);
  // The result's blob is allocated FIRST, for the largest possible node count (2 N): a caller that rebuilds trees
  // gets the block of its previous tree back, where a late request for 2 GB in one piece makes the stream-ordered
  // pool remap its fragments (measured: 15-180 ms).  Truncated trees (min_split > 16) are small next to that bound and
  // get an exact blob at the end instead.
  KdTreePtr res;
  const bool early = min_split <= 16;
  if (early && (rc = kd_alloc(ctx, kd_layout(N, D, 2 * N, with_pts), &res))) return rc;
  // ---- 1. the top, on every rank ---------------------------------------------------------------------------------------
  // (the top and the subtree are scaffolding: their blobs carry no copy of the points)
  KdTreePtr top, sub;
  rc = build_tree(ctx, d_pts, N, D, low, high, (int)ms_top, false, &top);
  // A rank that fails here still takes part in the agreement below (as "not complete"): every rank then builds alone
  // and the failing rank reports its own error, instead of the others waiting in a collective for ever.
  const int rc_top = rc;
  phase("top build");
  static const KdHeader no_header{};
  const KdHeader &th = rc_top == MG_OK ? top->h : no_header;
  const char *tb = rc_top == MG_OK ? (const char *)top->d_blob : nullptr;
  std::vector<KdNode> tnodes((size_t)th.nnodes);
  std::vector<int32_t> tcount((size_t)th.nnodes), tbegin((size_t)th.nnodes);
  bool complete = rc_top == MG_OK && th.nnodes == 2 * (int64_t)R - 1;
  if (complete) {
    MG_CUDA(ctx, cudaMemcpyAsync(tnodes.data(), tb + th.off_nodes, sizeof(KdNode) * tnodes.size(), cudaMemcpyDeviceToHost, s));
    MG_CUDA(ctx, cudaMemcpyAsync(tcount.data(), tb + th.off_count, 4 * tcount.size(), cudaMemcpyDeviceToHost, s));
    MG_CUDA(ctx, cudaMemcpyAsync(tbegin.data(), tb + th.off_begin, 4 * tbegin.size(), cudaMemcpyDeviceToHost, s));
    MG_CUDA(ctx, cudaStreamSynchronize(s));
    for (int i = 0; i < R - 1; ++i) complete = complete && tnodes[i].left == 2 * i + 1;      // a complete binary top
    for (int i = R - 1; i < 2 * R - 1; ++i) complete = complete && tnodes[i].left < 0 && tcount[i] >= 2;
  }
  phase("top d2h");
  // every rank must take the same branch: the tops are identical, but agree explicitly
  {
    int64_t mine = complete ? 1 : 0;
    std::vector<int64_t> all((size_t)R);
    if ((rc = mg_comm_allgather(c, &mine, all.data(), sizeof mine))) return rc;
    for (int r = 0; r < R; ++r) complete = complete && all[r] == 1;
  }
  if (!complete) return rc_top != MG_OK ? rc_top : build_tree(ctx, d_pts, N, D, low, high, min_split, with_pts, out);
  phase("top");
  // ---- 2. this rank's subtree -------------------------------------------------------------------------------------------
  const int me = c->rank;
  const int32_t my_b = tbegin[R - 1 + me], my_n = tcount[R - 1 + me];
  const int32_t *top_perm = (const int32_t *)(tb + th.off_perm);
  DevBuf<double> rows;
  MG_CUDA(ctx, rows.alloc((size_t)my_n * D, s));
  kdd_gather_rows_kernel<<<(unsigned)(((int64_t)my_n * D + 255) / 256), 256, 0, s>>>(d_pts, top_perm + my_b, my_n, D, rows.get());
  MG_CHECK_LAUNCH(ctx);
  phase("gather");
  rc = build_tree(ctx, rows.get(), my_n, D, low, high, min_split, false, &sub);
  const int rc_sub = rc;                         // a failure travels in the record below, so that no rank is left waiting
  phase("subtree");
  const KdHeader &sh = rc_sub == MG_OK ? sub->h : no_header;
  const char *sb = rc_sub == MG_OK ? (const char *)sub->d_blob : nullptr;
  struct Rec { int32_t nl, nn, npts, pbegin; int32_t lb[KDD_MAXL + 1]; int32_t bad; };
  Rec mine{};
  if (rc_sub == MG_OK) {                         // the builder's level table, cut at KDD_MAXL levels (then flagged below)
    const std::vector<int32_t> &lvb = sub->level_begin;
    mine.nl = (int32_t)std::min<size_t>(lvb.size() - 1, KDD_MAXL);
    for (int l = 0; l <= mine.nl; ++l) mine.lb[l] = lvb[l];
  }
  mine.nn = (int32_t)sh.nnodes; mine.npts = my_n; mine.pbegin = my_b;
  mine.bad = rc_sub != MG_OK ? 2 : ((mine.nl >= KDD_MAXL || mine.lb[mine.nl] != mine.nn) ? 1 : 0);
  std::vector<Rec> recs((size_t)R);
  if ((rc = mg_comm_allgather(c, &mine, recs.data(), sizeof mine))) return rc;
  phase("tables");
  // ---- 3. numbering of the whole tree and the exchange -------------------------------------------------------------------
  std::vector<KddTables> Tv(1);
  KddTables &T = Tv[0];
  memset(&T, 0, sizeof T);
  int maxl = 0; int64_t chunk = 0;
  for (int r = 0; r < R; ++r) {
    const Rec &q = recs[r];
    if (q.bad == 2) return (r == c->rank) ? rc_sub : set_err(ctx, MG_EFAIL, "kd-tree (distributed): rank %d failed to build its subtree", r);
    if (q.bad) return set_err(ctx, MG_EFAIL, "kd-tree (distributed): rank %d built a subtree deeper than %d levels", r, KDD_MAXL);
    T.nl[r] = q.nl; T.nn[r] = q.nn; T.npts[r] = q.npts; T.pbegin[r] = q.pbegin;
    memcpy(T.lb[r], q.lb, sizeof q.lb);
    for (int l = q.nl + 1; l <= KDD_MAXL; ++l) T.lb[r][l] = q.nn;
    maxl = std::max(maxl, (int)q.nl);
    T.off_count[r] = align256(16LL * q.nn); T.off_begin[r] = align256(T.off_count[r] + 4LL * q.nn);
    T.off_perm[r] = align256(T.off_begin[r] + 4LL * q.nn);
    chunk = std::max<int64_t>(chunk, align256(T.off_perm[r] + 4LL * q.npts));
  }
  T.gbase[0] = R - 1;                               // level k of the whole tree starts after the 2^k - 1 nodes above it
  for (int l = 0; l <= maxl; ++l) {
    int64_t tot = 0;
    for (int r = 0; r < R; ++r) { T.goff[r][l] = (int32_t)tot; tot += T.lb[r][l + 1] - T.lb[r][l]; }
    T.gbase[l + 1] = T.gbase[l] + (int32_t)tot;
  }
  const int64_t nnodes = T.gbase[maxl];
  MG_REQUIRE(ctx, nnodes <= 2 * N, "kd-tree (distributed): node count out of range");
  DevBuf<uint8_t> sendb, recvb;
  DevBuf<KddTables> d_T;
  MG_CUDA(ctx, sendb.alloc((size_t)chunk, s)); MG_CUDA(ctx, recvb.alloc((size_t)chunk * R, s));
  MG_CUDA(ctx, upload(d_T, &T, 1, s));
  MG_CUDA(ctx, cudaMemcpyAsync(sendb.get(), sb + sh.off_nodes, 16 * (size_t)sh.nnodes, cudaMemcpyDeviceToDevice, s));
  MG_CUDA(ctx, cudaMemcpyAsync(sendb.get() + T.off_count[me], sb + sh.off_count, 4 * (size_t)sh.nnodes, cudaMemcpyDeviceToDevice, s));
  MG_CUDA(ctx, cudaMemcpyAsync(sendb.get() + T.off_begin[me], sb + sh.off_begin, 4 * (size_t)sh.nnodes, cudaMemcpyDeviceToDevice, s));
  MG_CUDA(ctx, cudaMemcpyAsync(sendb.get() + T.off_perm[me], sb + sh.off_perm, 4 * (size_t)my_n, cudaMemcpyDeviceToDevice, s));
  {
    CollTimer tm(c);
    if ((rc = comm_allgather_dev(c, sendb.get(), recvb.get(), (size_t)chunk))) return rc;
    tm.stop();
  }
  phase("allgather");
  // ---- the blob: the nodes of the top, then every rank's subtree ------------------------------------------------------------
  if (!early && (rc = kd_alloc(ctx, kd_layout(N, D, nnodes, with_pts), &res))) return rc;
  KdHeader &h = res->h;
  h.nnodes = nnodes; h.nlevels = k + maxl; h.min_split = min_split;
  char *blob = (char *)res->d_blob;
  phase("blob alloc");
  // the 2^k - 1 nodes above the subtrees: numbers, counts and positions are those of the top tree
  MG_CUDA(ctx, cudaMemcpyAsync(blob + h.off_nodes, tb + th.off_nodes, 16 * (size_t)(R - 1), cudaMemcpyDeviceToDevice, s));
  MG_CUDA(ctx, cudaMemcpyAsync(blob + h.off_count, tb + th.off_count, 4 * (size_t)(R - 1), cudaMemcpyDeviceToDevice, s));
  MG_CUDA(ctx, cudaMemcpyAsync(blob + h.off_begin, tb + th.off_begin, 4 * (size_t)(R - 1), cudaMemcpyDeviceToDevice, s));
  for (int r = 0; r < R; ++r) {
    const uint8_t *ch = recvb.get() + (size_t)chunk * r;
    kdd_unpack_nodes_kernel<<<(unsigned)((T.nn[r] + 255) / 256), 256, 0, s>>>(d_T.get(), r, ch, (KdNode *)(blob + h.off_nodes),
                                                                              (int32_t *)(blob + h.off_count), (int32_t *)(blob + h.off_begin));
    MG_CHECK_LAUNCH(ctx);
    kdd_unpack_perm_kernel<<<(unsigned)((T.npts[r] + 255) / 256), 256, 0, s>>>(d_T.get(), r, ch, top_perm, (int32_t *)(blob + h.off_perm));
    MG_CHECK_LAUNCH(ctx);
  }
  phase("unpack");
  rc = kd_finish(ctx, std::move(res), low, high, d_pts, out);
  phase("finish");
  return rc;
}

}  // namespace mg

extern "C" int mg_kdtree_build_distributed(mg_comm *c, const double *d_pts, int64_t N, int32_t D, const double *low,
                                           const double *high, int32_t min_split, mg_kdtree **out) {
  if (!c) return MG_EINVAL;
  MG_REQUIRE(c->ctx, d_pts && low && high && out, "kd-tree (distributed): null argument");
  KdTreePtr t;
  const int rc = build_tree_distributed(c, d_pts, N, D, low, high, min_split, true, &t);
  *out = t.release();
  return rc;
}

// Ensemble diagnostics (diagnostics.cu) of chains sharded over the ranks: every rank runs the local pass on its own
// [n][D+2][C_r] block and pools it into one record per field, (count, mean and M2 of the sequence means, sum s_m^2,
// sum_m gamma_m(t)) = F (L + 4) doubles, plus its status; the records are all-gathered and folded in rank order by the
// same host step as the single-GPU call, so every rank gets the same bytes and one rank gives the single-GPU bits.
namespace mg {
int diag_check_cfg(mg_ctx *ctx, const mg_diag_cfg *cfg);
int diag_local_record(mg_ctx *ctx, const double *d_x, const mg_diag_cfg *cfg, double *d_seq_tau, std::vector<double> &rec);
void diag_finish(const double *recs, int R, int F, int L, int64_t N, double *rhat, double *ess, double *tau,
                 int32_t *closed, double *rho);
}  // namespace mg

extern "C" int mg_comm_chain_diagnostics(mg_comm *c, const double *d_samples_local, const mg_diag_cfg *cfg_local,
                                         double *out_rhat, double *out_ess, double *out_tau, int32_t *out_window_closed,
                                         double *out_rho, double *d_seq_tau) {
  if (!c) return MG_EINVAL;
  mg_ctx *ctx = c->ctx;
  // dim and maxlag size the exchanged record: every rank must pass the same values (include/mcmc_gpu.h).  A rank that
  // fails this check returns before the collective and the others wait for it, as in mg_comm_pool_moments; every
  // later failure (other checks, the local pass) still takes part in the all-gather and is reported on every rank.
  MG_REQUIRE(ctx, cfg_local && cfg_local->dim >= 1 && cfg_local->maxlag >= 2 && cfg_local->maxlag <= MG_DIAG_MAXLAG,
             "chain_diagnostics (comm): bad configuration");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  const int F = cfg_local->dim + 2, L = cfg_local->maxlag, W = L + 4;
  int rc = diag_check_cfg(ctx, cfg_local);
  if (rc == MG_OK && !(d_samples_local && out_rhat && out_ess && out_tau && out_window_closed))
    rc = set_err(ctx, MG_EINVAL, "chain_diagnostics (comm): null argument");
  std::vector<double> rec;
  if (rc == MG_OK) rc = diag_local_record(ctx, d_samples_local, cfg_local, d_seq_tau, rec);
  std::vector<double> mine((size_t)F * W + 3, 0.0), all(mine.size() * c->nranks);
  if (rc == MG_OK) std::copy(rec.begin(), rec.end(), mine.begin());
  const int64_t N = cfg_local->split ? cfg_local->n / 2 : cfg_local->n;
  mine[(size_t)F * W] = (double)rc;
  mine[(size_t)F * W + 1] = (double)N;
  mine[(size_t)F * W + 2] = (double)cfg_local->split;
  const int rc2 = mg_comm_allgather(c, mine.data(), all.data(), (int64_t)(sizeof(double) * mine.size()));
  if (rc) return rc;
  if (rc2) return rc2;
  std::vector<double> recs((size_t)F * W * c->nranks);
  for (int r = 0; r < c->nranks; ++r) {
    const double *q = all.data() + mine.size() * r;
    if (q[(size_t)F * W] != 0.0) return set_err(ctx, (int)q[(size_t)F * W], "chain_diagnostics (comm): rank %d failed", r);
    if (q[(size_t)F * W + 1] != (double)N || q[(size_t)F * W + 2] != (double)cfg_local->split)
      return set_err(ctx, MG_EINVAL, "chain_diagnostics (comm): rank %d has another n or split", r);
    std::copy(q, q + (size_t)F * W, recs.begin() + (size_t)F * W * r);
  }
  diag_finish(recs.data(), c->nranks, F, L, N, out_rhat, out_ess, out_tau, out_window_closed, out_rho);
  return MG_OK;
}

// Quantiles (quantiles.cu) of the union of every rank's block: one header exchange checks that n, D and the probs
// agree and gives the pooled size; the order statistics then run on every rank with their exchanges (brackets, region
// counts, select histograms) summed in rank order, so every rank gets the same bytes and one rank the single-GPU bits.
namespace mg {
int qt_check(mg_ctx *ctx, const void *x, int64_t n, int32_t D, int64_t C, const void *list, int32_t nq,
             const double *out);
int qt_prob_ranks(mg_ctx *ctx, const double *probs, int32_t nq, int64_t N, std::vector<int64_t> &ranks);
int qt_order_keys(mg_ctx *ctx, mg_comm *comm, const double *d_x, int64_t n, int32_t D, int64_t C, int64_t N,
                  const std::vector<int64_t> &ranks, std::vector<uint64_t> &keys, std::vector<int> &nan_f);
void qt_finish_quantiles(const double *probs, int32_t nq, int64_t N, int F, const std::vector<int64_t> &ranks,
                         const std::vector<uint64_t> &keys, const std::vector<int> &nan_f, double *out);
}  // namespace mg

extern "C" int mg_comm_quantiles(mg_comm *c, const double *d_samples_local, int64_t n, int32_t D, int64_t C_local,
                                 const double *probs, int32_t nq, double *out) {
  if (!c) return MG_EINVAL;
  mg_ctx *ctx = c->ctx;
  std::vector<int64_t> ranks;
  int rc = qt_check(ctx, d_samples_local, n, D, C_local, probs, nq, out);
  if (rc == MG_OK) rc = qt_prob_ranks(ctx, probs, nq, n * C_local, ranks);
  if (rc == MG_OK && cudaSetDevice(ctx->device) != cudaSuccess) rc = set_err(ctx, MG_ECUDA, "cuda: cannot select the device");
  // header: status, n, D, C_r, nq, the bits of probs
  const size_t H = 5 + MG_QUANT_MAX;
  std::vector<uint64_t> mine(H, 0), all(H * c->nranks);
  mine[0] = (uint64_t)rc;
  if (rc == MG_OK) {
    mine[1] = (uint64_t)n; mine[2] = (uint64_t)D; mine[3] = (uint64_t)C_local; mine[4] = (uint64_t)nq;
    memcpy(&mine[5], probs, sizeof(double) * nq);
  }
  const int rc2 = mg_comm_allgather(c, mine.data(), all.data(), (int64_t)(sizeof(uint64_t) * H));
  if (rc) return rc;
  if (rc2) return rc2;
  int64_t Ctot = 0;
  for (int r = 0; r < c->nranks; ++r) {
    const uint64_t *q = all.data() + H * r;
    if (q[0] != 0) return set_err(ctx, (int)q[0], "quantiles (comm): rank %d failed", r);
    if (!std::equal(q + 1, q + 3, mine.begin() + 1) || !std::equal(q + 4, q + H, mine.begin() + 4))
      return set_err(ctx, MG_EINVAL, "quantiles (comm): rank %d has another n, D or probs", r);
    Ctot += (int64_t)q[3];
  }
  const int64_t N = n * Ctot;
  if ((rc = qt_prob_ranks(ctx, probs, nq, N, ranks))) return rc;
  std::vector<uint64_t> keys;
  std::vector<int> nan_f;
  if ((rc = qt_order_keys(ctx, c, d_samples_local, n, D, C_local, N, ranks, keys, nan_f))) return rc;
  qt_finish_quantiles(probs, nq, N, D + 2, ranks, keys, nan_f, out);
  return MG_OK;
}
