// kdtree.cu -- Kd_tree.tree_of_objects (kd_tree.ml:155-175) built on the GPU,
// bit-exact with the reference rule, plus the Interpolate_pdf kernels
// (interpolate_pdf.ml:101-159).
//
// Build.  The reference recurses over OCaml lists and finds the pivot with a
// randomized quickselect (kd_tree.ml:69-86).  Here every coordinate is sorted
// ONCE (stable radix sort of order-preserving uint64 keys, one batch row per
// dimension), giving D index lists; a (D+1)-th list keeps the input order.
// The tree is then grown level by level on flat node arrays: inside a node's
// range every list holds the same points, so
//   tight bounds        = first / last element of each sorted list  (:96-110)
//   n/2-th order stat.  = element at offset n/2 of the split dim's list (:162-167)
//   <= pivot / > pivot  = a position threshold in that list (binary search)
//   max L, min R        = the two elements around the threshold (:170-171)
// and a level costs one flag pass plus one STABLE partition of the D+1 lists
// (tile reduce -> scan -> scatter), which keeps each list sorted and the
// input-order list in the reference's List.partition order (:168).
// Algorithmic traffic per level: (D+1) lists x N x ~18 B (SURVEY.md 8d gives
// (16 D + 16) N for a row-permuting build; index lists move 4-byte ids instead
// of 8 D-byte rows).  All kernels are HBM / L2-gather bound.
#include "kdtree.cuh"

#include <cmath>
#include <cstdlib>
#include <vector>

#include "common.cuh"
#include "radix_sort.cuh"
#include "scan.cuh"

namespace mg {

constexpr int KB = 256;  // generic block size

__global__ void check_finite_kernel(const double *__restrict__ x, int64_t n, int *__restrict__ flag) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    if (x[i] != x[i]) *flag = 1;
}

// keys[d][i] = ordered(pts[i][d]), vals[d][i] = i; row D of vals = identity.  A CTA transposes a tile of
// MK_TILE points through shared memory: the rows are read as one contiguous chunk, each dimension's keys are
// written as one contiguous run (a thread-per-(d, i) kernel reads with a stride of D doubles).
constexpr int MK_TILE = 128;
__global__ void __launch_bounds__(KB)
make_keys_kernel(const double *__restrict__ pts, int64_t N, int D, uint64_t *__restrict__ keys,
                 int32_t *__restrict__ vals) {
  extern __shared__ double mk_tile[];            // [MK_TILE][DP], DP odd: conflict-free column reads
  const int DP = D | 1;
  for (int64_t i0 = (int64_t)blockIdx.x * MK_TILE; i0 < N; i0 += (int64_t)gridDim.x * MK_TILE) {
    const int cnt = (int)((N - i0 < MK_TILE) ? N - i0 : MK_TILE);
    const double *src = pts + i0 * D;
    for (int k = threadIdx.x; k < cnt * D; k += KB) { const int r = k / D, c = k - r * D; mk_tile[r * DP + c] = src[k]; }
    __syncthreads();
    for (int k = threadIdx.x; k < D * MK_TILE; k += KB) {
      const int d = k / MK_TILE, r = k - d * MK_TILE;
      if (r < cnt) {
        keys[(int64_t)d * N + i0 + r] = f64_to_ordered(mk_tile[r * DP + d]);
        vals[(int64_t)d * N + i0 + r] = (int32_t)(i0 + r);
      }
    }
    for (int r = threadIdx.x; r < cnt; r += KB) vals[(int64_t)D * N + i0 + r] = (int32_t)(i0 + r);
    __syncthreads();
  }
}

// ---- sorting the D coordinate lists on a 32-bit window of the keys ------------------------------------------------
// The tree needs the index lists only, not the sorted keys.  The coordinates of one dimension usually share their
// top bytes (sign, most of the exponent), so the order is decided by the 32 bits below the highest byte that
// varies: four radix passes over (4-byte key, 4-byte index) pairs instead of seven over (8-byte key, index) pairs.
// Elements whose windows tie keep their input order (the passes are stable); tie_fix_kernel then orders each run of
// equal windows by the full key (stable insertion, runs are a handful of elements for continuous data, equal full
// keys -- duplicated samples -- stay in input order).  A run longer than KD_TIE_MAX raises a flag and the build
// falls back to the 64-bit sort.
constexpr int KD_TIE_MAX = 64;

__global__ void make_key32_kernel(const uint64_t *__restrict__ keys, int64_t N, const int *__restrict__ shift /* [D] */,
                                  uint32_t *__restrict__ key32) {
  const int d = blockIdx.y;
  const int sh = shift[d];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x)
    key32[(int64_t)d * N + i] = (uint32_t)(__ldcs(keys + (int64_t)d * N + i) >> sh);
}

__global__ void tie_fix_kernel(const uint32_t *__restrict__ key32 /* sorted */, int32_t *__restrict__ lists,
                               const uint64_t *__restrict__ keys /* [D][N] by point id */, int64_t N,
                               const int *__restrict__ shift, int *__restrict__ overflow) {
  const int d = blockIdx.y;
  if (shift[d] == 0) return;                      // the window holds every varying bit: ties are equal keys
  const uint32_t *k32 = key32 + (int64_t)d * N;
  int32_t *lst = lists + (int64_t)d * N;
  const uint64_t *kf = keys + (int64_t)d * N;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t k = k32[i];
    if ((i > 0 && k32[i - 1] == k) || i + 1 >= N || k32[i + 1] != k) continue;   // not the head of a run
    int L = 2;
    while (i + L < N && L <= KD_TIE_MAX && k32[i + L] == k) ++L;
    if (L > KD_TIE_MAX) { *overflow = 1; continue; }
    int32_t id[KD_TIE_MAX];
    uint64_t full[KD_TIE_MAX];
    for (int j = 0; j < L; ++j) { id[j] = lst[i + j]; full[j] = kf[id[j]]; }
    for (int j = 1; j < L; ++j) {                 // stable insertion sort by the full key
      const uint64_t fk = full[j]; const int32_t fi = id[j];
      int m = j - 1;
      while (m >= 0 && full[m] > fk) { full[m + 1] = full[m]; id[m + 1] = id[m]; --m; }
      full[m + 1] = fk; id[m + 1] = fi;
    }
    for (int j = 0; j < L; ++j) lst[i + j] = id[j];
  }
}

struct BuildArrays {
  const double *pts;
  int64_t N;
  int D, min_split;
  int32_t *begin, *end, *dim, *left, *spos;
  double *split;
  int *err;   // mg_ctx::d_devflag
};

__device__ __forceinline__ double key_at(const BuildArrays &a, const int32_t *lists, int d, int64_t pos) {
  return a.pts[(int64_t)lists[(int64_t)d * a.N + pos] * a.D + d];
}

// kd_tree.ml:155-175 for the nodes [lb, le) of one level.
__global__ void node_split_kernel(BuildArrays a, const int32_t *__restrict__ lists, int32_t lb, int32_t le,
                                  int32_t *__restrict__ flags /* [2][nlvl]: is_split, nR */) {
  const int32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  const int32_t nlvl = le - lb;
  if (k >= nlvl) return;
  const int32_t id = lb + k;
  const int32_t b = a.begin[id], e = a.end[id], n = e - b;
  int is_split = 0, nR = 0;
  a.dim[id] = -1; a.left[id] = -1; a.split[id] = 0.0; a.spos[id] = e;
  if (n > 1 && n >= a.min_split) {                   // :157-158 (+ truncation)
    // bounds_of_objects (:96-110) and longest_dim (:120-130): first strictly largest spread
    int sd = -1;
    double dx_max = neg_inf();
    bool all_eq = true;
    for (int d = 0; d < a.D; ++d) {
      const double lo = key_at(a, lists, d, b), hi = key_at(a, lists, d, e - 1);
      if (lo != hi) all_eq = false;
      const double dx = hi - lo;
      if (dx > dx_max) { sd = d; dx_max = dx; }
    }
    if (!all_eq && sd >= 0) {                        // :159-160 identical coordinates -> leaf
      const double v = key_at(a, lists, sd, b + n / 2);  // :162-167
      // first position with key > v (List.partition (<= pvt), :168)
      int32_t lo = b + n / 2, hi = e;
      while (lo < hi) { const int32_t mid = lo + ((hi - lo) >> 1); if (key_at(a, lists, sd, mid) > v) hi = mid; else lo = mid + 1; }
      int32_t pos = lo;
      if (pos == e) {                                // adjust_for_empty_split :150-152: L = {k < max}
        lo = b; hi = b + n / 2;
        while (lo < hi) { const int32_t mid = lo + ((hi - lo) >> 1); if (key_at(a, lists, sd, mid) < v) lo = mid + 1; else hi = mid; }
        pos = lo;
      }
      if (pos > b && pos < e) {
        const double lt_bound = key_at(a, lists, sd, pos - 1), gt_bound = key_at(a, lists, sd, pos);  // :170-171
        a.dim[id] = sd;
        a.split[id] = 0.5 * (lt_bound + gt_bound);  // split_bounds :113
        a.spos[id] = pos;
        is_split = 1; nR = e - pos;
      }
    }
  }
  flags[k] = is_split;
  flags[nlvl + k] = nR;
}

__global__ void make_children_kernel(BuildArrays a, int32_t lb, int32_t le, const int32_t *__restrict__ flags,
                                     const int32_t *__restrict__ scans, int32_t next_base) {
  const int32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= le - lb) return;
  if (!flags[k]) return;
  const int32_t id = lb + k;
  const int32_t L = next_base + 2 * scans[k];
  a.left[id] = L;
  a.begin[L] = a.begin[id]; a.end[L] = a.spos[id];
  a.begin[L + 1] = a.spos[id]; a.end[L + 1] = a.end[id];
}

// side[point] = 1 iff the point goes to the right child of its (splitting) node
__global__ void mark_side_kernel(BuildArrays a, const int32_t *__restrict__ lists, const int32_t *__restrict__ seg,
                                 int32_t lb, int32_t le, uint8_t *__restrict__ side) {
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < a.N; p += (int64_t)gridDim.x * blockDim.x) {
    const int32_t id = seg[p];
    if (id < lb || id >= le) continue;
    const int32_t sd = a.dim[id];
    if (sd < 0) continue;
    side[lists[(int64_t)sd * a.N + p]] = (p >= a.spos[id]) ? 1 : 0;
  }
}

// Stable partition of every list inside every splitting node (List.partition,
// kd_tree.ml:168) in ONE pass per level: a chained scan with decoupled
// look-back over the tiles of each list gives every element the number of
// right-going elements before it; combined with the per-node offsets (a scan
// over the level's nodes) that is its destination.  Tiles take their index from
// a per-list ticket counter, so a tile only ever waits for tiles that are
// already running.
constexpr unsigned long long LB_AGG = 1ull << 62, LB_PREFIX = 2ull << 62, LB_MASK = 3ull << 62;

#ifndef MG_PART_MINBLOCKS
#define MG_PART_MINBLOCKS 5   /* 48 registers: 5 CTAs per SM; gather-latency bound (tools/part_occupancy_sweep.sh: 4 -> 5 CTAs, Lebesgue 73 -> 67 ms) */
#endif
template <bool VEC>
__global__ void __launch_bounds__(SCAN_BLOCK, MG_PART_MINBLOCKS)
part_fused_kernel(BuildArrays a, const int32_t *__restrict__ lists_in, int32_t *__restrict__ lists_out,
                  const int32_t *__restrict__ seg_in, int32_t *__restrict__ seg_out,
                  const uint8_t *__restrict__ side, int32_t lb, int32_t le, int64_t ntiles,
                  unsigned long long *__restrict__ status /* [NL][ntiles] */, unsigned int *__restrict__ ticket /* [NL] */,
                  const int32_t *__restrict__ ebegin /* [nlvl] */) {
  const int l = blockIdx.y;
  __shared__ unsigned int s_tile;
  __shared__ int s_base;
  if (threadIdx.x == 0) s_tile = atomicAdd(ticket + l, 1u);
  __syncthreads();
  const int64_t t = s_tile;
  const int32_t *list = lists_in + (int64_t)l * a.N;
  int32_t *out = lists_out + (int64_t)l * a.N;
  unsigned long long *st = status + (int64_t)l * ntiles;
  const int64_t base = t * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
  int f[SCAN_ITEMS]; int32_t nd[SCAN_ITEMS], ix[SCAN_ITEMS];
  if (VEC && base + SCAN_ITEMS <= a.N) {
    const int4 *lp = reinterpret_cast<const int4 *>(list + base), *sp = reinterpret_cast<const int4 *>(seg_in + base);
#pragma unroll
    for (int v = 0; v < SCAN_ITEMS / 4; ++v) {
      const int4 li = __ldcs(lp + v), si = __ldg(sp + v);   // lists stream through (evict first): keep L2 for side[] and seg[]
      ix[4 * v] = li.x; ix[4 * v + 1] = li.y; ix[4 * v + 2] = li.z; ix[4 * v + 3] = li.w;
      nd[4 * v] = si.x; nd[4 * v + 1] = si.y; nd[4 * v + 2] = si.z; nd[4 * v + 3] = si.w;
    }
  } else {
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
      const int64_t p = base + k;
      ix[k] = 0; nd[k] = -1;
      if (p < a.N) { ix[k] = __ldcs(list + p); nd[k] = seg_in[p]; }
    }
  }
  int acc = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    const int32_t id = nd[k];
    const bool active = (base + k < a.N) && id >= lb && id < le && a.dim[id] >= 0;
    f[k] = active ? (int)side[ix[k]] : 0;
    if (!active && base + k < a.N) nd[k] = -1 - id;   // remember the node id of a pass-through element as -1-id
    if (base + k >= a.N) nd[k] = -1;
    acc += f[k];
  }
  int total;
  const int ex = block_exclusive_scan<SCAN_BLOCK>(acc, &total);
  if (threadIdx.x < 32) {                  // warp 0: publish the aggregate, then look back 32 tiles at a time
    const int lane = threadIdx.x;
    if (lane == 0 && t > 0) atomicExch(st + t, LB_AGG | (unsigned long long)total);
    unsigned long long prefix = 0;
    int64_t end = t - 1;                   // nearest predecessor not yet accounted for
    bool done = (t == 0);
    while (!done) {
      const int64_t k = end - lane;
      unsigned long long v = LB_PREFIX;    // tiles before the list start: prefix 0
      if (k >= 0) {
        unsigned spins = 0;
        do {
          v = *reinterpret_cast<volatile unsigned long long *>(st + k);
          if (!(v & LB_MASK) && ((++spins & 1023u) == 0u)) {   // bounded wait: flag the context instead of trapping
            if (spins > (1u << 28)) atomicExch(a.err, MG_DEVERR_KD_LOOKBACK);
            if (*reinterpret_cast<volatile int *>(a.err) != 0) v = LB_PREFIX;   // give up: the build reports MG_ECUDA
          }
        } while (!(v & LB_MASK));
      }
      const unsigned has_prefix = __ballot_sync(0xffffffffu, (v & LB_MASK) == LB_PREFIX);
      const int first = __ffs(has_prefix) - 1;            // nearest tile that already knows its inclusive prefix
      unsigned long long part = (first < 0 || lane <= first) ? (v & ~LB_MASK) : 0ull;
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) part += __shfl_xor_sync(0xffffffffu, part, off);
      prefix += part;
      if (first >= 0) done = true; else end -= 32;        // (first is always >= 0 once k runs below 0)
    }
    if (lane == 0) {
      __threadfence();
      atomicExch(st + t, LB_PREFIX | (prefix + (unsigned long long)total));
      s_base = (int)prefix;
    }
  }
  __syncthreads();
  int E = ex + s_base;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    const int64_t p = base + k;
    if (p < a.N) {
      if (nd[k] < 0) {                       // element of a node that does not split at this level
        __stcs(out + p, ix[k]);
        if (l == 0) seg_out[p] = -1 - nd[k];
      } else {
        const int32_t id = nd[k];
        const int32_t b = a.begin[id], sp = a.spos[id];
        const int32_t r = E - ebegin[id - lb];            // right-goers in [b, p)
        const int64_t dst = f[k] ? (int64_t)sp + r : (int64_t)b + (p - b) - r;
        __stcs(out + dst, ix[k]);
        if (l == 0) seg_out[p] = (p < sp) ? a.left[id] : a.left[id] + 1;
      }
    }
    E += f[k];
  }
}

__global__ void pack_nodes_kernel(BuildArrays a, int64_t nnodes, KdNode *__restrict__ nodes, int32_t *__restrict__ count,
                                  int32_t *__restrict__ begin_out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nnodes; i += (int64_t)gridDim.x * blockDim.x) {
    KdNode nd; nd.split = a.split[i]; nd.left = a.left[i]; nd.dim = a.dim[i];
    nodes[i] = nd; count[i] = a.end[i] - a.begin[i]; begin_out[i] = a.begin[i];
  }
}

__global__ void fill_i32_kernel(int32_t *p, int64_t n, int32_t v) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = v;
}

static inline unsigned grid1d(mg_ctx *ctx, int64_t n, int block = KB) {
  int64_t g = (n + block - 1) / block;
  const int64_t cap = (int64_t)ctx->sm_count * 16;
  if (g > cap) g = cap;
  return (unsigned)(g < 1 ? 1 : g);
}

KdHeader kd_layout(int64_t N, int D, int64_t node_cap, bool with_pts) {
  KdHeader h{};
  h.magic = KD_MAGIC; h.N = N; h.nnodes = node_cap; h.D = D;
  int64_t off = align256(sizeof(KdHeader));
  h.off_low = off; off = align256(off + 8 * D);
  h.off_high = off; off = align256(off + 8 * D);
  h.off_nodes = off; off = align256(off + 16 * node_cap);
  h.off_count = off; off = align256(off + 4 * node_cap);
  h.off_begin = off; off = align256(off + 4 * node_cap);
  h.off_perm = off; off = align256(off + 4 * N);
  h.off_pts = off; off = align256(off + (with_pts ? 8 * N * D : 0));
  h.nbytes = off;
  return h;
}

int kd_alloc(mg_ctx *ctx, const KdHeader &h, KdTreePtr *out) {
  // from the stream-ordered pool (kept cached between builds: a synchronous cudaMalloc / cudaFree of a 2 GB blob
  // costs 0.1-0.4 s now and then and synchronises the device)
  void *blob = nullptr;
  const cudaError_t e = cudaMallocAsync(&blob, (size_t)h.nbytes, ctx->stream);
  if (e != cudaSuccess) return set_err(ctx, MG_ENOMEM, "cuda: %s (kd-tree blob of %lld bytes)", cudaGetErrorString(e), (long long)h.nbytes);
  out->reset(new mg_kdtree);
  (*out)->ctx = ctx; (*out)->d_blob = blob; (*out)->h = h;
  return MG_OK;
}

int kd_finish(mg_ctx *ctx, KdTreePtr t, const double *low, const double *high, const double *d_pts, KdTreePtr *out) {
  cudaStream_t s = ctx->stream;
  const KdHeader &h = t->h;
  char *blob = (char *)t->d_blob;
  MG_CUDA(ctx, cudaMemcpyAsync(blob, &h, sizeof(KdHeader), cudaMemcpyHostToDevice, s));
  MG_CUDA(ctx, cudaMemcpyAsync(blob + h.off_low, low, 8 * h.D, cudaMemcpyHostToDevice, s));
  MG_CUDA(ctx, cudaMemcpyAsync(blob + h.off_high, high, 8 * h.D, cudaMemcpyHostToDevice, s));
  if (h.off_pts < h.nbytes) MG_CUDA(ctx, cudaMemcpyAsync(blob + h.off_pts, d_pts, 8 * h.N * h.D, cudaMemcpyDeviceToDevice, s));
  const cudaError_t e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) return set_err(ctx, MG_ECUDA, "cuda: %s (kd-tree build)", cudaGetErrorString(e));
  if (int rc = poll_device_error(ctx)) return rc;
  *out = std::move(t);
  return MG_OK;
}

static int build_tree_v1(mg_ctx *ctx, const double *d_pts, int64_t N, int D, const double *low, const double *high,
                         int min_split, bool with_pts, KdTreePtr *out);

int build_tree(mg_ctx *ctx, const double *d_pts, int64_t N, int D, const double *low, const double *high,
               int min_split, bool with_pts, KdTreePtr *out) {
  cudaStream_t s = ctx->stream;
  MG_REQUIRE(ctx, N >= 1, "tree_of_objects: no objects");
  MG_REQUIRE(ctx, D >= 1 && D <= 64, "kd-tree: dim must be in 1..64");
  MG_REQUIRE(ctx, N < (1LL << 30), "kd-tree: too many points for int32 indices");
  if (min_split < 2) min_split = 2;
  // The second builder (key columns moved level by level, subtrees finished in shared memory) hands inputs it is not
  // made for back to the first one (presorted index lists)
  const int rc = build_tree_v2(ctx, d_pts, N, D, low, high, min_split, with_pts, out);
  if (rc != MG_V2_FALLBACK) return rc;
  if (getenv("MCMC_GPU_DEBUG")) fprintf(stderr, "kd-tree: second builder handed the input back (ties / depth), first builder runs\n");
  // NaN coordinates are rejected (Pervasives.compare orders them, IEEE does not)
  DevBuf<int> d_flag;
  MG_CUDA(ctx, d_flag.alloc(1, s));
  MG_CUDA(ctx, cudaMemsetAsync(d_flag.get(), 0, sizeof(int), s));
  check_finite_kernel<<<grid1d(ctx, N * D), KB, 0, s>>>(d_pts, N * D, d_flag.get());
  MG_CHECK_LAUNCH(ctx);
  int h_flag = 0;
  MG_CUDA(ctx, cudaMemcpyAsync(&h_flag, d_flag.get(), sizeof(int), cudaMemcpyDeviceToHost, s));
  MG_CUDA(ctx, cudaStreamSynchronize(s));
  MG_REQUIRE(ctx, h_flag == 0, "kd-tree: NaN coordinate");
  return build_tree_v1(ctx, d_pts, N, D, low, high, min_split, with_pts, out);
}

static int build_tree_v1(mg_ctx *ctx, const double *d_pts, int64_t N, int D, const double *low, const double *high,
                         int min_split, bool with_pts, KdTreePtr *out) {
  cudaStream_t s = ctx->stream;
  time_begin(ctx);
  kt_reset(ctx, N % 4 == 0 ? (const void *)part_fused_kernel<true> : (const void *)part_fused_kernel<false>);
  const int NL = D + 1;  // D sorted lists + the input-order list
  DevBuf<int32_t> listsA, listsB, segA, segB, nd_begin, nd_end, nd_dim, nd_left, nd_spos, flags, scans, tsum, totals;
  DevBuf<double> nd_split;
  DevBuf<uint8_t> side;
  MG_CUDA(ctx, listsA.alloc((size_t)NL * N, s));
  MG_CUDA(ctx, listsB.alloc((size_t)NL * N, s));
  {
    DevBuf<uint64_t> keys;
    MG_CUDA(ctx, keys.alloc((size_t)D * N, s));
    const size_t mk_smem = (size_t)MK_TILE * (D | 1) * sizeof(double);
    if (mk_smem > 48 * 1024)
      MG_CUDA(ctx, cudaFuncSetAttribute(make_keys_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mk_smem));
    make_keys_kernel<<<grid1d(ctx, (N + MK_TILE - 1) / MK_TILE * KB), KB, mk_smem, s>>>(d_pts, N, D, keys.get(), listsA.get());
    MG_CHECK_LAUNCH(ctx);
    int rc;
    bool sorted = false;
    if (N >= 65536) {
      // 32-bit window under the highest varying byte of each dimension (see make_key32_kernel)
      std::vector<unsigned char> cb;
      std::vector<double> veff;
      if ((rc = radix_constant_bytes<uint64_t>(ctx, keys.get(), N, D, cb, &veff))) return rc;
      std::vector<int> h_shift(D, 0);
      bool window_ok = true;
      for (int d = 0; d < D; ++d) {
        int top = 0;
        for (int p = 7; p >= 0; --p) if (!cb[(size_t)d * 8 + p]) { top = p; break; }
        h_shift[d] = 8 * std::max(0, top - 3);
        // Equal windows must be rare or the repair pass touches millions of runs.  Distinct windows are estimated
        // from the byte histograms as the product of the effective number of values (n^2 / sum count^2) of the
        // window's four bytes; N points then give ~N^2 / (2 distinct) tied pairs, accepted up to N / 16.  Coordinates whose sign or high exponent bits vary (top byte 7: only 20 mantissa bits are left in
        // the window) fail this at 1e7 points and take the 64-bit sort.
        if (h_shift[d] > 0) {
          double distinct = 1.0;
          for (int p = top - 3; p <= top; ++p) distinct *= veff[(size_t)d * 8 + p];
          if ((double)N * (double)N / (2.0 * distinct) > (double)N / 16.0) window_ok = false;
        }
      }
      if (window_ok) {
      DevBuf<int> d_shift, d_over;
      DevBuf<uint32_t> key32;
      MG_CUDA(ctx, upload(d_shift, h_shift.data(), (size_t)D, s));
      MG_CUDA(ctx, d_over.alloc(1, s));
      MG_CUDA(ctx, cudaMemsetAsync(d_over.get(), 0, sizeof(int), s));
      MG_CUDA(ctx, key32.alloc((size_t)D * N, s));
      make_key32_kernel<<<dim3(grid1d(ctx, N), (unsigned)D), KB, 0, s>>>(keys.get(), N, d_shift.get(), key32.get());
      MG_CHECK_LAUNCH(ctx);
      if ((rc = radix_sort_pairs_t<uint32_t>(ctx, key32.get(), listsA.get(), N, D))) return rc;
      tie_fix_kernel<<<dim3(grid1d(ctx, N), (unsigned)D), KB, 0, s>>>(key32.get(), listsA.get(), keys.get(), N, d_shift.get(), d_over.get());
      MG_CHECK_LAUNCH(ctx);
      int h_over = 0;
      MG_CUDA(ctx, cudaMemcpyAsync(&h_over, d_over.get(), sizeof(int), cudaMemcpyDeviceToHost, s));
      MG_CUDA(ctx, cudaStreamSynchronize(s));
      sorted = (h_over == 0);
      if (!sorted) {   // a long run of equal windows: start over with the full keys
        make_keys_kernel<<<grid1d(ctx, (N + MK_TILE - 1) / MK_TILE * KB), KB, mk_smem, s>>>(d_pts, N, D, keys.get(), listsA.get());
        MG_CHECK_LAUNCH(ctx);
      }
      }
    }
    if (!sorted && (rc = radix_sort_pairs(ctx, keys.get(), listsA.get(), N, D))) return rc;
  }
  const int64_t cap = 2 * N;
  MG_CUDA(ctx, nd_begin.alloc(cap, s)); MG_CUDA(ctx, nd_end.alloc(cap, s)); MG_CUDA(ctx, nd_dim.alloc(cap, s));
  MG_CUDA(ctx, nd_left.alloc(cap, s)); MG_CUDA(ctx, nd_spos.alloc(cap, s)); MG_CUDA(ctx, nd_split.alloc(cap, s));
  MG_CUDA(ctx, segA.alloc(N, s)); MG_CUDA(ctx, segB.alloc(N, s)); MG_CUDA(ctx, side.alloc(N, s));
  MG_CUDA(ctx, cudaMemsetAsync(segA.get(), 0, sizeof(int32_t) * N, s));
  MG_CUDA(ctx, cudaMemsetAsync(side.get(), 0, N, s));
  const int64_t ntiles = (N + SCAN_TILE - 1) / SCAN_TILE;
  DevBuf<unsigned long long> lb_status;
  DevBuf<unsigned int> lb_ticket;
  MG_CUDA(ctx, lb_status.alloc((size_t)NL * ntiles, s));
  MG_CUDA(ctx, lb_ticket.alloc((size_t)NL, s));
  MG_CUDA(ctx, totals.alloc(2, s));
  BuildArrays a{d_pts, N, D, min_split, nd_begin.get(), nd_end.get(), nd_dim.get(), nd_left.get(), nd_spos.get(),
                nd_split.get(), ctx->d_devflag};
  {
    const int32_t zero = 0, n32 = (int32_t)N;
    MG_CUDA(ctx, cudaMemcpyAsync(nd_begin.get(), &zero, 4, cudaMemcpyHostToDevice, s));
    MG_CUDA(ctx, cudaMemcpyAsync(nd_end.get(), &n32, 4, cudaMemcpyHostToDevice, s));
    MG_CUDA(ctx, cudaStreamSynchronize(s));
  }
  int32_t *lin = listsA.get(), *lout = listsB.get(), *sin = segA.get(), *sout = segB.get();
  int64_t lb = 0, le = 1, nnodes = 1;
  int nlevels = 0;
  int64_t flags_cap = 0;
  DevBuf<int32_t> scan_tmp;
  std::vector<int32_t> level_begin;
  for (;;) {
    ++nlevels;
    level_begin.push_back((int32_t)lb);
    if (nlevels > 100000) return set_err(ctx, MG_EFAIL, "kd-tree: too many levels");
    const int64_t nlvl = le - lb;
    if (2 * nlvl > flags_cap) {
      flags_cap = 2 * nlvl * 2;
      MG_CUDA(ctx, flags.alloc((size_t)flags_cap, s));
      MG_CUDA(ctx, scans.alloc((size_t)flags_cap, s));
      MG_CUDA(ctx, scan_tmp.alloc((size_t)scan_tmp_elems(flags_cap / 2, 2) + 2, s));
    }
    node_split_kernel<<<(unsigned)((nlvl + 127) / 128), 128, 0, s>>>(a, lin, (int32_t)lb, (int32_t)le, flags.get());
    MG_CHECK_LAUNCH(ctx);
    int rc = exclusive_scan_i32(ctx, flags.get(), scans.get(), nlvl, 2, scan_tmp.get(), totals.get());
    if (rc) return rc;
    int32_t h_tot[2];
    MG_CUDA(ctx, cudaMemcpyAsync(h_tot, totals.get(), 8, cudaMemcpyDeviceToHost, s));
    MG_CUDA(ctx, cudaStreamSynchronize(s));
    const int64_t nsplit = h_tot[0];
    if (nsplit == 0) break;
    if (nnodes + 2 * nsplit > cap) return set_err(ctx, MG_EFAIL, "kd-tree: node capacity exceeded");
    make_children_kernel<<<(unsigned)((nlvl + 127) / 128), 128, 0, s>>>(a, (int32_t)lb, (int32_t)le, flags.get(),
                                                                       scans.get(), (int32_t)nnodes);
    MG_CHECK_LAUNCH(ctx);
    mark_side_kernel<<<grid1d(ctx, N), KB, 0, s>>>(a, lin, sin, (int32_t)lb, (int32_t)le, side.get());
    MG_CHECK_LAUNCH(ctx);
    dim3 pgrid((unsigned)ntiles, (unsigned)NL);
    MG_CUDA(ctx, cudaMemsetAsync(lb_status.get(), 0, sizeof(unsigned long long) * NL * ntiles, s));
    MG_CUDA(ctx, cudaMemsetAsync(lb_ticket.get(), 0, sizeof(unsigned int) * NL, s));
    kt_start(ctx);
    if (N % 4 == 0)
      part_fused_kernel<true><<<pgrid, SCAN_BLOCK, 0, s>>>(a, lin, lout, sin, sout, side.get(), (int32_t)lb, (int32_t)le,
                                                           ntiles, lb_status.get(), lb_ticket.get(), scans.get() + nlvl);
    else
      part_fused_kernel<false><<<pgrid, SCAN_BLOCK, 0, s>>>(a, lin, lout, sin, sout, side.get(), (int32_t)lb, (int32_t)le,
                                                            ntiles, lb_status.get(), lb_ticket.get(), scans.get() + nlvl);
    kt_stop(ctx);
    MG_CHECK_LAUNCH(ctx);
    std::swap(lin, lout); std::swap(sin, sout);
    lb = le; le = nnodes + 2 * nsplit; nnodes = le;
  }
  level_begin.push_back((int32_t)nnodes);
  // ---- the blob: nodes, counts, begins and the order of the points are this builder's ------------------------------
  KdTreePtr t;
  if (int rc = kd_alloc(ctx, kd_layout(N, D, nnodes, with_pts), &t)) return rc;
  t->h.nlevels = nlevels; t->h.min_split = min_split; t->level_begin = std::move(level_begin);
  const KdHeader &h = t->h;
  char *blob = (char *)t->d_blob;
  pack_nodes_kernel<<<grid1d(ctx, nnodes), KB, 0, s>>>(a, nnodes, (KdNode *)(blob + h.off_nodes),
                                                      (int32_t *)(blob + h.off_count), (int32_t *)(blob + h.off_begin));
  MG_CHECK_LAUNCH(ctx);
  MG_CUDA(ctx, cudaMemcpyAsync(blob + h.off_perm, lin + (int64_t)D * N, 4 * N, cudaMemcpyDeviceToDevice, s));
  time_end(ctx);
  return kd_finish(ctx, std::move(t), low, high, d_pts, out);
}

// ---- Interpolate_pdf kernels ------------------------------------------------

__global__ void jump_prob_kernel(KdView t, const double *__restrict__ q, int64_t M, int nstop,
                                 double *__restrict__ out_prob, int32_t *__restrict__ out_node) {
  extern __shared__ double smem[];
  const KdScratch s = kd_scratch(smem, t.D);
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  for (int d = 0; d < t.D; ++d) s.Q(d) = q[i * t.D + d];
  int32_t node;
  const double p = kd_jump_prob(t, s, nstop, &node);
  if (out_prob) out_prob[i] = p;
  if (out_node) out_node[i] = node;
}

__global__ void draw_kernel(KdView t, CallKey key, uint64_t draw_offset, int64_t M, int nstop,
                            double *__restrict__ out, int *__restrict__ fail) {
  extern __shared__ double smem[];
  const KdScratch s = kd_scratch(smem, t.D);
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  Rng r(key, P_DRAW, draw_offset + (uint64_t)i, 0);
  if (!kd_draw(t, s, nstop, r)) { *fail = 1; for (int d = 0; d < t.D; ++d) out[i * t.D + d] = qnan(); return; }
  for (int d = 0; d < t.D; ++d) out[i * t.D + d] = s.Q(d);
}

// the cell (box, count, node) that find_cell reaches from every stored point: KdView::dcache
__global__ void draw_cache_kernel(KdView t, double *__restrict__ rec) {
  extern __shared__ double smem[];
  const KdScratch s = kd_scratch(smem, t.D);
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= t.N) return;
  for (int d = 0; d < t.D; ++d) s.Q(d) = t.pts[k * t.D + d];
  const int32_t id = kd_descend(t, s, 0);
  double *o = rec + k * (2 * t.D + 2);
  for (int d = 0; d < t.D; ++d) { o[d] = s.LO(d); o[t.D + d] = s.HI(d); }
  o[2 * t.D] = (double)__ldg(t.count + id);
  o[2 * t.D + 1] = (double)id;
}

static int query_block(int D) { return D <= 16 ? 128 : (D <= 32 ? 64 : 32); }

template <class K>
static int prep_smem(mg_ctx *ctx, K kernel, size_t bytes) {
  if (bytes > 48 * 1024) MG_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return MG_OK;
}

}  // namespace mg

using namespace mg;

extern "C" int mg_kdtree_build_dev(mg_ctx *ctx, const double *d_pts, int64_t N, int32_t D, const double *low,
                                   const double *high, int32_t min_split, mg_kdtree **out) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, d_pts && low && high && out, "kd-tree: null argument");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  KdTreePtr t;
  const int rc = build_tree(ctx, d_pts, N, D, low, high, min_split, true, &t);
  *out = t.release();
  return rc;
}

extern "C" int mg_kdtree_build(mg_ctx *ctx, const double *pts, int64_t N, int32_t D, const double *low,
                               const double *high, int32_t min_split, mg_kdtree **out) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, pts && low && high && out, "kd-tree: null argument");
  MG_REQUIRE(ctx, N >= 1, "tree_of_objects: no objects");
  MG_REQUIRE(ctx, D >= 1 && D <= 64, "kd-tree: dim must be in 1..64");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  DevBuf<double> d_pts;
  MG_CUDA(ctx, upload(d_pts, pts, (size_t)N * D, ctx->stream));
  KdTreePtr t;
  const int rc = build_tree(ctx, d_pts.get(), N, D, low, high, min_split, true, &t);
  *out = t.release();
  return rc;
}

extern "C" void mg_kdtree_destroy(mg_kdtree *t) {
  if (!t) return;
  if (t->ctx) { cudaSetDevice(t->ctx->device); cudaStreamSynchronize(t->ctx->stream); }
  if (t->owns_blob && t->d_blob) { if (t->ctx) cudaFreeAsync(t->d_blob, t->ctx->stream); else cudaFree(t->d_blob); }
  if (t->d_draw_cache) { if (t->ctx) cudaFreeAsync(t->d_draw_cache, t->ctx->stream); else cudaFree(t->d_draw_cache); }
  delete t;
}

// Interp.draw picks a STORED point and locates its cell by descent (interpolate_pdf.ml:114-119).  That cell depends on
// the point only, so it can be located once: this builds, for every stored point, the box / count / node the
// descent reaches (N x (2 D + 2) doubles, outside the blob; after a broadcast every rank builds its own).  Draws at
// leaf level (nstop = 0) then gather one record instead of walking ~log2 N dependent nodes; the values are the
// descent's own, so draws and densities do not change by a bit.
extern "C" int mg_kdtree_enable_draw_cache(mg_kdtree *t) {
  if (!t || !t->ctx) return MG_EINVAL;
  mg_ctx *ctx = t->ctx;
  if (t->d_draw_cache) return MG_OK;
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  const int D = t->h.D;
  const size_t bytes = (size_t)t->h.N * (2 * D + 2) * sizeof(double);
  double *rec = nullptr;
  cudaError_t e = cudaMallocAsync((void **)&rec, bytes, ctx->stream);
  if (e != cudaSuccess) return set_err(ctx, MG_ENOMEM, "cuda: %s (draw cache of %zu bytes)", cudaGetErrorString(e), bytes);
  const int block = query_block(D);
  const size_t smem = kd_scratch_bytes(D, block);
  int rc = prep_smem(ctx, draw_cache_kernel, smem);
  if (rc) { cudaFreeAsync(rec, ctx->stream); return rc; }
  draw_cache_kernel<<<(unsigned)((t->h.N + block - 1) / block), block, smem, ctx->stream>>>(t->view(), rec);
  ctx->launches++;
  e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) { cudaFreeAsync(rec, ctx->stream); return set_err(ctx, MG_ECUDA, "cuda: %s (draw cache)", cudaGetErrorString(e)); }
  t->d_draw_cache = rec;
  return MG_OK;
}

extern "C" int mg_kdtree_info(const mg_kdtree *t, int64_t *npoints, int32_t *dim, int64_t *nnodes, int32_t *nlevels) {
  if (!t) return MG_EINVAL;
  if (npoints) *npoints = t->h.N;
  if (dim) *dim = t->h.D;
  if (nnodes) *nnodes = t->h.nnodes;
  if (nlevels) *nlevels = t->h.nlevels;
  return MG_OK;
}

extern "C" int mg_kdtree_export(const mg_kdtree *t, int32_t *split_dim, double *split_val, int32_t *left,
                                int32_t *begin, int32_t *end, int32_t *perm) {
  if (!t) return MG_EINVAL;
  mg_ctx *ctx = t->ctx;
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  const int64_t nn = t->h.nnodes;
  const char *blob = (const char *)t->d_blob;
  std::vector<KdNode> nodes((size_t)nn);
  std::vector<int32_t> count((size_t)nn), b((size_t)nn);
  MG_CUDA(ctx, cudaMemcpyAsync(nodes.data(), blob + t->h.off_nodes, 16 * nn, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CUDA(ctx, cudaMemcpyAsync(count.data(), blob + t->h.off_count, 4 * nn, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CUDA(ctx, cudaMemcpyAsync(b.data(), blob + t->h.off_begin, 4 * nn, cudaMemcpyDeviceToHost, ctx->stream));
  if (perm) MG_CUDA(ctx, cudaMemcpyAsync(perm, blob + t->h.off_perm, 4 * t->h.N, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int64_t i = 0; i < nn; ++i) {
    if (split_dim) split_dim[i] = nodes[i].dim;
    if (split_val) split_val[i] = nodes[i].split;
    if (left) left[i] = nodes[i].left;
    if (begin) begin[i] = b[i];
    if (end) end[i] = b[i] + count[i];
  }
  return MG_OK;
}

extern "C" int mg_kdtree_blob_size(const mg_kdtree *t, int64_t *nbytes) {
  if (!t || !nbytes) return MG_EINVAL;
  *nbytes = t->h.nbytes;
  return MG_OK;
}
extern "C" int mg_kdtree_blob_dev(const mg_kdtree *t, void **d_blob) {
  if (!t || !d_blob) return MG_EINVAL;
  *d_blob = t->d_blob;
  return MG_OK;
}
// A blob arrives from another process (NCCL broadcast): nothing in it is trusted before the kernels index with it.
int mg::validate_blob_header(mg_ctx *ctx, const KdHeader &h) {
  MG_REQUIRE(ctx, h.magic == KD_MAGIC, "kd-tree blob: bad magic");
  MG_REQUIRE(ctx, h.D >= 1 && h.D <= 64 && h.N >= 1 && h.N < (1LL << 30), "kd-tree blob: bad N / D");
  MG_REQUIRE(ctx, h.nnodes >= 1 && h.nnodes <= 2 * h.N, "kd-tree blob: bad node count");
  const int64_t off[8] = {h.off_low, h.off_high, h.off_nodes, h.off_count, h.off_begin, h.off_perm, h.off_pts, h.nbytes};
  const int64_t need[7] = {8LL * h.D, 8LL * h.D, 16 * h.nnodes, 4 * h.nnodes, 4 * h.nnodes, 4 * h.N, 8 * h.N * h.D};
  MG_REQUIRE(ctx, off[0] >= (int64_t)sizeof(KdHeader), "kd-tree blob: sections overlap the header");
  for (int i = 0; i < 7; ++i)
    MG_REQUIRE(ctx, (off[i] & 255) == 0 && off[i] + need[i] <= off[i + 1], "kd-tree blob: section %d out of bounds or misaligned", i);
  return MG_OK;
}

extern "C" int mg_kdtree_from_blob_dev(mg_ctx *ctx, const void *d_blob, int64_t nbytes, mg_kdtree **out) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, d_blob && out && nbytes >= (int64_t)sizeof(KdHeader), "kd-tree: bad blob");
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  KdHeader h;
  MG_CUDA(ctx, cudaMemcpyAsync(&h, d_blob, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  MG_REQUIRE(ctx, h.magic == KD_MAGIC && h.nbytes == nbytes, "kd-tree: blob header mismatch");
  KdTreePtr t;
  int rc = validate_blob_header(ctx, h);
  if (rc == MG_OK) rc = kd_alloc(ctx, h, &t);
  if (rc) return rc;
  cudaError_t e = cudaMemcpyAsync(t->d_blob, d_blob, (size_t)nbytes, cudaMemcpyDeviceToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) return set_err(ctx, MG_ECUDA, "cuda: %s (kd-tree from blob)", cudaGetErrorString(e));
  *out = t.release();
  return MG_OK;
}

extern "C" double mg_bounds_volume(const double *low, const double *high, int32_t D) {
  double v = 1.0;  // kd_tree.ml:177-182
  for (int i = 0; i < D; ++i) v = v * (high[i] - low[i]);
  return v + 0.0;
}

extern "C" int mg_interp_jump_prob_dev(mg_ctx *ctx, const mg_kdtree *t, const double *d_q, int64_t M, int32_t nstop,
                                       double *d_out_prob, int32_t *d_out_node) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, t && d_q && M >= 0, "jump_prob: bad arguments");
  if (M == 0) return MG_OK;
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  const int block = query_block(t->h.D);
  const size_t smem = kd_scratch_bytes(t->h.D, block);
  int rc = prep_smem(ctx, jump_prob_kernel, smem);
  if (rc) return rc;
  time_begin(ctx);
  jump_prob_kernel<<<(unsigned)((M + block - 1) / block), block, smem, ctx->stream>>>(t->view(), d_q, M, nstop,
                                                                                      d_out_prob, d_out_node);
  MG_CHECK_LAUNCH(ctx);
  time_end(ctx);
  return MG_OK;
}

static int interp_query_host(mg_ctx *ctx, const mg_kdtree *t, const double *q, int64_t M, int32_t nstop,
                             double *out_prob, int32_t *out_node, const char *what) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, t && q && M >= 0, "%s: bad arguments", what);
  if (M == 0) return MG_OK;
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  DevBuf<double> d_q, d_p;
  DevBuf<int32_t> d_n;
  MG_CUDA(ctx, upload(d_q, q, (size_t)M * t->h.D, ctx->stream));
  MG_CUDA(ctx, d_p.alloc(M, ctx->stream));
  MG_CUDA(ctx, d_n.alloc(M, ctx->stream));
  int rc = mg_interp_jump_prob_dev(ctx, t, d_q.get(), M, nstop, d_p.get(), d_n.get());
  if (rc) return rc;
  std::vector<int32_t> nodes((size_t)M);
  if (out_prob) MG_CUDA(ctx, cudaMemcpyAsync(out_prob, d_p.get(), 8 * M, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CUDA(ctx, cudaMemcpyAsync(nodes.data(), d_n.get(), 4 * M, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  bool bad = false;
  for (int64_t i = 0; i < M; ++i) { if (out_node) out_node[i] = nodes[i]; if (nodes[i] < 0) bad = true; }
  if (bad) return set_err(ctx, MG_EFAIL, "%s: encountered empty tree!", what);  // interpolate_pdf.ml:124,149
  return MG_OK;
}

extern "C" int mg_interp_find_cell(mg_ctx *ctx, const mg_kdtree *t, const double *q, int64_t M, int32_t nstop,
                                   int32_t *out_node) {
  return interp_query_host(ctx, t, q, M, nstop, nullptr, out_node, "find_cell");
}
extern "C" int mg_interp_jump_prob(mg_ctx *ctx, const mg_kdtree *t, const double *q, int64_t M, int32_t nstop,
                                   double *out_prob) {
  return interp_query_host(ctx, t, q, M, nstop, out_prob, nullptr, "jump_prob_high_level");
}

extern "C" int mg_interp_draw_dev(mg_ctx *ctx, const mg_kdtree *t, int64_t M, int32_t nstop, double *d_out) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, t && d_out && M >= 0, "draw: bad arguments");
  if (M == 0) return MG_OK;
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  const int block = query_block(t->h.D);
  const size_t smem = kd_scratch_bytes(t->h.D, block);
  int rc = prep_smem(ctx, draw_kernel, smem);
  if (rc) return rc;
  DevBuf<int> d_fail;
  MG_CUDA(ctx, d_fail.alloc(1, ctx->stream));
  MG_CUDA(ctx, cudaMemsetAsync(d_fail.get(), 0, sizeof(int), ctx->stream));
  const CallKey key = next_key(ctx);
  time_begin(ctx);
  draw_kernel<<<(unsigned)((M + block - 1) / block), block, smem, ctx->stream>>>(t->view(), key, 0, M, nstop, d_out,
                                                                                 d_fail.get());
  MG_CHECK_LAUNCH(ctx);
  time_end(ctx);
  int h_fail = 0;
  MG_CUDA(ctx, cudaMemcpyAsync(&h_fail, d_fail.get(), sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  MG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (h_fail) return set_err(ctx, MG_EFAIL, "draw_high_level: encountered empty tree!");
  return MG_OK;
}

extern "C" int mg_interp_draw(mg_ctx *ctx, const mg_kdtree *t, int64_t M, int32_t nstop, double *out) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, t && out && M >= 0, "draw: bad arguments");
  if (M == 0) return MG_OK;
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  DevBuf<double> d_out;
  MG_CUDA(ctx, d_out.alloc((size_t)M * t->h.D, ctx->stream));
  int rc = mg_interp_draw_dev(ctx, t, M, nstop, d_out.get());
  if (rc) return rc;
  MG_CUDA(ctx, cudaMemcpyAsync(out, d_out.get(), 8 * M * t->h.D, cudaMemcpyDeviceToHost, ctx->stream));
  MG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MG_OK;
}
