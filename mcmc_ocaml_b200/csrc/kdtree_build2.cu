// kdtree_build2.cu -- Kd_tree.tree_of_objects (kd_tree.ml:155-175), second builder: no presort.
//
// The first builder (kdtree.cu) sorts every coordinate once and then carries D + 1 index lists through one stable
// partition per level; its partition pass is bound by the L2 gathers of a per-point side flag (14 % of HBM).
// This builder moves the DATA instead of index lists, so that every pass is a coalesced stream:
//
//   top phase (level-synchronous, nodes larger than NMAX points).  The points live as D key columns
//   K[d][position] (order-preserving uint64 keys) in the current node order.  Per level:
//     bounds    per-node min / max of every column: the root's come with the key pass, the children's are found by
//               the scatter pass of their parent                          (bounds_of_objects :96-110)
//     node      first strictly largest spread -> split dimension          (longest_dim :120-130), leaves (:157-160)
//     select    the n/2-th order statistic of the split column by MSB-first radix select on the keys: 8-bit digits
//               from the highest bit in which the node's keys differ, over as soon as the order statistic is alone in
//               its bin (the scatter only compares keys with it)           (find_ith :69-86 -- its RESULT)
//     scatter   stable partition (<= pivot | > pivot, or < max | >= max after adjust_for_empty_split :144-153) of
//               all D columns + the index column by one chained scan with decoupled look-back; the same pass
//               finds max L / min R for the split plane 0.5 (max L + min R)  (:113,170-172) and the children's bounds
//   Traffic per level ~ (2 * 8 D + 16) N bytes for the scatter -- SURVEY.md 8d's figure for a row-permuting build --
//   plus 3-4 x 12 N for the select.  A truncated build stops the level loop where no node can split any more.
//
//   bottom phase (one CTA per subtree of <= NMAX points).  The subtree's raw key columns live in shared memory and are
//   never moved: nodes are ranges of a 16-bit local-id list.  One warp per node (all warps for the bounds of a level's
//   few large nodes, one lane per dimension for nodes of <= 128 points, one thread per node of <= 8 points): bounds,
//   split dimension, radix select on the split column finished by ranking <= 32 candidates, stable partition of the
//   ids by ballots.  Nodes are written with subtree-local numbers; a scan over (subtree, level) node counts turns them
//   into the breadth-first numbers of the whole tree (children adjacent), which is the numbering of the first
//   builder and of the oracle.  The builder keeps the first node of every level (mg_kdtree::level_begin) for the
//   distributed build (comm.cu).
//
// Inputs on which the top phase cannot reach subtrees of <= NMAX points within its level budget (heavy ties), or
// whose subtrees are deeper than the local level budget, return MG_V2_FALLBACK and take the first builder.
#include <algorithm>
#include <cstdlib>
#include <vector>

#include "common.cuh"
#include "kdtree.cuh"
#include "radix_sort.cuh"
#include "scan.cuh"

namespace mg {

constexpr int V2_MAXLEV = 72;        // top-phase levels (2^30 points, NMAX >= 1024: 20 + extra)
constexpr int V2_MAXL = 64;          // levels inside one subtree
constexpr int V2_EXTRA = 3;          // top levels beyond the predicted hand-over level before giving up
constexpr int V2_TB = 256, V2_ITEMS = 8, V2_TILE = V2_TB * V2_ITEMS;

struct V2Level { int32_t lb, le; };
struct V2Info {
  V2Level lvl[V2_MAXLEV + 1];
  int32_t maxsize[V2_MAXLEV + 1];   // largest node of each level
  int32_t nnodes;                   // nodes created so far
  int32_t nlevels;                  // levels holding at least one node
  int32_t sel_active;               // nodes of the current level whose select is still running
  int32_t overflow;                 // a capacity was exceeded
};
// shift: position of the next 8-bit digit (< 0: no (more) select work); dim: split dimension in the low byte, and in the
// second byte the lowest key bit already decided (64: none) -- digits start at the highest bit in which the node's keys
// differ, not at a byte boundary, so the first pass already resolves eight bits
struct V2Sel { uint64_t prefix; int32_t shift; int32_t dim; };

struct V2Top {
  int64_t N; int D, min_split; int32_t LC, cap;
  V2Info *info;
  int32_t *nb, *ne, *ndim, *nleft, *nspos; double *nsplit;      // node arrays [cap]
  uint64_t *lo, *hi;                                            // [LC][D] bounds of the current level's nodes
  V2Sel *sel; int32_t *kth, *below; uint32_t *hist;             // [LC], [LC][256]
  uint64_t *v, *maxL, *minR; uint8_t *fix; int32_t *nR, *ebegin; // [LC]
};

__device__ __forceinline__ double ordered_to_f64(uint64_t k) {
  const uint64_t b = (k >> 63) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k;
  return __longlong_as_double((long long)b);
}

__device__ __forceinline__ uint64_t warp_min_u64(uint64_t v);
__device__ __forceinline__ uint64_t warp_max_u64(uint64_t v);

// ---- key columns ----------------------------------------------------------------------------------------------
constexpr int V2_MK = 128;
// Rows -> key columns through a shared-memory transpose; the same pass finds the root's bounds (bounds_of_objects of
// level 0) and rejects NaN coordinates, so the data are read once for all three.
__global__ void __launch_bounds__(256)
v2_make_keys_kernel(const double *__restrict__ pts, int64_t N, int D, uint64_t *__restrict__ K, int32_t *__restrict__ perm,
                    int32_t *__restrict__ seg, uint64_t *__restrict__ root_lo, uint64_t *__restrict__ root_hi, int *__restrict__ nan_flag) {
  extern __shared__ double v2_mk_tile[];          // [V2_MK][DP], DP odd
  __shared__ unsigned long long s_lo[64], s_hi[64];
  const int DP = D | 1;
  if (threadIdx.x < 64) { s_lo[threadIdx.x] = ~0ull; s_hi[threadIdx.x] = 0ull; }
  bool bad = false;
  for (int64_t i0 = (int64_t)blockIdx.x * V2_MK; i0 < N; i0 += (int64_t)gridDim.x * V2_MK) {
    const int cnt = (int)((N - i0 < V2_MK) ? N - i0 : V2_MK);
    const double *src = pts + i0 * D;
    __syncthreads();
    for (int k = threadIdx.x; k < cnt * D; k += 256) { const int r = k / D, c = k - r * D; const double v = src[k]; bad |= (v != v); v2_mk_tile[r * DP + c] = v; }
    __syncthreads();
    for (int k = threadIdx.x; k < D * V2_MK; k += 256) {      // a warp covers 32 consecutive points of ONE dimension
      const int d = k / V2_MK, r = k - d * V2_MK;
      uint64_t key = 0ull;
      if (r < cnt) { key = f64_to_ordered(v2_mk_tile[r * DP + d]); K[(int64_t)d * N + i0 + r] = key; }
      const uint64_t mn = warp_min_u64(r < cnt ? key : ~0ull), mx = warp_max_u64(r < cnt ? key : 0ull);
      if ((threadIdx.x & 31) == 0 && mn <= mx) { atomicMin(&s_lo[d], (unsigned long long)mn); atomicMax(&s_hi[d], (unsigned long long)mx); }
    }
    for (int r = threadIdx.x; r < cnt; r += 256) { perm[i0 + r] = (int32_t)(i0 + r); seg[i0 + r] = 0; }
  }
  __syncthreads();
  if (threadIdx.x < D && s_lo[threadIdx.x] <= s_hi[threadIdx.x]) {
    atomicMin((unsigned long long *)root_lo + threadIdx.x, s_lo[threadIdx.x]);
    atomicMax((unsigned long long *)root_hi + threadIdx.x, s_hi[threadIdx.x]);
  }
  if (bad) *nan_flag = 1;
}

__global__ void v2_init_kernel(V2Top t) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    V2Info *in = t.info;
    for (int l = 0; l <= V2_MAXLEV; ++l) { in->lvl[l].lb = in->lvl[l].le = 0; in->maxsize[l] = 0; }
    in->lvl[0].lb = 0; in->lvl[0].le = 1; in->maxsize[0] = (int32_t)t.N;
    in->nnodes = 1; in->nlevels = 0; in->sel_active = 0; in->overflow = 0;
    t.nb[0] = 0; t.ne[0] = (int32_t)t.N; t.ndim[0] = -1; t.nleft[0] = -1; t.nspos[0] = (int32_t)t.N; t.nsplit[0] = 0.0;
  }
}

// ---- per-level: bounds ------------------------------------------------------------------------------------------
__global__ void v2_level_init_kernel(V2Top t, int L, uint64_t *__restrict__ lo, uint64_t *__restrict__ hi) {
  const V2Level lv = t.info->lvl[L];
  const int64_t tot = (int64_t)(lv.le - lv.lb) * t.D;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += (int64_t)gridDim.x * blockDim.x) {
    lo[i] = ~0ull; hi[i] = 0ull;
  }
}

// 64-bit warp min / max from the 32-bit redux instruction: high words first, then the low words of the lanes that hold
// the winning high word (2 REDUX instead of 10 shuffle + compare steps)
__device__ __forceinline__ uint64_t warp_min_u64(uint64_t v) {
  const unsigned h = (unsigned)(v >> 32), l = (unsigned)v;
  const unsigned mh = __reduce_min_sync(0xffffffffu, h);
  const unsigned ml = __reduce_min_sync(0xffffffffu, h == mh ? l : 0xffffffffu);
  return ((uint64_t)mh << 32) | ml;
}
__device__ __forceinline__ uint64_t warp_max_u64(uint64_t v) {
  const unsigned h = (unsigned)(v >> 32), l = (unsigned)v;
  const unsigned mh = __reduce_max_sync(0xffffffffu, h);
  const unsigned ml = __reduce_max_sync(0xffffffffu, h == mh ? l : 0u);
  return ((uint64_t)mh << 32) | ml;
}

// min / max of a per-lane (node, lo, hi) triple into global per-node slots.  Lanes of a warp cover consecutive
// positions, so at most the first and the last node of the warp have many lanes: those two groups are reduced in the
// warp and flushed by one lane each, the (rare) lanes of other nodes flush themselves.  node < 0: nothing to flush.
__device__ __forceinline__ void warp_minmax_flush(int node, uint64_t mn, uint64_t mx, uint64_t *lo, uint64_t *hi) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int n_first = __shfl_sync(full, node, 0), n_last = __shfl_sync(full, node, 31);
  if (__all_sync(full, node < 0)) return;
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    const int target = g == 0 ? n_first : n_last;
    if (g == 1 && n_last == n_first) break;
    if (target < 0) continue;                                  // warp-uniform
    const uint64_t a = lo ? warp_min_u64(node == target ? mn : ~0ull) : 0ull;
    const uint64_t b = hi ? warp_max_u64(node == target ? mx : 0ull) : 0ull;
    if (lane == 0) {
      if (lo && a != ~0ull) atomicMin((unsigned long long *)lo + target, (unsigned long long)a);
      if (hi && b != 0ull) atomicMax((unsigned long long *)hi + target, (unsigned long long)b);
    }
  }
  if (node >= 0 && node != n_first && node != n_last) {
    if (lo && mn != ~0ull) atomicMin((unsigned long long *)lo + node, (unsigned long long)mn);
    if (hi && mx != 0ull) atomicMax((unsigned long long *)hi + node, (unsigned long long)mx);
  }
}

// V2_ITEMS consecutive elements of one thread (blocked arrangement), 16-byte loads when the column allows it
__device__ __forceinline__ void v2_load8(const uint64_t *__restrict__ col, int64_t base, int64_t N, bool vec, uint64_t (&key)[V2_ITEMS]) {
  if (vec && base + V2_ITEMS <= N) {
    const ulonglong2 *p = reinterpret_cast<const ulonglong2 *>(col + base);
#pragma unroll
    for (int q = 0; q < V2_ITEMS / 2; ++q) { const ulonglong2 x = __ldcs(p + q); key[2 * q] = x.x; key[2 * q + 1] = x.y; }
  } else {
#pragma unroll
    for (int k = 0; k < V2_ITEMS; ++k) key[k] = (base + k < N) ? __ldcs(col + base + k) : 0ull;
  }
}
__device__ __forceinline__ void v2_load8_i32(const int32_t *__restrict__ a, int64_t base, int64_t N, int32_t (&v)[V2_ITEMS], int32_t fill) {
  if (base + V2_ITEMS <= N) {
    const int4 *p = reinterpret_cast<const int4 *>(a + base);
    const int4 x = p[0], y = p[1];
    v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w; v[4] = y.x; v[5] = y.y; v[6] = y.z; v[7] = y.w;
  } else {
#pragma unroll
    for (int k = 0; k < V2_ITEMS; ++k) v[k] = (base + k < N) ? a[base + k] : fill;
  }
}
static_assert(V2_ITEMS == 8, "v2_load8 helpers assume 8 items per thread");

// One tile of positions, all D columns (used for the root level; deeper levels get their bounds from the scatter pass
// of their parents).  A thread owns V2_ITEMS consecutive positions; positions of one thread that straddle a node
// boundary flush the minority directly.
__global__ void __launch_bounds__(V2_TB)
v2_bounds_kernel(V2Top t, int L, const uint64_t *__restrict__ K, const int32_t *__restrict__ seg, uint64_t *__restrict__ lo,
                 uint64_t *__restrict__ hi) {
  const V2Level lv = t.info->lvl[L];
  if (lv.le <= lv.lb) return;
  const int64_t base = ((int64_t)blockIdx.x * V2_TB + threadIdx.x) * V2_ITEMS;
  const bool vec = (t.N & 1) == 0;
  int nd[V2_ITEMS];
  v2_load8_i32(seg, base, t.N, nd, -1);
  int first = -1;                       // the node of this thread's first active position (level-relative), or -1
  bool uniform = true;
#pragma unroll
  for (int k = 0; k < V2_ITEMS; ++k) {
    int id = (base + k < t.N) ? nd[k] : -1;
    id = (id >= lv.lb && id < lv.le) ? id - lv.lb : -1;
    nd[k] = id;
    if (id >= 0) { if (first < 0) first = id; else if (id != first) uniform = false; }
  }
  for (int d = 0; d < t.D; ++d) {
    uint64_t key[V2_ITEMS];
    v2_load8(K + (int64_t)d * t.N, base, t.N, vec, key);
    uint64_t mn = ~0ull, mx = 0ull;
#pragma unroll
    for (int k = 0; k < V2_ITEMS; ++k) {
      if (nd[k] < 0) continue;
      if (uniform || nd[k] == first) { mn = key[k] < mn ? key[k] : mn; mx = key[k] > mx ? key[k] : mx; }
      else { atomicMin((unsigned long long *)lo + (int64_t)nd[k] * t.D + d, (unsigned long long)key[k]);
             atomicMax((unsigned long long *)hi + (int64_t)nd[k] * t.D + d, (unsigned long long)key[k]); }
    }
    // slot of (node, d) = node * D + d: the node index handed to the flush is node * D, the pointers carry + d
    warp_minmax_flush(first < 0 ? -1 : first * t.D, mn, mx, lo + d, hi + d);
  }
}

// ---- per-level: leaves, split dimension, select set-up ---------------------------------------------------------------
__global__ void v2_node_kernel(V2Top t, int L) {
  const V2Level lv = t.info->lvl[L];
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= lv.le - lv.lb) return;
  const int id = lv.lb + k;
  const int32_t b = t.nb[id], e = t.ne[id], n = e - b;
  int sd = -1;
  if (n > 1 && n >= t.min_split) {                        // kd_tree.ml:157-158 (+ truncation)
    double dx_max = neg_inf();
    bool all_eq = true;
    for (int d = 0; d < t.D; ++d) {                        // :96-110, :120-130 first strictly largest spread
      const uint64_t l = t.lo[(int64_t)k * t.D + d], h = t.hi[(int64_t)k * t.D + d];
      if (l != h) all_eq = false;
      const double dx = ordered_to_f64(h) - ordered_to_f64(l);
      if (dx > dx_max) { sd = d; dx_max = dx; }
    }
    if (all_eq) sd = -1;                                   // :159-160 identical coordinates -> leaf
  }
  t.ndim[id] = sd; t.nleft[id] = -1; t.nsplit[id] = 0.0; t.nspos[id] = e;
  V2Sel s; s.prefix = 0; s.shift = -1; s.dim = sd;
  t.kth[k] = n / 2; t.below[k] = 0; t.nR[k] = 0; t.fix[k] = 0; t.v[k] = 0; t.maxL[k] = 0ull; t.minR[k] = ~0ull;
  if (sd >= 0) {
    const uint64_t l = t.lo[(int64_t)k * t.D + sd], h = t.hi[(int64_t)k * t.D + sd];
    const int top = 63 - __clzll((long long)(l ^ h));      // highest differing bit (l != h here)
    const int df = top + 1;                                // bits df .. 63 are shared by all keys of the node
    s.shift = top >= 7 ? top - 7 : 0;
    s.prefix = df >= 64 ? 0ull : (l >> df) << df;
    s.dim = sd | (df << 8);
    atomicAdd(&t.info->sel_active, 1);
  }
  t.sel[k] = s;
}

// ---- per-level: radix select -------------------------------------------------------------------------------------------
constexpr int V2_NH = 4;       // nodes of a tile with a private shared-memory histogram
__global__ void __launch_bounds__(V2_TB)
v2_hist_kernel(V2Top t, int L, const uint64_t *__restrict__ K, const int32_t *__restrict__ seg) {
  if (t.info->sel_active <= 0) return;
  const V2Level lv = t.info->lvl[L];
  __shared__ uint32_t sh[V2_NH][256];
  __shared__ int s_first;
  for (int i = threadIdx.x; i < V2_NH * 256; i += V2_TB) (&sh[0][0])[i] = 0u;
  if (threadIdx.x == 0) s_first = 0x7fffffff;
  __syncthreads();
  const int64_t base = (int64_t)blockIdx.x * V2_TILE;
  int nd[V2_ITEMS]; uint32_t bin[V2_ITEMS];
  int mymin = 0x7fffffff;
#pragma unroll
  for (int k = 0; k < V2_ITEMS; ++k) {                      // striped: coalesced 4-byte / 8-byte loads
    const int64_t p = base + (int64_t)k * V2_TB + threadIdx.x;
    nd[k] = -1;
    if (p >= t.N) continue;
    int id = seg[p];
    if (id < lv.lb || id >= lv.le) continue;
    id -= lv.lb;
    const V2Sel s = t.sel[id];
    if (s.shift < 0) continue;
    const uint64_t key = K[(int64_t)(s.dim & 255) * t.N + p];
    const int df = s.dim >> 8;
    if (df < 64 && ((key ^ s.prefix) >> df) != 0ull) continue;
    nd[k] = id; bin[k] = (uint32_t)(key >> s.shift) & 255u;
    mymin = id < mymin ? id : mymin;
  }
  if (mymin != 0x7fffffff) atomicMin(&s_first, mymin);
  __syncthreads();
  const int first = s_first;
#pragma unroll
  for (int k = 0; k < V2_ITEMS; ++k) {
    if (nd[k] < 0) continue;
    const int rel = nd[k] - first;
    if (rel < V2_NH) atomicAdd(&sh[rel][bin[k]], 1u);
    else atomicAdd(t.hist + (int64_t)nd[k] * 256 + bin[k], 1u);
  }
  __syncthreads();
  if (first == 0x7fffffff) return;
  const int nlvl = lv.le - lv.lb;
  for (int i = threadIdx.x; i < V2_NH * 256; i += V2_TB) {
    const uint32_t c = (&sh[0][0])[i];
    const int node = first + (i >> 8);
    if (c && node < nlvl) atomicAdd(t.hist + (int64_t)node * 256 + (i & 255), c);
  }
}

// one warp per node: the bin that holds the kth key; when the last byte is decided, the node's split position
__global__ void __launch_bounds__(256)
v2_pick_kernel(V2Top t, int L) {
  if (t.info->sel_active <= 0) return;
  const V2Level lv = t.info->lvl[L];
  const int k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (k >= lv.le - lv.lb) return;
  V2Sel s = t.sel[k];
  if (s.shift < 0) return;
  uint32_t *h = t.hist + (int64_t)k * 256;
  uint32_t c[8]; uint32_t sum = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) { c[j] = h[lane * 8 + j]; sum += c[j]; h[lane * 8 + j] = 0u; }
  uint32_t incl = sum;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) { const uint32_t x = __shfl_up_sync(0xffffffffu, incl, off); if (lane >= off) incl += x; }
  const uint32_t excl = incl - sum;
  const uint32_t kth = (uint32_t)t.kth[k];
  const bool mine = kth >= excl && kth < incl;              // exactly one lane
  const unsigned who = __ballot_sync(0xffffffffu, mine);
  const int src = __ffs(who) - 1;
  int bin = 0; uint32_t below = 0, cnt = 0;
  if (mine) {
    uint32_t run = excl;
#pragma unroll
    for (int j = 0; j < 8; ++j) { if (kth >= run && kth < run + c[j]) { bin = lane * 8 + j; below = run; cnt = c[j]; } run += c[j]; }
  }
  bin = __shfl_sync(0xffffffffu, bin, src); below = __shfl_sync(0xffffffffu, below, src); cnt = __shfl_sync(0xffffffffu, cnt, src);
  if (lane != 0) return;
  if (src < 0) { t.info->overflow = 1; return; }            // cannot happen: the histogram holds >= kth + 1 keys
  s.prefix |= (uint64_t)bin << s.shift;
  t.kth[k] = (int32_t)(kth - below);
  const int32_t below_tot = t.below[k] + (int32_t)below;
  t.below[k] = below_tot;
  // The select is over as soon as the bin of the order statistic holds ONE key: the scatter only compares keys with
  // the pivot, and a pivot that is alone in its bin is ordered against every other key by the bits decided so far
  // (the split plane comes from max L / min R, which the scatter finds).  Otherwise all 64 bits are decided.
  if (s.shift == 0 || cnt == 1u) {
    const int id = lv.lb + k;
    const int32_t b = t.nb[id], e = t.ne[id], n = e - b;
    int32_t cntL = below_tot + (int32_t)cnt;                // keys <= v   (List.partition (<= pvt), :168)
    uint8_t fix = 0;
    if (cntL == n) { cntL = below_tot; fix = 1; }           // adjust_for_empty_split :150-152: L = {k < max}
    // undecided low bits: all ones for "key > v goes right", all zeros for "key >= v goes right" (the pivot itself)
    const uint64_t low = (s.shift > 0 && !fix) ? ((1ull << s.shift) - 1ull) : 0ull;
    t.v[k] = s.prefix | low; t.fix[k] = fix; t.nR[k] = n - cntL; t.nspos[id] = b + cntL;
    if (cntL <= 0 || cntL >= n) t.info->overflow = 1;       // cannot happen (lo != hi on the split dimension)
    s.shift = -1;
    atomicSub(&t.info->sel_active, 1);
  } else {
    s.dim = (s.dim & 255) | (s.shift << 8);                 // decided down to this digit; the last digit may overlap it
    s.shift = s.shift >= 8 ? s.shift - 8 : 0;
  }
  t.sel[k] = s;
}

// ---- per-level: children (breadth-first numbering) -------------------------------------------------------------------
__global__ void __launch_bounds__(1024)
v2_children_kernel(V2Top t, int L) {
  V2Info *in = t.info;
  const V2Level lv = in->lvl[L];
  const int nlvl = lv.le - lv.lb;
  __shared__ int carry_s, carry_r, s_max;
  if (threadIdx.x == 0) { carry_s = 0; carry_r = 0; s_max = 0; }
  __syncthreads();
  const int next_base = lv.le;                 // levels are numbered consecutively: the next level starts where this one ends
  for (int base = 0; base < nlvl; base += 1024) {
    const int k = base + threadIdx.x;
    int is = 0, nr = 0;
    if (k < nlvl) { is = t.ndim[lv.lb + k] >= 0 ? 1 : 0; nr = is ? t.nR[k] : 0; }
    int tot_s, tot_r;
    const int ex_s = block_exclusive_scan<1024>(is, &tot_s);
    const int ex_r = block_exclusive_scan<1024>(nr, &tot_r);
    const int cs = carry_s, cr = carry_r;
    if (k < nlvl) {
      t.ebegin[k] = cr + ex_r;
      if (is) {
        const int id = lv.lb + k;
        const int64_t Lc = (int64_t)next_base + 2 * (int64_t)(cs + ex_s);
        if (Lc + 1 < t.cap) {
          const int32_t b = t.nb[id], e = t.ne[id], sp = t.nspos[id];
          t.nleft[id] = (int32_t)Lc;
          t.nb[Lc] = b; t.ne[Lc] = sp; t.nb[Lc + 1] = sp; t.ne[Lc + 1] = e;
          atomicMax(&s_max, max(sp - b, e - sp));
        }
      }
    }
    __syncthreads();
    if (threadIdx.x == 0) { carry_s = cs + tot_s; carry_r = cr + tot_r; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const int nsplit = carry_s;
    if (nlvl > 0) in->nlevels = L + 1;
    const int64_t nle = (int64_t)next_base + 2 * (int64_t)nsplit;
    if (nle > t.cap || 2 * nsplit > t.LC || L + 1 > V2_MAXLEV) { in->overflow = 1; in->lvl[L + 1].lb = in->lvl[L + 1].le = next_base; }
    else { in->lvl[L + 1].lb = next_base; in->lvl[L + 1].le = (int32_t)nle; in->nnodes = (int32_t)nle; in->maxsize[L + 1] = s_max; }
  }
}

// ---- per-level: stable partition of every column ------------------------------------------------------------------------
// One tile: flags from the split column, chained scan with decoupled look-back for the global offsets, then every
// column is moved through shared memory -- a thread writes its keys at the tile-local compact index of their
// destination stream (left-goers and pass-through elements first, right-goers after them; inside a stream consecutive
// elements have consecutive destinations), and the tile leaves in that order: coalesced 8-byte stores instead of one
// 32-byte sector per key.  While a column passes through, the bounds of the CHILD nodes (the next level's
// bounds_of_objects) are reduced from it, so the next level needs no pass of its own over the data.
constexpr unsigned long long V2_AGG = 1ull << 62, V2_PRE = 2ull << 62, V2_MSK = 3ull << 62;

#ifndef MG_V2_SCATTER_MINBLOCKS
#define MG_V2_SCATTER_MINBLOCKS 3
#endif
__global__ void __launch_bounds__(V2_TB, MG_V2_SCATTER_MINBLOCKS)
v2_scatter_kernel(V2Top t, int L, const uint64_t *__restrict__ Kin, uint64_t *__restrict__ Kout,
                  const int32_t *__restrict__ perm_in, int32_t *__restrict__ perm_out, const int32_t *__restrict__ seg_in,
                  int32_t *__restrict__ seg_out, unsigned long long *__restrict__ status, unsigned int *__restrict__ ticket,
                  uint64_t *__restrict__ lo_next, uint64_t *__restrict__ hi_next, int *__restrict__ err) {
  const V2Level lv = t.info->lvl[L];
  __shared__ unsigned int s_tile;
  __shared__ int s_base;
  __shared__ uint64_t sk0[V2_TILE], sk1[V2_TILE];   // two columns of the tile in destination order
  int32_t *sdst = reinterpret_cast<int32_t *>(sk1);  // first: destination of every compact slot ...
  int32_t *schild = sdst + V2_TILE;                  // ... and its child node relative to the next level (-1: none)
  if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1u);
  __syncthreads();
  const int64_t tile = s_tile;
  const int64_t tbase = tile * V2_TILE;
  const int64_t base = tbase + (int64_t)threadIdx.x * V2_ITEMS;
  const bool vec = (t.N & 1) == 0;
  const int next_lb = lv.le;
  int nd[V2_ITEMS]; int f[V2_ITEMS];
  v2_load8_i32(seg_in, base, t.N, nd, -1);
  int acc = 0;
  int first = -1; bool uniform = true;
  uint64_t rmn = ~0ull, lmx = 0ull;          // min of right-goers / max of left-goers of node `first`
#pragma unroll
  for (int k = 0; k < V2_ITEMS; ++k) {
    const int64_t p = base + k;
    f[k] = 0;
    if (p >= t.N) { nd[k] = -1; continue; }
    const int id = nd[k];
    if (id < lv.lb || id >= lv.le) { nd[k] = -2 - id; continue; }       // pass-through: remember the node as -2 - id
    const int kk = id - lv.lb;
    const int sd = t.ndim[id];
    if (sd < 0) { nd[k] = -2 - id; continue; }
    nd[k] = kk;
    const uint64_t key = Kin[(int64_t)sd * t.N + p];
    const uint64_t v = t.v[kk];
    const bool right = t.fix[kk] ? (key >= v) : (key > v);
    f[k] = right ? 1 : 0;
    acc += f[k];
    if (first < 0) first = kk; else if (kk != first) uniform = false;
    if (uniform || kk == first) { if (right) rmn = key < rmn ? key : rmn; else lmx = key > lmx ? key : lmx; }
    else { if (right) atomicMin((unsigned long long *)t.minR + kk, (unsigned long long)key);
           else atomicMax((unsigned long long *)t.maxL + kk, (unsigned long long)key); }
  }
  // max L / min R of the split plane (:170-171), aggregated per warp
  warp_minmax_flush(first, rmn, ~0ull, t.minR, nullptr);
  warp_minmax_flush(first, 0ull, lmx, nullptr, t.maxL);
  int total;
  const int ex = block_exclusive_scan<V2_TB>(acc, &total);
  if (threadIdx.x < 32) {                  // chained scan with decoupled look-back over the tiles
    const int lane = threadIdx.x;
    if (lane == 0 && tile > 0) atomicExch(status + tile, V2_AGG | (unsigned long long)total);
    unsigned long long prefix = 0;
    int64_t end = tile - 1;
    bool done = (tile == 0);
    while (!done) {
      const int64_t kq = end - lane;
      unsigned long long vv = V2_PRE;
      if (kq >= 0) {
        unsigned spins = 0;
        do {
          vv = *reinterpret_cast<volatile unsigned long long *>(status + kq);
          if (!(vv & V2_MSK) && ((++spins & 1023u) == 0u)) {
            if (spins > (1u << 28)) atomicExch(err, MG_DEVERR_KD_LOOKBACK);
            if (*reinterpret_cast<volatile int *>(err) != 0) vv = V2_PRE;
          }
        } while (!(vv & V2_MSK));
      }
      const unsigned has_prefix = __ballot_sync(0xffffffffu, (vv & V2_MSK) == V2_PRE);
      const int firstp = __ffs(has_prefix) - 1;
      unsigned long long part = (firstp < 0 || lane <= firstp) ? (vv & ~V2_MSK) : 0ull;
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) part += __shfl_xor_sync(0xffffffffu, part, off);
      prefix += part;
      if (firstp >= 0) done = true; else end -= 32;
    }
    if (lane == 0) {
      __threadfence();
      atomicExch(status + tile, V2_PRE | (prefix + (unsigned long long)total));
      s_base = (int)prefix;
    }
  }
  __syncthreads();
  const int tile_cnt = (int)((t.N - tbase < V2_TILE) ? t.N - tbase : V2_TILE);
  const int tile_left = tile_cnt - total;    // left-goers and pass-through elements of the tile
  int E = ex + s_base, el = ex;              // global / tile-local exclusive count of right-goers
  int ci[V2_ITEMS];
  const int lpos0 = threadIdx.x * V2_ITEMS;
#pragma unroll
  for (int k = 0; k < V2_ITEMS; ++k) {
    const int64_t p = base + k;
    ci[k] = -1;
    if (p < t.N) {
      int64_t dst; int32_t child = -1, sg;
      if (nd[k] < 0) { dst = p; sg = -2 - nd[k]; }
      else {
        const int kk = nd[k], id = lv.lb + kk;
        const int32_t b = t.nb[id], sp = t.nspos[id];
        const int32_t r = E - t.ebegin[kk];                   // right-goers in [b, p)
        dst = f[k] ? (int64_t)sp + r : (int64_t)b + (p - b) - r;
        sg = f[k] ? t.nleft[id] + 1 : t.nleft[id];
        child = sg - next_lb;
      }
      ci[k] = f[k] ? tile_left + el : (lpos0 + k) - el;
      sdst[ci[k]] = (int32_t)dst; schild[ci[k]] = child;
      seg_out[dst] = sg;
      perm_out[dst] = perm_in[p];
    }
    E += f[k]; el += f[k];
  }
  __syncthreads();
  // copy-out slots of this thread: tid, tid + TB, ... (consecutive lanes hold consecutive destinations);
  // bounds slots of this thread: 8 consecutive compact slots (mostly one child), read in a rotated order
  int32_t odst[V2_ITEMS], bch[V2_ITEMS];
#pragma unroll
  for (int q = 0; q < V2_ITEMS; ++q) {
    const int j = q * V2_TB + threadIdx.x;
    odst[q] = j < tile_cnt ? sdst[j] : -1;
    const int jb = lpos0 + ((q + threadIdx.x) & (V2_ITEMS - 1));
    bch[q] = jb < tile_cnt ? schild[jb] : -1;
  }
  int cA = -1, cB = -1;                       // the children at the two ends of my 8 bounds slots
#pragma unroll
  for (int q = 0; q < V2_ITEMS; ++q) {
    const int jq = (q + threadIdx.x) & (V2_ITEMS - 1);       // position of rotated slot q inside my 8
    if (jq == 0) cA = bch[q];
    if (jq == V2_ITEMS - 1) cB = bch[q];
  }
  if (cA < 0) { cA = cB; }
  __syncthreads();                            // sdst / schild are in registers now: their memory becomes the second column buffer
  for (int d0 = 0; d0 < t.D; d0 += 2) {       // two columns per barrier pair
    const bool two = d0 + 1 < t.D;
    uint64_t key[V2_ITEMS], key2[V2_ITEMS];
    v2_load8(Kin + (int64_t)d0 * t.N, base, t.N, vec, key);
    if (two) v2_load8(Kin + (int64_t)(d0 + 1) * t.N, base, t.N, vec, key2);
#pragma unroll
    for (int k = 0; k < V2_ITEMS; ++k) if (ci[k] >= 0) { sk0[ci[k]] = key[k]; if (two) sk1[ci[k]] = key2[k]; }
    __syncthreads();
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (h == 1 && !two) break;
      const int d = d0 + h;
      const uint64_t *sk = h == 0 ? sk0 : sk1;
      uint64_t *co = Kout + (int64_t)d * t.N;
#pragma unroll
      for (int q = 0; q < V2_ITEMS; ++q)
        if (odst[q] >= 0) __stcs(co + odst[q], sk[q * V2_TB + threadIdx.x]);
      // bounds of the children (the next level's bounds_of_objects)
      uint64_t mnA = ~0ull, mxA = 0ull, mnB = ~0ull, mxB = 0ull;
#pragma unroll
      for (int q = 0; q < V2_ITEMS; ++q) {
        const int c = bch[q];
        if (c < 0) continue;
        const uint64_t x = sk[lpos0 + ((q + threadIdx.x) & (V2_ITEMS - 1))];
        if (c == cA) { mnA = x < mnA ? x : mnA; mxA = x > mxA ? x : mxA; }
        else if (c == cB) { mnB = x < mnB ? x : mnB; mxB = x > mxB ? x : mxB; }
        else { atomicMin((unsigned long long *)lo_next + (int64_t)c * t.D + d, (unsigned long long)x);
               atomicMax((unsigned long long *)hi_next + (int64_t)c * t.D + d, (unsigned long long)x); }
      }
      warp_minmax_flush(cA < 0 ? -1 : cA * t.D, mnA, mxA, lo_next + d, hi_next + d);
      if (__any_sync(0xffffffffu, cB >= 0 && cB != cA))
        warp_minmax_flush((cB < 0 || cB == cA) ? -1 : cB * t.D, mnB, mxB, lo_next + d, hi_next + d);
    }
    __syncthreads();
  }
}

__global__ void v2_split_kernel(V2Top t, int L) {
  const V2Level lv = t.info->lvl[L];
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= lv.le - lv.lb) return;
  const int id = lv.lb + k;
  if (t.ndim[id] < 0) return;
  // max L is the pivot itself unless the empty-side fix-up moved it; min R likewise -- both were gathered by the
  // scatter pass from the keys that actually went left / right
  t.nsplit[id] = 0.5 * (ordered_to_f64(t.maxL[k]) + ordered_to_f64(t.minR[k]));   // split_bounds :113
}

// ---- bottom phase ---------------------------------------------------------------------------------------------------------
struct V2Bottom {
  int64_t N; int D, min_split, L0;
  const V2Info *info;
  const int32_t *nb, *ne;              // top node arrays (subtree roots)
  const uint64_t *K; const int32_t *perm_in; int32_t *perm_out;
  int32_t *l_dim, *l_child, *l_begin, *l_end; double *l_split;   // local nodes at [2 * b + k]
  int32_t *cnt;                         // [nsub][V2_MAXL]
  int32_t *depth;                       // [nsub]
  int *overflow;
};

template <int NMAX, int BT>
constexpr size_t v2_bottom_smem(int D) {
  return (size_t)D * NMAX * 8 /* key columns */ + (size_t)(BT / 32) * 256 * 4 /* per-warp histograms */ +
         (size_t)NMAX * 2 * 8 /* ids x2, cur b/e, next b/e, spl, sps */ + 64;
}

// One CTA per subtree; the subtree's key columns live in shared memory, one warp works on one node at a time.
template <int NMAX, int BT>
__global__ void __launch_bounds__(BT)
v2_bottom_kernel(V2Bottom a) {
  extern __shared__ __align__(16) unsigned char v2_smem[];
  uint64_t *skeys = reinterpret_cast<uint64_t *>(v2_smem);                    // [D][NMAX] keys by local id
  uint32_t *hist_all = reinterpret_cast<uint32_t *>(skeys + (size_t)a.D * NMAX);   // [warps][256]
  uint16_t *ids0 = reinterpret_cast<uint16_t *>(hist_all + (BT / 32) * 256), *ids1 = ids0 + NMAX;   // local ids in node order
  uint16_t *cb0 = ids1 + NMAX, *ce0 = cb0 + NMAX, *cb1 = ce0 + NMAX, *ce1 = cb1 + NMAX;              // level nodes: begin / end
  uint16_t *spl = ce1 + NMAX, *sps = spl + NMAX;                              // is_split / local split position
  __shared__ int s_scan[BT / 32], s_tot;
  const V2Level lv = a.info->lvl[a.L0];
  const int s = blockIdx.x;
  if (s >= lv.le - lv.lb) return;
  const int g = lv.lb + s;
  const int32_t b = a.nb[g], e = a.ne[g];
  const int n = e - b;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = BT / 32;
  const unsigned full = 0xffffffffu, lt = (1u << lane) - 1u;
  int32_t *cnt = a.cnt + (size_t)s * V2_MAXL;
  if (n > NMAX || n <= 0) { if (tid == 0) { *a.overflow = 1; a.depth[s] = 0; } return; }
  for (int d = 0; d < a.D; ++d) {
    const uint64_t *col = a.K + (int64_t)d * a.N + b;
    for (int j = tid; j < n; j += BT) skeys[(size_t)d * NMAX + j] = col[j];
  }
  for (int j = tid; j < n; j += BT) ids0[j] = (uint16_t)j;
  if (tid == 0) { cb0[0] = 0; ce0[0] = (uint16_t)n; }
  __syncthreads();
  uint16_t *ids = ids0, *idn = ids1, *cb = cb0, *ce = ce0, *nb_ = cb1, *ne_ = ce1;
  uint32_t *h = hist_all + warp * 256;
  uint64_t *cand = reinterpret_cast<uint64_t *>(h);      // the same 1 KB holds up to 32 candidate keys
  int cur_n = 1, lbase = 0, l = 0, level_max = n;
  const int64_t gbase = 2 * (int64_t)b;
  constexpr int kLaneDimMax = 128;     // nodes up to this size: one lane per dimension walks the node's points
  constexpr int kTinyMax = 8;          // nodes up to this size: one thread per node
  uint64_t *pair_lo = reinterpret_cast<uint64_t *>(hist_all), *pair_hi = pair_lo + (BT / 32) * 64;   // [warps][64] (aliases the histograms)
  static_assert((BT / 32) * 64 * 16 <= (BT / 32) * 256 * 4, "pair bounds fit the histogram area");
  for (;;) {
    if (tid == 0) cnt[l] = cur_n;
    // Large nodes exist only while the level has few nodes (at most one per warp): their bounds are then computed by
    // ALL warps, one (node, dimension) pair at a time, instead of by the node's own warp alone.
    // (level_max estimates the level's largest node: without ties a child holds at most n / 2 + 1 of its parent's n
    // points.  Once that is <= kLaneDimMax the pair pass would only skip its pairs; a node kept large by ties then gets
    // its bounds from its own warp below -- slower, same result.)
    const bool pair_mode = cur_n <= nwarps && level_max > kLaneDimMax;
    uint64_t pre_lo[2] = {~0ull, ~0ull}, pre_hi[2] = {0ull, 0ull};
    bool have_pre = false;
    if (pair_mode) {
      for (int pair = warp; pair < cur_n * a.D; pair += nwarps) {
        const int node = pair / a.D, d = pair - node * a.D;
        const int nb0 = cb[node], ne0 = ce[node];
        if (ne0 - nb0 <= kLaneDimMax) continue;
        const uint64_t *col = skeys + (size_t)d * NMAX;
        uint64_t mn = ~0ull, mx = 0ull;
        for (int j = nb0 + lane; j < ne0; j += 32) { const uint64_t k = col[ids[j]]; mn = k < mn ? k : mn; mx = k > mx ? k : mx; }
        mn = warp_min_u64(mn); mx = warp_max_u64(mx);
        if (lane == 0) { pair_lo[node * 64 + d] = mn; pair_hi[node * 64 + d] = mx; }
      }
      __syncthreads();
      if (warp < cur_n && ce[warp] - cb[warp] > kLaneDimMax) {
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const int d = hh * 32 + lane;
          if (d < a.D) { pre_lo[hh] = pair_lo[warp * 64 + d]; pre_hi[hh] = pair_hi[warp * 64 + d]; }
        }
        have_pre = true;
      }
      __syncthreads();          // the histogram area is free again
    }
    // Tiny nodes (the last levels of a full tree hold 7/8 of all nodes): one THREAD per node, everything in
    // registers -- same rule, scalar code.
    for (int node = tid; node < cur_n; node += BT) {
      const int nb0 = cb[node], ne0 = ce[node], m = ne0 - nb0;
      if (m > kTinyMax) continue;
      int sd = -1; double split = 0.0; int spos = ne0;
      uint16_t id[kTinyMax];
#pragma unroll
      for (int j = 0; j < kTinyMax; ++j) id[j] = j < m ? ids[nb0 + j] : (uint16_t)0;
      if (m > 1 && m >= a.min_split) {                                // kd_tree.ml:157-158 (+ truncation)
        double dx_max = neg_inf(); bool all_eq = true;
        for (int d = 0; d < a.D; ++d) {                               // :96-110, :120-130
          const uint64_t *col = skeys + (size_t)d * NMAX;
          uint64_t mn = ~0ull, mx = 0ull;
#pragma unroll
          for (int j = 0; j < kTinyMax; ++j) if (j < m) { const uint64_t k = col[id[j]]; mn = k < mn ? k : mn; mx = k > mx ? k : mx; }
          if (mn != mx) all_eq = false;
          const double dx = ordered_to_f64(mx) - ordered_to_f64(mn);
          if (dx > dx_max) { sd = d; dx_max = dx; }
        }
        if (all_eq) sd = -1;                                          // :159-160
        if (sd >= 0) {
          const uint64_t *col = skeys + (size_t)sd * NMAX;
          uint64_t key[kTinyMax];
#pragma unroll
          for (int j = 0; j < kTinyMax; ++j) key[j] = j < m ? col[id[j]] : ~0ull;
          uint64_t v = 0ull;                                          // the m/2-th order statistic (:162-167)
#pragma unroll
          for (int j = 0; j < kTinyMax; ++j) {
            int r = 0;
#pragma unroll
            for (int i = 0; i < kTinyMax; ++i) r += (i < m && (key[i] < key[j] || (key[i] == key[j] && i < j))) ? 1 : 0;
            if (j < m && r == m / 2) v = key[j];
          }
          int below = 0, eq = 0;
#pragma unroll
          for (int j = 0; j < kTinyMax; ++j) if (j < m) { below += key[j] < v; eq += key[j] == v; }
          int cntL = below + eq;                                      // List.partition (<= pvt), :168
          const bool fix = cntL == m;                                 // adjust_for_empty_split :150-152
          if (fix) cntL = below;
          spos = nb0 + cntL;
          uint64_t ml = 0ull, mr = ~0ull;
          int lc = 0, rc = 0;
#pragma unroll
          for (int j = 0; j < kTinyMax; ++j) {
            if (j >= m) continue;
            const bool left = fix ? (key[j] < v) : (key[j] <= v);
            if (left) { ml = key[j] > ml ? key[j] : ml; idn[nb0 + lc++] = id[j]; }
            else { mr = key[j] < mr ? key[j] : mr; idn[spos + rc++] = id[j]; }
          }
          split = 0.5 * (ordered_to_f64(ml) + ordered_to_f64(mr));    // split_bounds :113
        }
      }
      if (sd < 0) {
#pragma unroll
        for (int j = 0; j < kTinyMax; ++j) if (j < m) idn[nb0 + j] = id[j];
      }
      spl[node] = sd >= 0 ? 1 : 0; sps[node] = (uint16_t)spos;
      const int64_t gk = gbase + lbase + node;
      a.l_dim[gk] = sd; a.l_split[gk] = split; a.l_begin[gk] = nb0; a.l_end[gk] = ne0; a.l_child[gk] = -1;
    }
    for (int node = warp; node < cur_n; node += nwarps) {
      const int nb0 = cb[node], ne0 = ce[node], m = ne0 - nb0;
      if (m <= kTinyMax) continue;                                    // done by its own thread above
      int sd = -1; double split = 0.0; int spos = ne0;
      if (m > 1 && m >= a.min_split) {                                // kd_tree.ml:157-158 (+ truncation)
        // bounds_of_objects (:96-110); lane d keeps dimension d (and d + 32)
        uint64_t klo[2] = {~0ull, ~0ull}, khi[2] = {0ull, 0ull};
        bool all_eq = true;
        if (have_pre) {
          klo[0] = pre_lo[0]; klo[1] = pre_lo[1]; khi[0] = pre_hi[0]; khi[1] = pre_hi[1];
        } else if (m <= kLaneDimMax) {
          // small node: lane d walks the node's points along its own dimension(s); no cross-lane reduction
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            const int d = hh * 32 + lane;
            if (hh * 32 >= a.D) break;
            const uint64_t *col = skeys + (size_t)(d < a.D ? d : 0) * NMAX;
            uint64_t mn = ~0ull, mx = 0ull;
            for (int j = nb0; j < ne0; ++j) { const uint64_t k = col[ids[j]]; mn = k < mn ? k : mn; mx = k > mx ? k : mx; }
            if (d < a.D) { klo[hh] = mn; khi[hh] = mx; }
          }
        } else {
          for (int d = 0; d < a.D; ++d) {
            const uint64_t *col = skeys + (size_t)d * NMAX;
            uint64_t mn = ~0ull, mx = 0ull;
            for (int j = nb0 + lane; j < ne0; j += 32) { const uint64_t k = col[ids[j]]; mn = k < mn ? k : mn; mx = k > mx ? k : mx; }
            mn = warp_min_u64(mn); mx = warp_max_u64(mx);
            if ((d & 31) == lane) { klo[d >> 5] = mn; khi[d >> 5] = mx; }
          }
        }
        {
          const bool differs = (lane < a.D && klo[0] != khi[0]) || (lane + 32 < a.D && klo[1] != khi[1]);
          all_eq = !__any_sync(full, differs);
        }
        if (!all_eq) {                                                // :159-160
          // longest_dim (:120-130): first strictly largest spread, in float64
          double dx_best = neg_inf(); int d_best = -1;
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            const int d = hh * 32 + lane;
            double dx = neg_inf(); bool ok = false;
            if (d < a.D) { dx = ordered_to_f64(khi[hh]) - ordered_to_f64(klo[hh]); ok = dx > neg_inf(); }   // NaN never wins (`dx > !dx_max`)
            if (!ok) dx = neg_inf();
            double mxv = dx;
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) { const double o = __shfl_xor_sync(full, mxv, off); mxv = o > mxv ? o : mxv; }
            const unsigned who = __ballot_sync(full, ok && dx == mxv);
            if (who && mxv > dx_best) { dx_best = mxv; d_best = hh * 32 + __ffs(who) - 1; }
          }
          sd = d_best;
        }
        if (sd >= 0) {
          const uint64_t *col = skeys + (size_t)sd * NMAX;
          const uint64_t lo = __shfl_sync(full, klo[sd >> 5], sd & 31), hi = __shfl_sync(full, khi[sd >> 5], sd & 31);
          // the m/2-th order statistic (:162-167): MSB-first radix select below the bytes lo and hi share, finished
          // by ranking once at most 32 candidates are left
          int shift = ((63 - __clzll((long long)(lo ^ hi))) >> 3) << 3;
          uint64_t prefix = shift >= 56 ? 0ull : (lo >> (shift + 8)) << (shift + 8);
          int kth = m / 2, below_tot = 0, cnt_eq = 0, cand_n = m, cshift = 64;
          uint64_t v = 0ull;
          while (cand_n > 32 && cshift != 0) {
            for (int q = lane; q < 256; q += 32) h[q] = 0u;
            __syncwarp();
            for (int j = nb0 + lane; j < ne0; j += 32) {
              const uint64_t k = col[ids[j]];
              if (shift >= 56 || ((k ^ prefix) >> (shift + 8)) == 0ull) atomicAdd(&h[(unsigned)(k >> shift) & 255u], 1u);
            }
            __syncwarp();
            uint32_t c[8]; uint32_t sum = 0;
#pragma unroll
            for (int q = 0; q < 8; ++q) { c[q] = h[lane * 8 + q]; sum += c[q]; }
            uint32_t incl = sum;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) { const uint32_t x = __shfl_up_sync(full, incl, off); if (lane >= off) incl += x; }
            const uint32_t excl = incl - sum;
            const bool mine = (uint32_t)kth >= excl && (uint32_t)kth < incl;
            const int src = __ffs(__ballot_sync(full, mine)) - 1;
            int bin = 0; uint32_t below = 0, cn = 0;
            if (mine) {
              uint32_t run = excl;
#pragma unroll
              for (int q = 0; q < 8; ++q) { if ((uint32_t)kth >= run && (uint32_t)kth < run + c[q]) { bin = lane * 8 + q; below = run; cn = c[q]; } run += c[q]; }
            }
            bin = __shfl_sync(full, bin, src); below = __shfl_sync(full, below, src); cn = __shfl_sync(full, cn, src);
            prefix |= (uint64_t)bin << shift;
            kth -= (int)below; below_tot += (int)below; cand_n = (int)cn; cshift = shift; shift -= 8;
            __syncwarp();
          }
          if (cand_n > 32) { v = prefix; cnt_eq = cand_n; }          // every bit decided: cand_n copies of one key
          else {
            int pos = 0;
            for (int j0 = nb0; j0 < ne0; j0 += 32) {
              const int j = j0 + lane;
              const uint64_t k = j < ne0 ? col[ids[j]] : 0ull;
              const bool match = j < ne0 && (cshift >= 64 || ((k ^ prefix) >> cshift) == 0ull);
              const unsigned mk = __ballot_sync(full, match);
              if (match) cand[pos + __popc(mk & lt)] = k;
              pos += __popc(mk);
            }
            __syncwarp();
            const bool have = lane < cand_n;
            const uint64_t mine = have ? cand[lane] : ~0ull;
            int rank = 0;
            for (int q = 0; q < cand_n; ++q) { const uint64_t o = __shfl_sync(full, mine, q); rank += (o < mine || (o == mine && q < lane)) ? 1 : 0; }
            const int src = __ffs(__ballot_sync(full, have && rank == kth)) - 1;
            v = __shfl_sync(full, mine, src < 0 ? 0 : src);
            below_tot += __popc(__ballot_sync(full, have && mine < v));
            cnt_eq = __popc(__ballot_sync(full, have && mine == v));
            __syncwarp();
          }
          int cntL = below_tot + cnt_eq;                              // keys <= v   (List.partition (<= pvt), :168)
          const bool fix = (cntL == m);                               // adjust_for_empty_split :150-152: L = {k < max}
          if (fix) cntL = below_tot;
          spos = nb0 + cntL;
          // max L / min R (:170-171) and the stable partition (:168)
          uint64_t ml = 0ull, mr = ~0ull;
          int lc = 0, rc = 0;
          for (int j0 = nb0; j0 < ne0; j0 += 32) {
            const int j = j0 + lane;
            const bool valid = j < ne0;
            const unsigned id = valid ? ids[j] : 0u;
            const uint64_t k = valid ? col[id] : 0ull;
            const bool left = valid && (fix ? (k < v) : (k <= v)), right = valid && !left;
            if (left) ml = k > ml ? k : ml;
            if (right) mr = k < mr ? k : mr;
            const unsigned Lm = __ballot_sync(full, left), Rm = __ballot_sync(full, right);
            if (left) idn[nb0 + lc + __popc(Lm & lt)] = (uint16_t)id;
            if (right) idn[spos + rc + __popc(Rm & lt)] = (uint16_t)id;
            lc += __popc(Lm); rc += __popc(Rm);
          }
          ml = warp_max_u64(ml); mr = warp_min_u64(mr);
          split = 0.5 * (ordered_to_f64(ml) + ordered_to_f64(mr));    // split_bounds :113
        }
      }
      if (sd < 0) for (int j = nb0 + lane; j < ne0; j += 32) idn[j] = ids[j];
      if (lane == 0) {
        spl[node] = sd >= 0 ? 1 : 0; sps[node] = (uint16_t)spos;
        const int64_t gk = gbase + lbase + node;
        a.l_dim[gk] = sd; a.l_split[gk] = split; a.l_begin[gk] = nb0; a.l_end[gk] = ne0; a.l_child[gk] = -1;
      }
    }
    __syncthreads();
    // children in parent order: exclusive scan of is_split over the level's nodes
    int carry = 0;
    for (int base = 0; base < cur_n; base += BT) {
      const int node = base + tid;
      const int is = node < cur_n ? spl[node] : 0;
      int incl = is;
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) { const int x = __shfl_up_sync(full, incl, off); if (lane >= off) incl += x; }
      if (lane == 31) s_scan[warp] = incl;
      __syncthreads();
      if (warp == 0) {
        int x = lane < nwarps ? s_scan[lane] : 0, xi = x;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) { const int y = __shfl_up_sync(full, xi, off); if (lane >= off) xi += y; }
        if (lane < nwarps) s_scan[lane] = xi - x;
        if (lane == nwarps - 1) s_tot = xi;
      }
      __syncthreads();
      const int ex = carry + incl - is + s_scan[warp];
      if (is) {
        const int c = 2 * ex;
        a.l_child[gbase + lbase + node] = c;
        nb_[c] = cb[node]; ne_[c] = sps[node]; nb_[c + 1] = sps[node]; ne_[c + 1] = ce[node];
      }
      carry += s_tot;
      __syncthreads();
    }
    const int nsplit = carry;
    if (nsplit == 0) break;
    lbase += cur_n; cur_n = 2 * nsplit; ++l; level_max = level_max / 2 + 1;
    if (l >= V2_MAXL) { if (tid == 0) *a.overflow = 1; --l; break; }
    { uint16_t *x = ids; ids = idn; idn = x; x = cb; cb = nb_; nb_ = x; x = ce; ce = ne_; ne_ = x; }
    __syncthreads();
  }
  // the last level's nodes were all leaves: idn holds their (unchanged) order
  for (int j = tid; j < n; j += BT) a.perm_out[b + j] = a.perm_in[b + idn[j]];
  if (tid == 0) { a.depth[s] = l + 1; for (int q = l + 1; q < V2_MAXL; ++q) cnt[q] = 0; }
}

// prefix over the subtrees of the node counts of every local level: pre[s][l] = sum_{s' < s} cnt[s'][l]
__global__ void __launch_bounds__(1024)
v2_level_scan_kernel(const int32_t *__restrict__ cnt, int32_t *__restrict__ pre, int nsub, int32_t *__restrict__ totals) {
  const int l = blockIdx.x;
  __shared__ int carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < nsub; base += 1024) {
    const int s = base + threadIdx.x;
    const int v = s < nsub ? cnt[(size_t)s * V2_MAXL + l] : 0;
    int tot;
    const int ex = block_exclusive_scan<1024>(v, &tot);
    const int c = carry;
    if (s < nsub) pre[(size_t)s * V2_MAXL + l] = c + ex;
    __syncthreads();
    if (threadIdx.x == 0) carry = c + tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) totals[l] = carry;
}

struct V2LevelBase { int32_t base[V2_MAXL + 1]; };

__global__ void v2_emit_top_kernel(V2Top t, int64_t nn_top, KdNode *__restrict__ nodes, int32_t *__restrict__ count,
                                   int32_t *__restrict__ begin_out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nn_top; i += (int64_t)gridDim.x * blockDim.x) {
    KdNode nd; nd.split = t.nsplit[i]; nd.left = t.nleft[i]; nd.dim = t.ndim[i];
    nodes[i] = nd; count[i] = t.ne[i] - t.nb[i]; begin_out[i] = t.nb[i];
  }
}

__global__ void __launch_bounds__(256)
v2_emit_bottom_kernel(V2Bottom a, const int32_t *__restrict__ pre, V2LevelBase lb, KdNode *__restrict__ nodes,
                      int32_t *__restrict__ count, int32_t *__restrict__ begin_out) {
  const V2Level lv = a.info->lvl[a.L0];
  const int s = blockIdx.x;
  if (s >= lv.le - lv.lb) return;
  const int g = lv.lb + s;
  const int32_t b = a.nb[g];
  const int32_t *cnt = a.cnt + (size_t)s * V2_MAXL, *pr = pre + (size_t)s * V2_MAXL;
  const int depth = a.depth[s];
  int lstart = 0;
  for (int l = 0; l < depth; ++l) {
    const int c = cnt[l];
    for (int i = threadIdx.x; i < c; i += blockDim.x) {
      const int64_t gk = 2 * (int64_t)b + lstart + i;
      const int gid = l == 0 ? g : lb.base[l] + pr[l] + i;
      const int ch = a.l_child[gk];
      KdNode nd; nd.split = a.l_split[gk]; nd.dim = a.l_dim[gk];
      nd.left = ch < 0 ? -1 : lb.base[l + 1] + pr[l + 1] + ch;
      nodes[gid] = nd; count[gid] = a.l_end[gk] - a.l_begin[gk]; begin_out[gid] = b + a.l_begin[gk];
    }
    lstart += c;
  }
}

template <int NMAX, int BT>
static int v2_launch_bottom(mg_ctx *ctx, const V2Bottom &a, int nsub, int D) {
  const size_t smem = v2_bottom_smem<NMAX, BT>(D);
  MG_CUDA(ctx, cudaFuncSetAttribute(v2_bottom_kernel<NMAX, BT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  v2_bottom_kernel<NMAX, BT><<<(unsigned)nsub, BT, smem, ctx->stream>>>(a);
  MG_CHECK_LAUNCH(ctx);
  return MG_OK;
}

// Returns MG_OK, an error, or MG_V2_FALLBACK (the caller then runs the first builder).
int build_tree_v2(mg_ctx *ctx, const double *d_pts, int64_t N, int D, const double *low, const double *high, int min_split,
                  bool with_pts, KdTreePtr *out) {
  cudaStream_t s = ctx->stream;
  // the largest subtree whose key columns fit the shared memory of one SM
  constexpr size_t smem_cap = 224 * 1024;
  const int NMAX = v2_bottom_smem<2048, 1024>(D) <= smem_cap ? 2048 : v2_bottom_smem<1024, 1024>(D) <= smem_cap ? 1024
                   : v2_bottom_smem<512, 512>(D) <= smem_cap ? 512 : 256;
  if (N >= (1LL << 30)) return MG_V2_FALLBACK;
  int L0 = 0;
  { int64_t sz = N; while (sz > NMAX) { sz = sz / 2 + 1; ++L0; } }
  if (L0 + V2_EXTRA >= V2_MAXLEV) return MG_V2_FALLBACK;
  const int32_t LC = (int32_t)std::min<int64_t>(std::max<int64_t>(N, 1), 1LL << std::min(L0 + V2_EXTRA, 30));
  const int64_t cap_top = std::min<int64_t>(2 * N + 2, 2LL * LC * 2 + 4);       // nodes of all top levels
  time_begin(ctx);
  kt_reset(ctx, (const void *)v2_scatter_kernel);
  DevBuf<uint64_t> KA, KB, lo, hi, lo2, hi2, v, maxL, minR;
  DevBuf<int32_t> permA, permB, segA, segB, nb, ne, ndim, nleft, nspos, kth, below, nR, ebegin;
  DevBuf<double> nsplit;
  DevBuf<V2Sel> sel; DevBuf<uint32_t> hist; DevBuf<uint8_t> fix; DevBuf<V2Info> info;
  DevBuf<unsigned long long> status; DevBuf<unsigned int> ticket; DevBuf<int> nan_flag;
  const int64_t ntiles = (N + V2_TILE - 1) / V2_TILE;
  MG_CUDA(ctx, KA.alloc((size_t)D * N, s)); MG_CUDA(ctx, KB.alloc((size_t)D * N, s));
  MG_CUDA(ctx, permA.alloc(N, s)); MG_CUDA(ctx, permB.alloc(N, s)); MG_CUDA(ctx, segA.alloc(N, s)); MG_CUDA(ctx, segB.alloc(N, s));
  MG_CUDA(ctx, nb.alloc(cap_top, s)); MG_CUDA(ctx, ne.alloc(cap_top, s)); MG_CUDA(ctx, ndim.alloc(cap_top, s));
  MG_CUDA(ctx, nleft.alloc(cap_top, s)); MG_CUDA(ctx, nspos.alloc(cap_top, s)); MG_CUDA(ctx, nsplit.alloc(cap_top, s));
  MG_CUDA(ctx, lo.alloc((size_t)LC * D, s)); MG_CUDA(ctx, hi.alloc((size_t)LC * D, s));
  MG_CUDA(ctx, lo2.alloc((size_t)LC * D, s)); MG_CUDA(ctx, hi2.alloc((size_t)LC * D, s));
  MG_CUDA(ctx, sel.alloc(LC, s)); MG_CUDA(ctx, kth.alloc(LC, s)); MG_CUDA(ctx, below.alloc(LC, s)); MG_CUDA(ctx, hist.alloc((size_t)LC * 256, s));
  MG_CUDA(ctx, v.alloc(LC, s)); MG_CUDA(ctx, maxL.alloc(LC, s)); MG_CUDA(ctx, minR.alloc(LC, s)); MG_CUDA(ctx, fix.alloc(LC, s));
  MG_CUDA(ctx, nR.alloc(LC, s)); MG_CUDA(ctx, ebegin.alloc(LC, s)); MG_CUDA(ctx, info.alloc(1, s));
  MG_CUDA(ctx, status.alloc((size_t)ntiles, s)); MG_CUDA(ctx, ticket.alloc(1, s)); MG_CUDA(ctx, nan_flag.alloc(1, s));
  MG_CUDA(ctx, cudaMemsetAsync(hist.get(), 0, sizeof(uint32_t) * (size_t)LC * 256, s));
  V2Top t{N, D, min_split, LC, (int32_t)cap_top, info.get(), nb.get(), ne.get(), ndim.get(), nleft.get(), nspos.get(), nsplit.get(),
          lo.get(), hi.get(), sel.get(), kth.get(), below.get(), hist.get(), v.get(), maxL.get(), minR.get(), fix.get(), nR.get(), ebegin.get()};
  const unsigned gtile = (unsigned)ntiles;
  {
    const size_t mk_smem = (size_t)V2_MK * (D | 1) * sizeof(double);
    if (mk_smem > 48 * 1024) MG_CUDA(ctx, cudaFuncSetAttribute(v2_make_keys_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mk_smem));
    const int64_t gb = std::min<int64_t>((N + V2_MK - 1) / V2_MK, (int64_t)ctx->sm_count * 16);
    v2_init_kernel<<<1, 32, 0, s>>>(t);
    MG_CHECK_LAUNCH(ctx);
    v2_level_init_kernel<<<1, 64, 0, s>>>(t, 0, t.lo, t.hi);          // the root's bounds: filled by the key pass
    MG_CHECK_LAUNCH(ctx);
    MG_CUDA(ctx, cudaMemsetAsync(nan_flag.get(), 0, sizeof(int), s));
    v2_make_keys_kernel<<<(unsigned)gb, 256, mk_smem, s>>>(d_pts, N, D, KA.get(), permA.get(), segA.get(), t.lo, t.hi, nan_flag.get());
    MG_CHECK_LAUNCH(ctx);
  }
  uint64_t *lo_next = lo2.get(), *hi_next = hi2.get();
  uint64_t *Kin = KA.get(), *Kout = KB.get();
  int32_t *pin = permA.get(), *pout = permB.get(), *sin = segA.get(), *sout = segB.get();
  auto run_level = [&](int L) -> int {
    const int64_t nodes_cap = std::min<int64_t>(LC, 1LL << std::min(L, 30));
    const unsigned gnode = (unsigned)((nodes_cap + 127) / 128);
    // (the root's bounds came with the key pass, deeper levels received theirs from the scatter pass of their parents)
    v2_node_kernel<<<gnode, 128, 0, s>>>(t, L);
    MG_CHECK_LAUNCH(ctx);
    for (int pass = 0; pass < 8; ++pass) {
      v2_hist_kernel<<<gtile, V2_TB, 0, s>>>(t, L, Kin, sin);
      MG_CHECK_LAUNCH(ctx);
      v2_pick_kernel<<<(unsigned)((nodes_cap * 32 + 255) / 256), 256, 0, s>>>(t, L);
      MG_CHECK_LAUNCH(ctx);
    }
    v2_children_kernel<<<1, 1024, 0, s>>>(t, L);
    MG_CHECK_LAUNCH(ctx);
    MG_CUDA(ctx, cudaMemsetAsync(status.get(), 0, sizeof(unsigned long long) * (size_t)ntiles, s));
    MG_CUDA(ctx, cudaMemsetAsync(ticket.get(), 0, sizeof(unsigned int), s));
    {
      const int64_t next_cap = std::min<int64_t>(LC, 2 * nodes_cap);
      v2_level_init_kernel<<<(unsigned)std::min<int64_t>((next_cap * D + 255) / 256, 4096), 256, 0, s>>>(t, L + 1, lo_next, hi_next);
      MG_CHECK_LAUNCH(ctx);
    }
    kt_start(ctx);
    v2_scatter_kernel<<<gtile, V2_TB, 0, s>>>(t, L, Kin, Kout, pin, pout, sin, sout, status.get(), ticket.get(), lo_next, hi_next,
                                              ctx->d_devflag);
    kt_stop(ctx);
    MG_CHECK_LAUNCH(ctx);
    v2_split_kernel<<<gnode, 128, 0, s>>>(t, L);
    MG_CHECK_LAUNCH(ctx);
    std::swap(Kin, Kout); std::swap(pin, pout); std::swap(sin, sout);
    std::swap(t.lo, lo_next); std::swap(t.hi, hi_next);
    return MG_OK;
  };
  int rc;
  // A truncated build (min_split above the subtree size: Evidence with a large n, the top of a distributed build)
  // stops splitting long before the hand-over level: without ties a node of level L holds at most (N >> L) + 2
  // points (s' <= s / 2 + 1), so the level loop is cut where that falls below min_split and the read-back below
  // decides the rest.
  int Lrun = L0;
  if (min_split > NMAX) { Lrun = 0; while (Lrun < L0 && (N >> Lrun) + 2 >= (int64_t)min_split) ++Lrun; }
  for (int L = 0; L < Lrun; ++L) if ((rc = run_level(L))) return rc;
  V2Info h_info;
  int Lh = Lrun;                                 // the hand-over level
  bool leaves_only = false;                      // no node of level Lh splits: the top phase has built the whole tree
  for (;;) {
    int h_nan = 0;
    MG_CUDA(ctx, cudaMemcpyAsync(&h_info, info.get(), sizeof h_info, cudaMemcpyDeviceToHost, s));
    MG_CUDA(ctx, cudaMemcpyAsync(&h_nan, nan_flag.get(), sizeof(int), cudaMemcpyDeviceToHost, s));
    MG_CUDA(ctx, cudaStreamSynchronize(s));
    // NaN coordinates are rejected (Pervasives.compare orders them, IEEE does not); as keys they are ordinary
    // integers, so the levels above ran to completion on them
    MG_REQUIRE(ctx, h_nan == 0, "kd-tree: NaN coordinate");
    if (h_info.overflow) return MG_V2_FALLBACK;
    if (h_info.maxsize[Lh] < min_split && h_info.maxsize[Lh] > NMAX) { leaves_only = true; break; }
    if (h_info.maxsize[Lh] <= NMAX) break;
    if (Lh >= L0 + V2_EXTRA) return MG_V2_FALLBACK;   // heavy ties: subtrees do not shrink -> first builder
    if ((rc = run_level(Lh))) return rc;
    ++Lh;
  }
  int nsub = h_info.lvl[Lh].le - h_info.lvl[Lh].lb;
  const int64_t nn_top = h_info.nnodes;
  if (leaves_only) {                             // the nodes of level Lh are leaves: give them their fields, no bottom phase
    if (nsub > 0) {
      v2_node_kernel<<<(unsigned)((nsub + 127) / 128), 128, 0, s>>>(t, Lh);
      MG_CHECK_LAUNCH(ctx);
      h_info.nlevels = std::max(h_info.nlevels, Lh + 1);   // (counted by the children pass of a level, which did not run)
    }
    nsub = 0;
  }
  // ---- bottom phase ----------------------------------------------------------------------------------------------
  DevBuf<int32_t> l_dim, l_child, l_begin, l_end, cnt, pre, depth, totals, perm_fin;
  DevBuf<double> l_split;
  DevBuf<int> b_over;
  int64_t nnodes = nn_top;
  int nlevels = h_info.nlevels;
  V2LevelBase lbase{};
  V2Bottom a{};
  if (nsub > 0) {
    MG_CUDA(ctx, l_dim.alloc((size_t)2 * N, s)); MG_CUDA(ctx, l_child.alloc((size_t)2 * N, s)); MG_CUDA(ctx, l_begin.alloc((size_t)2 * N, s));
    MG_CUDA(ctx, l_end.alloc((size_t)2 * N, s)); MG_CUDA(ctx, l_split.alloc((size_t)2 * N, s));
    MG_CUDA(ctx, cnt.alloc((size_t)nsub * V2_MAXL, s)); MG_CUDA(ctx, pre.alloc((size_t)nsub * V2_MAXL, s));
    MG_CUDA(ctx, depth.alloc(nsub, s)); MG_CUDA(ctx, totals.alloc(V2_MAXL, s)); MG_CUDA(ctx, b_over.alloc(1, s));
    MG_CUDA(ctx, cudaMemsetAsync(b_over.get(), 0, sizeof(int), s));
    MG_CUDA(ctx, cudaMemcpyAsync(pout, pin, sizeof(int32_t) * N, cudaMemcpyDeviceToDevice, s));   // positions outside the subtrees
    a = V2Bottom{N, D, min_split, Lh, info.get(), nb.get(), ne.get(), Kin, pin, pout, l_dim.get(), l_child.get(), l_begin.get(),
                 l_end.get(), l_split.get(), cnt.get(), depth.get(), b_over.get()};
    rc = NMAX == 2048 ? v2_launch_bottom<2048, 1024>(ctx, a, nsub, D)
         : NMAX == 1024 ? v2_launch_bottom<1024, 1024>(ctx, a, nsub, D)
         : NMAX == 512 ? v2_launch_bottom<512, 512>(ctx, a, nsub, D) : v2_launch_bottom<256, 256>(ctx, a, nsub, D);
    if (rc) return rc;
    v2_level_scan_kernel<<<V2_MAXL, 1024, 0, s>>>(cnt.get(), pre.get(), nsub, totals.get());
    MG_CHECK_LAUNCH(ctx);
    int32_t h_tot[V2_MAXL]; int h_over = 0;
    MG_CUDA(ctx, cudaMemcpyAsync(h_tot, totals.get(), sizeof h_tot, cudaMemcpyDeviceToHost, s));
    MG_CUDA(ctx, cudaMemcpyAsync(&h_over, b_over.get(), sizeof(int), cudaMemcpyDeviceToHost, s));
    MG_CUDA(ctx, cudaStreamSynchronize(s));
    if (h_over) return MG_V2_FALLBACK;             // a subtree deeper than the local level budget
    lbase.base[0] = 0; lbase.base[1] = (int32_t)nn_top;
    int dmax = 1;
    for (int l = 1; l < V2_MAXL; ++l) {
      lbase.base[l + 1] = lbase.base[l] + h_tot[l];
      if (h_tot[l] > 0) dmax = l + 1;
    }
    nnodes = lbase.base[V2_MAXL];
    nlevels = std::max(nlevels, Lh + dmax);
    std::swap(pin, pout);                           // pin = final order
  }
  if (nnodes > 2 * N) return set_err(ctx, MG_EFAIL, "kd-tree: node capacity exceeded");
  // ---- the blob: nodes, counts, begins and the order of the points are this builder's --------------------------------
  KdTreePtr tr;
  if ((rc = kd_alloc(ctx, kd_layout(N, D, nnodes, with_pts), &tr))) return rc;
  tr->h.nlevels = nlevels; tr->h.min_split = min_split;
  // first node of every level: the top levels as the level loop numbered them, the subtree levels from the scan
  for (int L = 0; L <= Lh && L < nlevels; ++L) tr->level_begin.push_back(h_info.lvl[L].lb);
  for (int l = 1; Lh + l < nlevels; ++l) tr->level_begin.push_back(lbase.base[l]);
  tr->level_begin.push_back((int32_t)nnodes);
  const KdHeader &h = tr->h;
  char *blob = (char *)tr->d_blob;
  KdNode *nodes = (KdNode *)(blob + h.off_nodes);
  int32_t *count = (int32_t *)(blob + h.off_count), *begin_out = (int32_t *)(blob + h.off_begin);
  v2_emit_top_kernel<<<(unsigned)std::min<int64_t>((nn_top + 255) / 256, 4096), 256, 0, s>>>(t, nn_top, nodes, count, begin_out);
  MG_CHECK_LAUNCH(ctx);
  if (nsub > 0) {
    v2_emit_bottom_kernel<<<(unsigned)nsub, 256, 0, s>>>(a, pre.get(), lbase, nodes, count, begin_out);
    MG_CHECK_LAUNCH(ctx);
  }
  MG_CUDA(ctx, cudaMemcpyAsync(blob + h.off_perm, pin, 4 * N, cudaMemcpyDeviceToDevice, s));
  time_end(ctx);
  return kd_finish(ctx, std::move(tr), low, high, d_pts, out);
}

}  // namespace mg
