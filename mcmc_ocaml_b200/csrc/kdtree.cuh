// kdtree.cuh -- flat kd-tree in HBM and the point-location descent
// (interpolate_pdf.ml:88-109) shared by the Interpolate_pdf kernels and the
// reversible-jump sampler.
//
// Layout.  One contiguous device blob (so that a tree can be broadcast to the
// other GPUs with a single NCCL call):
//   header | root low[D] | root high[D] | nodes[nnodes] (16 B: split value,
//   left child, split dim) | count[nnodes] | begin[nnodes] | perm[N] |
//   pts[N][D]
// Nodes are numbered breadth first, children of a split node adjacent
// (left, left + 1); a leaf has left = -1.  A node does not store its box:
// boxes are inherited (kd_tree.ml:174-175) and are rebuilt during the descent
// from the root box and the (dim, split) pairs on the path, exactly as
// split_bounds (kd_tree.ml:112-118) builds them.
#pragma once
#ifndef __CUDACC_RTC__
#include <cstdint>
#endif

#include "models.cuh"

namespace mg {

struct KdNode {
  double split;
  int32_t left;   // -1: leaf
  int32_t dim;
};
static_assert(sizeof(KdNode) == 16, "KdNode must be 16 bytes");

struct KdHeader {
  uint64_t magic;
  int64_t N, nnodes, nbytes;
  int32_t D, nlevels, min_split, pad;
  int64_t off_low, off_high, off_nodes, off_count, off_begin, off_perm, off_pts;
};
constexpr uint64_t KD_MAGIC = 0x6b64747265653031ull;  // "kdtree01"

struct KdView {
  const KdNode *nodes;
  const int32_t *count;
  const double *low, *high;  // root box
  const double *pts;         // [N][D]
  int64_t N;
  int32_t D;
  // optional: for every stored point the cell that find_cell reaches from it -- box low[D], high[D], object count,
  // node id (2 D + 2 doubles per point), written by the same descent (mg_kdtree_enable_draw_cache).  Interp.draw
  // then costs one gather instead of one dependent node load per level.
  const double *dcache;
};

// Shared-memory scratch of one thread: q, lo, hi, each D doubles, laid out
// [d][blockDim.x] so that a warp touching one coordinate is conflict free.
struct KdScratch {
  double *q, *lo, *hi;
  int stride;
  __device__ __forceinline__ double &Q(int d) const { return q[d * stride]; }
  __device__ __forceinline__ double &LO(int d) const { return lo[d * stride]; }
  __device__ __forceinline__ double &HI(int d) const { return hi[d * stride]; }
};

__device__ __forceinline__ KdScratch kd_scratch(double *smem_base, int D) {
  KdScratch s;
  s.stride = blockDim.x;
  s.q = smem_base + threadIdx.x;
  s.lo = s.q + (size_t)D * blockDim.x;
  s.hi = s.lo + (size_t)D * blockDim.x;
  return s;
}
#ifndef __CUDACC_RTC__
inline size_t kd_scratch_bytes(int D, int block) { return (size_t)3 * D * block * sizeof(double); }
#endif

// find_cell (interpolate_pdf.ml:101-109) / the *_high_level descents
// (:121-133,144-159).  The query is in s.Q(.).  Go left iff the point lies in
// the left child's box on ALL dimensions, bounds inclusive (:88-99,106);
// otherwise go right without checking.  `out_mask` tracks on which
// dimensions the point is outside the current box, so the all-dimension test
// costs O(1) per level.  On return s.LO / s.HI hold the cell's box.
// Returns the node id, or -1 where the reference raises (high-level descent
// reaching an Empty child).
__device__ __forceinline__ int32_t kd_descend(const KdView &t, const KdScratch &s, int nstop) {
  uint64_t out_mask = 0;
  for (int d = 0; d < t.D; ++d) {
    const double lo = __ldg(t.low + d), hi = __ldg(t.high + d), q = s.Q(d);
    s.LO(d) = lo; s.HI(d) = hi;
    if (!(q >= lo && q <= hi)) out_mask |= (1ull << d);
  }
  int32_t id = 0;
  for (;;) {
    const KdNode nd = *reinterpret_cast<const KdNode *>(
        __builtin_assume_aligned(t.nodes + id, 16));
    if (nstop > 0) {
      if (__ldg(t.count + id) <= nstop) return id;
      if (nd.left < 0) return -1;
    } else if (nd.left < 0) {
      return id;
    }
    const int sd = nd.dim;
    const double q = s.Q(sd);
    const uint64_t bit = 1ull << sd;
    const bool in_left = ((out_mask & ~bit) == 0) && (q >= s.LO(sd)) && (q <= nd.split);
    if (in_left) {
      s.HI(sd) = nd.split;
      out_mask &= ~bit;
      id = nd.left;
    } else {
      s.LO(sd) = nd.split;
      if (q >= nd.split && q <= s.HI(sd)) out_mask &= ~bit; else out_mask |= bit;
      id = nd.left + 1;
    }
  }
}

// Kd_tree.bounds_volume (kd_tree.ml:177-182): left-to-right product from 1.0
__device__ __forceinline__ double kd_cell_volume(const KdScratch &s, int D) {
  double v = 1.0;
  for (int i = 0; i < D; ++i) v = v * (s.HI(i) - s.LO(i));
  return v + 0.0;
}

// Interpolate_pdf.jump_prob (interpolate_pdf.ml:135-159) for the query in s.Q
__device__ __forceinline__ double kd_jump_prob(const KdView &t, const KdScratch &s, int nstop, int32_t *node) {
  const int32_t id = kd_descend(t, s, nstop);
  if (node) *node = id;
  if (id < 0) return qnan();
  const double nobjs = (double)__ldg(t.count + id);
  const double v = kd_cell_volume(s, t.D);
  return nobjs / (v * (double)t.N);
}

// Interpolate_pdf.draw (interpolate_pdf.ml:114-133): pick a stored point,
// locate its cell by descent, draw uniformly in the cell's box.  The result is
// written to s.Q(.).  Returns false where the reference raises.
__device__ __forceinline__ bool kd_draw(const KdView &t, const KdScratch &s, int nstop, Rng &r, int32_t *node = nullptr) {
  const int64_t k = (int64_t)r.below((uint64_t)t.N);
  if (t.dcache != nullptr && nstop == 0) {       // the cell of stored point k, located once by the same descent
    const double *rec = t.dcache + k * (2 * t.D + 2);
    for (int d = 0; d < t.D; ++d) {              // random_in_volume :80-86
      const double lo = __ldg(rec + d), hi = __ldg(rec + t.D + d);
      s.LO(d) = lo; s.HI(d) = hi;
      s.Q(d) = lo + (hi - lo) * r.uniform();
    }
    if (node) *node = (int32_t)__ldg(rec + 2 * t.D + 1);
    return true;
  }
  const double *p = t.pts + k * t.D;
  for (int d = 0; d < t.D; ++d) s.Q(d) = __ldg(p + d);
  const int32_t id = kd_descend(t, s, nstop);
  if (node) *node = id;
  if (id < 0) return false;
  for (int d = 0; d < t.D; ++d) {  // random_in_volume :80-86
    const double lo = s.LO(d), hi = s.HI(d);
    s.Q(d) = lo + (hi - lo) * r.uniform();
  }
  return true;
}

}  // namespace mg

#ifndef __CUDACC_RTC__
#include <memory>
#include <vector>
// host-side handle
struct mg_kdtree {
  mg_ctx *ctx = nullptr;
  void *d_blob = nullptr;
  bool owns_blob = true;
  double *d_draw_cache = nullptr;   // [N][2 D + 2], see KdView::dcache (not part of the blob: rebuilt per rank)
  mg::KdHeader h{};
  std::vector<int32_t> level_begin;  // first node of every level and nnodes at the end (nlevels + 1 entries, either builder)
  mg::KdView view() const {
    const char *b = (const char *)d_blob;
    mg::KdView v;
    v.nodes = (const mg::KdNode *)(b + h.off_nodes);
    v.count = (const int32_t *)(b + h.off_count);
    v.low = (const double *)(b + h.off_low);
    v.high = (const double *)(b + h.off_high);
    v.pts = (const double *)(b + h.off_pts);
    v.N = h.N; v.D = h.D;
    v.dcache = d_draw_cache;
    return v;
  }
};

namespace mg {

// A tree this code still owns (being built, or not yet handed to the caller): destroyed with its blob unless released.
struct KdTreeDelete { void operator()(mg_kdtree *t) const { mg_kdtree_destroy(t); } };
using KdTreePtr = std::unique_ptr<mg_kdtree, KdTreeDelete>;

inline int64_t align256(int64_t x) { return (x + 255) & ~255LL; }

// ---- the blob (kdtree.cu) ----------------------------------------------------------------------------------------------
// kd_layout is the one place that states the section order and alignment.  It leaves room for node_cap nodes and sets
// h.nnodes = node_cap (a builder that fills fewer sets h.nnodes itself); without the points, off_pts == nbytes.
KdHeader kd_layout(int64_t N, int D, int64_t node_cap, bool with_pts);
// a handle that owns a fresh blob of h.nbytes bytes and holds h
int kd_alloc(mg_ctx *ctx, const KdHeader &h, KdTreePtr *out);
// Writes the header, the root box and, where the layout has room for them, the points into t's blob, then waits for
// the stream: a failed copy, kernel or device-side wait is reported and t is freed; otherwise t moves to *out.
int kd_finish(mg_ctx *ctx, KdTreePtr t, const double *low, const double *high, const double *d_pts, KdTreePtr *out);
// checks a blob that arrives from another process before any kernel indexes with it
int validate_blob_header(mg_ctx *ctx, const KdHeader &h);

// Kd_tree.tree_of_objects.  with_pts: the blob carries a copy of the points (Interpolate_pdf draws from it; callers
// that keep the rows themselves leave it out).
int build_tree(mg_ctx *ctx, const double *d_pts, int64_t N, int D, const double *low, const double *high,
               int min_split, bool with_pts, KdTreePtr *out);
// the second builder (kdtree_build2.cu); MG_V2_FALLBACK: this input is for the first builder (not an error)
constexpr int MG_V2_FALLBACK = -1000;
int build_tree_v2(mg_ctx *ctx, const double *d_pts, int64_t N, int D, const double *low, const double *high,
                  int min_split, bool with_pts, KdTreePtr *out);
// the same tree of the N points every rank holds, built by all ranks of c together (comm.cu)
int build_tree_distributed(mg_comm *c, const double *d_pts, int64_t N, int D, const double *low, const double *high,
                           int min_split, bool with_pts, KdTreePtr *out);

}  // namespace mg
#endif  // !__CUDACC_RTC__
