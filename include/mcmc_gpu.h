/* mcmc_gpu.h -- C ABI of the B200-native sampling-and-evidence path.
 *
 * Every entry point replaces one piece of the OCaml interface of
 * farr/mcmc-ocaml (citations are file:line in the reference tree).  The
 * reference has no FFI at all (SURVEY.md F3); this header is the boundary a
 * maintainer binds from OCaml with thin C stubs over float64 Bigarrays
 * (see INTEGRATION.md and ocaml/).  Plain C: opaque handles, plain pointers
 * and sizes, int status codes.  No torch / C++ types cross this boundary.
 *
 * Conventions
 *   - all reals are IEEE float64, all arrays C layout, caller allocated.
 *   - "host" entry points take host pointers (pinned or pageable) and do the
 *     H2D / D2H copies themselves; "*_dev" entry points take device pointers
 *     on the context's device and never touch host memory.
 *   - status: MG_OK or an error; mg_last_error(ctx) gives the message.
 *     MG_EINVAL <-> Invalid_argument, MG_EFAIL <-> Failure,
 *     MG_ECUDA <-> Failure "cuda: ..." on the OCaml side.
 *   - a context is single-caller (the reference is non-reentrant:
 *     global counters mcmc.ml:27-28 and the global Random state).
 *   - there is NO CPU fallback: without a CUDA device mg_ctx_create fails.
 */
#ifndef MCMC_GPU_H
#define MCMC_GPU_H

#ifndef __CUDACC_RTC__
#include <stdint.h>
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define MG_ABI_VERSION 1

enum {
  MG_OK = 0,
  MG_EINVAL = 1, /* Invalid_argument */
  MG_EFAIL = 2,  /* Failure */
  MG_ECUDA = 3,  /* Failure "cuda: ..." */
  MG_ENOMEM = 4
};

typedef struct mg_ctx mg_ctx;
typedef struct mg_kdtree mg_kdtree;
typedef struct mg_comm mg_comm;

/* ------------------------------------------------------------------ */
/* context                                                             */
/* ------------------------------------------------------------------ */

int mg_abi_version(void);
/* Random.init seed (bin/rjmcmc_gaussian_cauchy.ml:24): one Philox4x32-10 key
 * per context; every sampling call consumes one "epoch" of it. */
int mg_ctx_create(int device, uint64_t seed, mg_ctx **out);
void mg_ctx_destroy(mg_ctx *ctx);
const char *mg_last_error(const mg_ctx *ctx);
int mg_ctx_set_seed(mg_ctx *ctx, uint64_t seed);    /* resets epoch to 0 */
int mg_ctx_set_epoch(mg_ctx *ctx, uint64_t epoch);  /* next call uses it  */
uint64_t mg_ctx_get_epoch(const mg_ctx *ctx);
int mg_ctx_set_stream(mg_ctx *ctx, void *cuda_stream); /* NULL = own stream */
void *mg_ctx_get_stream(const mg_ctx *ctx);
int mg_ctx_sync(mg_ctx *ctx);
/* Temporaries are taken from the device's stream-ordered memory pool and kept
 * cached there between calls; this returns the cached memory to the driver
 * (for processes that share the GPU with another allocator). */
int mg_ctx_trim_pool(mg_ctx *ctx);
/* The opposite: make the pool hold at least nbytes in ONE piece (a pool grown
 * request by request answers some 1-2 GB requests by remapping its fragments,
 * 15-180 ms).  mg_ctx_create reserves 12 GB when the device has 48 GB free
 * (MCMC_GPU_POOL_RESERVE_GB overrides, 0 = none); call this after a trim. */
int mg_ctx_reserve_pool(mg_ctx *ctx, int64_t nbytes);
/* Mcmc.reset_counters / Mcmc.get_counters (mcmc.ml:30-35). */
int mg_reset_counters(mg_ctx *ctx);
int mg_get_counters(mg_ctx *ctx, int64_t *naccept, int64_t *nreject);
/* number of kernels this context has launched (bench.py gpu_launches). */
int64_t mg_ctx_launch_count(const mg_ctx *ctx);
/* duration in ms of the dominant kernel of the last sampling / build call,
 * from CUDA events recorded on the context's stream around that launch. */
double mg_ctx_last_kernel_ms(const mg_ctx *ctx);
/* the dominant kernel of the last sampling / build / evidence call: its
 * (demangled) name, how many times the call launched it and the mean duration
 * of a launch in ms (CUDA event pairs on the context's stream around EVERY
 * launch).  bench.py derives roofline.achieved from these. */
int mg_ctx_last_kernel_stats(mg_ctx *ctx, char *name, int64_t name_cap,
                             int64_t *launches, double *mean_ms);

/* diagnostics: device microbenchmarks for the roofline denominators that
 * MEASURED_PEAKS.json lacks (FP64 FMA TFLOP/s; streaming-store GB/s). */
int mg_measure_fp64_tflops(mg_ctx *ctx, int reps, double *out_tflops);
int mg_measure_store_gbs(mg_ctx *ctx, int64_t nbytes, int reps, double *out_gbs);
/* FP64 tensor-core throughput (mma.sync m8n8k4.f64, DMMA) in TFLOP/s. */
int mg_measure_dmma_tflops(mg_ctx *ctx, int reps, double *out_tflops);
/* decision experiment for the north star's tensor-core clause: the quadratic
 * form logc - 1/2 |L (x - mu)|^2 of M device points [D][M], D in {32, 64}, by
 * variant 0 (one thread per point, the sampler plugin's FMA order) or 1 (one
 * warp per 32 points on the FP64 tensor cores).  *ms: kernel time, best of reps. */
int mg_debug_quadform(mg_ctx *ctx, int32_t variant, int32_t D, const double *mu,
                      const double *Lpacked, double logc, const double *d_x,
                      int64_t M, double *d_out, int32_t reps, double *ms);
/* diagnostic: stable radix sort of n float64 keys on the device (the sort
 * under Kd_tree and Evidence); counts order / stability violations. */
int mg_debug_sort_check(mg_ctx *ctx, const double *d_x, int64_t n, int64_t *violations);
/* diagnostic: the sampler's accept test  log u < delta  (mcmc.ml:47) for n host
 * (u, delta) pairs, as the kernels decide it (single-precision estimate with an
 * error bound, float64 log on near-ties) and by the float64 comparison alone;
 * out_fast[i], out_exact[i] in {0, 1}.  The two must agree everywhere. */
int mg_debug_accept_test(mg_ctx *ctx, const double *u, const double *delta, int64_t n,
                         uint8_t *out_fast, uint8_t *out_exact);

/* device / pinned memory helpers for callers without their own allocator */
int mg_malloc_device(mg_ctx *ctx, int64_t nbytes, void **out);
int mg_free_device(mg_ctx *ctx, void *p);
int mg_malloc_pinned(mg_ctx *ctx, int64_t nbytes, void **out);
int mg_free_pinned(mg_ctx *ctx, void *p);
int mg_memcpy_h2d(mg_ctx *ctx, void *dst_dev, const void *src_host, int64_t nbytes);
int mg_memcpy_d2h(mg_ctx *ctx, void *dst_host, const void *src_dev, int64_t nbytes);
int mg_memcpy_d2d(mg_ctx *ctx, void *dst_dev, const void *src_dev, int64_t nbytes);

/* ------------------------------------------------------------------ */
/* plugins: log-density functions and jump proposals                   */
/* ------------------------------------------------------------------ */
/* The reference passes OCaml closures (mcmc.mli:58-60).  Closures cannot
 * cross to the GPU, so the GPU path takes *registered plugins*: a kind id
 * plus a float64 parameter blob.  Built-in kinds cover the models the
 * reference ships in bin/ and test/.  User kinds are added at run time with
 * mg_plugin_register_source (NVRTC, inlined into the sampler kernels) and are
 * accepted wherever a log_likelihood / log_prior is: mg_mcmc_array*,
 * mg_rjmcmc_array*, mg_nested_evidence, mg_evidence_tempered*, mg_logfn_eval. */

enum {
  /* 0.0 */
  MG_FN_ZERO = 0,
  /* params: c -> c */
  MG_FN_CONST = 1,
  /* params: lo[D], hi[D], c -> c if lo<=x<=hi on every dim else -inf
   * (bin/gaussian_cauchy_efficiency.ml:60-67, test/mcmc_test.ml:157-159) */
  MG_FN_BOX_CLOSED = 2,
  /* as above with strict inequalities (test/nested_test.ml:24-28) */
  MG_FN_BOX_OPEN = 3,
  /* params: mu[D], sigma[D] -> Stats.log_multi_gaussian (stats.ml:98-108) */
  MG_FN_GAUSS_DIAG = 4,
  /* params: mu[D], L[D(D+1)/2] (row-major lower triangle of the whitening
   * matrix, L^T L = Sigma^-1), logc -> logc - 1/2 |L (x-mu)|^2
   * (BASELINE.json config 2: 10-D correlated Gaussian) */
  MG_FN_GAUSS_CORR = 5,
  /* D = 2, x = (mu, sigma); params: data[nd] -> sum_i Stats.log_gaussian
   * (bin/gaussian_cauchy_efficiency.ml:69-77) */
  MG_FN_GAUSS_DATA = 6,
  /* D = 2, x = (x0, gamma); params: data[nd] -> sum_i Stats.log_cauchy
   * (bin/gaussian_cauchy_efficiency.ml:79-87) */
  MG_FN_CAUCHY_DATA = 7,
  /* params: c[D], r, w -> log N(|x-c| ; r, w)   (BASELINE.json config 4) */
  MG_FN_SHELL = 8,
  /* params: K, mu[K][D], sigma[D] -> log sum_k exp log_multi_gaussian
   * (test/nested_test.ml:41-53) */
  MG_FN_GAUSS_MIX = 9,
  MG_FN_NKINDS = 10,
  /* ids >= MG_FN_USER are returned by mg_plugin_register_source */
  MG_FN_USER = 1000
};

typedef struct {
  int32_t kind;
  int32_t dim;
  double scale;          /* result = scale * f(x); 1.0 for plain */
  const double *params;  /* host pointer, copied by the call */
  int64_t nparams;
} mg_logfn;

enum {
  /* params: h[D]; x_i + random_between(-h_i, h_i); symmetric
   * (bin/evidence_direct.ml:24-43) */
  MG_PROP_BOX = 0,
  /* params: lo[D], hi[D], dx[D]; Mcmc.uniform_wrapping per coordinate
   * (mcmc.ml:187-196; reflects at the bounds, SURVEY F5c); symmetric */
  MG_PROP_WRAP = 1,
  /* params: mu[D], sigma[D]; y_i = Stats.draw_gaussian mu_i sigma_i
   * independent of x; log q = sum log_gaussian (test/mcmc_test.ml:119-127) */
  MG_PROP_INDEP_GAUSS = 2,
  /* 1-D; params: sigma; left with p=0.75 (test/mcmc_test.ml:66-73) */
  MG_PROP_LEFT_BIASED = 3,
  /* 1-D; params: sign, width; y = x + sign * width * u; log q = -log width
   * on the reachable side, -inf elsewhere (test/mcmc_test.ml:186-199) */
  MG_PROP_ONE_SIDED = 4,
  /* Mcmc.combine_jump_proposals (mcmc.ml:165-185): params: K, then for each
   * component: weight, kind, nparams, params[nparams].  A component is
   * chosen with probability weight / sum; log q is the log-sum-exp over ALL
   * components (Mcmc.log_sum_logs, mcmc.ml:155-163). */
  MG_PROP_MIXTURE = 5,
  /* Mcmc.differential_evolution_proposal ?mode_hopping_frac to_float from_float
   * samples (mcmc.ml:198-218; mcmc.mli:215-218): params: mode_hopping_frac, M,
   * samples[M][D] (the `value`s of the 'a mcmc_sample array, M >= 2).
   * z' = z + d (y - x), x = samples.(i), y = samples.(j), i <> j drawn with
   * Random.int; d = 1 with probability mode_hopping_frac, else
   * Stats.draw_gaussian 0 (2.38 / sqrt (2 D)) (the code, not the doc: SURVEY
   * F5b).  Symmetric: log q = 0. */
  MG_PROP_DE = 6,
  MG_PROP_NKINDS = 7
};

typedef struct {
  int32_t kind;
  int32_t dim;
  const double *params;
  int64_t nparams;
} mg_proposal;

/* Compile a user log-density as CUDA source with NVRTC and register it.
 * `body` is the body of
 *   __device__ double f(const double* x, int dim, const double* p, long np)
 * The function is inlined into freshly compiled sampler kernels (no
 * indirect call in the hot loop).  Returns the new kind id in *kind. */
int mg_plugin_register_source(mg_ctx *ctx, const char *name, const char *body,
                              int32_t *kind);

/* Evaluate a log-density plugin on M points (host [M][D]); used by the
 * parity tests and by Nested for the initial live points. */
int mg_logfn_eval(mg_ctx *ctx, const mg_logfn *fn, const double *x, int64_t M,
                  double *out);

/* ------------------------------------------------------------------ */
/* Mcmc: ensembles of independent Metropolis-Hastings chains           */
/* ------------------------------------------------------------------ */

/* Sample block layout (device and host): [n][D+2][C] float64 -- sample s,
 * field f (0..D-1 coordinates, D log_likelihood, D+1 log_prior), chain c.
 * A warp of 32 chains stores 256 contiguous bytes per field per step.
 * MG_LAYOUT_CHAIN_MAJOR asks the host entry points for [C][n][D+2] instead
 * (one 'a mcmc_sample array per chain, mcmc.mli:33-42), transposed on the
 * device before the D2H copy. */
enum { MG_LAYOUT_STEP_MAJOR = 0, MG_LAYOUT_CHAIN_MAJOR = 1 };

typedef struct {
  int64_t nchains;      /* C */
  int32_t dim;          /* D */
  int32_t layout;       /* MG_LAYOUT_* of out_samples (host entry only) */
  int64_t nbin;         /* ?nbin, default 0   (mcmc.ml:58) */
  int64_t nskip;        /* ?nskip, default 1  (mcmc.ml:58) */
  int64_t n;            /* samples per chain; slot 0 = state after nbin */
  uint64_t chain_offset;/* global id of chain 0 (shards across GPUs) */
  int32_t x0_shared;    /* 1: x0 is one start point [D] used by all chains */
  int32_t reserved;
} mg_mcmc_cfg;

/* Mcmc.mcmc_array (mcmc.ml:58-72) for C independent chains.
 * x0: host [C][D] (or [D] if x0_shared).  out_samples: host, layout above,
 * may be NULL (then only counters / final state are produced).
 * out_accept / out_reject: per chain [C], may be NULL. */
int mg_mcmc_array(mg_ctx *ctx, const mg_logfn *like, const mg_logfn *prior,
                  const mg_proposal *prop, const mg_mcmc_cfg *cfg,
                  const double *x0, double *out_samples, int64_t *out_accept,
                  int64_t *out_reject);

/* Device-resident form.  d_state: [D+2][C] in/out (coordinates, ll, lp; ll
 * and lp are recomputed from the coordinates on entry, mcmc.ml:59-61).
 * d_samples: [n][D+2][C] or NULL.  d_accept: int32 [C] accumulated, or NULL.
 * Asynchronous on the context stream. */
int mg_mcmc_array_dev(mg_ctx *ctx, const mg_logfn *like, const mg_logfn *prior,
                      const mg_proposal *prop, const mg_mcmc_cfg *cfg,
                      double *d_state, double *d_samples, int32_t *d_accept);

/* Mcmc.mcmc_array whose sample block stays in HBM for the GPU consumers that
 * follow it in every reference program (Interp.make, Evidence.*, Stats.*;
 * e.g. bin/gaussian_cauchy_efficiency.ml:99-130), returning to the host what
 * a caller inspects after a run: the final sample of every chain, the
 * accept / reject counters and the per-field mean and std over all recorded
 * samples (Stats.multi_mean / multi_std over the pooled chains).
 * x0: host [C][D] or [D].  d_samples: device [n][D+2][C], caller owned.
 * out_final: host [C][D+2] or NULL.  out_mean / out_std: host [D+2] or NULL. */
int mg_mcmc_array_resident(mg_ctx *ctx, const mg_logfn *like,
                           const mg_logfn *prior, const mg_proposal *prop,
                           const mg_mcmc_cfg *cfg, const double *x0,
                           double *d_samples, double *out_final,
                           int64_t *out_accept, int64_t *out_reject,
                           double *out_mean, double *out_std);

/* Mcmc.remove_repeat_samples (mcmc.ml:74-81) on one chain: host [n][D+2]
 * rows; writes kept rows to out, returns count in *nkept. */
int mg_remove_repeat_samples(mg_ctx *ctx, const double *rows, int64_t n,
                             int32_t dim, double *out, int64_t *nkept);

/* ------------------------------------------------------------------ */
/* Kd_tree + Interpolate_pdf                                           */
/* ------------------------------------------------------------------ */

/* Kd_tree.Make.tree_of_objects objs low high (kd_tree.ml:155-175), as flat
 * node arrays in breadth-first order (node 0 = root; children of a split
 * node are adjacent: left, left+1).  Bit-exact split dims / values / cell
 * membership w.r.t. the reference rule (SURVEY.md 8a K1, F7).
 * min_split: nodes with fewer objects are not split (2 = the reference's
 * full tree; Evidence passes its ?n because collect_subvolumes never looks
 * below the first cell with < n objects, evidence.ml:83-89).
 * pts: host [N][D].  NaN coordinates -> MG_EINVAL. */
int mg_kdtree_build(mg_ctx *ctx, const double *pts, int64_t N, int32_t D,
                    const double *low, const double *high, int32_t min_split,
                    mg_kdtree **out);
/* d_pts: device [N][D] */
int mg_kdtree_build_dev(mg_ctx *ctx, const double *d_pts, int64_t N, int32_t D,
                        const double *low, const double *high,
                        int32_t min_split, mg_kdtree **out);
void mg_kdtree_destroy(mg_kdtree *t);
int mg_kdtree_info(const mg_kdtree *t, int64_t *npoints, int32_t *dim,
                   int64_t *nnodes, int32_t *nlevels);
/* Export for bit-exact comparison; any pointer may be NULL.
 * split_dim[nnodes] (-1 = leaf), split_val[nnodes], left[nnodes] (-1 = leaf),
 * begin/end[nnodes]: the node's objects are perm[begin..end) in the
 * reference's list order (stable partitions of the input order). */
int mg_kdtree_export(const mg_kdtree *t, int32_t *split_dim, double *split_val,
                     int32_t *left, int32_t *begin, int32_t *end,
                     int32_t *perm);
/* Serialise / rebuild the flat arrays, e.g. to broadcast a tree to the
 * other GPUs of the box (NCCL broadcast of one contiguous device blob). */
int mg_kdtree_blob_size(const mg_kdtree *t, int64_t *nbytes);
int mg_kdtree_blob_dev(const mg_kdtree *t, void **d_blob); /* borrowed */
int mg_kdtree_from_blob_dev(mg_ctx *ctx, const void *d_blob, int64_t nbytes,
                            mg_kdtree **out);
/* Interp.draw locates the cell of a STORED point by descent
 * (interpolate_pdf.ml:114-119); that cell depends on the point only.  This
 * locates it once for every stored point (N x (2 D + 2) doubles next to the
 * tree, not inside the blob); leaf-level draws then gather one record instead
 * of ~log2 N dependent node loads, with bit-identical results.
 * mg_rjmcmc_array* enable it by themselves for leaf-level draws (nstop = 0)
 * from trees of at most 8 dimensions, when the run takes at least as many
 * chain-steps as the tree has points. */
int mg_kdtree_enable_draw_cache(mg_kdtree *t);
/* Kd_tree.bounds_volume (kd_tree.ml:177-182) */
double mg_bounds_volume(const double *low, const double *high, int32_t D);

/* Interpolate_pdf.find_cell (interpolate_pdf.ml:101-109): node id reached
 * by descent for each query (host [M][D]).  nstop = 0: descend to a leaf;
 * nstop > 0: stop at the first cell with <= nstop objects (the *_high_level
 * forms, interpolate_pdf.ml:121-133,144-159). */
int mg_interp_find_cell(mg_ctx *ctx, const mg_kdtree *t, const double *q,
                        int64_t M, int32_t nstop, int32_t *out_node);
/* Interpolate_pdf.jump_prob / jump_prob_high_level
 * (interpolate_pdf.ml:135-159): nobjs / (V * N), a density, not a log. */
int mg_interp_jump_prob(mg_ctx *ctx, const mg_kdtree *t, const double *q,
                        int64_t M, int32_t nstop, double *out_prob);
int mg_interp_jump_prob_dev(mg_ctx *ctx, const mg_kdtree *t, const double *d_q,
                            int64_t M, int32_t nstop, double *d_out_prob,
                            int32_t *d_out_node);
/* Interpolate_pdf.draw / draw_high_level (interpolate_pdf.ml:114-133):
 * M independent draws, host out [M][D]. */
int mg_interp_draw(mg_ctx *ctx, const mg_kdtree *t, int64_t M, int32_t nstop,
                   double *out);
int mg_interp_draw_dev(mg_ctx *ctx, const mg_kdtree *t, int64_t M,
                       int32_t nstop, double *d_out);

/* ------------------------------------------------------------------ */
/* Mcmc: two-model reversible jump                                     */
/* ------------------------------------------------------------------ */

/* how a chain proposes INTO a model (jintoa / jintob, mcmc.mli:132-140) */
enum {
  /* Interp.draw / log (Interp.jump_prob ...)  (test/mcmc_test.ml:175-178) */
  MG_INTO_INTERP = 0,
  /* independent Gaussian, params mu[D], sigma[D] (test/mcmc_test.ml:123-127) */
  MG_INTO_INDEP_GAUSS = 1
};

typedef struct {
  int32_t kind;
  int32_t nstop;            /* MG_INTO_INTERP: 0 = draw, >0 = *_high_level */
  const mg_kdtree *tree;    /* MG_INTO_INTERP */
  const double *params;     /* MG_INTO_INDEP_GAUSS */
  int64_t nparams;
} mg_into;

typedef struct {
  mg_logfn like, prior;
  mg_proposal prop;
  mg_into into;             /* proposal into THIS model */
  double p;                 /* model prior pa / pb */
} mg_rj_model;

typedef struct {
  int64_t nchains;
  int64_t nbin, nskip, n;
  uint64_t chain_offset;
  int32_t layout;
  int32_t reserved;
} mg_rjmcmc_cfg;

/* Mcmc.rjmcmc_array (mcmc.ml:121-139) for C independent chains.
 * a0 / b0: host start points [dA], [dB] shared by all chains.
 * out_model: uint8 [n][C] (0 = A, 1 = B) or NULL.
 * out_samples: [n][Dmax+2][C] or NULL (unused coordinates are 0).
 * out_counts: {#A, #B} over all recorded samples (rjmcmc_model_counts,
 * mcmc.ml:141-149). */
int mg_rjmcmc_array(mg_ctx *ctx, const mg_rj_model *A, const mg_rj_model *B,
                    const mg_rjmcmc_cfg *cfg, const double *a0,
                    const double *b0, uint8_t *out_model, double *out_samples,
                    int64_t out_counts[2]);
/* k-model reversible jump -- an EXTENSION (SURVEY.md 8f rank 3): the reference's
 * sampler is strictly two-model (type rjmcmc_value = A | B, mcmc.ml:83-87).
 * Structure kept from make_rjmcmc_sampler / rjmcmc_array: the model prior p_k
 * is part of the log prior (mcmc.ml:116-118,128), jump densities are
 * log p_target + log q_into_target (mcmc.ml:103-112), the priors' sum is checked
 * one-sidedly (mcmc.ml:90).  A step walks the priors cyclically from the current
 * model with one uniform (stay with probability p_current, as mcmc.ml:92-102)
 * and the initial model is uniform over the K (the fair coin of mcmc.ml:123).
 * With nmodels = 2 the chains equal mg_rjmcmc_array's draw for draw.
 * models: [nmodels]; starts: nmodels host pointers, starts[k] = [dim_k];
 * out_model: uint8 [n][C] (model index) or NULL; out_samples: [n][Dmax+2][C] or
 * NULL; out_counts: [nmodels] samples per model. */
#define MG_RJ_MAX_MODELS 8
int mg_rjmcmc_array_k(mg_ctx *ctx, const mg_rj_model *models, int32_t nmodels,
                      const mg_rjmcmc_cfg *cfg, const double *const *starts,
                      uint8_t *out_model, double *out_samples,
                      int64_t *out_counts);
/* Diagnostics of the last mg_rjmcmc_array call on this context: how many steps
 * proposed a jump into the other model (mcmc.ml:97,102) and how many of those
 * were accepted -- the mixing rate of the interpolated jumps. */
int mg_rjmcmc_jump_counters(const mg_ctx *ctx, int64_t *proposed, int64_t *accepted);

/* ------------------------------------------------------------------ */
/* Ellipse (ellipse.ml) -- SURVEY.md 8f rank 4                          */
/* ------------------------------------------------------------------ */
typedef struct mg_ellipse_tree mg_ellipse_tree;

/* Ellipse.enclosing_ellipse sf to_coord pts (ellipse.ml:98-103): centre =
 * mean (:36-46), covariance (:48-66), eigen-system (:58-61, eigenvalues
 * ascending as LAPACK returns them), axes = eigenvalue * sf^(1/D) * r_max
 * (:83-86).  pts: host [N][D], D <= 32.  center[D], axes[D], orientation[D][D]
 * with orientation[i][j] = component i of eigenvector j (Lacaml's z); the
 * eigenvector sign, which LAPACK leaves open, is fixed here (largest
 * component positive). */
int mg_ellipse_enclosing(mg_ctx *ctx, const double *pts, int64_t N, int32_t D,
                         double sf, double *center, double *axes,
                         double *orientation);
/* Ellipse.elliptical_range ell pt (ellipse.ml:63-73) of M host points q[M][D] */
int mg_ellipse_range(mg_ctx *ctx, const double *center, const double *axes,
                     const double *orientation, int32_t D, const double *q,
                     int64_t M, double *out);
/* Ellipse.ellipse_tree sf to_coord pts (ellipse.ml:150-173).  Nodes are
 * numbered breadth first; a child with fewer than D + 1 points is Empty (-1).
 * N < D + 1 is the reference's Assert_failure (MG_EINVAL); a node whose points
 * all lie on one side of its centre makes the reference recurse forever and
 * is MG_EFAIL here. */
int mg_ellipse_tree_build(mg_ctx *ctx, const double *pts, int64_t N, int32_t D,
                          double sf, mg_ellipse_tree **out);
int mg_ellipse_tree_build_dev(mg_ctx *ctx, const double *d_pts, int64_t N,
                              int32_t D, double sf, mg_ellipse_tree **out);
void mg_ellipse_tree_destroy(mg_ellipse_tree *t);
int mg_ellipse_tree_info(const mg_ellipse_tree *t, int64_t *npoints,
                         int32_t *dim, int64_t *nnodes, int32_t *nlevels);
/* Flat arrays of the tree (any pointer may be NULL): left / right child or -1
 * (Empty); the node's points are perm[begin..end) -- as a set: the reference's
 * `pts` field lists them in input order, i.e. sorted by id; `ellipse` =
 * center[D], axes[D], orientation[D][D]; `circumcircle` (:159-167) =
 * cc_center[D], cc_radius. */
int mg_ellipse_tree_export(const mg_ellipse_tree *t, int32_t *left,
                           int32_t *right, int32_t *begin, int32_t *end,
                           int32_t *perm, double *center, double *axes,
                           double *orientation, double *cc_center,
                           double *cc_radius);

/* ------------------------------------------------------------------ */
/* Evidence + Stats                                                    */
/* ------------------------------------------------------------------ */

/* Evidence.evidence_harmonic_mean (evidence.ml:101-107).  ll: host [N]. */
int mg_evidence_harmonic_mean(mg_ctx *ctx, const double *ll, int64_t N,
                              double *out);
int mg_evidence_harmonic_mean_dev(mg_ctx *ctx, const double *d_ll, int64_t N,
                                  double *out);
/* bin/harmonic_evidence.ml:41-52: nbstrap bootstrap replicates of the
 * harmonic-mean evidence (n indices resampled with Random.int n each).
 * out_evs: host [nbstrap], unsorted (replicate b uses Philox stream b). */
int mg_evidence_harmonic_bootstrap(mg_ctx *ctx, const double *ll, int64_t N,
                                   int32_t nbstrap, double *out_evs);
/* Evidence.evidence_lebesgue ?n ?eps (evidence.ml:202-221).
 * pts host [N][D]; ll, lp host [N].  Defaults n = 64, eps = 0.1. */
int mg_evidence_lebesgue(mg_ctx *ctx, const double *pts, const double *ll,
                         const double *lp, int64_t N, int32_t D, int32_t n,
                         double eps, double *out);
int mg_evidence_lebesgue_dev(mg_ctx *ctx, const double *d_pts,
                             const double *d_ll, const double *d_lp, int64_t N,
                             int32_t D, int32_t n, double eps, double *out);
/* Evidence.evidence_direct ?n (evidence.ml:148-165). */
int mg_evidence_direct(mg_ctx *ctx, const double *pts, const double *ll,
                       const double *lp, int64_t N, int32_t D, int32_t n,
                       double *out);
int mg_evidence_direct_dev(mg_ctx *ctx, const double *d_pts,
                           const double *d_ll, const double *d_lp, int64_t N,
                           int32_t D, int32_t n, double *out);

/* Stats.mean / Stats.std ?mean (stats.ml:17-43); have_mean=0 computes it. */
int mg_stats_mean(mg_ctx *ctx, const double *x, int64_t n, double *out);
int mg_stats_std(mg_ctx *ctx, const double *x, int64_t n, int have_mean,
                 double mean, double *out);
/* Stats.multi_mean / multi_std (stats.ml:58-87); xs host [n][D]. */
int mg_stats_multi_mean(mg_ctx *ctx, const double *xs, int64_t n, int32_t D,
                        double *out);
int mg_stats_multi_std(mg_ctx *ctx, const double *xs, int64_t n, int32_t D,
                       const double *mean_or_null, double *out);
/* The same over a device sample block [n][D+2][C] (all chains pooled):
 * per-field mean and std, fields 0..D+1.  out_mean/out_std: host [D+2]. */
int mg_stats_sample_block_dev(mg_ctx *ctx, const double *d_samples, int64_t n,
                              int32_t D, int64_t C, double *out_mean,
                              double *out_std);
/* Stats.slow_autocorrelation nslides x (stats.ml:223-238) for lags
 * 0..nslides-1 (the reference's loop bound overruns by one, SURVEY F6:
 * parity unpinned).  Also the integrated autocorrelation length
 * 1 + 2 sum_{i>=1} r_i up to the first non-positive r_i (an addition). */
int mg_stats_autocorrelation(mg_ctx *ctx, const double *x, int64_t n,
                             int32_t nslides, double *out_r,
                             double *out_length);

/* Ensemble convergence diagnostics of a sample block (an addition beyond the
 * reference, like the integrated length above; DESIGN.md 4b).  Block
 * x[s][f][c], s < n, f < F = D+2, c < C.
 * Sequences: split = 1 -> N = n/2 (floor), M = 2C, sequence c = rows [0, N) of
 * chain c, sequence C+c = rows [n-N, n) (an odd n drops its middle row);
 * split = 0 -> N = n, M = C.  Per sequence m and field f:
 *   xbar_m = (1/N) sum_s x_s,  s2_m = N/(N-1) gamma_m(0),
 *   gamma_m(t) = (1/N) sum_{s=0}^{N-1-t} (x_s - xbar_m)(x_{s+t} - xbar_m).
 * Pooled: W = mean_m s2_m, B = N/(M-1) sum_m (xbar_m - xbar)^2 (0 if M = 1),
 *   var+ = (N-1)/N W + B/N, Rhat = sqrt(var+/W) (NaN if M = 1, +inf if W = 0
 *   and the means differ), rho_0 = 1, rho_t = 1 - (W - mean_m gamma_m(t))/var+.
 * Geyer's initial monotone sequence: P_k = rho_2k + rho_2k+1 (k < L/2),
 *   K = first k with P_k <= 0 (none: K = L/2, window_closed = 0), P'_0 = P_0,
 *   P'_k = min(P_k, P'_k-1), tau = -1 + 2 sum_{k<K} P'_k, ESS = M N / tau.
 * Per sequence: the same rule on gamma_m(t)/gamma_m(0) gives seq_tau (NaN for a
 * constant sequence or one with a non-finite value).  A field that is constant
 * over the block or holds a non-finite value has NaN Rhat, ESS, tau and rho.
 * MG_EINVAL: null or inconsistent arguments, L < 2, L >= N, L > MG_DIAG_MAXLAG,
 * split with n < 4.  The definition holds for any 2 <= L <= N-1; the kernel
 * keeps a sequence's lag sums in registers and so stops at MG_DIAG_MAXLAG = 256
 * (a known gap: a chain with tau above ~50-100 may need a longer window, which
 * then shows as window_closed = 0 and tau as a lower bound). */
#define MG_DIAG_MAXLAG 256
typedef struct {
  int64_t n;        /* rows of the block (samples per chain) */
  int64_t nchains;  /* C */
  int32_t dim;      /* D: fields 0..D+1 are diagnosed */
  int32_t maxlag;   /* L: lags 0..L-1, 2 <= L <= min(N-1, MG_DIAG_MAXLAG) */
  int32_t split;    /* 1: each chain is two sequences (split-R-hat) */
  int32_t reserved;
} mg_diag_cfg;
/* d_samples: device [n][D+2][C] (the layout of mg_mcmc_array_dev /
 * _resident), not modified.  out_rhat, out_ess, out_tau: host [D+2];
 * out_window_closed: host int32 [D+2]; out_rho: host [D+2][L] or NULL;
 * d_seq_tau: device [D+2][M] or NULL. */
int mg_stats_chain_diagnostics_dev(mg_ctx *ctx, const double *d_samples,
                                   const mg_diag_cfg *cfg, double *out_rhat,
                                   double *out_ess, double *out_tau,
                                   int32_t *out_window_closed, double *out_rho,
                                   double *d_seq_tau);
/* the same on a host block; seq_tau: host [D+2][M] or NULL */
int mg_stats_chain_diagnostics(mg_ctx *ctx, const double *samples,
                               const mg_diag_cfg *cfg, double *out_rhat,
                               double *out_ess, double *out_tau,
                               int32_t *out_window_closed, double *out_rho,
                               double *seq_tau);

/* Exact per-field order statistics and quantiles of a sample block (Stats
 * order statistics, stats.mli:19-110; DESIGN.md 4c).  Block x[s][f][c],
 * s < n, f < F = D+2, c < C.  For each field f, the pool is the N = n*C values
 * x[s][f][c] (all chains pooled, as mg_stats_sample_block_dev pools them).
 * Order is the total order of f64_to_ordered: -inf is the smallest value and
 * +inf the largest; -0.0 equals +0.0, and a zero is returned as +0.0.
 * To drop a burn-in, pass d_samples + r*F*C and n - r (the block base need
 * only be 8-byte aligned).
 * Order statistic of rank k (0 <= k < N, 0-based: k = 0 is the minimum): the
 *   k-th smallest value of the pool, exact (one of the block's values, bit for
 *   bit, except for the sign of a zero).
 * Quantile at p in [0, 1] (numpy's default "linear" rule, Hyndman-Fan 7, with
 *   one rounding):
 *   h = (double)(N-1) * p, lo = floor(h), g = h - lo, a = x_(lo),
 *   b = x_(min(lo+1, N-1));
 *   if g = 0 or a = b, q = a;
 *   else if a = -inf: q = NaN when b = +inf, and -inf otherwise;
 *   else if b = +inf, q = +inf;
 *   otherwise q = a + g*(b - a), evaluated exactly as written (the library
 *   builds with -fmad=false).
 * NaN: if a field holds any NaN, every output for that field is NaN; other
 *   fields are unaffected.
 * MG_EINVAL: null pointers, n < 1, C < 1, D < 1, nq (or nk) outside
 *   [1, MG_QUANT_MAX], a p outside [0, 1] or NaN, a k outside [0, N).
 * The device block is read and never modified.  out: host [D+2][nq]
 * ([D+2][nk] for order statistics). */
#define MG_QUANT_MAX 64
int mg_stats_quantiles_dev(mg_ctx *ctx, const double *d_samples, int64_t n,
                           int32_t D, int64_t C, const double *probs,
                           int32_t nq, double *out);
/* the same on a host block [n][D+2][C] */
int mg_stats_quantiles(mg_ctx *ctx, const double *samples, int64_t n,
                       int32_t D, int64_t C, const double *probs, int32_t nq,
                       double *out);
int mg_stats_order_statistics_dev(mg_ctx *ctx, const double *d_samples,
                                  int64_t n, int32_t D, int64_t C,
                                  const int64_t *ranks, int32_t nk,
                                  double *out);

/* Stats.draw_uniform a b / draw_gaussian mu sigma / draw_cauchy x0 gamma
 * (stats.ml:126-128, 113-124 [Leva's ratio of uniforms], 89-91), n draws at
 * once.  Draw i comes from the call's Philox stream; the reference's global
 * Random stream is not reproduced, parity is in distribution (and value for
 * value against the oracle, which addresses the same stream). */
enum { MG_DRAW_UNIFORM = 0, MG_DRAW_GAUSSIAN = 1, MG_DRAW_CAUCHY = 2 };
int mg_stats_draw(mg_ctx *ctx, int32_t kind, double a, double b, int64_t n,
                  double *out);
int mg_stats_draw_dev(mg_ctx *ctx, int32_t kind, double a, double b,
                      int64_t n, double *d_out);

/* ------------------------------------------------------------------ */
/* Evidence by parallel tempering                                      */
/* ------------------------------------------------------------------ */
/* M ladders of T tempered chains ("rungs"): rung k samples
 * pi_k ~ L^beta_k * prior, neighbouring rungs swap states, and log Z follows
 * from thermodynamic integration (TI, log Z = int_0^1 E_beta[log L] dbeta) and
 * from stepping stones (SS, Xie et al. 2011:
 * log Z = sum_k log E_beta_k[L^(beta_k+1 - beta_k)]).
 *
 * Definition (the oracle, oracle/tempered_oracle.cpp, transcribes it):
 * - Inputs: like, prior; props[T], one proposal per rung (pass the same one T
 *   times for one proposal); betas[T] finite, strictly increasing,
 *   betas[0] >= 0, betas[T-1] == 1; M ladders whose rungs all start at x0_m
 *   (x0 [M][D], or [D] with x0_shared), evaluated as in mcmc.ml:59-61;
 *   nbin >= 0, nsteps >= 1, swap_every >= 0, ladder_offset = global id of
 *   ladder 0 (sharding).
 * - Tempered step: rung k runs mcmc.ml:37-56 with the log posterior replaced
 *   by tl(x) = (beta_k == 0 ? 0.0 : beta_k * ll(x)) + lp(x), in mh_step's
 *   order: log_accept = tl(y) - tl(x), then + log_backward - log_forward for
 *   asymmetric proposals; accepted iff log u < log_accept (strict, NaN rejects).
 * - Draws: the uniforms of step t (t = 0 .. nbin + nsteps - 1) of rung k of
 *   ladder m are those of (P_MH, g = (ladder_offset + m) * T + k, t).  With
 *   swap_every = 0 the rung at beta = 1 is, draw for draw, chain g of
 *   mg_mcmc_array on the same seed and epoch.
 * - Swaps (even-odd): when swap_every > 0, a swap round follows every step t
 *   with (t + 1) % swap_every == 0; its number is r = (t + 1) / swap_every - 1
 *   and it tries the pairs (k, k+1) with k = r (mod 2).  The pair's uniform is
 *   the first draw of (P_PT_SWAP, g = (ladder_offset + m) * 32 + k, r); the
 *   swap is accepted iff log u < (beta_k+1 - beta_k) * (ll_k - ll_k+1) and
 *   exchanges x, ll and lp.
 * - Measurement: for t >= nbin, after the swap round that follows step t (if
 *   any), rung k records its ll.  The pivot p is the first measured ll (0.0 if
 *   that is not finite).  S1 = sum (ll - p) in step order, Neumaier-compensated
 *   over the finite terms, the non-finite terms added apart (so a -inf gives
 *   -inf and a NaN gives NaN).  For k < T-1, (a, s) accumulates
 *   w = (beta_k+1 - beta_k) * ll as a log-sum-exp: a the running maximum,
 *   s = sum exp(w - a), rescaled when a grows; w = -inf adds nothing.
 *   Accepted MH steps per rung and accepted swaps per pair are counted over
 *   the measured phase.
 * - Per ladder: L_mk = p + S1 / nsteps;  TI_m = sum_k (beta_k+1 - beta_k) *
 *   (L_mk + L_m,k+1) / 2 in k order;  SS_m = sum_k (a_mk + log(s_mk / nsteps)).
 * - Pooled (every sum over ladders in ladder order; means and spreads by
 *   Welford's / Chan's update over the finite values, non-finite values summed
 *   apart and taking the result over): mean_ll[k] = mean over ladders of L_.k,
 *   mean_ll_err[k] = sd / sqrt(M); log_z_ti = trapezoid over mean_ll,
 *   log_z_ti_err = sd(TI_m) / sqrt(M); log_z_ss = sum_k [lse_m(a_mk + log s_mk)
 *   - log(M * nsteps)], log_z_ss_err = sd(SS_m) / sqrt(M).  sd has M - 1 in
 *   its denominator: M = 1, or a non-finite value, gives errors of NaN.
 * - A rung at beta = 0 that measures ll = -inf (a prior draw outside the
 *   likelihood's support) makes mean_ll[0] and log_z_ti -inf; SS is unaffected
 *   (exp(-inf) = 0).  SS is the primary estimate; TI also carries the
 *   trapezoid bias of its ladder (DESIGN 4d).
 * - One call key (epoch); the context's accept / reject counters are left
 *   unchanged.  MG_EINVAL: null pointers, M < 1, T outside [2, 32], betas that
 *   break the rules above, nsteps < 1, nbin < 0, swap_every < 0, nbin + nsteps
 *   >= 2^31, D outside 1..64, a plugin or proposal whose dim != D, ladder ids
 *   that overflow the 48-bit chain id of the Philox counter. */
#define MG_TEMPERED_MAX_T 32
typedef struct {
  int64_t nladders;       /* M (this rank's ladders in the sharded call) */
  int32_t ntemps;         /* T, 2..32 */
  int32_t dim;            /* D */
  int64_t nbin;           /* steps before the measured phase */
  int64_t nsteps;         /* measured steps */
  int64_t swap_every;     /* a swap round every swap_every steps; 0 = none */
  uint64_t ladder_offset; /* global id of ladder 0 */
  int32_t x0_shared;      /* 1: x0 is one start point [D] */
  int32_t reserved;
} mg_tempered_cfg;

/* Results.  The four log Z numbers are always written; every pointer may be
 * NULL.  mean_ll, mean_ll_err, accept: [T]; swaps_accepted, swaps_tried:
 * [T-1]; final: [M][T][D+2] (x, ll, lp of every replica at the end);
 * ladder_mean_ll: [M][T] (L_mk).  final and ladder_mean_ll cover this rank's
 * ladders in the sharded call, everything else all ladders. */
typedef struct {
  double log_z_ss, log_z_ss_err;
  double log_z_ti, log_z_ti_err;
  double *mean_ll, *mean_ll_err;
  int64_t *accept, *swaps_accepted, *swaps_tried;
  double *final;
  double *ladder_mean_ll;
} mg_tempered_out;

/* The definition above on one GPU: one warp holds floor(32 / T) ladders, the
 * swaps are warp shuffles, and every replica keeps its state and sums in
 * registers for the whole run (DESIGN 4d).  Host arrays. */
int mg_evidence_tempered(mg_ctx *ctx, const mg_logfn *like, const mg_logfn *prior,
                         const mg_proposal *props, const double *betas,
                         const mg_tempered_cfg *cfg, const double *x0,
                         mg_tempered_out *out);

/* ------------------------------------------------------------------ */
/* Nested sampling                                                     */
/* ------------------------------------------------------------------ */

typedef struct {
  int32_t dim;
  int32_t nlive;            /* ?nlive  default 1000 (nested.ml:122) */
  int32_t nmcmc;            /* ?nmcmc  default 1000 */
  int32_t batch;            /* K live points replaced per iteration; 1 =
                               the reference's one-at-a-time schedule */
  double epsrel;            /* ?epsrel default 0.01 */
  double mode_hopping_frac; /* ?mode_hopping_frac default 0.1 */
  int64_t max_points;       /* capacity of the output arrays */
} mg_nested_cfg;

/* Nested.nested_evidence (nested.ml:122-146).  draw_prior is uniform on the
 * box [prior_lo, prior_hi] (every reference caller: nested_test.ml:34-35).
 * Outputs: log_ev, log_dev, *npts points ascending in ll with their log
 * weights.  pts host [max_points][D]; ll, lp, logw host [max_points].
 * MG_EFAIL if a replacement ends below its threshold (nested.ml:70-72) or
 * max_points is too small. */
int mg_nested_evidence(mg_ctx *ctx, const mg_logfn *like, const mg_logfn *prior,
                       const double *prior_lo, const double *prior_hi,
                       const mg_nested_cfg *cfg, double *log_ev,
                       double *log_dev, int64_t *npts, double *pts, double *ll,
                       double *lp, double *logw);
/* ?observer (nested.ml:123-125,136): called on the calling thread with every
 * retired point, in retirement order (K calls after each batch of K), before
 * nested_evidence returns.  fn = NULL removes it.  The library and the plugins
 * may NOT be re-entered from the callback. */
typedef void (*mg_nested_observer)(void *user, const double *value, int32_t dim,
                                   double log_likelihood, double log_prior);
int mg_nested_set_observer(mg_ctx *ctx, mg_nested_observer fn, void *user);
/* Nested.evidence_error_and_weights generalised to K-at-a-time shrinkage
 * (nested.ml:81-120 when batch = 1).  ll: host [n] ascending. */
int mg_nested_weights(mg_ctx *ctx, const double *ll, int64_t n, int32_t nlive,
                      int32_t batch, double *log_ev, double *log_dev,
                      double *logw);
/* Nested.posterior_samples n nested_output (nested.ml:152-178): indices of n
 * draws from the weighted points (inverse CDF over the running sums of
 * exp log_weight, weight_binary_search_index :152-165).  logw: host [npts];
 * out_idx: host [n].  Consumes one epoch of the context's Philox key. */
int mg_nested_posterior_indices(mg_ctx *ctx, const double *logw, int64_t npts,
                                int64_t n, int64_t *out_idx);
/* Nested.log_total_error_estimate (nested.ml:148-150) */
double mg_nested_log_total_error(double log_ev, double log_dev, int32_t nlive);

/* ------------------------------------------------------------------ */
/* Several GPUs of one box: one process (one context) per GPU, NCCL     */
/* ------------------------------------------------------------------ */
/* The reference is single-threaded; what it computes shards naturally
 * (SURVEY.md 8e): chains and queries are independent, a kd-tree is built on
 * one rank and replicated, per-rank statistics and per-cell evidence terms are
 * gathered and combined in a fixed order.  NCCL is loaded at run time
 * (libnccl.so.2); without it only the entry points below fail (MG_EFAIL).
 * Every entry point here is COLLECTIVE: all ranks of the communicator call it.
 * The rank-pooled calls (the sharded evidence estimators, the distributed
 * kd-tree build, mg_rjmcmc_array_sharded, mg_comm_pool_moments,
 * mg_comm_chain_diagnostics, mg_comm_quantiles and mg_evidence_tempered_sharded)
 * exchange every rank's status
 * before they use another rank's data: an argument error or a failure on any
 * rank is returned on every rank, and the arguments that must be the same on
 * every rank are checked ("rank r has another ..." is MG_EINVAL).  A null comm
 * returns MG_EINVAL at once. */
#define MG_COMM_ID_BYTES 128
/* ncclGetUniqueId: called by one rank, which hands the 128 bytes to the others
 * through any channel of the host program (a file, a socket, MPI, ...). */
int mg_comm_get_unique_id(uint8_t id[MG_COMM_ID_BYTES]);
/* ncclCommInitRank on the context's device; nranks == 1 needs no NCCL. */
int mg_comm_create(mg_ctx *ctx, int32_t nranks, int32_t rank,
                   const uint8_t id[MG_COMM_ID_BYTES], mg_comm **out);
void mg_comm_destroy(mg_comm *comm);
int32_t mg_comm_rank(const mg_comm *comm);
int32_t mg_comm_size(const mg_comm *comm);
int mg_comm_nccl_version(int32_t *version);
int mg_comm_barrier(mg_comm *comm);
/* device time (ms, CUDA events on the context's stream) this rank spent in the
 * NCCL calls of the last collective entry point. */
double mg_comm_last_collective_ms(const mg_comm *comm);
/* ncclAllGather of a small host record: recv[nranks][nbytes] in rank order. */
int mg_comm_allgather(mg_comm *comm, const void *send, void *recv, int64_t nbytes);
/* Interp.make on `root`, used everywhere: ONE ncclBroadcast of the tree's
 * contiguous device blob, from the builder's blob straight into the receivers'
 * (no staging copy).  tree: the root's tree (ignored elsewhere, may be NULL).
 * *out: on the root `tree` itself, on the other ranks a new tree (destroy it).
 * An argument error on one rank is not propagated to the others. */
int mg_kdtree_broadcast(mg_comm *comm, mg_kdtree *tree, int32_t root,
                        mg_kdtree **out);
/* Kd_tree.tree_of_objects (kd_tree.ml:155-175) built by all ranks together
 * (SURVEY.md 8f rank 3).  d_pts: the same N x D device rows on every rank.  Every
 * rank builds the top log2(nranks) levels, rank r builds the subtree under node
 * r of that level from its N / nranks rows, one ncclAllGather exchanges the
 * subtrees; every rank receives the whole tree, bit-identical to
 * mg_kdtree_build_dev on one GPU.  A rank count that is not a power of two,
 * fewer than 4096 points per rank, min_split above N / nranks or ties that keep
 * the top from being a complete tree make every rank build the tree alone.
 * An argument error on one rank is not propagated to the others. */
int mg_kdtree_build_distributed(mg_comm *comm, const double *d_pts, int64_t N,
                                int32_t D, const double *low, const double *high,
                                int32_t min_split, mg_kdtree **out);
/* Evidence.evidence_lebesgue / evidence_direct (evidence.ml:148-221) with the
 * kd-cells shared out: `root` holds the samples (device pointers; ignored on
 * the other ranks), does the global steps (sort, prefix cut, de-duplication,
 * tree), the tree is broadcast, every rank integrates a contiguous range of
 * nodes, the per-node terms are all-gathered and summed by the same
 * deterministic reduction everywhere: *out is bit-identical on every rank and
 * to the single-GPU call. */
int mg_evidence_lebesgue_sharded(mg_comm *comm, int32_t root, const double *d_pts,
                                 const double *d_ll, const double *d_lp,
                                 int64_t N, int32_t D, int32_t n, double eps,
                                 double *out);
int mg_evidence_direct_sharded(mg_comm *comm, int32_t root, const double *d_pts,
                               const double *d_ll, const double *d_lp, int64_t N,
                               int32_t D, int32_t n, double *out);
/* Evidence.evidence_harmonic_mean over samples sharded across the ranks
 * (d_ll_shard: this rank's log-likelihoods, device). */
int mg_evidence_harmonic_mean_sharded(mg_comm *comm, const double *d_ll_shard,
                                      int64_t n_shard, double *out);
/* Mcmc.rjmcmc_array with the cfg->nchains chains cut into one contiguous range
 * per rank (global chain ids: results do not depend on the number of ranks);
 * out_counts = rjmcmc_model_counts over ALL ranks; out_model / out_samples get
 * this rank's chains only, which *shard_begin / *shard_count identify. */
int mg_rjmcmc_array_sharded(mg_comm *comm, const mg_rj_model *A,
                            const mg_rj_model *B, const mg_rjmcmc_cfg *cfg,
                            const double *a0, const double *b0,
                            uint8_t *out_model, double *out_samples,
                            int64_t out_counts[2], int64_t *shard_begin,
                            int64_t *shard_count);
/* Stats.multi_mean / multi_std of samples held by several ranks, pooled from
 * each rank's (count, mean[F], std[F]) in rank order (same F on every rank). */
int mg_comm_pool_moments(mg_comm *comm, int64_t n_local, const double *mean_local,
                         const double *std_local, int32_t F, int64_t *n_total,
                         double *out_mean, double *out_std);
/* mg_stats_chain_diagnostics_dev over chains sharded across the ranks: each
 * rank passes its own [n][D+2][C_r] block (same n, dim, maxlag and split on
 * every rank).  The pooled outputs are identical on every rank (one rank: the
 * bits of the single-GPU call); d_seq_tau covers the local sequences [D+2][M_r]. */
int mg_comm_chain_diagnostics(mg_comm *comm, const double *d_samples_local,
                              const mg_diag_cfg *cfg_local, double *out_rhat,
                              double *out_ess, double *out_tau,
                              int32_t *out_window_closed, double *out_rho,
                              double *d_seq_tau);
/* mg_stats_quantiles_dev of the union of every rank's block: each rank passes
 * its own [n][D+2][C_r] block (same n, D, nq and probs on every rank, C_r of
 * its own).  The result is the same on every rank and bit-identical to
 * mg_stats_quantiles_dev on the concatenated block. */
int mg_comm_quantiles(mg_comm *comm, const double *d_samples_local, int64_t n,
                      int32_t D, int64_t C_local, const double *probs,
                      int32_t nq, double *out);
/* mg_evidence_tempered (definition in the parallel-tempering section) with
 * the ladders split over the ranks: each rank runs cfg->nladders ladders from
 * global id cfg->ladder_offset (x0 covers its own ladders) and reduces them to
 * a per-rank record, the records are pooled in rank order.  T, betas, nbin,
 * nsteps, swap_every and dim must agree.  One rank: the single-GPU call's
 * bits; several: per-ladder outputs and counts equal the single-GPU run on the
 * union, pooled values agree to rounding. */
int mg_evidence_tempered_sharded(mg_comm *comm, const mg_logfn *like,
                                 const mg_logfn *prior, const mg_proposal *props,
                                 const double *betas, const mg_tempered_cfg *cfg,
                                 const double *x0, mg_tempered_out *out);

/* ------------------------------------------------------------------ */
/* Read_write: the text format of the reference's tools (host only)    */
/* ------------------------------------------------------------------ */
/* Read_write.write / read (read_write.ml:19-58): one sample per line,
 * "%g " per coordinate then "%g %g\n" (log_likelihood, log_prior).
 * rows: [n][D+2].  precision 0 = the reference's "%g" (6 digits, lossy),
 * 17 = "%.17g" (same grammar, exact round trip).  path "-" = stdout / stdin.
 * Readers return malloc'ed arrays: release with mg_free_host.
 * MG_EFAIL <-> Sys_error / Scanf failure / End_of_file. */
int mg_write_samples(const char *path, const double *rows, int64_t n,
                     int32_t D, int32_t precision);
int mg_read_samples(const char *path, double **rows, int64_t *n, int32_t *D);
/* Read_write.write_nested / read_nested (read_write.ml:60-101) */
int mg_write_nested(const char *path, double log_ev, double log_dev,
                    const double *rows, const double *logw, int64_t n,
                    int32_t D, int32_t precision);
int mg_read_nested(const char *path, double *log_ev, double *log_dev,
                   double **rows, double **logw, int64_t *n, int32_t *D);
void mg_free_host(void *p);

#ifdef __cplusplus
}
#endif
#endif /* MCMC_GPU_H */
