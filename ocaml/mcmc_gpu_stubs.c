/* mcmc_gpu_stubs.c -- thin OCaml C stubs over include/mcmc_gpu.h.
 *
 * NOT COMPILED IN THIS REPOSITORY'S IMAGE: there is no OCaml toolchain here
 * (no caml/*.h, ocamlfind, ocamlopt; SURVEY.md F1).  The file is the binding a
 * maintainer of farr/mcmc-ocaml adds next to mcmc.ml; it is kept small enough
 * to review by eye.  Build (on a machine with OCaml >= 4.08 and CUDA):
 *
 *   ocamlfind ocamlopt -package bigarray -c mcmc_gpu_stubs.c -ccopt -I../include
 *   ocamlfind ocamlopt -package bigarray mcmc_gpu.mli mcmc_gpu.ml mcmc_gpu_stubs.o \
 *       -cclib -L../mcmc_ocaml_b200 -cclib -lmcmcgpu -a -o mcmc_gpu.cmxa
 *
 * Conventions: float64 Bigarray.Array{1,2,3} in c_layout carry all bulk data
 * (the host entry points copy to / from the device themselves; `Mcmc_gpu.Pinned`
 * allocates page-locked ones, mcmcgpu_pinned_raw below); contexts, trees and pinned
 * buffers are custom blocks with finalisers that share a reference-counted context; every status other than MG_OK raises the
 * exception the reference raises in the same situation:
 *   MG_EINVAL -> Invalid_argument, MG_EFAIL / MG_ECUDA / MG_ENOMEM -> Failure.
 * The runtime lock is released around every call that launches kernels.
 */
#include <stdlib.h>
#include <string.h>

#include <caml/alloc.h>
#include <caml/bigarray.h>
#include <caml/custom.h>
#include <caml/fail.h>
#include <caml/memory.h>
#include <caml/mlvalues.h>
#include <caml/threads.h>

#include "mcmc_gpu.h"

/* ---- handles ----------------------------------------------------------
 * OCaml does not order finalisers: a tree (or a pinned buffer) may be finalised after the context it belongs to.
 * Every handle therefore holds a reference on a small C box around the mg_ctx; the context is destroyed by whoever
 * drops the last reference, so mg_kdtree_destroy / mg_free_pinned never see a dead context. */
typedef struct { mg_ctx *ctx; long refs; } ctx_box;
typedef struct { mg_kdtree *tree; ctx_box *box; } tree_box;
typedef struct { void *ptr; ctx_box *box; } pinned_box;
#define Box_val(v) (*((ctx_box **)Data_custom_val(v)))
#define Ctx_val(v) (Box_val(v)->ctx)
#define Treebox_val(v) ((tree_box *)Data_custom_val(v))
#define Tree_val(v) (Treebox_val(v)->tree)
#define Pinned_val(v) ((pinned_box *)Data_custom_val(v))

static void box_release(ctx_box *b) {
  if (b && --b->refs == 0) { if (b->ctx) mg_ctx_destroy(b->ctx); free(b); }
}
static void ctx_finalize(value v) { box_release(Box_val(v)); Box_val(v) = NULL; }
static void tree_finalize(value v) {
  tree_box *t = Treebox_val(v);
  if (t->tree) { mg_kdtree_destroy(t->tree); t->tree = NULL; }
  box_release(t->box); t->box = NULL;
}
static void pinned_finalize(value v) {
  pinned_box *p = Pinned_val(v);
  if (p->ptr && p->box) { mg_free_pinned(p->box->ctx, p->ptr); p->ptr = NULL; }
  box_release(p->box); p->box = NULL;
}

static struct custom_operations ctx_ops = {"mcmc_gpu.ctx", ctx_finalize, custom_compare_default, custom_hash_default,
                                           custom_serialize_default, custom_deserialize_default,
                                           custom_compare_ext_default, custom_fixed_length_default};
static struct custom_operations tree_ops = {"mcmc_gpu.kdtree", tree_finalize, custom_compare_default,
                                            custom_hash_default, custom_serialize_default, custom_deserialize_default,
                                            custom_compare_ext_default, custom_fixed_length_default};
static struct custom_operations pinned_ops = {"mcmc_gpu.pinned", pinned_finalize, custom_compare_default,
                                              custom_hash_default, custom_serialize_default, custom_deserialize_default,
                                              custom_compare_ext_default, custom_fixed_length_default};

static void check(mg_ctx *ctx, int rc) {
  if (rc == MG_OK) return;
  const char *msg = ctx ? mg_last_error(ctx) : "mcmc_gpu: no context";
  if (rc == MG_EINVAL) caml_invalid_argument(msg);
  caml_failwith(msg);
}

/* ---- plugins: OCaml records -> mg_logfn / mg_proposal -------------------
 * type logfn = { kind : int; dim : int; scale : float; params : (float, float64_elt, c_layout) Array1.t }
 * type proposal = { pkind : int; pdim : int; pparams : (float, float64_elt, c_layout) Array1.t } */
static mg_logfn logfn_of_value(value v) {
  mg_logfn f;
  f.kind = Int_val(Field(v, 0)); f.dim = Int_val(Field(v, 1)); f.scale = Double_val(Field(v, 2));
  f.params = (const double *)Caml_ba_data_val(Field(v, 3));
  f.nparams = Caml_ba_array_val(Field(v, 3))->dim[0];
  return f;
}
static mg_proposal proposal_of_value(value v) {
  mg_proposal p;
  p.kind = Int_val(Field(v, 0)); p.dim = Int_val(Field(v, 1));
  p.params = (const double *)Caml_ba_data_val(Field(v, 2));
  p.nparams = Caml_ba_array_val(Field(v, 2))->dim[0];
  return p;
}

/* ---- context ---------------------------------------------------------- */
CAMLprim value mcmcgpu_ctx_create(value device, value seed) {
  CAMLparam2(device, seed);
  CAMLlocal1(v);
  mg_ctx *ctx = NULL;
  int rc = mg_ctx_create(Int_val(device), (uint64_t)Int64_val(seed), &ctx);
  if (rc != MG_OK) caml_failwith("cuda: cannot create a GPU context (no CPU fallback)");
  ctx_box *b = (ctx_box *)malloc(sizeof(ctx_box));
  b->ctx = ctx; b->refs = 1;
  v = caml_alloc_custom(&ctx_ops, sizeof(ctx_box *), 0, 1);
  Box_val(v) = b;
  CAMLreturn(v);
}

/* ---- pinned float64 Bigarrays -------------------------------------------------------------------------------
 * external pinned_raw : ctx -> int array (dims, 1..3) -> (float, float64_elt, c_layout) Genarray.t * pinned_handle
 * The Bigarray is a view of page-locked host memory (mg_malloc_pinned): the host entry points then copy with DMA at
 * full PCIe rate.  The handle's finaliser frees the memory; Mcmc_gpu.Pinned keeps handle and view together. */
CAMLprim value mcmcgpu_pinned_raw(value ctx, value dims) {
  CAMLparam2(ctx, dims);
  CAMLlocal3(ba, h, r);
  const int nd = (int)Wosize_val(dims);
  if (nd < 1 || nd > 3) caml_invalid_argument("Mcmc_gpu.Pinned: 1 to 3 dimensions");
  intnat d[3]; int64_t count = 1;
  for (int i = 0; i < nd; ++i) { d[i] = Long_val(Field(dims, i)); if (d[i] < 0) caml_invalid_argument("Mcmc_gpu.Pinned: negative dimension"); count *= d[i]; }
  void *p = NULL;
  check(Ctx_val(ctx), mg_malloc_pinned(Ctx_val(ctx), count * (int64_t)sizeof(double), &p));
  h = caml_alloc_custom(&pinned_ops, sizeof(pinned_box), 0, 1);
  Pinned_val(h)->ptr = p; Pinned_val(h)->box = Box_val(ctx); Box_val(ctx)->refs++;
  ba = caml_ba_alloc(CAML_BA_FLOAT64 | CAML_BA_C_LAYOUT | CAML_BA_EXTERNAL, nd, p, d);
  r = caml_alloc_tuple(2);
  Store_field(r, 0, ba); Store_field(r, 1, h);
  CAMLreturn(r);
}
/* Random.init seed */
CAMLprim value mcmcgpu_set_seed(value ctx, value seed) {
  check(Ctx_val(ctx), mg_ctx_set_seed(Ctx_val(ctx), (uint64_t)Int64_val(seed)));
  return Val_unit;
}
/* Mcmc.reset_counters / Mcmc.get_counters (mcmc.ml:30-35) */
CAMLprim value mcmcgpu_reset_counters(value ctx) { check(Ctx_val(ctx), mg_reset_counters(Ctx_val(ctx))); return Val_unit; }
CAMLprim value mcmcgpu_get_counters(value ctx) {
  CAMLparam1(ctx);
  CAMLlocal1(r);
  int64_t a = 0, b = 0;
  check(Ctx_val(ctx), mg_get_counters(Ctx_val(ctx), &a, &b));
  r = caml_alloc_tuple(2);
  Store_field(r, 0, Val_long(a)); Store_field(r, 1, Val_long(b));
  CAMLreturn(r);
}

/* ---- Mcmc.mcmc_array (mcmc.ml:58-72) -----------------------------------
 * external mcmc_array : ctx -> logfn -> logfn -> proposal -> nbin:int -> nskip:int -> n:int -> nchains:int ->
 *   chain_offset:int -> (float, float64_elt, c_layout) Array2.t (* x0 [C][D] *) ->
 *   (float, float64_elt, c_layout) Array3.t (* out [C][n][D+2] *) -> unit
 * More than 5 arguments: bytecode / native pair. */
CAMLprim value mcmcgpu_mcmc_array_native(value ctx, value like, value prior, value prop, value nbin, value nskip,
                                         value n, value nchains, value chain_offset, value x0, value out) {
  CAMLparam5(ctx, like, prior, prop, x0);
  CAMLxparam1(out);
  mg_logfn l = logfn_of_value(like), p = logfn_of_value(prior);
  mg_proposal j = proposal_of_value(prop);
  mg_mcmc_cfg cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.nchains = Long_val(nchains); cfg.dim = l.dim; cfg.layout = MG_LAYOUT_CHAIN_MAJOR;
  cfg.nbin = Long_val(nbin); cfg.nskip = Long_val(nskip); cfg.n = Long_val(n);
  cfg.chain_offset = (uint64_t)Long_val(chain_offset);
  cfg.x0_shared = (Caml_ba_array_val(x0)->dim[0] == 1 && cfg.nchains > 1);
  const double *px0 = (const double *)Caml_ba_data_val(x0);
  double *pout = (double *)Caml_ba_data_val(out);
  mg_ctx *c = Ctx_val(ctx);
  caml_release_runtime_system();   /* Bigarray data does not move */
  int rc = mg_mcmc_array(c, &l, &p, &j, &cfg, px0, pout, NULL, NULL);
  caml_acquire_runtime_system();
  check(c, rc);
  CAMLreturn(Val_unit);
}
CAMLprim value mcmcgpu_mcmc_array_bytecode(value *a, int argn) {
  (void)argn;
  return mcmcgpu_mcmc_array_native(a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7], a[8], a[9], a[10]);
}

/* ---- Kd_tree / Interpolate_pdf ----------------------------------------- */
/* Interpolate_pdf.make pts low high (interpolate_pdf.ml:111-112) */
CAMLprim value mcmcgpu_interp_make(value ctx, value pts, value low, value high) {
  CAMLparam4(ctx, pts, low, high);
  CAMLlocal1(v);
  mg_kdtree *t = NULL;
  struct caml_ba_array *b = Caml_ba_array_val(pts);
  mg_ctx *c = Ctx_val(ctx);
  const double *pp = (const double *)Caml_ba_data_val(pts), *pl = (const double *)Caml_ba_data_val(low),
               *ph = (const double *)Caml_ba_data_val(high);
  int64_t N = b->dim[0]; int32_t D = (int32_t)b->dim[1];
  caml_release_runtime_system();
  int rc = mg_kdtree_build(c, pp, N, D, pl, ph, 2, &t);
  caml_acquire_runtime_system();
  check(c, rc);
  v = caml_alloc_custom(&tree_ops, sizeof(tree_box), 0, 1);
  Treebox_val(v)->tree = t; Treebox_val(v)->box = Box_val(ctx); Box_val(ctx)->refs++;
  CAMLreturn(v);
}
/* Interpolate_pdf.jump_prob / jump_prob_high_level n (interpolate_pdf.ml:135-159) on a batch */
CAMLprim value mcmcgpu_interp_jump_prob(value ctx, value tree, value nstop, value q, value out) {
  CAMLparam5(ctx, tree, nstop, q, out);
  mg_ctx *c = Ctx_val(ctx);
  int rc = mg_interp_jump_prob(c, Tree_val(tree), (const double *)Caml_ba_data_val(q),
                               Caml_ba_array_val(q)->dim[0], Int_val(nstop), (double *)Caml_ba_data_val(out));
  check(c, rc);
  CAMLreturn(Val_unit);
}
/* Interpolate_pdf.draw / draw_high_level n (interpolate_pdf.ml:114-133), m draws */
CAMLprim value mcmcgpu_interp_draw(value ctx, value tree, value nstop, value out) {
  CAMLparam4(ctx, tree, nstop, out);
  mg_ctx *c = Ctx_val(ctx);
  int rc = mg_interp_draw(c, Tree_val(tree), Caml_ba_array_val(out)->dim[0], Int_val(nstop),
                          (double *)Caml_ba_data_val(out));
  check(c, rc);
  CAMLreturn(Val_unit);
}

/* ---- Evidence (evidence.ml:101-107,148-165,202-221) ---------------------- */
CAMLprim value mcmcgpu_evidence_harmonic_mean(value ctx, value ll) {
  CAMLparam2(ctx, ll);
  double out = 0.0;
  mg_ctx *c = Ctx_val(ctx);
  check(c, mg_evidence_harmonic_mean(c, (const double *)Caml_ba_data_val(ll), Caml_ba_array_val(ll)->dim[0], &out));
  CAMLreturn(caml_copy_double(out));
}
CAMLprim value mcmcgpu_evidence_lebesgue_native(value ctx, value n, value eps, value pts, value ll, value lp) {
  CAMLparam5(ctx, n, eps, pts, ll);
  CAMLxparam1(lp);
  double out = 0.0;
  mg_ctx *c = Ctx_val(ctx);
  struct caml_ba_array *b = Caml_ba_array_val(pts);
  const double *pp = (const double *)Caml_ba_data_val(pts), *pll = (const double *)Caml_ba_data_val(ll),
               *plp = (const double *)Caml_ba_data_val(lp);
  int64_t N = b->dim[0]; int32_t D = (int32_t)b->dim[1]; int32_t nn = Int_val(n); double e = Double_val(eps);
  caml_release_runtime_system();
  int rc = mg_evidence_lebesgue(c, pp, pll, plp, N, D, nn, e, &out);
  caml_acquire_runtime_system();
  check(c, rc);
  CAMLreturn(caml_copy_double(out));
}
CAMLprim value mcmcgpu_evidence_lebesgue_bytecode(value *a, int argn) {
  (void)argn;
  return mcmcgpu_evidence_lebesgue_native(a[0], a[1], a[2], a[3], a[4], a[5]);
}
CAMLprim value mcmcgpu_evidence_direct(value ctx, value n, value pts, value ll, value lp) {
  CAMLparam5(ctx, n, pts, ll, lp);
  double out = 0.0;
  mg_ctx *c = Ctx_val(ctx);
  struct caml_ba_array *b = Caml_ba_array_val(pts);
  check(c, mg_evidence_direct(c, (const double *)Caml_ba_data_val(pts), (const double *)Caml_ba_data_val(ll),
                              (const double *)Caml_ba_data_val(lp), b->dim[0], (int32_t)b->dim[1], Int_val(n), &out));
  CAMLreturn(caml_copy_double(out));
}

/* ---- Stats (stats.ml:17-87) ---------------------------------------------- */
CAMLprim value mcmcgpu_stats_multi_mean(value ctx, value xs, value out) {
  CAMLparam3(ctx, xs, out);
  mg_ctx *c = Ctx_val(ctx);
  struct caml_ba_array *b = Caml_ba_array_val(xs);
  check(c, mg_stats_multi_mean(c, (const double *)Caml_ba_data_val(xs), b->dim[0], (int32_t)b->dim[1],
                               (double *)Caml_ba_data_val(out)));
  CAMLreturn(Val_unit);
}
/* mean_opt: float array option as a Bigarray of length 0 (None) or D (Some mu) */
CAMLprim value mcmcgpu_stats_multi_std(value ctx, value xs, value mean_opt, value out) {
  CAMLparam4(ctx, xs, mean_opt, out);
  mg_ctx *c = Ctx_val(ctx);
  struct caml_ba_array *b = Caml_ba_array_val(xs);
  const double *mu = Caml_ba_array_val(mean_opt)->dim[0] > 0 ? (const double *)Caml_ba_data_val(mean_opt) : NULL;
  check(c, mg_stats_multi_std(c, (const double *)Caml_ba_data_val(xs), b->dim[0], (int32_t)b->dim[1], mu,
                              (double *)Caml_ba_data_val(out)));
  CAMLreturn(Val_unit);
}

/* ---- ensemble convergence diagnostics (mg_stats_chain_diagnostics*, an addition beyond the reference) ------------
 * out: [4][F] = rhat, ess, tau, window_closed (0. / 1.); rho: [F][L]; seq_tau: [F][M], or [0][0] for none.
 * external chain_diagnostics : ctx -> int (* maxlag *) -> int (* split *) -> (float, float64_elt, c_layout) Array3.t
 *   (* block [n][D+2][C] *) -> Array2.t (* out *) -> Array2.t (* rho *) -> Array2.t (* seq_tau *) -> unit
 * More than 5 arguments: bytecode / native pair. */
static void diag_run(mg_ctx *c, const double *blk_host, const double *blk_dev, mg_diag_cfg *cfg, value out, value rho,
                     double *seq_tau) {
  const int F = cfg->dim + 2;
  int32_t *closed = (int32_t *)malloc(sizeof(int32_t) * (size_t)F);
  double *o = (double *)Caml_ba_data_val(out);
  double *prho = (double *)Caml_ba_data_val(rho);
  if (!closed) caml_failwith("chain_diagnostics: out of memory");
  caml_release_runtime_system();
  int rc = blk_host ? mg_stats_chain_diagnostics(c, blk_host, cfg, o, o + F, o + 2 * F, closed, prho, seq_tau)
                    : mg_stats_chain_diagnostics_dev(c, blk_dev, cfg, o, o + F, o + 2 * F, closed, prho, seq_tau);
  caml_acquire_runtime_system();
  if (rc == MG_OK)
    for (int f = 0; f < F; ++f) o[3 * F + f] = (double)closed[f];
  free(closed);
  check(c, rc);
}
CAMLprim value mcmcgpu_chain_diagnostics_native(value ctx, value maxlag, value split, value blk, value out, value rho,
                                                value seq_tau) {
  CAMLparam5(ctx, maxlag, split, blk, out);
  CAMLxparam2(rho, seq_tau);
  struct caml_ba_array *b = Caml_ba_array_val(blk);
  mg_diag_cfg cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.n = b->dim[0]; cfg.dim = (int32_t)b->dim[1] - 2; cfg.nchains = b->dim[2];
  cfg.maxlag = Int_val(maxlag); cfg.split = Int_val(split);
  double *st = Caml_ba_array_val(seq_tau)->dim[0] > 0 ? (double *)Caml_ba_data_val(seq_tau) : NULL;
  diag_run(Ctx_val(ctx), (const double *)Caml_ba_data_val(blk), NULL, &cfg, out, rho, st);
  CAMLreturn(Val_unit);
}
CAMLprim value mcmcgpu_chain_diagnostics_bytecode(value *a, int argn) {
  (void)argn;
  return mcmcgpu_chain_diagnostics_native(a[0], a[1], a[2], a[3], a[4], a[5], a[6]);
}
/* the same on a device block (its device address as int64, e.g. from another CUDA library); seq_tau: device
 * address of [F][M] doubles or 0L.
 * external chain_diagnostics_dev : ctx -> int64 -> int (* n *) -> int (* dim *) -> int (* nchains *) ->
 *   int (* maxlag *) -> int (* split *) -> Array2.t (* out *) -> Array2.t (* rho *) -> int64 -> unit */
CAMLprim value mcmcgpu_chain_diagnostics_dev_native(value ctx, value ptr, value n, value dim, value nchains, value maxlag,
                                                    value split, value out, value rho, value seq_tau) {
  CAMLparam5(ctx, ptr, n, dim, nchains);
  CAMLxparam3(maxlag, split, out);
  CAMLxparam2(rho, seq_tau);
  mg_diag_cfg cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.n = Long_val(n); cfg.dim = Int_val(dim); cfg.nchains = Long_val(nchains);
  cfg.maxlag = Int_val(maxlag); cfg.split = Int_val(split);
  diag_run(Ctx_val(ctx), NULL, (const double *)(intptr_t)Int64_val(ptr), &cfg, out, rho, (double *)(intptr_t)Int64_val(seq_tau));
  CAMLreturn(Val_unit);
}
CAMLprim value mcmcgpu_chain_diagnostics_dev_bytecode(value *a, int argn) {
  (void)argn;
  return mcmcgpu_chain_diagnostics_dev_native(a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7], a[8], a[9]);
}

/* ---- exact quantiles of a sample block (mg_stats_quantiles*) ------------------------------------------------
 * external quantiles : ctx -> (float, float64_elt, c_layout) Array3.t (* block [n][D+2][C] *) ->
 *   Array1.t (* probs *) -> Array2.t (* out [D+2][nq] *) -> unit */
CAMLprim value mcmcgpu_quantiles(value ctx, value blk, value probs, value out) {
  CAMLparam4(ctx, blk, probs, out);
  struct caml_ba_array *b = Caml_ba_array_val(blk);
  mg_ctx *c = Ctx_val(ctx);
  const double *x = (const double *)Caml_ba_data_val(blk), *p = (const double *)Caml_ba_data_val(probs);
  double *o = (double *)Caml_ba_data_val(out);
  const int64_t n = b->dim[0], C = b->dim[2];
  const int32_t D = (int32_t)b->dim[1] - 2, nq = (int32_t)Caml_ba_array_val(probs)->dim[0];
  caml_release_runtime_system();
  int rc = mg_stats_quantiles(c, x, n, D, C, p, nq, o);
  caml_acquire_runtime_system();
  check(c, rc);
  CAMLreturn(Val_unit);
}
/* the same on a device block (its device address as int64)
 * external quantiles_dev : ctx -> int64 -> int (* n *) -> int (* dim *) -> int (* nchains *) -> Array1.t (* probs *) ->
 *   Array2.t (* out *) -> unit */
CAMLprim value mcmcgpu_quantiles_dev_native(value ctx, value ptr, value n, value dim, value nchains, value probs,
                                            value out) {
  CAMLparam5(ctx, ptr, n, dim, nchains);
  CAMLxparam2(probs, out);
  mg_ctx *c = Ctx_val(ctx);
  const double *x = (const double *)(intptr_t)Int64_val(ptr), *p = (const double *)Caml_ba_data_val(probs);
  double *o = (double *)Caml_ba_data_val(out);
  const int32_t nq = (int32_t)Caml_ba_array_val(probs)->dim[0];
  const int64_t nn = Long_val(n), C = Long_val(nchains);
  const int32_t D = Int_val(dim);
  caml_release_runtime_system();
  int rc = mg_stats_quantiles_dev(c, x, nn, D, C, p, nq, o);
  caml_acquire_runtime_system();
  check(c, rc);
  CAMLreturn(Val_unit);
}
CAMLprim value mcmcgpu_quantiles_dev_bytecode(value *a, int argn) {
  (void)argn;
  return mcmcgpu_quantiles_dev_native(a[0], a[1], a[2], a[3], a[4], a[5], a[6]);
}

/* ---- Stats.draw_uniform / draw_gaussian / draw_cauchy (stats.ml:89-91,113-128), n draws per call ----------
 * external stats_draw : ctx -> int -> float -> float -> (float, float64_elt, c_layout) Array1.t -> unit
 * kind: 0 uniform a b | 1 gaussian mu sigma | 2 cauchy x0 gamma (MG_DRAW_*) */
CAMLprim value mcmcgpu_stats_draw(value ctx, value kind, value a, value b, value out) {
  CAMLparam5(ctx, kind, a, b, out);
  mg_ctx *c = Ctx_val(ctx);
  check(c, mg_stats_draw(c, Int_val(kind), Double_val(a), Double_val(b), Caml_ba_array_val(out)->dim[0],
                         (double *)Caml_ba_data_val(out)));
  CAMLreturn(Val_unit);
}

/* ---- Nested.posterior_samples (nested.ml:152-178): indices of n weighted draws ------------------------------
 * external posterior_indices : ctx -> (float, float64_elt, c_layout) Array1.t -> (int64, int64_elt, c_layout) Array1.t -> unit */
CAMLprim value mcmcgpu_nested_posterior_indices(value ctx, value logw, value out) {
  CAMLparam3(ctx, logw, out);
  mg_ctx *c = Ctx_val(ctx);
  check(c, mg_nested_posterior_indices(c, (const double *)Caml_ba_data_val(logw), Caml_ba_array_val(logw)->dim[0],
                                       Caml_ba_array_val(out)->dim[0], (int64_t *)Caml_ba_data_val(out)));
  CAMLreturn(Val_unit);
}

/* ---- Mcmc.rjmcmc_array (mcmc.ml:121-139) -----------------------------------
 * type rj_model = { like : logfn; prior : logfn; prop : proposal; into : tree option;
 *                   into_gauss : (float, float64_elt, c_layout) Array1.t; nstop : int; p : float }
 * Returns (#A, #B) = Mcmc.rjmcmc_model_counts; out_model : (int, int8_unsigned_elt, c_layout) Array2.t [n][C]. */
static mg_rj_model rj_of_value(value v) {
  mg_rj_model m;
  memset(&m, 0, sizeof m);
  m.like = logfn_of_value(Field(v, 0));
  m.prior = logfn_of_value(Field(v, 1));
  m.prop = proposal_of_value(Field(v, 2));
  if (Is_block(Field(v, 3))) {              /* Some tree: Interp.draw / log (Interp.jump_prob) */
    m.into.kind = MG_INTO_INTERP;
    m.into.tree = Tree_val(Field(Field(v, 3), 0));
    m.into.nstop = Int_val(Field(v, 5));
  } else {                                  /* None: independent Gaussian (mu, sigma) */
    m.into.kind = MG_INTO_INDEP_GAUSS;
    m.into.params = (const double *)Caml_ba_data_val(Field(v, 4));
    m.into.nparams = Caml_ba_array_val(Field(v, 4))->dim[0];
  }
  m.p = Double_val(Field(v, 6));
  return m;
}
CAMLprim value mcmcgpu_rjmcmc_array_native(value ctx, value ma, value mb, value nbin, value nskip, value n,
                                           value nchains, value a0, value b0, value out_model) {
  CAMLparam5(ctx, ma, mb, a0, b0);
  CAMLxparam1(out_model);
  CAMLlocal1(r);
  mg_rj_model A = rj_of_value(ma), B = rj_of_value(mb);
  mg_rjmcmc_cfg cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.nchains = Long_val(nchains); cfg.nbin = Long_val(nbin); cfg.nskip = Long_val(nskip); cfg.n = Long_val(n);
  int64_t counts[2] = {0, 0};
  mg_ctx *c = Ctx_val(ctx);
  const double *pa = (const double *)Caml_ba_data_val(a0), *pb = (const double *)Caml_ba_data_val(b0);
  uint8_t *pm = (uint8_t *)Caml_ba_data_val(out_model);
  caml_release_runtime_system();
  int rc = mg_rjmcmc_array(c, &A, &B, &cfg, pa, pb, pm, NULL, counts);
  caml_acquire_runtime_system();
  check(c, rc);                             /* incl. Assert_failure mcmc.ml:90 -> Failure */
  r = caml_alloc_tuple(2);
  Store_field(r, 0, Val_long(counts[0])); Store_field(r, 1, Val_long(counts[1]));
  CAMLreturn(r);
}
CAMLprim value mcmcgpu_rjmcmc_array_bytecode(value *a, int argn) {
  (void)argn;
  return mcmcgpu_rjmcmc_array_native(a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7], a[8], a[9]);
}

/* k-model extension (mg_rjmcmc_array_k; the reference's sum type is two-model, mcmc.ml:83-87).
 * external rjmcmc_array_k_raw : ctx -> raw_model array -> int -> int -> int -> int ->
 *   (float, float64_elt, c_layout) Array1.t array -> (int, int8_unsigned_elt, c_layout) Array2.t -> int array */
CAMLprim value mcmcgpu_rjmcmc_array_k_native(value ctx, value models, value nbin, value nskip, value n, value nchains,
                                             value starts, value out_model) {
  CAMLparam4(ctx, models, starts, out_model);
  CAMLlocal1(r);
  const int K = (int)Wosize_val(models);
  mg_ctx *c = Ctx_val(ctx);
  if (K < 2 || K > MG_RJ_MAX_MODELS || (int)Wosize_val(starts) != K) caml_invalid_argument("rjmcmc_array_k: 2..8 models, one start point each");
  mg_rj_model M[MG_RJ_MAX_MODELS];
  const double *st[MG_RJ_MAX_MODELS];
  for (int k = 0; k < K; ++k) { M[k] = rj_of_value(Field(models, k)); st[k] = (const double *)Caml_ba_data_val(Field(starts, k)); }
  mg_rjmcmc_cfg cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.nchains = Long_val(nchains); cfg.nbin = Long_val(nbin); cfg.nskip = Long_val(nskip); cfg.n = Long_val(n);
  int64_t counts[MG_RJ_MAX_MODELS] = {0};
  uint8_t *pm = (uint8_t *)Caml_ba_data_val(out_model);
  caml_release_runtime_system();
  int rc = mg_rjmcmc_array_k(c, M, K, &cfg, st, pm, NULL, counts);
  caml_acquire_runtime_system();
  check(c, rc);
  r = caml_alloc_tuple(K);
  for (int k = 0; k < K; ++k) Store_field(r, k, Val_long(counts[k]));
  CAMLreturn(r);
}
CAMLprim value mcmcgpu_rjmcmc_array_k_bytecode(value *a, int argn) {
  (void)argn;
  return mcmcgpu_rjmcmc_array_k_native(a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7]);
}

/* ---- Ellipse.enclosing_ellipse sf to_coord pts (ellipse.ml:98-103), to_coord = identity ------------------
 * external enclosing_ellipse_raw : ctx -> float -> (float, float64_elt, c_layout) Array2.t ->
 *   (float, float64_elt, c_layout) Array1.t -> (float, float64_elt, c_layout) Array1.t ->
 *   (float, float64_elt, c_layout) Array2.t -> unit        (center, axes, orientation are outputs) */
CAMLprim value mcmcgpu_enclosing_ellipse(value ctx, value sf, value pts, value center, value axes, value ori) {
  CAMLparam5(ctx, sf, pts, center, axes);
  CAMLxparam1(ori);
  mg_ctx *c = Ctx_val(ctx);
  const int64_t N = Caml_ba_array_val(pts)->dim[0]; const int32_t D = (int32_t)Caml_ba_array_val(pts)->dim[1];
  const double *pp = (const double *)Caml_ba_data_val(pts);
  double *pc = (double *)Caml_ba_data_val(center), *pa = (double *)Caml_ba_data_val(axes), *po = (double *)Caml_ba_data_val(ori);
  const double f = Double_val(sf);
  caml_release_runtime_system();
  int rc = mg_ellipse_enclosing(c, pp, N, D, f, pc, pa, po);
  caml_acquire_runtime_system();
  check(c, rc);
  CAMLreturn(Val_unit);
}
CAMLprim value mcmcgpu_enclosing_ellipse_bytecode(value *a, int argn) {
  (void)argn;
  return mcmcgpu_enclosing_ellipse(a[0], a[1], a[2], a[3], a[4], a[5]);
}

/* ---- Nested.nested_evidence (nested.ml:122-146) ----------------------------
 * external nested_evidence : ctx -> logfn -> logfn -> lo -> hi -> epsrel:float -> nmcmc:int -> nlive:int ->
 *   mode_hopping_frac:float -> batch:int -> pts [cap][D] -> ll [cap] -> lp [cap] -> logw [cap] ->
 *   float * float * int   (log_ev, log_dev, number of points) */
CAMLprim value mcmcgpu_nested_evidence_native(value ctx, value like, value prior, value lo, value hi, value epsrel,
                                              value nmcmc, value nlive, value mode_hop, value batch, value pts,
                                              value ll, value lp, value logw) {
  CAMLparam5(ctx, like, prior, lo, hi);
  CAMLxparam4(pts, ll, lp, logw);
  CAMLlocal1(r);
  mg_logfn l = logfn_of_value(like), p = logfn_of_value(prior);
  mg_nested_cfg cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.dim = l.dim; cfg.nlive = Int_val(nlive); cfg.nmcmc = Int_val(nmcmc); cfg.batch = Int_val(batch);
  cfg.epsrel = Double_val(epsrel); cfg.mode_hopping_frac = Double_val(mode_hop);
  cfg.max_points = Caml_ba_array_val(ll)->dim[0];
  double log_ev = 0.0, log_dev = 0.0; int64_t npts = 0;
  mg_ctx *c = Ctx_val(ctx);
  const double *plo = (const double *)Caml_ba_data_val(lo), *phi = (const double *)Caml_ba_data_val(hi);
  double *ppts = (double *)Caml_ba_data_val(pts), *pll = (double *)Caml_ba_data_val(ll),
         *plp = (double *)Caml_ba_data_val(lp), *plw = (double *)Caml_ba_data_val(logw);
  caml_release_runtime_system();
  int rc = mg_nested_evidence(c, &l, &p, plo, phi, &cfg, &log_ev, &log_dev, &npts, ppts, pll, plp, plw);
  caml_acquire_runtime_system();
  check(c, rc);                             /* nested.ml:70-72 -> Failure */
  r = caml_alloc_tuple(3);
  Store_field(r, 0, caml_copy_double(log_ev)); Store_field(r, 1, caml_copy_double(log_dev));
  Store_field(r, 2, Val_long(npts));
  CAMLreturn(r);
}
CAMLprim value mcmcgpu_nested_evidence_bytecode(value *a, int argn) {
  (void)argn;
  return mcmcgpu_nested_evidence_native(a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7], a[8], a[9], a[10], a[11],
                                        a[12], a[13]);
}
/* Nested.log_total_error_estimate (nested.ml:148-150) */
CAMLprim value mcmcgpu_log_total_error_estimate(value log_ev, value log_dev, value nlive) {
  return caml_copy_double(mg_nested_log_total_error(Double_val(log_ev), Double_val(log_dev), Int_val(nlive)));
}

/* ---- several GPUs: one OCaml process per GPU, one communicator per context (mg_comm_*, NCCL inside the library) ---------
 * The 128-byte NCCL id is made by rank 0 (comm_unique_id) and handed to the other ranks by the host program (a file, a
 * socket, MPI ...); it travels as a (int, int8_unsigned_elt, c_layout) Array1.t of length 128. */
typedef struct { mg_comm *comm; ctx_box *box; } comm_box;
#define Commbox_val(v) ((comm_box *)Data_custom_val(v))
#define Comm_val(v) (Commbox_val(v)->comm)
static void comm_finalize(value v) {
  comm_box *b = Commbox_val(v);
  if (b->comm) { mg_comm_destroy(b->comm); b->comm = NULL; }
  box_release(b->box); b->box = NULL;
}
static struct custom_operations comm_ops = {"mcmc_gpu.comm", comm_finalize, custom_compare_default, custom_hash_default,
                                            custom_serialize_default, custom_deserialize_default,
                                            custom_compare_ext_default, custom_fixed_length_default};
/* external comm_unique_id : (int, int8_unsigned_elt, c_layout) Array1.t -> unit */
CAMLprim value mcmcgpu_comm_unique_id(value id) {
  CAMLparam1(id);
  if (Caml_ba_array_val(id)->dim[0] != MG_COMM_ID_BYTES) caml_invalid_argument("comm_unique_id: the id holds 128 bytes");
  if (mg_comm_get_unique_id((uint8_t *)Caml_ba_data_val(id)) != MG_OK) caml_failwith("nccl: cannot create a unique id");
  CAMLreturn(Val_unit);
}
/* external comm_create : ctx -> int -> int -> (int, int8_unsigned_elt, c_layout) Array1.t -> comm   (nranks, rank, id) */
CAMLprim value mcmcgpu_comm_create(value ctx, value nranks, value rank, value id) {
  CAMLparam4(ctx, nranks, rank, id);
  CAMLlocal1(v);
  mg_ctx *c = Ctx_val(ctx);
  mg_comm *cm = NULL;
  const uint8_t *pid = (const uint8_t *)Caml_ba_data_val(id);
  const int n = Int_val(nranks), r = Int_val(rank);
  caml_release_runtime_system();                 /* ncclCommInitRank waits for the other ranks */
  int rc = mg_comm_create(c, n, r, pid, &cm);
  caml_acquire_runtime_system();
  check(c, rc);
  v = caml_alloc_custom(&comm_ops, sizeof(comm_box), 0, 1);
  Commbox_val(v)->comm = cm; Commbox_val(v)->box = Box_val(ctx); Box_val(ctx)->refs++;
  CAMLreturn(v);
}
static value wrap_tree(value ctx, mg_kdtree *t) {
  CAMLparam1(ctx);
  CAMLlocal1(v);
  v = caml_alloc_custom(&tree_ops, sizeof(tree_box), 0, 1);
  Treebox_val(v)->tree = t; Treebox_val(v)->box = Box_val(ctx); Box_val(ctx)->refs++;
  CAMLreturn(v);
}
/* Interp.make on `root`, the tree replicated on every rank (one ncclBroadcast of the blob).
 * external interp_broadcast : ctx -> comm -> interp_tree option -> int -> interp_tree */
CAMLprim value mcmcgpu_interp_broadcast(value ctx, value comm, value tree_opt, value root) {
  CAMLparam4(ctx, comm, tree_opt, root);
  mg_ctx *c = Ctx_val(ctx);
  mg_kdtree *mine = Is_block(tree_opt) ? Tree_val(Field(tree_opt, 0)) : NULL, *out = NULL;
  mg_comm *cm = Comm_val(comm);
  const int r = Int_val(root);
  caml_release_runtime_system();
  int rc = mg_kdtree_broadcast(cm, mine, r, &out);
  caml_acquire_runtime_system();
  check(c, rc);
  if (out == mine && Is_block(tree_opt)) CAMLreturn(Field(tree_opt, 0));   /* the root keeps its own tree */
  CAMLreturn(wrap_tree(ctx, out));
}
/* Interp.make by all ranks together (every rank passes the same points): mg_kdtree_build_distributed.
 * external interp_make_distributed : ctx -> comm -> pts -> low -> high -> interp_tree */
CAMLprim value mcmcgpu_interp_make_distributed(value ctx, value comm, value pts, value low, value high) {
  CAMLparam5(ctx, comm, pts, low, high);
  mg_ctx *c = Ctx_val(ctx);
  mg_comm *cm = Comm_val(comm);
  struct caml_ba_array *b = Caml_ba_array_val(pts);
  const int64_t N = b->dim[0]; const int32_t D = (int32_t)b->dim[1];
  const double *pp = (const double *)Caml_ba_data_val(pts), *pl = (const double *)Caml_ba_data_val(low),
               *ph = (const double *)Caml_ba_data_val(high);
  mg_kdtree *t = NULL;
  void *d_pts = NULL;
  caml_release_runtime_system();
  int rc = mg_malloc_device(c, (int64_t)sizeof(double) * N * D, &d_pts);
  if (rc == MG_OK) rc = mg_memcpy_h2d(c, d_pts, pp, (int64_t)sizeof(double) * N * D);
  if (rc == MG_OK) rc = mg_kdtree_build_distributed(cm, (const double *)d_pts, N, D, pl, ph, 2, &t);
  if (d_pts) mg_free_device(c, d_pts);
  caml_acquire_runtime_system();
  check(c, rc);
  CAMLreturn(wrap_tree(ctx, t));
}
/* Evidence.evidence_lebesgue ?n ?eps with the kd-tree built by all ranks and the cells shared out; the samples live on
 * `root` (the other ranks pass empty arrays).  Every rank receives the same value.
 * external evidence_lebesgue_sharded : ctx -> comm -> int -> pts -> ll -> lp -> int -> float -> float */
CAMLprim value mcmcgpu_evidence_lebesgue_sharded_native(value ctx, value comm, value root, value pts, value ll, value lp,
                                                        value n, value eps) {
  CAMLparam5(ctx, comm, root, pts, ll);
  CAMLxparam3(lp, n, eps);
  mg_ctx *c = Ctx_val(ctx);
  mg_comm *cm = Comm_val(comm);
  const int r = Int_val(root), nn = Int_val(n);
  const double e = Double_val(eps);
  const int is_root = mg_comm_rank(cm) == r;
  struct caml_ba_array *b = Caml_ba_array_val(pts);
  const int64_t N = b->dim[0]; const int32_t D = (int32_t)b->dim[1];
  const double *pp = (const double *)Caml_ba_data_val(pts), *pll = (const double *)Caml_ba_data_val(ll),
               *plp = (const double *)Caml_ba_data_val(lp);
  void *dp = NULL, *dl = NULL, *dq = NULL;
  double z = 0.0;
  caml_release_runtime_system();
  int rc = MG_OK;
  if (is_root) {
    rc = mg_malloc_device(c, (int64_t)sizeof(double) * N * D, &dp);
    if (rc == MG_OK) rc = mg_malloc_device(c, (int64_t)sizeof(double) * N, &dl);
    if (rc == MG_OK) rc = mg_malloc_device(c, (int64_t)sizeof(double) * N, &dq);
    if (rc == MG_OK) rc = mg_memcpy_h2d(c, dp, pp, (int64_t)sizeof(double) * N * D);
    if (rc == MG_OK) rc = mg_memcpy_h2d(c, dl, pll, (int64_t)sizeof(double) * N);
    if (rc == MG_OK) rc = mg_memcpy_h2d(c, dq, plp, (int64_t)sizeof(double) * N);
  }
  /* (a root that failed above still enters the collective: the library broadcasts its status first) */
  int rc2 = mg_evidence_lebesgue_sharded(cm, r, rc == MG_OK ? (const double *)dp : NULL, (const double *)dl, (const double *)dq, N, D, nn, e, &z);
  if (dp) mg_free_device(c, dp);
  if (dl) mg_free_device(c, dl);
  if (dq) mg_free_device(c, dq);
  caml_acquire_runtime_system();
  check(c, rc != MG_OK ? rc : rc2);
  CAMLreturn(caml_copy_double(z));
}
CAMLprim value mcmcgpu_evidence_lebesgue_sharded_bytecode(value *a, int argn) {
  (void)argn;
  return mcmcgpu_evidence_lebesgue_sharded_native(a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7]);
}
/* Mcmc.rjmcmc_array with the chains cut into one range per rank (global chain ids: results do not depend on the number
 * of ranks); returns the counts of ALL ranks.
 * external rjmcmc_array_sharded_raw : ctx -> comm -> rj_model_raw -> rj_model_raw -> int -> int -> int -> int -> a0 -> b0 -> int * int */
CAMLprim value mcmcgpu_rjmcmc_array_sharded_native(value ctx, value comm, value ma, value mb, value nbin, value nskip,
                                                   value n, value nchains, value a0, value b0) {
  CAMLparam5(ctx, comm, ma, mb, a0);
  CAMLxparam1(b0);
  CAMLlocal1(r);
  mg_rj_model A = rj_of_value(ma), B = rj_of_value(mb);
  mg_rjmcmc_cfg cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.nchains = Long_val(nchains); cfg.nbin = Long_val(nbin); cfg.nskip = Long_val(nskip); cfg.n = Long_val(n);
  int64_t counts[2] = {0, 0}, sb = 0, sc = 0;
  mg_ctx *c = Ctx_val(ctx);
  mg_comm *cm = Comm_val(comm);
  const double *pa = (const double *)Caml_ba_data_val(a0), *pb = (const double *)Caml_ba_data_val(b0);
  caml_release_runtime_system();
  int rc = mg_rjmcmc_array_sharded(cm, &A, &B, &cfg, pa, pb, NULL, NULL, counts, &sb, &sc);
  caml_acquire_runtime_system();
  check(c, rc);
  r = caml_alloc_tuple(2);
  Store_field(r, 0, Val_long(counts[0])); Store_field(r, 1, Val_long(counts[1]));
  CAMLreturn(r);
}
CAMLprim value mcmcgpu_rjmcmc_array_sharded_bytecode(value *a, int argn) {
  (void)argn;
  return mcmcgpu_rjmcmc_array_sharded_native(a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7], a[8], a[9]);
}
