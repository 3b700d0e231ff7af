(* mcmc_gpu.ml -- OCaml side of the binding (see mcmc_gpu.mli).
   NOT COMPILED in this repository's image (no OCaml toolchain). *)
open Bigarray

type ctx
type tree

type logfn = { kind : int; dim : int; scale : float; params : (float, float64_elt, c_layout) Array1.t }
type proposal = { pkind : int; pdim : int; pparams : (float, float64_elt, c_layout) Array1.t }

external ctx_create : int -> int64 -> ctx = "mcmcgpu_ctx_create"
external set_seed : ctx -> int64 -> unit = "mcmcgpu_set_seed"
external reset_counters : ctx -> unit = "mcmcgpu_reset_counters"
external get_counters : ctx -> int * int = "mcmcgpu_get_counters"
external mcmc_array_raw :
  ctx -> logfn -> logfn -> proposal -> int -> int -> int -> int -> int ->
  (float, float64_elt, c_layout) Array2.t -> (float, float64_elt, c_layout) Array3.t -> unit
  = "mcmcgpu_mcmc_array_bytecode" "mcmcgpu_mcmc_array_native"
external interp_make_raw :
  ctx -> (float, float64_elt, c_layout) Array2.t -> (float, float64_elt, c_layout) Array1.t ->
  (float, float64_elt, c_layout) Array1.t -> tree = "mcmcgpu_interp_make"
external interp_jump_prob_raw :
  ctx -> tree -> int -> (float, float64_elt, c_layout) Array2.t -> (float, float64_elt, c_layout) Array1.t -> unit
  = "mcmcgpu_interp_jump_prob"
external interp_draw_raw : ctx -> tree -> int -> (float, float64_elt, c_layout) Array2.t -> unit = "mcmcgpu_interp_draw"
external stats_draw_raw : ctx -> int -> float -> float -> (float, float64_elt, c_layout) Array1.t -> unit = "mcmcgpu_stats_draw"
external posterior_indices_raw :
  ctx -> (float, float64_elt, c_layout) Array1.t -> (int64, int64_elt, c_layout) Array1.t -> unit = "mcmcgpu_nested_posterior_indices"
external harmonic_raw : ctx -> (float, float64_elt, c_layout) Array1.t -> float = "mcmcgpu_evidence_harmonic_mean"
external lebesgue_raw :
  ctx -> int -> float -> (float, float64_elt, c_layout) Array2.t -> (float, float64_elt, c_layout) Array1.t ->
  (float, float64_elt, c_layout) Array1.t -> float
  = "mcmcgpu_evidence_lebesgue_bytecode" "mcmcgpu_evidence_lebesgue_native"
external direct_raw :
  ctx -> int -> (float, float64_elt, c_layout) Array2.t -> (float, float64_elt, c_layout) Array1.t ->
  (float, float64_elt, c_layout) Array1.t -> float = "mcmcgpu_evidence_direct"
type pinned_handle
external pinned_raw : ctx -> int array -> (float, float64_elt, c_layout) Genarray.t * pinned_handle = "mcmcgpu_pinned_raw"
external multi_mean_raw :
  ctx -> (float, float64_elt, c_layout) Array2.t -> (float, float64_elt, c_layout) Array1.t -> unit = "mcmcgpu_stats_multi_mean"
external multi_std_raw :
  ctx -> (float, float64_elt, c_layout) Array2.t -> (float, float64_elt, c_layout) Array1.t ->
  (float, float64_elt, c_layout) Array1.t -> unit = "mcmcgpu_stats_multi_std"
external chain_diagnostics_raw :
  ctx -> int -> int -> (float, float64_elt, c_layout) Array3.t -> (float, float64_elt, c_layout) Array2.t ->
  (float, float64_elt, c_layout) Array2.t -> (float, float64_elt, c_layout) Array2.t -> unit
  = "mcmcgpu_chain_diagnostics_bytecode" "mcmcgpu_chain_diagnostics_native"
external chain_diagnostics_dev_raw :
  ctx -> int64 -> int -> int -> int -> int -> int -> (float, float64_elt, c_layout) Array2.t ->
  (float, float64_elt, c_layout) Array2.t -> int64 -> unit
  = "mcmcgpu_chain_diagnostics_dev_bytecode" "mcmcgpu_chain_diagnostics_dev_native"
external quantiles_raw :
  ctx -> (float, float64_elt, c_layout) Array3.t -> (float, float64_elt, c_layout) Array1.t ->
  (float, float64_elt, c_layout) Array2.t -> unit = "mcmcgpu_quantiles"
external quantiles_dev_raw :
  ctx -> int64 -> int -> int -> int -> (float, float64_elt, c_layout) Array1.t -> (float, float64_elt, c_layout) Array2.t ->
  unit = "mcmcgpu_quantiles_dev_bytecode" "mcmcgpu_quantiles_dev_native"
external evidence_tempered_raw :
  ctx -> logfn -> logfn -> proposal array -> (float, float64_elt, c_layout) Array1.t -> int array ->
  (float, float64_elt, c_layout) Array2.t -> (float, float64_elt, c_layout) Array1.t ->
  (int64, int64_elt, c_layout) Array1.t -> unit = "mcmcgpu_evidence_tempered_bytecode" "mcmcgpu_evidence_tempered_native"
(* the record the stub reads field by field (rj_of_value in mcmc_gpu_stubs.c) *)
type rj_model_raw = {
  r_like : logfn; r_prior : logfn; r_prop : proposal; r_into : tree option;
  r_into_gauss : (float, float64_elt, c_layout) Array1.t; r_nstop : int; r_p : float }
external rjmcmc_array_raw :
  ctx -> rj_model_raw -> rj_model_raw -> int -> int -> int -> int -> (float, float64_elt, c_layout) Array1.t ->
  (float, float64_elt, c_layout) Array1.t -> (int, int8_unsigned_elt, c_layout) Array2.t -> int * int
  = "mcmcgpu_rjmcmc_array_bytecode" "mcmcgpu_rjmcmc_array_native"
external nested_evidence_raw :
  ctx -> logfn -> logfn -> (float, float64_elt, c_layout) Array1.t -> (float, float64_elt, c_layout) Array1.t ->
  float -> int -> int -> float -> int -> (float, float64_elt, c_layout) Array2.t -> (float, float64_elt, c_layout) Array1.t ->
  (float, float64_elt, c_layout) Array1.t -> (float, float64_elt, c_layout) Array1.t -> float * float * int
  = "mcmcgpu_nested_evidence_bytecode" "mcmcgpu_nested_evidence_native"
external log_total_error_estimate_raw : float -> float -> int -> float = "mcmcgpu_log_total_error_estimate"

let create ?(device = 0) ?(seed = 0L) () = ctx_create device seed

let ba1 a = Array1.of_array float64 c_layout a
let ba2 rows = Array2.of_array float64 c_layout rows

(* kind ids of include/mcmc_gpu.h *)
let flat dim = { kind = 0; dim; scale = 1.0; params = ba1 [||] }
let box_prior ?(value = 0.0) lo hi =
  { kind = 2; dim = Array.length lo; scale = 1.0; params = ba1 (Array.concat [lo; hi; [|value|]]) }
let gaussian mu sigma = { kind = 4; dim = Array.length mu; scale = 1.0; params = ba1 (Array.append mu sigma) }
let gaussian_data data = { kind = 6; dim = 2; scale = 1.0; params = ba1 data }
let cauchy_data data = { kind = 7; dim = 2; scale = 1.0; params = ba1 data }
let box_proposal h = { pkind = 0; pdim = Array.length h; pparams = ba1 h }
let uniform_wrapping lo hi dx = { pkind = 1; pdim = Array.length lo; pparams = ba1 (Array.concat [lo; hi; dx]) }
let independent_gaussian mu sigma = { pkind = 2; pdim = Array.length mu; pparams = ba1 (Array.append mu sigma) }
(* Mcmc.differential_evolution_proposal ?mode_hopping_frac to_float from_float samples (mcmc.ml:198-218) with
   to_float = from_float = identity: MG_PROP_DE, params = mode_hopping_frac, M, samples[M][D] *)
let differential_evolution_proposal ?(mode_hopping_frac = 0.0) (samples : float array Mcmc.mcmc_sample array) =
  let m = Array.length samples in
  if m < 2 then invalid_arg "differential_evolution_proposal: need at least two samples";
  let d = Array.length samples.(0).Mcmc.value in
  let blob = Array.concat ([| mode_hopping_frac; float_of_int m |] :: Array.to_list (Array.map (fun s -> s.Mcmc.value) samples)) in
  { pkind = 6; pdim = d; pparams = ba1 blob }

(* Page-locked float64 Bigarrays: the view and the handle that owns the memory travel together. *)
module Pinned = struct
  type 'a t = { data : 'a; handle : pinned_handle }
  let array1 ctx n = let g, h = pinned_raw ctx [| n |] in { data = array1_of_genarray g; handle = h }
  let array2 ctx n d = let g, h = pinned_raw ctx [| n; d |] in { data = array2_of_genarray g; handle = h }
  let array3 ctx a b c = let g, h = pinned_raw ctx [| a; b; c |] in { data = array3_of_genarray g; handle = h }
end

let mcmc_array ctx ?(nbin = 0) ?(nskip = 1) ?(nchains = 1) n like prior prop start =
  let d = like.dim in
  let out = Array3.create float64 c_layout nchains n (d + 2) in
  mcmc_array_raw ctx like prior prop nbin nskip n nchains 0 (ba2 [|start|]) out;
  Array.init nchains (fun c ->
      Array.init n (fun s ->
          { Mcmc.value = Array.init d (fun i -> out.{c, s, i});
            like_prior = { Mcmc.log_likelihood = out.{c, s, d}; log_prior = out.{c, s, d + 1} } }))

module Interp = struct
  type interp_pdf = { tree : tree; dim : int }
  let make ctx pts low high = { tree = interp_make_raw ctx (ba2 pts) (ba1 low) (ba1 high); dim = Array.length low }
  let draw_high_level ctx n ip =
    let out = Array2.create float64 c_layout 1 ip.dim in
    interp_draw_raw ctx ip.tree n out;
    Array.init ip.dim (fun i -> out.{0, i})
  let draw ctx ip = draw_high_level ctx 0 ip
  let jump_prob_batch ctx ?(n = 0) ip pts =
    let out = Array1.create float64 c_layout (Array.length pts) in
    interp_jump_prob_raw ctx ip.tree n (ba2 pts) out;
    Array.init (Array.length pts) (fun i -> out.{i})
  let jump_prob_high_level ctx n ip _ pt = (jump_prob_batch ctx ~n ip [|pt|]).(0)
  let jump_prob ctx ip src pt = jump_prob_high_level ctx 0 ip src pt
end

module Evidence = struct
  let columns samples =
    let pts = ba2 (Array.map (fun s -> s.Mcmc.value) samples) in
    let ll = ba1 (Array.map (fun s -> s.Mcmc.like_prior.Mcmc.log_likelihood) samples) in
    let lp = ba1 (Array.map (fun s -> s.Mcmc.like_prior.Mcmc.log_prior) samples) in
    (pts, ll, lp)
  let evidence_harmonic_mean ctx samples = let _, ll, _ = columns samples in harmonic_raw ctx ll
  let evidence_lebesgue ctx ?(n = 64) ?(eps = 0.1) samples =
    let pts, ll, lp = columns samples in lebesgue_raw ctx n eps pts ll lp
  let evidence_direct ctx ?(n = 64) samples =
    let pts, ll, lp = columns samples in direct_raw ctx n pts ll lp
end

(* Mcmc.rjmcmc_array (mcmc.ml:121-139; mcmc.mli:151-162) for [nchains] chains.  A model is its log-likelihood, log-prior,
   in-model proposal, model prior and the proposal INTO it: an Interp.interp_pdf (Interp.draw / log (Interp.jump_prob ..),
   test/mcmc_test.ml:175-178; ~nstop > 0 selects the *_high_level forms) or an independent Gaussian (mu, sigma). *)
type rj_into = Into_interp of Interp.interp_pdf * int | Into_gaussian of float array * float array
type rj_model = { rj_like : logfn; rj_prior : logfn; rj_prop : proposal; rj_into : rj_into; rj_p : float }
let raw_of_model m =
  match m.rj_into with
  | Into_interp (ip, nstop) ->
      { r_like = m.rj_like; r_prior = m.rj_prior; r_prop = m.rj_prop; r_into = Some ip.Interp.tree; r_into_gauss = ba1 [||];
        r_nstop = nstop; r_p = m.rj_p }
  | Into_gaussian (mu, sigma) ->
      { r_like = m.rj_like; r_prior = m.rj_prior; r_prop = m.rj_prop; r_into = None; r_into_gauss = ba1 (Array.append mu sigma);
        r_nstop = 0; r_p = m.rj_p }
(* returns the model of every recorded sample ([n][nchains], 0 = A, 1 = B) and Mcmc.rjmcmc_model_counts *)
let rjmcmc_array ctx ?(nbin = 0) ?(nskip = 1) ?(nchains = 1) n (ma : rj_model) (mb : rj_model) (a0 : float array) (b0 : float array) =
  let model = Array2.create int8_unsigned c_layout n nchains in
  let counts = rjmcmc_array_raw ctx (raw_of_model ma) (raw_of_model mb) nbin nskip n nchains (ba1 a0) (ba1 b0) model in
  (model, counts)
let rjmcmc_evidence_ratio (na, nb) = float_of_int na /. float_of_int nb     (* mcmc.ml:151-153 *)

(* k models (mg_rjmcmc_array_k): an extension, the reference's sum type is two-model (mcmc.ml:83-87); with two models
   the chains are those of [rjmcmc_array].  Returns the model index of every recorded sample and the counts per model. *)
external rjmcmc_array_k_raw :
  ctx -> rj_model_raw array -> int -> int -> int -> int -> (float, float64_elt, c_layout) Array1.t array ->
  (int, int8_unsigned_elt, c_layout) Array2.t -> int array
  = "mcmcgpu_rjmcmc_array_k_bytecode" "mcmcgpu_rjmcmc_array_k_native"
let rjmcmc_array_k ctx ?(nbin = 0) ?(nskip = 1) ?(nchains = 1) n (models : rj_model array) (starts : float array array) =
  let model = Array2.create int8_unsigned c_layout n nchains in
  let counts = rjmcmc_array_k_raw ctx (Array.map raw_of_model models) nbin nskip n nchains (Array.map ba1 starts) model in
  (model, counts)

(* Ellipse.enclosing_ellipse sf (fun x -> x) pts (ellipse.ml:98-103) *)
type ellipse = { center : float array; axes : float array; orientation : float array array }
external enclosing_ellipse_raw :
  ctx -> float -> (float, float64_elt, c_layout) Array2.t -> (float, float64_elt, c_layout) Array1.t ->
  (float, float64_elt, c_layout) Array1.t -> (float, float64_elt, c_layout) Array2.t -> unit
  = "mcmcgpu_enclosing_ellipse_bytecode" "mcmcgpu_enclosing_ellipse"
let enclosing_ellipse ctx sf (pts : float array array) =
  let d = Array.length pts.(0) in
  let c = Array1.create float64 c_layout d and a = Array1.create float64 c_layout d and o = Array2.create float64 c_layout d d in
  enclosing_ellipse_raw ctx sf (Array2.of_array float64 c_layout pts) c a o;
  { center = Array.init d (fun i -> c.{i}); axes = Array.init d (fun i -> a.{i});
    orientation = Array.init d (fun i -> Array.init d (fun j -> o.{i, j})) }

(* Stats.multi_mean / multi_std ?mean (stats.ml:58-87) *)
let multi_mean ctx (xs : float array array) =
  let out = Array1.create float64 c_layout (Array.length xs.(0)) in
  multi_mean_raw ctx (ba2 xs) out;
  Array.init (Array1.dim out) (fun i -> out.{i})
let multi_std ctx ?mean (xs : float array array) =
  let out = Array1.create float64 c_layout (Array.length xs.(0)) in
  multi_std_raw ctx (ba2 xs) (match mean with None -> ba1 [||] | Some mu -> ba1 mu) out;
  Array.init (Array1.dim out) (fun i -> out.{i})

(* Ensemble convergence diagnostics of a sample block (an addition beyond the reference, include/mcmc_gpu.h) *)
type chain_diagnostics = {
  rhat : float array; ess : float array; tau : float array; window_closed : bool array;
  rho : float array array; seq_tau : float array array option }
let diag_result f maxlag out rho seq_tau =
  { rhat = Array.init f (fun i -> out.{0, i}); ess = Array.init f (fun i -> out.{1, i});
    tau = Array.init f (fun i -> out.{2, i}); window_closed = Array.init f (fun i -> out.{3, i} <> 0.);
    rho = Array.init f (fun i -> Array.init maxlag (fun t -> rho.{i, t}));
    seq_tau = Option.map (fun s -> Array.init f (fun i -> Array.init (Array2.dim2 s) (fun m -> s.{i, m}))) seq_tau }
let chain_diagnostics ctx ?(split = true) ?(per_sequence = false) ~maxlag
    (block : (float, float64_elt, c_layout) Array3.t) =
  let f = Array3.dim2 block and c = Array3.dim3 block in
  let m = if split then 2 * c else c in
  let out = Array2.create float64 c_layout 4 f and rho = Array2.create float64 c_layout f maxlag in
  let st = if per_sequence then Array2.create float64 c_layout f m else Array2.create float64 c_layout 0 0 in
  chain_diagnostics_raw ctx maxlag (if split then 1 else 0) block out rho st;
  diag_result f maxlag out rho (if per_sequence then Some st else None)
let chain_diagnostics_dev ctx ?(split = true) ?(seq_tau = 0L) ~maxlag ~n ~dim ~nchains (block : int64) =
  let f = dim + 2 in
  let out = Array2.create float64 c_layout 4 f and rho = Array2.create float64 c_layout f maxlag in
  chain_diagnostics_dev_raw ctx block n dim nchains maxlag (if split then 1 else 0) out rho seq_tau;
  diag_result f maxlag out rho None

(* Exact per-field quantiles of a sample block [n][D+2][C], chains pooled (include/mcmc_gpu.h) *)
let quantiles_result f probs out =
  Array.init f (fun i -> Array.init (Array.length probs) (fun k -> out.{i, k}))
let quantiles ctx ~probs (block : (float, float64_elt, c_layout) Array3.t) =
  let f = Array3.dim2 block in
  let out = Array2.create float64 c_layout f (Array.length probs) in
  quantiles_raw ctx block (Array1.of_array float64 c_layout probs) out;
  quantiles_result f probs out
let quantiles_dev ctx ~probs ~n ~dim ~nchains (block : int64) =
  let f = dim + 2 in
  let out = Array2.create float64 c_layout f (Array.length probs) in
  quantiles_dev_raw ctx block n dim nchains (Array1.of_array float64 c_layout probs) out;
  quantiles_result f probs out

(* Evidence by parallel tempering (mg_evidence_tempered; the definition is in include/mcmc_gpu.h) *)
type tempered = {
  log_z_ss : float; log_z_ss_err : float; log_z_ti : float; log_z_ti_err : float;
  mean_ll : float array; mean_ll_err : float array;
  accept : int array; swaps_accepted : int array; swaps_tried : int array;
}
let evidence_tempered ctx ?(swap_every = 1) ~nladders ~nbin ~nsteps like prior props betas (start : float array array) =
  let t = Array.length betas in
  let x0 = Array2.of_array float64 c_layout start in
  let out = Array1.create float64 c_layout (4 + 2 * t) and cnt = Array1.create int64 c_layout (3 * t) in
  evidence_tempered_raw ctx like prior props (Array1.of_array float64 c_layout betas)
    [| nladders; nbin; nsteps; swap_every |] x0 out cnt;
  let ints o n = Array.init n (fun i -> Int64.to_int cnt.{o + i}) in
  { log_z_ss = out.{0}; log_z_ss_err = out.{1}; log_z_ti = out.{2}; log_z_ti_err = out.{3};
    mean_ll = Array.init t (fun k -> out.{4 + k}); mean_ll_err = Array.init t (fun k -> out.{4 + t + k});
    accept = ints 0 t; swaps_accepted = ints t (t - 1); swaps_tried = ints (2 * t) (t - 1) }

(* Nested.nested_evidence ?epsrel ?nmcmc ?nlive ?mode_hopping_frac (nested.ml:122-146; nested.mli:50-61) with draw_prior
   uniform on [prior_low, prior_high]; ?batch live points are replaced per iteration (1 = the reference's schedule).
   Result: 'a nested_output = (log_ev, log_dev, all points ascending in ll, log weights) (nested.ml:20). *)
let nested_evidence ctx ?(epsrel = 0.01) ?(nmcmc = 1000) ?(nlive = 1000) ?(mode_hopping_frac = 0.1) ?(batch = 1)
    ?max_points like prior prior_low prior_high =
  let d = like.dim in
  let cap = match max_points with Some c -> c | None -> nlive * 400 in
  let pts = Array2.create float64 c_layout cap d and ll = Array1.create float64 c_layout cap
  and lp = Array1.create float64 c_layout cap and lw = Array1.create float64 c_layout cap in
  let log_ev, log_dev, n =
    nested_evidence_raw ctx like prior (ba1 prior_low) (ba1 prior_high) epsrel nmcmc nlive mode_hopping_frac batch pts ll lp lw in
  let samples = Array.init n (fun i ->
      { Mcmc.value = Array.init d (fun k -> pts.{i, k});
        like_prior = { Mcmc.log_likelihood = ll.{i}; log_prior = lp.{i} } }) in
  (log_ev, log_dev, samples, Array.init n (fun i -> lw.{i}))
let log_total_error_estimate log_ev log_dev nlive = log_total_error_estimate_raw log_ev log_dev nlive   (* nested.ml:148-150 *)

(* Stats.draw_uniform / draw_gaussian / draw_cauchy (stats.ml:89-91,113-128): n draws from the context's stream *)
let draw kind ctx a b n =
  let out = Array1.create float64 c_layout n in
  stats_draw_raw ctx kind a b out;
  Array.init n (fun i -> out.{i})
let draw_uniform ctx a b n = draw 0 ctx a b n
let draw_gaussian ctx mu sigma n = draw 1 ctx mu sigma n
let draw_cauchy ctx x0 gamma n = draw 2 ctx x0 gamma n

(* Nested.posterior_samples n output (nested.ml:167-178): the sampled points *)
let posterior_samples ctx n (pts : float array array) (log_wts : float array) =
  let lw = Array1.of_array float64 c_layout log_wts in
  let idx = Array1.create int64 c_layout n in
  posterior_indices_raw ctx lw idx;
  Array.init n (fun i -> pts.(Int64.to_int idx.{i}))


(* Several GPUs: one OCaml process per GPU.  Rank 0 makes the 128-byte NCCL id ([Comm.unique_id]) and hands it to the other
   ranks (a file, a socket, MPI ...); every rank then creates its communicator.  All functions below are collective. *)
module Comm = struct
  type comm
  type id = (int, int8_unsigned_elt, c_layout) Array1.t
  external unique_id_raw : id -> unit = "mcmcgpu_comm_unique_id"
  external create : ctx -> int -> int -> id -> comm = "mcmcgpu_comm_create"
  external interp_broadcast_raw : ctx -> comm -> tree option -> int -> tree = "mcmcgpu_interp_broadcast"
  external interp_make_distributed_raw :
    ctx -> comm -> (float, float64_elt, c_layout) Array2.t -> (float, float64_elt, c_layout) Array1.t ->
    (float, float64_elt, c_layout) Array1.t -> tree = "mcmcgpu_interp_make_distributed"
  external evidence_lebesgue_sharded_raw :
    ctx -> comm -> int -> (float, float64_elt, c_layout) Array2.t -> (float, float64_elt, c_layout) Array1.t ->
    (float, float64_elt, c_layout) Array1.t -> int -> float -> float
    = "mcmcgpu_evidence_lebesgue_sharded_bytecode" "mcmcgpu_evidence_lebesgue_sharded_native"
  external rjmcmc_array_sharded_raw :
    ctx -> comm -> rj_model_raw -> rj_model_raw -> int -> int -> int -> int -> (float, float64_elt, c_layout) Array1.t ->
    (float, float64_elt, c_layout) Array1.t -> int * int
    = "mcmcgpu_rjmcmc_array_sharded_bytecode" "mcmcgpu_rjmcmc_array_sharded_native"
  let unique_id () = let id = Array1.create int8_unsigned c_layout 128 in unique_id_raw id; id
  (* Interp.make on [root], replicated on every rank by one broadcast *)
  let interp_broadcast ctx comm ?(root = 0) ~dim (ip : Interp.interp_pdf option) =
    let t = interp_broadcast_raw ctx comm (match ip with Some i -> Some i.Interp.tree | None -> None) root in
    { Interp.tree = t; dim }
  (* Interp.make by all ranks together; every rank passes the same points *)
  let interp_make_distributed ctx comm (pts : float array array) low high =
    { Interp.tree = interp_make_distributed_raw ctx comm (Array2.of_array float64 c_layout pts) (ba1 low) (ba1 high);
      dim = Array.length low }
  (* Evidence.evidence_lebesgue ?n ?eps of the samples held by [root] (the other ranks pass [||]) *)
  let evidence_lebesgue ctx comm ?(root = 0) ?(n = 64) ?(eps = 0.1) (pts : float array array) (ll : float array) (lp : float array) =
    let d = if Array.length pts > 0 then Array.length pts.(0) else 1 in
    let p = if Array.length pts > 0 then Array2.of_array float64 c_layout pts else Array2.create float64 c_layout 0 d in
    evidence_lebesgue_sharded_raw ctx comm root p (ba1 ll) (ba1 lp) n eps
  (* Mcmc.rjmcmc_array over all ranks: the model counts of the whole ensemble *)
  let rjmcmc_array ctx comm ?(nbin = 0) ?(nskip = 1) ?(nchains = 1) n (ma : rj_model) (mb : rj_model) a0 b0 =
    rjmcmc_array_sharded_raw ctx comm (raw_of_model ma) (raw_of_model mb) nbin nskip n nchains (ba1 a0) (ba1 b0)
end
