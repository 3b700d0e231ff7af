(** GPU path of the sampling-and-evidence modules, same shapes as [Mcmc],
    [Interpolate_pdf] and [Evidence], with closures replaced by registered
    plugins and ['a] fixed to [float array] (what every program in bin/ uses,
    e.g. bin/evidence_tool.ml:35-40).  NOT COMPILED in this repository's image
    (no OCaml toolchain, SURVEY.md F1). *)

open Bigarray

type ctx
(** One GPU, one Philox key, one CUDA stream.  Single caller, like the
    reference's global counters and [Random] state. *)

type logfn = { kind : int; dim : int; scale : float; params : (float, float64_elt, c_layout) Array1.t }
(** A registered log-likelihood / log-prior plugin (MG_FN_* kinds). *)

type proposal = { pkind : int; pdim : int; pparams : (float, float64_elt, c_layout) Array1.t }
(** A jump proposal with its log jump probability (MG_PROP_* kinds). *)

type pinned_handle

val create : ?device:int -> ?seed:int64 -> unit -> ctx
val set_seed : ctx -> int64 -> unit  (** [Random.init] *)

val reset_counters : ctx -> unit     (** [Mcmc.reset_counters] *)
val get_counters : ctx -> int * int  (** [Mcmc.get_counters] *)

(** Built-in plugins (the models shipped in bin/ and test/). *)
val gaussian : float array -> float array -> logfn           (* Stats.log_multi_gaussian mu sigma *)
val gaussian_data : float array -> logfn                      (* sum_i Stats.log_gaussian mu sigma data_i *)
val cauchy_data : float array -> logfn                        (* sum_i Stats.log_cauchy x0 gamma data_i *)
val box_prior : ?value:float -> float array -> float array -> logfn
val flat : int -> logfn
val box_proposal : float array -> proposal                    (* x_i + random_between (-h_i) h_i *)
val uniform_wrapping : float array -> float array -> float array -> proposal  (* Mcmc.uniform_wrapping *)
val independent_gaussian : float array -> float array -> proposal             (* test/mcmc_test.ml:119-127 *)
val differential_evolution_proposal :
  ?mode_hopping_frac:float -> float array Mcmc.mcmc_sample array -> proposal
(** [Mcmc.differential_evolution_proposal] (mcmc.mli:215-218) with [to_float] = [from_float] = identity. *)

(** Page-locked float64 Bigarrays (DMA at full PCIe rate for the host entry points).  Keep the record alive as long
    as [data] is in use: the handle's finaliser frees the memory. *)
module Pinned : sig
  type 'a t = { data : 'a; handle : pinned_handle }
  val array1 : ctx -> int -> (float, float64_elt, c_layout) Array1.t t
  val array2 : ctx -> int -> int -> (float, float64_elt, c_layout) Array2.t t
  val array3 : ctx -> int -> int -> int -> (float, float64_elt, c_layout) Array3.t t
end

val mcmc_array :
  ctx -> ?nbin:int -> ?nskip:int -> ?nchains:int -> int -> logfn -> logfn -> proposal -> float array ->
  float array Mcmc.mcmc_sample array array
(** [mcmc_array ctx ?nbin ?nskip ?nchains n log_likelihood log_prior
    jump_proposal start]: [Mcmc.mcmc_array] for [nchains] independent chains
    (default 1); element [c] of the result is chain [c]'s sample array. *)

module Interp : sig
  type interp_pdf
  val make : ctx -> float array array -> float array -> float array -> interp_pdf
  val draw : ctx -> interp_pdf -> float array
  val draw_high_level : ctx -> int -> interp_pdf -> float array
  val jump_prob : ctx -> interp_pdf -> 'a -> float array -> float
  val jump_prob_high_level : ctx -> int -> interp_pdf -> 'a -> float array -> float
  val jump_prob_batch : ctx -> ?n:int -> interp_pdf -> float array array -> float array
end

module Evidence : sig
  val evidence_harmonic_mean : ctx -> float array Mcmc.mcmc_sample array -> float
  val evidence_lebesgue : ctx -> ?n:int -> ?eps:float -> float array Mcmc.mcmc_sample array -> float
  val evidence_direct : ctx -> ?n:int -> float array Mcmc.mcmc_sample array -> float
end

(** {2 Mcmc.rjmcmc_array (mcmc.mli:132-162)} *)
type rj_into = Into_interp of Interp.interp_pdf * int | Into_gaussian of float array * float array
(** how a chain proposes INTO a model: [Interp.draw] / [log (Interp.jump_prob ..)] ([int] > 0: the [*_high_level] forms
    with that many objects per cell), or an independent Gaussian [(mu, sigma)] *)
type rj_model = { rj_like : logfn; rj_prior : logfn; rj_prop : proposal; rj_into : rj_into; rj_p : float }
val rjmcmc_array :
  ctx -> ?nbin:int -> ?nskip:int -> ?nchains:int -> int -> rj_model -> rj_model -> float array -> float array ->
  (int, int8_unsigned_elt, c_layout) Array2.t * (int * int)
(** [rjmcmc_array ctx ?nbin ?nskip ?nchains n model_a model_b a b]: the model of every recorded sample ([n][nchains],
    0 = A) and [Mcmc.rjmcmc_model_counts].  Raises [Failure] where the reference's [assert] on the priors fails. *)
val rjmcmc_evidence_ratio : int * int -> float
val rjmcmc_array_k :
  ctx -> ?nbin:int -> ?nskip:int -> ?nchains:int -> int -> rj_model array -> float array array ->
  (int, int8_unsigned_elt, c_layout) Array2.t * int array
(** k-model reversible jump (2..8 models): an extension -- the reference's sum type is two-model (mcmc.ml:83-87).
    With two models the chains are those of [rjmcmc_array]. *)

(** {2 Ellipse (ellipse.ml:21-24, 98-103)} *)
type ellipse = { center : float array; axes : float array; orientation : float array array }
val enclosing_ellipse : ctx -> float -> float array array -> ellipse
(** [enclosing_ellipse ctx sf pts] = [Ellipse.enclosing_ellipse sf (fun x -> x) pts] *)

(** {2 Stats (stats.mli:41-55)} *)
val multi_mean : ctx -> float array array -> float array
val multi_std : ctx -> ?mean:float array -> float array array -> float array

type chain_diagnostics = {
  rhat : float array; ess : float array; tau : float array; window_closed : bool array;
  rho : float array array; seq_tau : float array array option }
val chain_diagnostics :
  ctx -> ?split:bool -> ?per_sequence:bool -> maxlag:int -> (float, Bigarray.float64_elt, Bigarray.c_layout) Bigarray.Array3.t ->
  chain_diagnostics
(** Ensemble convergence diagnostics of a sample block [n][D+2][C] (an addition beyond the reference): per field
    split-Rhat, ESS, Geyer's integrated autocorrelation time, whether the lag window closed and the ensemble
    autocorrelation at lags [0, maxlag); [?per_sequence] adds tau of every sequence.  Definitions in mcmc_gpu.h.
    [Invalid_argument] for maxlag < 2, maxlag >= N or above 256, split with n < 4. *)
val chain_diagnostics_dev :
  ctx -> ?split:bool -> ?seq_tau:int64 -> maxlag:int -> n:int -> dim:int -> nchains:int -> int64 ->
  chain_diagnostics
(** The same on a device block (its address); [?seq_tau] is the device address of a [D+2][M] float64 array. *)
val quantiles :
  ctx -> probs:float array -> (float, Bigarray.float64_elt, Bigarray.c_layout) Bigarray.Array3.t -> float array array
(** Exact quantiles [D+2][nq] of a sample block [n][D+2][C], all chains pooled: numpy's "linear" rule on the exact
    order statistics; a field holding a NaN gives NaN.  Definitions in mcmc_gpu.h.  [Invalid_argument] for no probs or
    more than 64, or a p outside [0, 1]. *)
val quantiles_dev : ctx -> probs:float array -> n:int -> dim:int -> nchains:int -> int64 -> float array array
(** The same on a device block (its address), which is not modified. *)

type tempered = {
  log_z_ss : float; log_z_ss_err : float; log_z_ti : float; log_z_ti_err : float;
  mean_ll : float array; mean_ll_err : float array;
  accept : int array; swaps_accepted : int array; swaps_tried : int array;
}
val evidence_tempered :
  ctx -> ?swap_every:int -> nladders:int -> nbin:int -> nsteps:int -> logfn -> logfn -> proposal array -> float array ->
  float array array -> tempered
(** log Z by parallel tempering: [nladders] ladders of [Array.length betas] tempered chains (one proposal per rung,
    betas strictly increasing from >= 0 to 1), all rungs of a ladder starting at its row of [start] (one row: shared).
    [log_z_ss] (stepping stones) is the primary estimate; [log_z_ti] also carries the trapezoid bias of the ladder.
    Definitions in mcmc_gpu.h.  [Invalid_argument] for fewer than 2 or more than 32 rungs, bad betas, nsteps < 1. *)

(** {2 Nested (nested.mli:50-69)} *)
val nested_evidence :
  ctx -> ?epsrel:float -> ?nmcmc:int -> ?nlive:int -> ?mode_hopping_frac:float -> ?batch:int -> ?max_points:int ->
  logfn -> logfn -> float array -> float array ->
  float * float * float array Mcmc.mcmc_sample array * float array
(** ['a nested_output] of [Nested.nested_evidence] with [draw_prior] uniform on the box; [?batch] (default 1, the
    reference's schedule) live points are replaced per iteration.  [Failure] as nested.ml:70-72. *)
val log_total_error_estimate : float -> float -> int -> float

(** [Stats.draw_uniform a b], [draw_gaussian mu sigma], [draw_cauchy x0 gamma] (stats.ml:89-91,113-128),
    [n] draws per call from the context's Philox stream. *)
val draw_uniform : ctx -> float -> float -> int -> float array
val draw_gaussian : ctx -> float -> float -> int -> float array
val draw_cauchy : ctx -> float -> float -> int -> float array

(** [Nested.posterior_samples n output] (nested.ml:167-178) given the points and their log weights. *)
val posterior_samples : ctx -> int -> float array array -> float array -> float array array


(** {2 Several GPUs} one OCaml process per GPU; rank 0 makes the NCCL id and hands it to the others; every function is
    collective.  Results do not depend on the number of ranks (global chain ids; evidences bit-identical to one GPU). *)
module Comm : sig
  type comm
  type id = (int, int8_unsigned_elt, c_layout) Array1.t
  val unique_id : unit -> id
  val create : ctx -> int -> int -> id -> comm
  (** [create ctx nranks rank id] *)
  val interp_broadcast : ctx -> comm -> ?root:int -> dim:int -> Interp.interp_pdf option -> Interp.interp_pdf
  (** the root passes [Some tree], the other ranks [None]; [dim] is the tree's dimension (known to every rank) *)
  val interp_make_distributed : ctx -> comm -> float array array -> float array -> float array -> Interp.interp_pdf
  val evidence_lebesgue :
    ctx -> comm -> ?root:int -> ?n:int -> ?eps:float -> float array array -> float array -> float array -> float
  val rjmcmc_array :
    ctx -> comm -> ?nbin:int -> ?nskip:int -> ?nchains:int -> int -> rj_model -> rj_model -> float array -> float array -> int * int
end
