"""Host-side mirror of ``Evidence.Make`` (evidence.ml:31-58) for the GPU path.
Samples are given as coordinate rows [N][D] with their ``log_likelihood`` and
``log_prior`` (the fields of ``'a Mcmc.mcmc_sample``), or as ``McmcSamples``."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _abi
from .context import Context, default_context
from .kd_tree import KdTree


def _unpack(samples, ll=None, lp=None):
    if hasattr(samples, "values") and ll is None:          # McmcSamples
        return _abi.as_f64(samples.values()), _abi.as_f64(samples.log_likelihood()), _abi.as_f64(samples.log_prior())
    pts = _abi.as_f64(samples)
    if pts.ndim == 1:
        pts = pts.reshape(-1, 1)
    ll, lp = _abi.as_f64(ll), _abi.as_f64(lp)
    if ll.ndim and lp.ndim and (ll.size != pts.shape[0] or lp.size != pts.shape[0]):   # the library reads N of each
        raise _abi.InvalidArgument("evidence: log_likelihood / log_prior must have one entry per sample")
    return pts, ll, lp


def kd_tree_of_samples(samples, low, high, *, ctx: Context | None = None) -> KdTree:
    """``Evidence.kd_tree_of_samples`` (evidence.ml:70)."""
    pts, _, _ = _unpack(samples, 0, 0) if not hasattr(samples, "values") else _unpack(samples)
    return KdTree(pts, low, high, ctx=ctx)


def evidence_harmonic_mean(samples=None, ll=None, *, ctx: Context | None = None) -> float:
    """``Evidence.evidence_harmonic_mean`` (evidence.ml:101-107)."""
    ctx = ctx or default_context()
    if ll is None:
        ll = samples.log_likelihood()
    ll = _abi.as_f64(ll)
    out = C.c_double()
    ctx.check(ctx.lib.mg_evidence_harmonic_mean(ctx.h, _abi.ptr(ll), C.c_int64(ll.size), C.byref(out)))
    return out.value


def harmonic_bootstrap(ll, nbstrap: int = 10000, *, ctx: Context | None = None) -> np.ndarray:
    """Bootstrap replicates of the harmonic-mean evidence (bin/harmonic_evidence.ml:41-52),
    sorted ascending like the reference's ``Array.fast_sort``."""
    ctx = ctx or default_context()
    ll = _abi.as_f64(ll)
    out = np.empty(nbstrap)
    ctx.check(ctx.lib.mg_evidence_harmonic_bootstrap(ctx.h, _abi.ptr(ll), C.c_int64(ll.size), C.c_int32(nbstrap), _abi.ptr(out)))
    return np.sort(out)


def evidence_lebesgue(samples, ll=None, lp=None, *, n: int = 64, eps: float = 0.1, ctx: Context | None = None) -> float:
    """``Evidence.evidence_lebesgue ?n ?eps`` (evidence.ml:202-221), Weinberg's
    Lebesgue integral of 1/L over kd-tree cells."""
    ctx = ctx or default_context()
    pts, ll, lp = _unpack(samples, ll, lp)
    out = C.c_double()
    ctx.check(ctx.lib.mg_evidence_lebesgue(ctx.h, _abi.ptr(pts), _abi.ptr(ll), _abi.ptr(lp), C.c_int64(pts.shape[0]),
                                           C.c_int32(pts.shape[1]), C.c_int32(n), C.c_double(eps), C.byref(out)))
    return out.value


def evidence_direct(samples, ll=None, lp=None, *, n: int = 64, ctx: Context | None = None) -> float:
    """``Evidence.evidence_direct ?n`` (evidence.ml:148-165)."""
    ctx = ctx or default_context()
    pts, ll, lp = _unpack(samples, ll, lp)
    out = C.c_double()
    ctx.check(ctx.lib.mg_evidence_direct(ctx.h, _abi.ptr(pts), _abi.ptr(ll), _abi.ptr(lp), C.c_int64(pts.shape[0]),
                                         C.c_int32(pts.shape[1]), C.c_int32(n), C.byref(out)))
    return out.value


def evidence_lebesgue_dev(pts_ptr: int, ll_ptr: int, lp_ptr: int, N: int, D: int, *, n: int = 64, eps: float = 0.1,
                          ctx: Context | None = None) -> float:
    """Device-resident form: pointers to float64 [N][D], [N], [N] on the context's GPU."""
    ctx = ctx or default_context()
    out = C.c_double()
    ctx.check(ctx.lib.mg_evidence_lebesgue_dev(ctx.h, C.c_void_p(pts_ptr), C.c_void_p(ll_ptr), C.c_void_p(lp_ptr),
                                               C.c_int64(N), C.c_int32(D), C.c_int32(n), C.c_double(eps), C.byref(out)))
    return out.value


def evidence_direct_dev(pts_ptr: int, ll_ptr: int, lp_ptr: int, N: int, D: int, *, n: int = 64,
                        ctx: Context | None = None) -> float:
    ctx = ctx or default_context()
    out = C.c_double()
    ctx.check(ctx.lib.mg_evidence_direct_dev(ctx.h, C.c_void_p(pts_ptr), C.c_void_p(ll_ptr), C.c_void_p(lp_ptr),
                                             C.c_int64(N), C.c_int32(D), C.c_int32(n), C.byref(out)))
    return out.value


def evidence_harmonic_mean_dev(ll_ptr: int, N: int, *, ctx: Context | None = None) -> float:
    ctx = ctx or default_context()
    out = C.c_double()
    ctx.check(ctx.lib.mg_evidence_harmonic_mean_dev(ctx.h, C.c_void_p(ll_ptr), C.c_int64(N), C.byref(out)))
    return out.value


class TemperedEvidence:
    """Result of ``evidence_tempered``: log Z by stepping stones (``log_z_ss``, the primary estimate) and by
    thermodynamic integration (``log_z_ti``, which also carries the trapezoid bias of its ladder), each with its
    spread over ladders / sqrt(M); per rung the mean log-likelihood over ladders (``mean_ll``, ``mean_ll_err``) and
    the accepted MH steps (``accept``); per pair (k, k+1) the accepted and tried swaps; per ladder and rung the mean
    log-likelihood (``ladder_mean_ll`` [M][T]) and the final state (``final`` [M][T][D+2])."""

    def __init__(self, d):
        self.__dict__.update(d)

    def __repr__(self):
        return (f"TemperedEvidence(log_z_ss={self.log_z_ss:.6g} +- {self.log_z_ss_err:.2g}, "
                f"log_z_ti={self.log_z_ti:.6g} +- {self.log_z_ti_err:.2g})")


def _tempered_args(like, prior, props, betas, start, nladders, nbin, nsteps, swap_every, ladder_offset):
    b = _abi.as_f64(betas).ravel()
    T, D = b.size, like.dim
    if not isinstance(props, (list, tuple)):
        props = [props] * T
    if len(props) != T:
        raise _abi.InvalidArgument("evidence_tempered: one proposal per beta")
    specs = [p.spec() for p in props]
    pa = (_abi.mg_proposal * max(T, 1))(*specs)
    x0 = _abi.as_f64(start)
    shared = x0.size == D
    if not shared and x0.size != nladders * D:
        raise _abi.InvalidArgument("evidence_tempered: start must be [D] or [nladders][D]")
    cfg = _abi.mg_tempered_cfg(nladders, T, D, nbin, nsteps, swap_every, ladder_offset, 1 if shared else 0, 0)
    return cfg, pa, (props, specs), x0, b


def _tempered_outputs(cfg):
    T, M, D = cfg.ntemps, cfg.nladders, cfg.dim
    res = dict(mean_ll=np.empty(T), mean_ll_err=np.empty(T), accept=np.empty(T, np.int64),
               swaps_accepted=np.empty(max(T - 1, 0), np.int64), swaps_tried=np.empty(max(T - 1, 0), np.int64),
               final=np.empty((M, T, D + 2)), ladder_mean_ll=np.empty((M, T)))
    out = _abi.mg_tempered_out(0.0, 0.0, 0.0, 0.0, _abi.ptr(res["mean_ll"]), _abi.ptr(res["mean_ll_err"]),
                               _abi.ptr(res["accept"], _abi.c_int64_p), _abi.ptr(res["swaps_accepted"], _abi.c_int64_p),
                               _abi.ptr(res["swaps_tried"], _abi.c_int64_p), _abi.ptr(res["final"]),
                               _abi.ptr(res["ladder_mean_ll"]))
    return res, out


def _evidence_tempered_call(fn, handle, like, prior, jump_proposals, betas, start, nladders, nbin, nsteps, swap_every,
                            ladder_offset, check):
    cfg, pa, keep, x0, b = _tempered_args(like, prior, jump_proposals, betas, start, nladders, nbin, nsteps,
                                          swap_every, ladder_offset)
    res, out = _tempered_outputs(cfg)
    ls, ps = like.spec(), prior.spec()
    check(fn(handle, C.byref(ls), C.byref(ps), pa, _abi.ptr(b), C.byref(cfg), _abi.ptr(x0), C.byref(out)))
    res.update(log_z_ss=out.log_z_ss, log_z_ss_err=out.log_z_ss_err, log_z_ti=out.log_z_ti,
               log_z_ti_err=out.log_z_ti_err)
    return TemperedEvidence(res)


def evidence_tempered(log_likelihood, log_prior, jump_proposals, betas, start, *, nladders: int, nbin: int, nsteps: int,
                      swap_every: int = 1, ladder_offset: int = 0, ctx: Context | None = None) -> TemperedEvidence:
    """log Z by parallel tempering (``mg_evidence_tempered``; include/mcmc_gpu.h has the definition): ``nladders``
    ladders of ``len(betas)`` tempered chains (betas strictly increasing from >= 0 to 1), ``jump_proposals`` one
    proposal for every rung or a list with one per rung, ``start`` [D] or [nladders][D], ``nbin`` steps before
    ``nsteps`` measured ones, a swap round every ``swap_every`` steps (0: none)."""
    ctx = ctx or default_context()
    return _evidence_tempered_call(ctx.lib.mg_evidence_tempered, ctx.h, log_likelihood, log_prior, jump_proposals,
                                   betas, start, nladders, nbin, nsteps, swap_every, ladder_offset, ctx.check)
